// ogb_map.cuh -- per-sample read depth of the unitigs of the last ogb_graph_spell (ogb_spell.cuh): every read of a sample is looked
// up in the unitig sequences with up to d substitutions and counts wherever it occurs with the fewest.
//
// S_u = the sequence of unitig u (the spell's word-aligned layout). A sample read is kept iff it passes the Dataset filter for the
// build's minOverlap m (k_ds_filter). For a kept read s of length L and the caller's d (0 <= d <= OGB_MAP_MAX_MISMATCHES):
//   d_r = min(d, floor(L / K) - 1), K = min(32, m + 1) the key length of the index: pigeonhole needs d_r + 1 disjoint K-mers in s.
//   candidate (u, p, strand): [p, p + L) inside S_u; H = the Hamming distance of S_u[p, p + L) and s (strand 0) or rc(s) (strand 1).
//   b(s) = the least H over the candidates of both strands; s is mapped iff b(s) <= d_r. Its placements are the distinct (u, p) with
//   min(H_fw, H_rc) == b(s): a (u, p) reached on both strands counts once (for a palindrome: tested on one strand only).
// Every placement adds 1 on [p, p + L) of S_u; hits(s) = its placements, strat(s) = b(s) (OGB_MAP_UNPLACED when unmapped). Raw reads
// count one by one, so duplicates count as often as they occur. d = 0 is the exact lookup: S_u[p, p + L) == s or rc(s). Raising d
// never removes a placement: a read mapped at b counts the same placements at every d >= b.
//
// Index (built on the first mapping after a spell, kept for the later samples and every d): one entry per layout position p of u
// with p + K <= |S_u|, in B = mp_buckets(bases) buckets (a power of two, 1 to 2 positions per bucket) of a CSR: entry = tag << 32 | p,
// bucket and tag from one 64-bit mix of the K-mer at p.
//   k_map_count   thread per layout word (binary search for its unitig, as sp_word): the <= 32 K-mers that start in it, counted per
//                 bucket; an exclusive scan gives the bucket starts
//   k_map_fill    the same walk, entries scattered to their buckets (the order inside a bucket does not change any sum)
// Sample, in chunks of at most OGB_MAP_CHUNK_READS reads, so device memory does not grow with the sample: upload, k_ds_filter +
// scan + k_ds_compact, k_map_geom + scan + k_map_meta (the chunk's read store, laid out like the build's), k_pack_ascii (forward
// strand and reverse complement), then
//   k_map_reads   thread per kept read, straight-line like k_verify (mp_read): per strand, seed j = the K bases at read offset jK
//                 (j = 0 .. d_r) selects one bucket; every entry whose tag matches and whose read would lie inside the unitig is a
//                 candidate p = q - jK. Pass 1 (d_r > 0) finds b(s) with cv_mismatches (popcount of the 2-bit xor, early exit above
//                 the bound); pass 2 places the candidates with H == b(s), each from the lowest seed exact at p only, on strand 1
//                 only where H_fw(p) > b(s). At d_r = 0 pass 2 alone runs: one seed per strand, verified base for base (cv_equal).
//                 A placement adds +1 at p and -1 at p + L to a u32 difference array over the layout and counts in its unitig's
//                 record. The difference array accumulates over the chunks.
//   k_map_hits    per raw read: hits and strata scattered from the kept reads, OGB_MAP_FILTERED / OGB_MAP_UNPLACED for a dropped one
// Depth: one exclusive scan and k_cov_reduce into ogb_unitig_coverage records (reads = read_count = placements, contained = 0).
//
// Integer atomics only, so a run is deterministic. The per-thread bodies are `__host__ __device__`: tests/map_emul.cpp (d = 0) and
// tests/map_approx_emul.cpp (any d) run them on the CPU.
#ifndef OGB_MAP_CUH_
#define OGB_MAP_CUH_

#include "ogb_coverage.cuh"

struct MapArgs {
	const cu64 *layout;             // the spell's packed words, followed by one zero word (sp_extract32 reads word w + 1)
	const cu64 *wpos;               // n_rec + 1: first layout word of each record, total last
	const ogb_unitig *rec;
	cu64 n_rec;
	cu32 K;
	cu64 bmask;                     // buckets - 1
	const cu64 *bstart;             // buckets + 1: bucket b holds ent[bstart[b] .. bstart[b + 1])
	const cu64 *ent;                // tag << 32 | layout position
	const cu64 *rwords;             // the chunk's read store: read i forward at word off, reverse complement at off + pw
	const cu64 *rmeta;              // off << 16 | L per kept read of the chunk
	cu32 d = 0;                     // max_mismatches (0: exact placements only)
};

// buckets of the index over a layout of `bases` bases: the smallest power of two >= bases / 2
OGB_HD cu64 mp_buckets(cu64 bases)
{
	cu64 b = 1;
	while (2 * b < bases) b <<= 1;
	return b;
}

// 64-bit finaliser (MurmurHash3 fmix64): the low bits pick the bucket, the high 32 are the tag
OGB_HD cu64 mp_hash(cu64 x)
{
	x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
	return x;
}

// thread = layout word w: emit(bucket, tag, position) for every indexed position 32 w + j (p + K <= length of its unitig)
template <class EMIT>
OGB_HD void mp_word(const MapArgs &A, cu64 w, EMIT emit)
{
	const cu64 u = cv_owner(A.wpos, A.n_rec, w);
	const cu64 p0 = 32 * (w - A.wpos[u]), len = A.rec[u].length;
	if (p0 + A.K > len) return;
	const cu32 n = len - A.K - p0 + 1 < 32 ? (cu32)(len - A.K - p0 + 1) : 32;
	const cu64 a = A.layout[w], b = A.layout[w + 1], mask = sp_top_bases(A.K);
	for (cu32 j = 0; j < n; j++) {
		const cu64 x = j ? (a << (2 * j)) | (b >> (64 - 2 * j)) : a;
		const cu64 h = mp_hash(x & mask);
		emit(h & A.bmask, (cu32)(h >> 32), 32 * w + j);
	}
}

// the K bases of strand t at read offset o, in the top bits (the key the index hashed at a layout position)
OGB_HD cu64 mp_seed(const cu64 *t, cu64 o, cu32 K)
{
	return ((o & 31) ? sp_extract32(t, o) : t[o >> 5]) & sp_top_bases(K);
}

// every candidate (u, p) of seed j of strand t: an index entry q of the seed's bucket with its tag, p = q - jK, [p, p + L) inside the
// unitig that owns q. visit(p, u) returns false to stop the walk; mp_walk then returns false too.
template <class VISIT>
OGB_HD bool mp_walk(const MapArgs &A, const cu64 *t, cu32 j, cu32 L, VISIT visit)
{
	const cu64 jk = (cu64)j * A.K;
	const cu64 h = mp_hash(mp_seed(t, jk, A.K)), b = h & A.bmask;
	const cu32 tag = (cu32)(h >> 32);
	for (cu64 e = A.bstart[b], ee = A.bstart[b + 1]; e < ee; e++) {
		const cu64 x = A.ent[e];
		if ((cu32)(x >> 32) != tag) continue;
		const cu64 q = (cu32)x;
		const cu64 u = cv_owner(A.wpos, A.n_rec, q >> 5), u0 = 32 * A.wpos[u];
		if (q < u0 + jk || q - jk + L > u0 + A.rec[u].length) continue;
		if (!visit(q - jk, u)) return false;
	}
	return true;
}

// thread = kept read i of the chunk: its placements in the best stratum b <= d_r = min(A.d, L / K - 1), each passed to add (the
// difference array, as cv_place) and to place(unitig). Returns the read's hit count; *strat = b, or OGB_MAP_UNPLACED without one.
//   pass 1 (d_r > 0): b = the least Hamming distance over the candidates of seeds 0 .. d_r of both strands. A candidate below the
//          best so far has an exact seed among the first `best`, so the seeds walked shrink with it.
//   pass 2: the candidates with H == b, each counted from the lowest seed that occurs exactly at p (<= b by pigeonhole, and the index
//          holds that seed's position, so it finds p itself); on the reverse strand p is skipped when H_fw(p) == b, strand 0 owns it.
// With d_r = 0, b = 0 and pass 2 is the exact lookup: seed 0 of each strand, cv_equal, no dedupe (H == 0 matches every seed) and no
// strand test (H_fw(p) == H_rc(p) == 0 only for a palindrome, tested on one strand).
// EXACT compiles the d = 0 body alone (k_map_reads<true>): the same work as before substitutions were searched.
// mp_search reports each placement as visit(p, u, L, strand): p the layout position, L the read's length, strand 0 iff H_fw(p) == b
// (ogb_sam.cuh writes it); mp_read passes it to add (the difference array, as cv_place) and place(unitig).
template <bool EXACT = false, class VISIT>
OGB_HD cu32 mp_search(const MapArgs &A, cu64 i, VISIT visit, cu32 &strat)
{
	const cu64 m = A.rmeta[i];
	const cu32 L = (cu32)(m & 0xFFFF), pw = ((L + 63) >> 6) << 1;
	const cu64 *fw = A.rwords + (m >> 16);
	const int strands = cv_equal(fw, 0, fw + pw, L) ? 1 : 2;          // a palindrome occurs at the same places on both strands
	const cu32 dr = EXACT ? 0 : (A.d < L / A.K - 1 ? A.d : L / A.K - 1);
	cu32 b = 0;
	if (dr) {
		cu32 best = dr + 1;
		for (int s = 0; s < strands && best; s++) {
			const cu64 *t = fw + (s ? pw : 0);
			for (cu32 j = 0; j < best; j++)
				mp_walk(A, t, j, L, [&](cu64 p, cu64) {
					const cu32 H = cv_mismatches(A.layout, p, t, L, best - 1);
					if (H < best) best = H;
					return best > j;                                   // seeds >= best cannot find anything better
				});
		}
		if (best > dr) { strat = OGB_MAP_UNPLACED; return 0; }
		b = best;
	}
	cu32 hits = 0;
	for (int s = 0; s < strands; s++) {
		const cu64 *t = fw + (s ? pw : 0);
		for (cu32 j = 0; j <= b; j++)
			mp_walk(A, t, j, L, [&](cu64 p, cu64 u) {
				if (!b) {
					if (!cv_equal(A.layout, p, t, L)) return true;
				} else {
					if (cv_mismatches(A.layout, p, t, L, b) != b) return true;
					cu32 k = 0;                                             // the lowest seed exact at p must be j
					while (k <= j && (sp_extract32(A.layout, p + (cu64)k * A.K) ^ mp_seed(t, (cu64)k * A.K, A.K)) & sp_top_bases(A.K)) k++;
					if (k != j) return true;
					if (s && cv_mismatches(A.layout, p, fw, L, b) <= b) return true;
				}
				visit(p, u, L, s);
				hits++;
				return true;
			});
	}
	strat = hits ? b : OGB_MAP_UNPLACED;
	return hits;
}
template <bool EXACT = false, class ADD, class PLACE>
OGB_HD cu32 mp_read(const MapArgs &A, cu64 i, ADD add, PLACE place, cu32 &strat)
{
	return mp_search<EXACT>(A, i, [&](cu64 p, cu64 u, cu32 L, int) {
		add(p, 1u);
		add(p + L, 0xFFFFFFFFu);
		place(u);
	}, strat);
}
template <class ADD, class PLACE>
OGB_HD cu32 mp_read(const MapArgs &A, cu64 i, ADD add, PLACE place)
{
	cu32 strat;
	return mp_read(A, i, add, place, strat);
}

// place() of mp_read: the unitig's placement counts, atomic on the device, plain on the host (tests/map_emul.cpp)
struct MpPlace {
	ogb_unitig_coverage *out;
	OGB_HD void operator()(cu64 u) const
	{
#if defined(__CUDA_ARCH__)
		atomicAdd(&out[u].reads, 1u);
		atomicAdd((unsigned long long *)&out[u].read_count, 1ull);
#else
		out[u].reads++;
		out[u].read_count++;
#endif
	}
};

#if defined(__CUDACC__)
__global__ void __launch_bounds__(256) k_map_count(MapArgs A, cu64 n_words, cu32 *cnt)
{
	OGB_SP_LOOP(w, n_words) mp_word(A, w, [&](cu64 b, cu32, cu64) { atomicAdd(cnt + b, 1u); });
}
__global__ void __launch_bounds__(256) k_map_fill(MapArgs A, cu64 n_words, cu32 *fill, cu64 *ent)
{
	OGB_SP_LOOP(w, n_words) mp_word(A, w, [&](cu64 b, cu32 tag, cu64 p) { ent[A.bstart[b] + atomicAdd(fill + b, 1u)] = (cu64)tag << 32 | p; });
}
// words of each kept read's two strands (scanned into its store offset), then meta = off << 16 | L in place
__global__ void __launch_bounds__(256) k_map_geom(const unsigned short *__restrict__ len, cu32 n, cu32 *nw)
{
	OGB_SP_LOOP(i, n) nw[i] = ((((cu32)len[i] + 63) >> 6) << 1) * 2;
}
__global__ void __launch_bounds__(256) k_map_meta(const unsigned short *__restrict__ len, cu32 n, cu64 *meta)
{
	OGB_SP_LOOP(i, n) meta[i] = meta[i] << 16 | len[i];
}
// ctr[0] mapped reads, [1] reads with >= 2 placements, [2] placements: one atomic each per warp. strat: NULL or the best stratum per
// kept read (OGB_MAP_UNPLACED when unmapped). EXACT: launched for A.d == 0
template <bool EXACT>
__global__ void __launch_bounds__(256) k_map_reads(MapArgs A, cu32 n, cu32 *diff, ogb_unitig_coverage *out, cu32 *__restrict__ hits, unsigned char *__restrict__ strat,
                                                   cu64 *ctr)
{
	const CvAdd add{diff};
	const MpPlace place{out};
	const cu32 lane = threadIdx.x & 31;
	for (cu64 i0 = (cu64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); i0 < n; i0 += (cu64)gridDim.x * blockDim.x) {   // warp-uniform
		const cu64 i = i0 + lane;
		cu32 h = 0, b;
		if (i < n) {
			h = mp_read<EXACT>(A, i, add, place, b);
			hits[i] = h;
			if (strat) strat[i] = (unsigned char)b;
		}
		const cu32 mapped = __reduce_add_sync(0xFFFFFFFFu, h > 0), multi = __reduce_add_sync(0xFFFFFFFFu, h > 1);
		cu64 pl = h;
		for (int d = 16; d > 0; d >>= 1) pl += __shfl_down_sync(0xFFFFFFFFu, pl, d);
		if (lane == 0 && mapped) {
			atomicAdd((unsigned long long *)ctr, (unsigned long long)mapped);
			if (multi) atomicAdd((unsigned long long *)ctr + 1, (unsigned long long)multi);
			atomicAdd((unsigned long long *)ctr + 2, (unsigned long long)pl);
		}
	}
}
// per raw read of the chunk: its kept read's hit count, or OGB_MAP_FILTERED, into hits; its stratum, or OGB_MAP_UNPLACED, into strat
// (either may be NULL)
__global__ void __launch_bounds__(256) k_map_hits(const cu32 *__restrict__ good, const cu64 *__restrict__ pos, const cu32 *__restrict__ khits,
                                                  const unsigned char *__restrict__ kstrat, cu32 n, cu32 *__restrict__ hits, unsigned char *__restrict__ strat)
{
	OGB_SP_LOOP(i, n) {
		if (hits) hits[i] = good[i] ? khits[pos[i]] : OGB_MAP_FILTERED;
		if (strat) strat[i] = good[i] ? kstrat[pos[i]] : (unsigned char)OGB_MAP_UNPLACED;
	}
}
#endif

#endif

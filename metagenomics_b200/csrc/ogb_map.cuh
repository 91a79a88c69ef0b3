// ogb_map.cuh -- per-sample read depth of the unitigs of the last ogb_graph_spell (ogb_spell.cuh): every read of a sample is looked
// up in the unitig sequences, exactly, and counts wherever it occurs.
//
// S_u = the sequence of unitig u (the spell's word-aligned layout). A sample read is kept iff it passes the Dataset filter for the
// build's minOverlap m (k_ds_filter); a placement of a kept read s of length L is (u, p) with S_u[p, p + L) == s or rc(s), a read
// equal to its own reverse complement tested on one strand only. Every placement adds 1 on [p, p + L) of S_u; hits(s) = its
// placements. Raw reads count one by one, so duplicates count as often as they occur.
//
// Index (built on the first mapping after a spell, kept for the later samples): K = min(32, m + 1) <= the length of every kept read,
// one entry per layout position p of u with p + K <= |S_u|, in B = mp_buckets(bases) buckets (a power of two, 1 to 2 positions per
// bucket) of a CSR: entry = tag << 32 | p, bucket and tag from one 64-bit mix of the K-mer at p.
//   k_map_count   thread per layout word (binary search for its unitig, as sp_word): the <= 32 K-mers that start in it, counted per
//                 bucket; an exclusive scan gives the bucket starts
//   k_map_fill    the same walk, entries scattered to their buckets (the order inside a bucket does not change any sum)
// Sample, in chunks of at most OGB_MAP_CHUNK_READS reads, so device memory does not grow with the sample: upload, k_ds_filter +
// scan + k_ds_compact, k_map_geom + scan + k_map_meta (the chunk's read store, laid out like the build's), k_pack_ascii (forward
// strand and reverse complement), then
//   k_map_reads   thread per kept read, straight-line like k_verify: per strand the first K bases select one bucket; every entry
//                 whose tag matches and whose read would end inside the unitig is verified base for base (cv_equal against the
//                 layout); a verified placement adds +1 at p and -1 at p + L to a u32 difference array over the layout and counts in
//                 its unitig's record. The difference array accumulates over the chunks.
// Depth: one exclusive scan and k_cov_reduce into ogb_unitig_coverage records (reads = read_count = placements, contained = 0).
//
// Integer atomics only, so a run is deterministic. The per-thread bodies are `__host__ __device__`: tests/map_emul.cpp runs them on
// the CPU.
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

// thread = kept read i of the chunk: its placements, each passed to add (the difference array, as cv_place) and to place(unitig).
// Returns the read's hit count.
template <class ADD, class PLACE>
OGB_HD cu32 mp_read(const MapArgs &A, cu64 i, ADD add, PLACE place)
{
	const cu64 m = A.rmeta[i];
	const cu32 L = (cu32)(m & 0xFFFF), pw = ((L + 63) >> 6) << 1;
	const cu64 *fw = A.rwords + (m >> 16);
	const int strands = cv_equal(fw, 0, fw + pw, L) ? 1 : 2;          // a palindrome occurs at the same places on both strands
	cu32 hits = 0;
	for (int s = 0; s < strands; s++) {
		const cu64 *t = fw + (s ? pw : 0);
		const cu64 h = mp_hash(t[0] & sp_top_bases(A.K)), b = h & A.bmask;
		const cu32 tag = (cu32)(h >> 32);
		for (cu64 e = A.bstart[b], ee = A.bstart[b + 1]; e < ee; e++) {
			const cu64 x = A.ent[e];
			if ((cu32)(x >> 32) != tag) continue;
			const cu64 p = (cu32)x;
			const cu64 u = cv_owner(A.wpos, A.n_rec, p >> 5);
			if (p + L > 32 * A.wpos[u] + A.rec[u].length || !cv_equal(A.layout, p, t, L)) continue;
			add(p, 1u);
			add(p + L, 0xFFFFFFFFu);
			place(u);
			hits++;
		}
	}
	return hits;
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
// ctr[0] mapped reads, [1] reads with >= 2 placements, [2] placements: one atomic each per warp
__global__ void __launch_bounds__(256) k_map_reads(MapArgs A, cu32 n, cu32 *diff, ogb_unitig_coverage *out, cu32 *__restrict__ hits, cu64 *ctr)
{
	const CvAdd add{diff};
	const MpPlace place{out};
	const cu32 lane = threadIdx.x & 31;
	for (cu64 i0 = (cu64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); i0 < n; i0 += (cu64)gridDim.x * blockDim.x) {   // warp-uniform
		const cu64 i = i0 + lane;
		cu32 h = 0;
		if (i < n) { h = mp_read(A, i, add, place); hits[i] = h; }
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
// per raw read of the chunk: its kept read's hit count, or OGB_MAP_FILTERED
__global__ void __launch_bounds__(256) k_map_hits(const cu32 *__restrict__ good, const cu64 *__restrict__ pos, const cu32 *__restrict__ khits, cu32 n,
                                                  cu32 *__restrict__ hits)
{
	OGB_SP_LOOP(i, n) hits[i] = good[i] ? khits[pos[i]] : OGB_MAP_FILTERED;
}
#endif

#endif

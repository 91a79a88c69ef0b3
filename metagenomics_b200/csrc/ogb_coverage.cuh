// ogb_coverage.cuh -- per-base read depth and abundance of the unitigs of the last ogb_graph_spell (ogb_spell.cuh), contained
// reads included.
//
// Unitig u = composite edge e with placements k = 0..c+1 (read r_k, strand, P_k, L_k as in ogb_spell.cuh). f(r) = the read's
// frequency (Dataset dedupe count). The depth profile D_u[p], 0 <= p < length(u), is
//   graph reads:     every placement k adds f(r_k) on [P_k, P_k + L_k);
//   contained reads: every read x with superReadID(x) = r_k adds f(x) on [a, a + L(x)), where q_x is the smallest shift in
//                    [0, L(r_k) - L(x)] at which x's stored strand equals r_k's forward strand, else the smallest at which x's
//                    reverse complement does, and a = P_k + q_x (r_k forward in u) or P_k + L(r_k) - q_x - L(x) (reverse).
// q_x depends on x and its super read only, so the twin unitig's profile is the reverse of u's, and a contained read whose super
// read is a branch node counts in every unitig that holds the node.
//
//   k_cov_locate   thread per read with sup != 0 (K2's packed L_super << 32 | ~super_idx): q_x by shifted compares against the super
//                  read's forward strand (cv_locate), counted per super read; an exclusive scan and k_cov_scatter build the CSR
//                  super read -> contained reads. Skipped when no read is contained (one read length: K2 is a no-op).
//   k_cov_init     thread per record: its ogb_unitig_coverage with zero sums, and its c + 2 placements; an exclusive scan gives the
//                  flat placement index, and a binary search over it the record of a placement (as sp_word finds its unitig). Without
//                  nplace (sample mapping, ogb_map.cuh) the records start with reads = 0.
//   k_cov_place    thread per placement (cv_place): +f at start + a, -f at start + a + L of a u32 difference array over the spell's
//                  word-aligned layout (atomicAdd mod 2^32), for the read and for each contained read of it
//   (scan)         one GLOBAL exclusive scan of the difference array: every +f/-f pair of a unitig lies in [start, start + length],
//                  so each unitig's net sum is 0 before the next start and no segment resets are needed. The scan sums in u64;
//                  its low 32 bits are the depth, which is < 2^32 (ogb_graph_coverage refuses frequencies that sum to 2^32 or more).
//   k_cov_reduce   warp per 32 words, lane per base: D[p] = low 32 bits of scan[p + 1] written as the u32 profile, and sum, sum of
//                  squares, min and max per unitig over [start, start + length); padding bases are written (as 0) but not reduced
//
// The compare of cv_locate uses the spell's sp_extract32 rather than region_equal of ogb_kernels.cuh (device loads and funnel
// intrinsics): the same code then runs in tests/coverage_emul.cpp. A shift almost always fails on its first 32 bases.
//
// Integer atomics only, so a run is deterministic. depth_sq_sum is exact while max(D)^2 * length < 2^64.
#ifndef OGB_COVERAGE_CUH_
#define OGB_COVERAGE_CUH_

#include "ogb_spell.cuh"

#define OGB_CV_UNPLACED 0xFFFFFFFFu

struct CovArgs {
	SpellArgs S;                    // read store, composite edges, item scan, spell records
	const cu64 *ppos;               // n_rec + 1: exclusive scan of the placements per record (c + 2)
	const cu32 *freq;               // per read idx
	const cu64 *sup;                // per read idx: K2's L_super << 32 | ~super_idx, 0 = not contained; null = none contained
	const cu32 *q;                  // per read idx: q_x of a contained read (OGB_CV_UNPLACED: no occurrence)
	const cu64 *cstart;             // n + 1: contained reads of super read idx s are clist[cstart[s] .. cstart[s + 1])
	const cu32 *clist;
};

// s[a .. a + len) == t[0 .. len) on packed strands, 32 bases at a time, stopping at the first differing word
OGB_HD bool cv_equal(const cu64 *s, cu64 a, const cu64 *t, cu32 len)
{
	for (cu32 k = 0; k < len; k += 32) {
		const cu32 n = len - k < 32 ? len - k : 32;
		if ((sp_extract32(s, a + k) ^ t[k >> 5]) & sp_top_bases(n)) return false;
	}
	return true;
}

// Hamming distance of s[a .. a + len) and t[0 .. len) on packed strands, 32 bases at a time; once it passes `limit` the count so far
// (> limit) is returned
OGB_HD cu32 cv_mismatches(const cu64 *s, cu64 a, const cu64 *t, cu32 len, cu32 limit)
{
	cu32 h = 0;
	for (cu32 k = 0; k < len; k += 32) {
		const cu32 n = len - k < 32 ? len - k : 32;
		const cu64 x = sp_extract32(s, a + k) ^ t[k >> 5];
#if defined(__CUDA_ARCH__)
		h += __popcll((x | x >> 1) & 0x5555555555555555ull & sp_top_bases(n));
#else
		h += __builtin_popcountll((x | x >> 1) & 0x5555555555555555ull & sp_top_bases(n));
#endif
		if (h > limit) return h;
	}
	return h;
}

// thread = read idx i with sup[i] != 0: q_x against its super read (OGB_CV_UNPLACED when neither strand occurs); *super_idx = its idx
OGB_HD cu32 cv_locate(const CovArgs &A, cu32 i, cu32 &super_idx)
{
	super_idx = 0xFFFFFFFFu - (cu32)(A.sup[i] & 0xFFFFFFFFull);
	cu64 ox, os; cu32 Lx, Ls, pwx, pws;
	sp_geom(A.S, i + 1, ox, Lx, pwx);
	sp_geom(A.S, super_idx + 1, os, Ls, pws);
	if (Lx > Ls) return OGB_CV_UNPLACED;
	const cu64 *sf = A.S.words + os;
	for (int strand = 0; strand < 2; strand++) {
		const cu64 *x = A.S.words + ox + (strand ? pwx : 0);
		for (cu32 q = 0; q + Lx <= Ls; q++)
			if (cv_equal(sf, q, x, Lx)) return q;
	}
	return OGB_CV_UNPLACED;
}

// largest u with pos[u] <= j (pos non-decreasing, pos[0] = 0)
OGB_HD cu64 cv_owner(const cu64 *pos, cu64 n, cu64 j)
{
	cu64 lo = 0, hi = n;
	while (hi - lo > 1) { const cu64 mid = (lo + hi) >> 1; if (pos[mid] <= j) lo = mid; else hi = mid; }
	return lo;
}

// thread = flat placement j: the record u it belongs to, and the +f / -f pairs of its read and of the reads contained in it, passed
// to add(position in the word-aligned layout, u32 value). Returns the reads' frequency sum; *contained = contained reads placed.
template <class ADD>
OGB_HD cu64 cv_place(const CovArgs &A, cu64 j, cu64 &u, cu32 &contained, ADD add)
{
	u = cv_owner(A.ppos, A.S.n_rec, j);
	const ogb_unitig R = A.S.rec[u];
	const ogb_cedge E = A.S.edges[R.edge];
	cu32 id; bool fwd; cu64 P;
	sp_piece(A.S, E, (cu32)(j - A.ppos[u]), id, fwd, P);
	cu64 off; cu32 L, pw;
	sp_geom(A.S, id, off, L, pw);
	const cu32 f = A.freq[id - 1];
	add(R.start + P, f);
	add(R.start + P + L, 0u - f);
	cu64 reads = f;
	contained = 0;
	if (A.cstart) {
		for (cu64 t = A.cstart[id - 1], te = A.cstart[id]; t < te; t++) {
			const cu32 x = A.clist[t];
			cu64 ox; cu32 Lx, pwx;
			sp_geom(A.S, x + 1, ox, Lx, pwx);
			const cu64 a = P + (fwd ? A.q[x] : L - A.q[x] - Lx);
			const cu32 fx = A.freq[x];
			add(R.start + a, fx);
			add(R.start + a + Lx, 0u - fx);
			reads += fx;
			contained++;
		}
	}
	return reads;
}

// the depth at base p of the layout from the exclusive scan of the difference array
OGB_HD cu32 cv_depth(const cu64 *scan, cu64 p) { return (cu32)scan[p + 1]; }

struct CovAcc {
	cu64 sum, sq;
	cu32 mn, mx;
};
OGB_HD void cv_acc_init(CovAcc &a) { a.sum = 0; a.sq = 0; a.mn = 0xFFFFFFFFu; a.mx = 0; }
OGB_HD void cv_acc_add(CovAcc &a, cu32 d) { a.sum += d; a.sq += (cu64)d * d; if (d < a.mn) a.mn = d; if (d > a.mx) a.mx = d; }

// add() of cv_place: atomic on the device, plain on the host (tests/coverage_emul.cpp); both mod 2^32
struct CvAdd {
	cu32 *diff;
	OGB_HD void operator()(cu64 p, cu32 v) const
	{
#if defined(__CUDA_ARCH__)
		atomicAdd(diff + p, v);
#else
		diff[p] += v;
#endif
	}
};

OGB_HD void cv_record(const ogb_unitig &R, ogb_unitig_coverage &o, cu32 count)
{
	o.edge = R.edge; o.reads = count + 2; o.contained = 0; o.depth_min = 0xFFFFFFFFu; o.depth_max = 0; o.reserved = 0;
	o.length = R.length; o.start = R.start; o.read_count = 0; o.depth_sum = 0; o.depth_sq_sum = 0;
}

#if defined(__CUDACC__)
__global__ void __launch_bounds__(256) k_cov_locate(CovArgs A, cu32 n, cu32 *q, cu32 *cnt, cu64 *unplaced)
{
	OGB_SP_LOOP(i, n) {
		if (!A.sup[i]) continue;
		cu32 s;
		const cu32 v = cv_locate(A, (cu32)i, s);
		q[i] = v;
		if (v == OGB_CV_UNPLACED) atomicAdd((unsigned long long *)unplaced, 1ull);
		else atomicAdd(cnt + s, 1u);
	}
}
__global__ void __launch_bounds__(256) k_cov_scatter(const cu64 *__restrict__ sup, const cu32 *__restrict__ q, cu32 n, const cu64 *__restrict__ cstart,
                                                     cu32 *fill, cu32 *clist)
{
	OGB_SP_LOOP(i, n) {
		const cu64 sv = sup[i];
		if (!sv || q[i] == OGB_CV_UNPLACED) continue;
		const cu32 s = 0xFFFFFFFFu - (cu32)(sv & 0xFFFFFFFFull);
		clist[cstart[s] + atomicAdd(fill + s, 1u)] = (cu32)i;        // the order inside a list does not change any sum
	}
}
__global__ void __launch_bounds__(256) k_cov_init(const ogb_unitig *__restrict__ rec, const ogb_cedge *__restrict__ edges, cu64 n_rec,
                                                  ogb_unitig_coverage *out, cu32 *nplace)
{
	OGB_SP_LOOP(u, n_rec) {
		const ogb_unitig R = rec[u];
		const cu32 c = edges[R.edge].count;
		cv_record(R, out[u], c);
		if (nplace) nplace[u] = c + 2;
		else out[u].reads = 0;                                 // sample mapping (ogb_map.cuh): reads counts its placements
	}
}
// n_place on the device (the scan's total): no host round trip before the launch
__global__ void __launch_bounds__(256) k_cov_place(CovArgs A, const cu64 *__restrict__ n_place, cu32 *diff, ogb_unitig_coverage *out,
                                                   cu64 *n_contained)
{
	const cu64 np = *n_place;
	const CvAdd add{diff};
	const cu32 lane = threadIdx.x & 31;
	for (cu64 j0 = (cu64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); j0 < np; j0 += (cu64)gridDim.x * blockDim.x) {   // warp-uniform
		const cu64 j = j0 + lane;
		cu64 u = ~0ull, reads = 0;
		cu32 nc = 0;
		if (j < np) reads = cv_place(A, j, u, nc, add);
		// consecutive placements mostly share a record: one atomic per warp then
		const cu64 u0 = __shfl_sync(0xFFFFFFFFu, u, 0);
		if (__all_sync(0xFFFFFFFFu, u == u0 || u == ~0ull)) {
			for (int d = 16; d > 0; d >>= 1) { reads += __shfl_down_sync(0xFFFFFFFFu, reads, d); nc += __shfl_down_sync(0xFFFFFFFFu, nc, d); }
			if (lane == 0) {
				atomicAdd((unsigned long long *)&out[u0].read_count, (unsigned long long)reads);
				if (nc) { atomicAdd(&out[u0].contained, nc); atomicAdd((unsigned long long *)n_contained, (unsigned long long)nc); }
			}
		} else if (u != ~0ull) {
			atomicAdd((unsigned long long *)&out[u].read_count, (unsigned long long)reads);
			if (nc) { atomicAdd(&out[u].contained, nc); atomicAdd((unsigned long long *)n_contained, (unsigned long long)nc); }
		}
	}
}
// the warp's sums of one record into the record (every lane calls it)
__device__ __forceinline__ void cv_flush(CovAcc a, ogb_unitig_coverage *o)
{
	for (int d = 16; d > 0; d >>= 1) {
		a.sum += __shfl_down_sync(0xFFFFFFFFu, a.sum, d); a.sq += __shfl_down_sync(0xFFFFFFFFu, a.sq, d);
		a.mn = min(a.mn, __shfl_down_sync(0xFFFFFFFFu, a.mn, d)); a.mx = max(a.mx, __shfl_down_sync(0xFFFFFFFFu, a.mx, d));
	}
	if ((threadIdx.x & 31) == 0) {
		atomicAdd((unsigned long long *)&o->depth_sum, (unsigned long long)a.sum);
		atomicAdd((unsigned long long *)&o->depth_sq_sum, (unsigned long long)a.sq);
		atomicMin(&o->depth_min, a.mn); atomicMax(&o->depth_max, a.mx);
	}
}
// warp per 32 consecutive words, lane per base: coalesced loads of the scan and stores of the profile; the sums of a record are
// flushed when the owner changes (a unitig of config 3 spans about 60 words on average)
__global__ void __launch_bounds__(256) k_cov_reduce(const cu64 *__restrict__ scan, const cu64 *__restrict__ wpos, cu64 n_rec, cu64 n_words,
                                                    cu32 *__restrict__ depth, ogb_unitig_coverage *out)
{
	const cu32 lane = threadIdx.x & 31;
	const cu64 warp = ((cu64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((cu64)gridDim.x * blockDim.x) >> 5;
	for (cu64 w0 = warp * 32; w0 < n_words; w0 += n_warps * 32) {
		const cu64 w1 = w0 + 32 < n_words ? w0 + 32 : n_words;
		cu64 u = cv_owner(wpos, n_rec, w0), uend = wpos[u + 1];
		cu64 len = out[u].length, base = 32 * wpos[u];
		CovAcc a; cv_acc_init(a);
		for (cu64 w = w0; w < w1; w++) {
			if (w == uend) {                                       // next record: flush the current one
				cv_flush(a, out + u);
				cv_acc_init(a);
				while (wpos[u + 1] <= w) u++;                          // (records of zero words do not exist: length >= 1)
				uend = wpos[u + 1]; len = out[u].length; base = 32 * wpos[u];
			}
			const cu64 p = 32 * w + lane;
			const cu32 d = cv_depth(scan, p);
			depth[p] = d;
			if (p - base < len) cv_acc_add(a, d);
		}
		cv_flush(a, out + u);
	}
}
#endif

#endif

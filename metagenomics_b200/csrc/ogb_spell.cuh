// ogb_spell.cuh -- the sequences of the unitigs of the simplified graph: what the reference's getStringInEdge (OverlapGraph.cpp:2009)
// returns for a composite edge, and what printGraph writes to the contigs file.
//
// Edge e = (src, dst, orient, offset) with items (read_k, off_k, or_k), k = 1..c, stands for reads r_0 = src, r_1..r_c, r_{c+1} = dst,
// src forward iff orient & 2, dst forward iff orient & 1, item k forward iff or_k == 1 (mergeList :760-785, mergedEdgeOrientation
// :803-829); positions P_0 = 0, P_k = off_1 + ... + off_k, P_{c+1} = offset. S(e) has offset + L[dst] bases; base p is base p - P_k of
// the oriented r_k, k the largest index with P_k <= p. Consecutive reads overlap by >= minOverlap (m) verified bases and no read in
// the graph is contained in another, so starts and ends both increase along the list and every read that covers p has the same base.
//
// Output: 2-bit packed like the read store (base p of a unitig in bits 63-2(p%32) .. 62-2(p%32) of its word p/32), every unitig
// starting on a word of its own, so one thread writes each output word and no two threads share one.
//
//   k_sp_select        thread per composite edge: selected (all, or canonical: src < dst, or src == dst and i < twin -- saveGraphToFile,
//                      OverlapGraph.cpp:321-326); an exclusive scan ranks the selected edges
//   k_sp_item_offsets  thread per item: its offset as u32; one flat exclusive scan gives P_k = scan[list_start + k] - scan[list_start]
//                      (lists are contiguous per edge)
//   k_sp_records       thread per edge whose rank lies in [first, first + count): its ogb_unitig record and its word count
//   k_spell_words      thread per output word (sp_word below)
//   k_spell_ascii      thread per packed word: 32 ACGT bytes
//
// Owner of a word's first base: a binary search over the edge's P_k (the scan above), not a word -> owner map written by one thread
// per read. With log-normal abundance (config 3) a high-coverage genome starts many reads inside one 32-base word; a map costs a thread
// and a scan position per READ whichever word it lands in, while the search costs O(log c) cached loads per WORD, so its work follows
// the output, not the depth of coverage. The read that owns the first base covers at least m + 1 bases from there, so for m >= 31 one
// unaligned 32-base extract from one stored strand fills the word; below that the loop moves on to the read that reaches furthest.
//
// The per-word body is `__host__ __device__` so that tests/spell_emul.cpp runs this very function on the CPU.
#ifndef OGB_SPELL_CUH_
#define OGB_SPELL_CUH_

#include <stdint.h>

#ifndef OGB_HD
#if defined(__CUDACC__)
#define OGB_HD __host__ __device__ __forceinline__
#else
#define OGB_HD inline
#endif
#endif

typedef unsigned int cu32;
typedef unsigned long long cu64;

struct SpellArgs {
	const cu64 *words;              // read store: forward strand of read idx at word off, reverse complement at off + pw
	const cu64 *meta;               // off << 16 | L per read idx; null = uniform_len / uniform_pw
	cu32 uniform_len, uniform_pw;
	const ogb_cedge *edges;
	const ogb_clist_item *items;
	const cu64 *ipos;               // n_items + 1: exclusive scan of the item offsets, total last
	const ogb_unitig *rec;
	cu64 n_rec;
	const cu64 *wpos;               // n_rec + 1: first output word of each record, total last
};

OGB_HD void sp_geom(const SpellArgs &A, cu32 id, cu64 &off, cu32 &L, cu32 &pw)
{
	if (A.meta) { const cu64 m = A.meta[id - 1]; L = (cu32)(m & 0xFFFF); off = m >> 16; pw = ((L + 63) >> 6) << 1; }
	else { L = A.uniform_len; pw = A.uniform_pw; off = (cu64)(id - 1) * 2 * pw; }
}

// 32 bases from base p of a packed strand (the words after a strand are always allocated; the caller masks what it does not own)
OGB_HD cu64 sp_extract32(const cu64 *w, cu64 p)
{
	const cu64 a = w[p >> 5], b = w[(p >> 5) + 1];
	const cu32 sh = (cu32)(p & 31) << 1;
	return sh ? (a << sh) | (b >> (64 - sh)) : a;
}

OGB_HD cu64 sp_top_bases(cu32 n) { return n >= 32 ? ~0ull : (n ? ~(~0ull >> (2 * n)) : 0ull); }   // the first n bases of a word

// r_k of edge E: read ID, forward?, P_k
OGB_HD void sp_piece(const SpellArgs &A, const ogb_cedge &E, cu32 k, cu32 &id, bool &fwd, cu64 &P)
{
	if (k == 0) { id = E.src; fwd = (E.orient & 2) != 0; P = 0; return; }
	if (k > E.count) { id = E.dst; fwd = (E.orient & 1) != 0; P = E.offset; return; }
	const ogb_clist_item it = A.items[E.list_start + k - 1];
	id = it.read; fwd = it.orient == 1; P = A.ipos[E.list_start + k] - A.ipos[E.list_start];
}
OGB_HD cu64 sp_pos(const SpellArgs &A, const ogb_cedge &E, cu32 k)
{
	if (k == 0) return 0;
	if (k > E.count) return E.offset;
	return A.ipos[E.list_start + k] - A.ipos[E.list_start];
}

// thread = output word w: the 32 bases S(e)[32j .. 32j+32) of the record u that owns w (j = w - wpos[u]); bases past the end are 0.
// Also writes the record's start (in bases of the word-aligned layout) when w is its first word.
OGB_HD cu64 sp_word(const SpellArgs &A, cu64 w, ogb_unitig *rec_out)
{
	cu64 lo = 0, hi = A.n_rec;                                 // largest u with wpos[u] <= w
	while (hi - lo > 1) { const cu64 mid = (lo + hi) >> 1; if (A.wpos[mid] <= w) lo = mid; else hi = mid; }
	const cu64 u = lo;
	const cu64 length = A.rec[u].length;                      // (not the whole record: the thread of its first word writes .start)
	if (w == A.wpos[u]) rec_out[u].start = 32 * w;
	const ogb_cedge E = A.edges[A.rec[u].edge];
	const cu64 p0 = 32 * (w - A.wpos[u]);
	const cu64 end = length - p0 < 32 ? length : p0 + 32;
	cu32 k = 0, kh = E.count + 1;                              // largest k with P_k <= p0
	while (kh > k) { const cu32 mid = k + ((kh - k + 1) >> 1); if (sp_pos(A, E, mid) <= p0) k = mid; else kh = mid - 1; }
	cu64 acc = 0, pos = p0;
	for (;;) {
		cu32 id, L, pw; bool fwd; cu64 P, off;
		sp_piece(A, E, k, id, fwd, P);
		sp_geom(A, id, off, L, pw);
		const cu64 q = pos - P;                                // r_k covers pos: P_k <= pos < P_k + L_k
		if (q >= L) break;                                     // cannot happen on a graph of verified overlaps
		const cu64 x = sp_extract32(A.words + off + (fwd ? 0 : pw), q);
		const cu64 stop = P + L < end ? P + L : end;
		const cu32 a = (cu32)(pos - p0), b = (cu32)(stop - p0);
		acc |= (x >> (2 * a)) & (sp_top_bases(b) & ~sp_top_bases(a));
		pos = stop;
		if (pos >= end) break;
		while (k <= E.count && sp_pos(A, E, k + 1) <= pos) k++;   // the read that reaches furthest (m < 31 only)
	}
	return acc;
}

OGB_HD bool sp_canonical(const ogb_cedge *edges, cu64 i)
{
	const ogb_cedge e = edges[i];
	return e.src < e.dst || (e.src == e.dst && i < e.twin);
}

// thread = composite edge i with rank r among the selected ones (exclusive scan of k_sp_select): its record when r is in the range.
// Returns the unitig's length (0: not in the range).
OGB_HD cu64 sp_record(const SpellArgs &A, cu64 i, cu64 r, cu64 first, cu64 count, ogb_unitig *rec, cu32 *nwords)
{
	if (r < first || r - first >= count) return 0;
	const ogb_cedge e = A.edges[i];
	cu64 off; cu32 L, pw;
	sp_geom(A, e.dst, off, L, pw);
	ogb_unitig o;
	o.edge = (cu32)i; o.src = e.src; o.dst = e.dst; o.orient = e.orient; o.reserved[0] = o.reserved[1] = o.reserved[2] = 0;
	o.length = e.offset + L; o.start = 0;
	rec[r - first] = o;
	nwords[r - first] = (cu32)((o.length + 31) / 32);
	return o.length;
}

#if defined(__CUDACC__)
#define OGB_SP_LOOP(i, n) for (cu64 i = (cu64)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (cu64)gridDim.x * blockDim.x)

__global__ void __launch_bounds__(256) k_sp_select(const ogb_cedge *__restrict__ edges, cu64 ne, int canonical_only, cu32 *sel)
{
	OGB_SP_LOOP(i, ne) sel[i] = canonical_only ? (sp_canonical(edges, i) ? 1u : 0u) : 1u;
}
__global__ void __launch_bounds__(256) k_sp_item_offsets(const ogb_clist_item *__restrict__ items, cu64 ni, cu32 *out)
{
	OGB_SP_LOOP(i, ni) out[i] = items[i].offset;
}
__global__ void __launch_bounds__(256) k_sp_records(SpellArgs A, cu64 ne, const cu32 *__restrict__ sel, const cu64 *__restrict__ rank, cu64 first,
                                                    cu64 count, ogb_unitig *rec, cu32 *nwords, cu64 *bases)
{
	OGB_SP_LOOP(i, ne) {
		const cu64 len = sel[i] ? sp_record(A, i, rank[i], first, count, rec, nwords) : 0;
		if (len) atomicAdd((unsigned long long *)bases, (unsigned long long)len);
	}
}
__global__ void __launch_bounds__(256) k_spell_words(SpellArgs A, cu64 n_words, ogb_unitig *rec, cu64 *__restrict__ out)
{
	OGB_SP_LOOP(w, n_words) out[w] = sp_word(A, w, rec);
}
// words [w0, w1) -> 32 bytes each at out[32 (w - w0)]
__global__ void __launch_bounds__(256) k_spell_ascii(const cu64 *__restrict__ words, cu64 w0, cu64 w1, char *__restrict__ out)
{
	OGB_SP_LOOP(i, w1 - w0) {
		const cu64 x = words[w0 + i];
		cu64 *o = reinterpret_cast<cu64 *>(out + 32 * i);
		#pragma unroll
		for (int q = 0; q < 4; q++) {
			cu64 v = 0;
			#pragma unroll
			for (int b = 0; b < 8; b++) {
				const cu32 code = (cu32)(x >> (62 - 2 * (8 * q + b))) & 3;
				v |= (cu64)(0x54474341u >> (8 * code) & 0xFF) << (8 * b);     // "ACGT" little-endian
			}
			o[q] = v;
		}
	}
}
#endif

#endif

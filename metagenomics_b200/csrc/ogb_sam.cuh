// ogb_sam.cuh -- the placements of a sample's reads on the unitigs of the last ogb_graph_spell as SAM text, formatted on the device
// (ogb_graph_map_reads_sam). The mapping is ogb_map.cuh's, unchanged; this file re-runs its search for the mapped reads of a chunk,
// keeps every placement and writes one line per record.
//
// Records of raw read i (0-based in the sample), in input order:
//   filtered                 1 record:  FLAG 4, SEQ = the raw bytes upper-cased, a non-letter as N ('*' if empty), tag YF:Z:filtered
//   kept, not mapped         1 record:  FLAG 4, SEQ = the read
//   mapped, h placements     h records, ascending (u, p): FLAG 16 strand + 256 (k > 0), RNAME unitig_<first + u>, POS p + 1,
//                            MAPQ 60 (h == 1) or 0, CIGAR <L>M, SEQ = the read (reverse complement on strand 1), NM:i:b MD:Z:<md> NH:i:h
// RNEXT *, PNEXT 0, TLEN 0 and QUAL * everywhere. A placement is on strand 0 iff H_fw(u, p) == b (the rule of mp_read's pass 2).
// QNAME: the caller's name of the read, or i in decimal.
//
// Per chunk, after k_map_reads (which also wrote each kept read's stratum):
//   scan          khits -> slot of each kept read's first placement
//   k_map_emit    thread per mapped kept read: mp_search again, (p << 1 | strand) into its slots, p the layout position (so the order
//                 of p is the order of (u, p)); then the read's slots sorted in the thread (sm_sort). The walk order of the index
//                 buckets (filled with atomics) changes from run to run; after the sort the slots do not.
//   k_sam_count   per raw read: its record count; scan -> first record of each raw read
//   k_sam_len     thread per record: the byte length of its line (sm_line with a counting sink); scan -> byte offsets
//   k_sam_cut     the records whose text starts in [s B, (s + 1) B) form slice s (B = OGB_SAM_SLICE)
//   k_sam_write   thread per record of one slice: its line (sm_line with a writing sink), then the slice goes to the host
// Lengths and text come from one body (sm_line), so a line fills exactly the bytes its length reserved.
#ifndef OGB_SAM_CUH_
#define OGB_SAM_CUH_

#include "ogb_map.cuh"

struct SamArgs {
	MapArgs M;                      // layout, unitig records, the chunk's read store (rwords / rmeta per kept read)
	const char *raw;                // the chunk's raw bytes: read i = raw[roffs[i] .. roffs[i + 1])
	const cu64 *roffs;
	const cu32 *good;               // per raw read: kept by the filter
	const cu64 *pos;                // per raw read: its kept index
	const cu32 *khits;              // per kept read: placements
	const unsigned char *kstrat;    // per kept read: stratum b
	const cu64 *kslot;              // per kept read: its first slot
	const cu64 *slot;               // per placement: p << 1 | strand, ascending per read
	const cu64 *rstart;             // n + 1: first record of each raw read, total last
	cu64 n;                         // raw reads of the chunk
	const char *names;              // NULL: QNAME = index0 + i; else read i's name = names[noffs[i] .. noffs[i + 1])
	const cu64 *noffs;
	cu64 index0;                    // sample index of the chunk's first read
	cu64 first;                     // name of unitig u = unitig_<first + u>
};

// sorts x[0 .. n) ascending (distinct keys): insertion sort for a few, heap sort beyond, both in the thread -- the search that filled
// them walked every candidate serially, so O(n log n) here stays of its order
OGB_HD void sm_sort(cu64 *x, cu32 n)
{
	if (n <= 16) {
		for (cu32 a = 1; a < n; a++) {
			const cu64 v = x[a];
			cu32 b = a;
			for (; b && x[b - 1] > v; b--) x[b] = x[b - 1];
			x[b] = v;
		}
		return;
	}
	auto sift = [&](cu32 r, cu32 end) {
		for (;;) {
			cu32 c = 2 * r + 1;
			if (c >= end) return;
			if (c + 1 < end && x[c + 1] > x[c]) c++;
			if (x[r] >= x[c]) return;
			const cu64 t = x[r]; x[r] = x[c]; x[c] = t;
			r = c;
		}
	};
	for (cu32 r = n / 2; r-- > 0;) sift(r, n);
	for (cu32 e = n - 1; e > 0; e--) {
		const cu64 t = x[0]; x[0] = x[e]; x[e] = t;
		sift(0, e);
	}
}

// thread = kept read i with khits[i] > 0: its placements into out[0 .. khits[i]), sorted. Returns their count.
template <bool EXACT>
OGB_HD cu32 sm_emit(const MapArgs &A, cu64 i, cu64 *out)
{
	cu32 k = 0, strat;
	mp_search<EXACT>(A, i, [&](cu64 p, cu64, cu32, int s) { out[k++] = p << 1 | (cu64)s; }, strat);
	sm_sort(out, k);
	return k;
}

// records of raw read i: max(1, hits) for a kept read, 1 for a filtered one
OGB_HD cu32 sm_records(const SamArgs &S, cu64 i)
{
	if (!S.good[i]) return 1;
	const cu32 h = S.khits[S.pos[i]];
	return h ? h : 1;
}

// Sinks of sm_line: SmCount adds up the bytes, SmWrite stores them. fill(n, f) emits f(0) .. f(n - 1).
struct SmCount {
	cu64 n = 0;
	OGB_HD void put(char) { n++; }
	template <class F> OGB_HD void fill(cu32 k, F) { n += k; }
};
struct SmWrite {
	char *o;
	OGB_HD void put(char c) { *o++ = c; }
	template <class F> OGB_HD void fill(cu32 k, F f) { for (cu32 j = 0; j < k; j++) *o++ = f(j); }
};

template <class OUT>
OGB_HD void sm_num(OUT &o, cu64 x)
{
	char d[20];
	cu32 n = 0;
	do { d[n++] = (char)('0' + x % 10); x /= 10; } while (x);
	o.fill(n, [&](cu32 j) { return d[n - 1 - j]; });
}
template <class OUT>
OGB_HD void sm_str(OUT &o, const char *s)
{
	while (*s) o.put(*s++);
}

OGB_HD char sm_base(const cu64 *t, cu64 k) { return "ACGT"[(t[k >> 5] >> (62 - 2 * (k & 31))) & 3]; }

OGB_HD cu32 sm_clz(cu64 x)
{
#if defined(__CUDA_ARCH__)
	return (cu32)__clzll((long long)x);
#else
	return (cu32)__builtin_clzll(x);
#endif
}

// MD of strand t (L bases) against layout bases [p, p + L): the xor of 32 bases at a time, one mismatch per set pair of bits
template <class OUT>
OGB_HD void sm_md(OUT &o, const cu64 *layout, cu64 p, const cu64 *t, cu32 L)
{
	cu32 run = 0;                                                         // read position after the last mismatch
	for (cu32 k = 0; k < L; k += 32) {
		const cu32 n = L - k < 32 ? L - k : 32;
		const cu64 ref = sp_extract32(layout, p + k);
		cu64 x = (ref ^ t[k >> 5]);
		x = (x | x >> 1) & 0x5555555555555555ull & sp_top_bases(n);
		while (x) {
			const cu32 j = sm_clz(x) >> 1;                                    // base j sits in bits 63 - 2j, 62 - 2j
			x &= ~(1ull << (62 - 2 * j));
			sm_num(o, k + j - run);
			o.put("ACGT"[(ref >> (62 - 2 * j)) & 3]);
			run = k + j + 1;
		}
	}
	sm_num(o, L - run);
}

// the line of record r of the chunk (owner: raw read i = the largest with rstart[i] <= r), newline included
template <class OUT>
OGB_HD void sm_line(const SamArgs &S, cu64 r, OUT &o)
{
	const cu64 i = cv_owner(S.rstart, S.n, r), k = r - S.rstart[i];
	if (S.names) {
		const char *q = S.names + S.noffs[i];
		o.fill((cu32)(S.noffs[i + 1] - S.noffs[i]), [&](cu32 j) { return q[j]; });
	} else {
		sm_num(o, S.index0 + i);
	}
	if (!S.good[i]) {
		const char *b = S.raw + S.roffs[i];
		const cu32 n = (cu32)(S.roffs[i + 1] - S.roffs[i]);
		sm_str(o, "\t4\t*\t0\t0\t*\t*\t0\t0\t");
		if (!n) o.put('*');
		o.fill(n, [&](cu32 j) {
			const char c = b[j];
			return c >= 'a' && c <= 'z' ? (char)(c - 32) : c >= 'A' && c <= 'Z' ? c : 'N';
		});
		sm_str(o, "\t*\tYF:Z:filtered\n");
		return;
	}
	const cu64 j = S.pos[i], m = S.M.rmeta[j];
	const cu32 L = (cu32)(m & 0xFFFF), pw = ((L + 63) >> 6) << 1, h = S.khits[j];
	const cu64 *fw = S.M.rwords + (m >> 16);
	if (!h) {
		sm_str(o, "\t4\t*\t0\t0\t*\t*\t0\t0\t");
		o.fill(L, [&](cu32 q) { return sm_base(fw, q); });
		sm_str(o, "\t*\n");
		return;
	}
	const cu64 x = S.slot[S.kslot[j] + k], p = x >> 1;
	const cu32 s = (cu32)(x & 1);
	const cu64 u = cv_owner(S.M.wpos, S.M.n_rec, p >> 5);
	const cu64 *t = fw + (s ? pw : 0);
	o.put('\t');
	sm_num(o, 16 * s + (k ? 256 : 0));
	sm_str(o, "\tunitig_");
	sm_num(o, S.first + u);
	o.put('\t');
	sm_num(o, p - 32 * S.M.wpos[u] + 1);
	sm_str(o, h == 1 ? "\t60\t" : "\t0\t");
	sm_num(o, L);
	sm_str(o, "M\t*\t0\t0\t");
	o.fill(L, [&](cu32 q) { return sm_base(t, q); });
	sm_str(o, "\t*\tNM:i:");
	sm_num(o, S.kstrat[j]);
	sm_str(o, "\tMD:Z:");
	sm_md(o, S.M.layout, p, t, L);
	sm_str(o, "\tNH:i:");
	sm_num(o, h);
	o.put('\n');
}

#if defined(__CUDACC__)
template <bool EXACT>
__global__ void __launch_bounds__(256) k_map_emit(MapArgs A, cu32 n, const cu32 *__restrict__ khits, const cu64 *__restrict__ kslot, cu64 *slot)
{
	OGB_SP_LOOP(i, n) if (khits[i]) sm_emit<EXACT>(A, i, slot + kslot[i]);
}
__global__ void __launch_bounds__(256) k_sam_count(SamArgs S, cu32 *cnt)
{
	OGB_SP_LOOP(i, S.n) cnt[i] = sm_records(S, i);
}
__global__ void __launch_bounds__(256) k_sam_len(SamArgs S, cu64 n_rec, cu32 *len)
{
	OGB_SP_LOOP(r, n_rec) {
		SmCount o;
		sm_line(S, r, o);
		len[r] = (cu32)o.n;
	}
}
// cut[s] = the first record whose text starts at or after s B (s = 0 .. ns - 1), cut[ns] = n_rec; at[s] = that record's offset
__global__ void __launch_bounds__(256) k_sam_cut(const cu64 *__restrict__ off, cu64 n_rec, cu64 B, cu64 ns, cu64 *cut, cu64 *at)
{
	OGB_SP_LOOP(s, ns + 1) {
		cu64 lo = 0, hi = n_rec;
		if (s < ns)
			while (lo < hi) { const cu64 mid = (lo + hi) >> 1; if (off[mid] < s * B) lo = mid + 1; else hi = mid; }
		else lo = n_rec;
		cut[s] = lo;
		at[s] = off[lo];
	}
}
__global__ void __launch_bounds__(256) k_sam_write(SamArgs S, cu64 r0, cu64 r1, const cu64 *__restrict__ off, char *text)
{
	const cu64 base = off[r0];
	OGB_SP_LOOP(k, r1 - r0) {
		SmWrite o{text + (off[r0 + k] - base)};
		sm_line(S, r0 + k, o);
	}
}
#endif

#endif

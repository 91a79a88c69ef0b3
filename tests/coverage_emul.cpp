// TEST INFRASTRUCTURE: runs the per-thread bodies of metagenomics_b200/csrc/ogb_coverage.cuh -- the functions the coverage kernels
// call -- on the CPU in the launch order of ogb_graph_coverage (csrc/ogb_device.cu), scans included, on the records and layout of a
// spell, so that the logic of the device coverage is checked against the plain restatement (oracle/unitig_coverage.py) where no
// GPU is present. The product never links or calls this file; the -m gpu tests check the kernels themselves.
//
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/_build/libcoverage_emul.so tests/coverage_emul.cpp
#include <vector>

#include "../include/ogb.h"
#include "../metagenomics_b200/csrc/ogb_coverage.cuh"

// words / meta: the read store (meta[idx] = off << 16 | L); edges / items: the simplified graph; rec / n_rec: the records of a spell
// of it (start included); freq / sup: per read idx (sup as K2 packs it, 0 = not contained). Writes n_rec coverage records and the
// depth of 32 * words bases; returns the number of unplaced contained reads, or -1 when the layout has a different size.
extern "C" long long emul_coverage(const cu64 *words, const cu64 *meta, uint32_t n_reads, const ogb_cedge *edges, const ogb_clist_item *items,
                                   uint64_t ni, const ogb_unitig *rec, uint64_t n_rec, const uint32_t *freq, const cu64 *sup,
                                   ogb_unitig_coverage *out, uint32_t *depth, uint64_t n_words, uint64_t *contained_placements)
{
	CovArgs A;
	A.S.words = words; A.S.meta = meta; A.S.uniform_len = 0; A.S.uniform_pw = 0; A.S.edges = edges; A.S.items = items;
	A.S.rec = rec; A.S.n_rec = n_rec; A.S.wpos = nullptr;
	std::vector<cu64> ipos(ni + 1, 0);
	for (cu64 i = 0; i < ni; i++) ipos[i + 1] = ipos[i] + items[i].offset;
	A.S.ipos = ipos.data();
	A.freq = freq;
	// locate, count per super read, scan, scatter (reverse thread order: the order inside a list must not matter)
	std::vector<cu32> q(n_reads, OGB_CV_UNPLACED), cnt(n_reads, 0), clist(n_reads);
	std::vector<cu64> cstart((cu64)n_reads + 1, 0);
	long long unplaced = 0;
	bool any = false;
	for (cu32 i = 0; i < n_reads; i++) any |= sup[i] != 0;
	A.sup = any ? sup : nullptr; A.q = nullptr; A.cstart = nullptr; A.clist = nullptr;
	if (any) {
		for (cu32 i = 0; i < n_reads; i++) {
			if (!sup[i]) continue;
			cu32 s;
			q[i] = cv_locate(A, i, s);
			if (q[i] == OGB_CV_UNPLACED) unplaced++;
			else cnt[s]++;
		}
		for (cu32 i = 0; i < n_reads; i++) cstart[i + 1] = cstart[i] + cnt[i];
		std::vector<cu32> fill(n_reads, 0);
		for (cu32 i = n_reads; i-- > 0;) {
			if (!sup[i] || q[i] == OGB_CV_UNPLACED) continue;
			const cu32 s = 0xFFFFFFFFu - (cu32)(sup[i] & 0xFFFFFFFFull);
			clist[cstart[s] + fill[s]++] = i;
		}
		A.q = q.data(); A.cstart = cstart.data(); A.clist = clist.data();
	}
	// records, placement scan, placements into the difference array (reverse order)
	std::vector<cu64> ppos(n_rec + 1, 0);
	for (cu64 u = 0; u < n_rec; u++) {
		cv_record(rec[u], out[u], edges[rec[u].edge].count);
		ppos[u + 1] = ppos[u] + out[u].reads;
		if (rec[u].start + rec[u].length > 32 * n_words) return -1;
	}
	A.ppos = ppos.data();
	std::vector<cu32> diff(32 * n_words + 1, 0);
	const CvAdd add{diff.data()};
	*contained_placements = 0;
	for (cu64 j = ppos[n_rec]; j-- > 0;) {
		cu64 u; cu32 nc;
		const cu64 reads = cv_place(A, j, u, nc, add);
		out[u].read_count += reads;
		out[u].contained += nc;
		*contained_placements += nc;
	}
	std::vector<cu64> scan(32 * n_words + 1, 0);
	for (cu64 p = 0; p < 32 * n_words; p++) scan[p + 1] = scan[p] + diff[p];
	for (cu64 p = 0; p < 32 * n_words; p++) depth[p] = cv_depth(scan.data(), p);
	for (cu64 u = 0; u < n_rec; u++) {
		CovAcc a;
		cv_acc_init(a);
		for (cu64 p = 0; p < rec[u].length; p++) cv_acc_add(a, depth[rec[u].start + p]);
		out[u].depth_sum = a.sum; out[u].depth_sq_sum = a.sq; out[u].depth_min = a.mn; out[u].depth_max = a.mx;
	}
	return unplaced;
}

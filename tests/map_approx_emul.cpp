// TEST INFRASTRUCTURE: runs the per-thread bodies of metagenomics_b200/csrc/ogb_map.cuh -- the index entries of a layout word
// (mp_word) and the seeded search of a read with up to d substitutions (mp_read) -- on the CPU in the launch order of
// ogb_graph_map_reads_approx (csrc/ogb_device.cu), CSR and scans included, with the coverage reduction's per-base accumulators
// (ogb_coverage.cuh), so that the logic of the device mapping is checked against the plain restatement
// (tests/map_approx_lib.py: map_sample_approx) where no GPU is present. The reads come kept and packed already (the filter is
// sample_map.kept, the packing unitig_lib.store_layout): tests/map_emul.cpp checks the filter and packer. The product never links or
// calls this file; the -m gpu tests check the kernels themselves.
//
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/_build/libmap_approx_emul.so tests/map_approx_emul.cpp
#include <vector>

#include "../include/ogb.h"
#include "../metagenomics_b200/csrc/ogb_map.cuh"

// layout: the spell's packed words (n_words of them); rec / n_rec: its records (start included); the kept reads: n_kept of them in
// the device read store (rwords, rmeta: off << 16 | L); m: the build's minOverlap, d: max_mismatches. Writes n_rec records, the depth
// of 32 * n_words bases, n_kept hit counts and strata and ctr = {mapped, multi, placements, index entries, index buckets}.
extern "C" void emul_map_approx(const cu64 *layout_in, uint64_t n_words, const ogb_unitig *rec, uint64_t n_rec, const cu64 *rwords,
                                const cu64 *rmeta, uint64_t n_kept, uint32_t m, uint32_t d, ogb_unitig_coverage *out, uint32_t *depth,
                                uint32_t *hits, uint8_t *strat, uint64_t *ctr)
{
	std::vector<cu64> layout(layout_in, layout_in + n_words);
	layout.push_back(0);                                                   // the spell's spare zero word
	std::vector<cu64> wpos(n_rec + 1, n_words);
	cu64 bases_total = 0;
	for (cu64 u = 0; u < n_rec; u++) { wpos[u] = rec[u].start / 32; bases_total += rec[u].length; }
	MapArgs A;
	A.layout = layout.data(); A.wpos = wpos.data(); A.rec = rec; A.n_rec = n_rec;
	A.K = m + 1 < 32 ? m + 1 : 32;
	A.d = d;
	const cu64 B = mp_buckets(bases_total);
	A.bmask = B - 1;
	// index: count, scan, fill (words in reverse order: the order inside a bucket must not matter)
	std::vector<cu32> cnt(B, 0);
	for (cu64 w = 0; w < n_words; w++) mp_word(A, w, [&](cu64 b, cu32, cu64) { cnt[b]++; });
	std::vector<cu64> bstart(B + 1, 0);
	for (cu64 b = 0; b < B; b++) bstart[b + 1] = bstart[b] + cnt[b];
	std::vector<cu64> ent(bstart[B] + 1);
	std::vector<cu32> fill(B, 0);
	A.bstart = bstart.data();
	for (cu64 w = n_words; w-- > 0;) mp_word(A, w, [&](cu64 b, cu32 tag, cu64 p) { ent[bstart[b] + fill[b]++] = (cu64)tag << 32 | p; });
	A.ent = ent.data();
	A.rwords = rwords; A.rmeta = rmeta;
	// records (k_cov_init without placements), mapping (reverse order), scan, reduction
	for (cu64 u = 0; u < n_rec; u++) { cv_record(rec[u], out[u], 0); out[u].reads = 0; }
	std::vector<cu32> diff(32 * n_words + 1, 0);
	const CvAdd add{diff.data()};
	const MpPlace place{out};
	for (int k = 0; k < 5; k++) ctr[k] = 0;
	for (cu64 i = n_kept; i-- > 0;) {
		cu32 b;
		hits[i] = mp_read(A, i, add, place, b);
		strat[i] = (uint8_t)b;
		ctr[0] += hits[i] > 0; ctr[1] += hits[i] > 1; ctr[2] += hits[i];
	}
	ctr[3] = bstart[B]; ctr[4] = B;
	std::vector<cu64> scan(32 * n_words + 1, 0);
	for (cu64 p = 0; p < 32 * n_words; p++) scan[p + 1] = scan[p] + diff[p];
	for (cu64 p = 0; p < 32 * n_words; p++) depth[p] = cv_depth(scan.data(), p);
	for (cu64 u = 0; u < n_rec; u++) {
		CovAcc a;
		cv_acc_init(a);
		for (cu64 p = 0; p < rec[u].length; p++) cv_acc_add(a, depth[rec[u].start + p]);
		out[u].depth_sum = a.sum; out[u].depth_sq_sum = a.sq; out[u].depth_min = a.mn; out[u].depth_max = a.mx;
	}
}

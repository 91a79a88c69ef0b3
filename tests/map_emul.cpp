// TEST INFRASTRUCTURE: runs the per-thread bodies of metagenomics_b200/csrc/ogb_map.cuh -- the index entries of a layout word
// (mp_word) and the query and verification of a read (mp_read) -- on the CPU in the launch order of ogb_graph_map_reads
// (csrc/ogb_device.cu), CSR and scans included, with the coverage reduction's per-base accumulators (ogb_coverage.cuh), so that the
// logic of the device mapping is checked against the plain restatement (oracle/sample_map.py) where no GPU is present. The filter
// and the packing are k_ds_filter's and k_pack_ascii's rules, restated. The product never links or calls this file; the -m gpu
// tests check the kernels themselves.
//
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/_build/libmap_emul.so tests/map_emul.cpp
#include <vector>

#include "../include/ogb.h"
#include "../metagenomics_b200/csrc/ogb_map.cuh"

// layout: the spell's packed words (n_words of them, plus room for one more); rec / n_rec: its records (start included); the sample:
// n reads, read i = bases[offsets[i] .. offsets[i+1]); m: the build's minOverlap. Writes n_rec records, the depth of 32 * n_words
// bases, n hit counts and ctr = {filtered, mapped, multi, placements, index entries, index buckets}.
extern "C" void emul_map(const cu64 *layout_in, uint64_t n_words, const ogb_unitig *rec, uint64_t n_rec, const char *bases, const uint64_t *offsets,
                         uint64_t n, uint32_t m, ogb_unitig_coverage *out, uint32_t *depth, uint32_t *hits, uint64_t *ctr)
{
	std::vector<cu64> layout(layout_in, layout_in + n_words);
	layout.push_back(0);                                                   // the spell's spare zero word
	std::vector<cu64> wpos(n_rec + 1, n_words);
	cu64 bases_total = 0;
	for (cu64 u = 0; u < n_rec; u++) { wpos[u] = rec[u].start / 32; bases_total += rec[u].length; }
	MapArgs A;
	A.layout = layout.data(); A.wpos = wpos.data(); A.rec = rec; A.n_rec = n_rec;
	A.K = m + 1 < 32 ? m + 1 : 32;
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
	// the sample: filter (k_ds_filter), read store with meta (k_map_geom / k_map_meta), packing (k_pack_ascii)
	std::vector<cu64> meta, words;
	std::vector<cu64> kept_of(n, ~0ull);
	for (cu64 i = 0; i < n; i++) {
		const cu64 len = offsets[i + 1] - offsets[i];
		const char *s = bases + offsets[i];
		bool ok = len > m && len < 65536;
		cu32 c4[4] = {0, 0, 0, 0};
		for (cu64 k = 0; ok && k < len; k++) {
			const cu32 ch = (cu32)(unsigned char)s[k] & ~0x20u;
			if (ch != 'A' && ch != 'C' && ch != 'G' && ch != 'T') ok = false;
			else c4[(ch >> 1) & 3]++;
		}
		if (ok) {
			const cu32 thr = (cu32)((cu32)len * .8);
			if (c4[0] >= thr || c4[1] >= thr || c4[2] >= thr || c4[3] >= thr) ok = false;
		}
		if (!ok) continue;
		const cu32 L = (cu32)len, pw = ((L + 63) >> 6) << 1;
		kept_of[i] = meta.size();
		meta.push_back((cu64)words.size() << 16 | L);
		const size_t off = words.size();
		words.resize(off + 2 * pw, 0);
		for (cu32 p = 0; p < L; p++) {
			cu32 c = ((cu32)s[p] >> 1) & 3; c ^= c >> 1;
			cu32 d = ((cu32)s[L - 1 - p] >> 1) & 3; d ^= d >> 1;
			words[off + p / 32] |= (cu64)c << (62 - 2 * (p % 32));
			words[off + pw + p / 32] |= (cu64)(3 - d) << (62 - 2 * (p % 32));
		}
	}
	words.resize(words.size() + 8, 0);
	A.rwords = words.data(); A.rmeta = meta.data();
	// records (k_cov_init without placements), mapping (reverse order), scan, reduction
	for (cu64 u = 0; u < n_rec; u++) { cv_record(rec[u], out[u], 0); out[u].reads = 0; }
	std::vector<cu32> diff(32 * n_words + 1, 0), khits(meta.size());
	const CvAdd add{diff.data()};
	const MpPlace place{out};
	for (cu64 i = meta.size(); i-- > 0;) khits[i] = mp_read(A, i, add, place);
	for (int k = 0; k < 6; k++) ctr[k] = 0;
	for (cu64 i = 0; i < n; i++) {
		if (kept_of[i] == ~0ull) { hits[i] = OGB_MAP_FILTERED; ctr[0]++; continue; }
		hits[i] = khits[kept_of[i]];
		ctr[1] += hits[i] > 0; ctr[2] += hits[i] > 1; ctr[3] += hits[i];
	}
	ctr[4] = bstart[B]; ctr[5] = B;
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

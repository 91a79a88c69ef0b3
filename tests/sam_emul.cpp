// TEST INFRASTRUCTURE: runs the per-thread bodies of metagenomics_b200/csrc/ogb_sam.cuh -- the search again with every placement
// kept and sorted (sm_emit), the record counts (sm_records) and the line of a record, counted (SmCount) and written (SmWrite) -- on
// the CPU in the launch order of ogb_graph_map_reads_sam (csrc/ogb_device.cu), over one chunk, so that the SAM records can be checked
// against the plain restatement (tests/sam_lib.py) where no GPU is present. The index, hits and strata come from the bodies of
// ogb_map.cuh as in tests/map_approx_emul.cpp. The reads come with the filter's verdict and kept reads packed already (the filter is
// sample_map.kept, the packing unitig_lib.store_layout). The product never links or calls this file; the -m gpu tests check the kernels.
//
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/_build/libsam_emul.so tests/sam_emul.cpp
#include <string>
#include <vector>

#include "../include/ogb.h"
#include "../metagenomics_b200/csrc/ogb_sam.cuh"

static std::string g_text;

// layout / n_words, rec / n_rec: the spell; raw / roffs / n: the raw reads; good: the filter's verdict per raw read; rwords / rmeta:
// the kept reads' store; names / noffs: NULL or the QNAMEs; m, d, first as in the product; reverse: fill the index buckets and run
// the emit threads in reverse order (the walk order changes, the text must not). Returns the records' text (no header) in *text.
extern "C" uint64_t emul_sam(const cu64 *layout_in, uint64_t n_words, const ogb_unitig *rec, uint64_t n_rec, const char *raw, const cu64 *roffs,
                             uint64_t n, const cu32 *good, const cu64 *rwords, const cu64 *rmeta, const char *names, const cu64 *noffs, uint32_t m,
                             uint32_t d, uint64_t first, int reverse, const char **text)
{
	std::vector<cu64> layout(layout_in, layout_in + n_words);
	layout.push_back(0);
	std::vector<cu64> wpos(n_rec + 1, n_words);
	cu64 bases_total = 0;
	for (cu64 u = 0; u < n_rec; u++) { wpos[u] = rec[u].start / 32; bases_total += rec[u].length; }
	MapArgs A;
	A.layout = layout.data(); A.wpos = wpos.data(); A.rec = rec; A.n_rec = n_rec;
	A.K = m + 1 < 32 ? m + 1 : 32;
	A.d = d;
	const cu64 B = mp_buckets(bases_total);
	A.bmask = B - 1;
	std::vector<cu32> cnt(B, 0);
	for (cu64 w = 0; w < n_words; w++) mp_word(A, w, [&](cu64 b, cu32, cu64) { cnt[b]++; });
	std::vector<cu64> bstart(B + 1, 0);
	for (cu64 b = 0; b < B; b++) bstart[b + 1] = bstart[b] + cnt[b];
	std::vector<cu64> ent(bstart[B] + 1);
	std::vector<cu32> fill(B, 0);
	A.bstart = bstart.data();
	for (cu64 k = 0; k < n_words; k++) {
		const cu64 w = reverse ? n_words - 1 - k : k;
		mp_word(A, w, [&](cu64 b, cu32 tag, cu64 p) { ent[bstart[b] + fill[b]++] = (cu64)tag << 32 | p; });
	}
	A.ent = ent.data();
	A.rwords = rwords; A.rmeta = rmeta;
	// the chunk: kept index per raw read, k_map_reads (hits, strata), slots, k_map_emit
	std::vector<cu64> pos(n + 1, 0);
	for (cu64 i = 0; i < n; i++) pos[i + 1] = pos[i] + (good[i] ? 1 : 0);
	const cu64 kept = pos[n];
	std::vector<cu32> khits(kept + 1, 0);
	std::vector<unsigned char> kstrat(kept + 1, 0);
	for (cu64 j = 0; j < kept; j++) {
		cu32 b;
		khits[j] = mp_read(A, j, [](cu64, cu32) {}, [](cu64) {}, b);
		kstrat[j] = (unsigned char)b;
	}
	std::vector<cu64> kslot(kept + 1, 0);
	for (cu64 j = 0; j < kept; j++) kslot[j + 1] = kslot[j] + khits[j];
	std::vector<cu64> slot(kslot[kept] + 1, 0);
	for (cu64 k = 0; k < kept; k++) {
		const cu64 j = reverse ? kept - 1 - k : k;
		if (khits[j]) {
			const cu32 h = d ? sm_emit<false>(A, j, slot.data() + kslot[j]) : sm_emit<true>(A, j, slot.data() + kslot[j]);
			if (h != khits[j]) return ~0ull;
		}
	}
	SamArgs S;
	S.M = A; S.raw = raw; S.roffs = roffs; S.good = good; S.pos = pos.data(); S.khits = khits.data(); S.kstrat = kstrat.data();
	S.kslot = kslot.data(); S.slot = slot.data(); S.n = n; S.names = names; S.noffs = noffs; S.index0 = 0; S.first = first;
	// k_sam_count + scan, k_sam_len + scan, k_sam_write
	std::vector<cu64> rstart(n + 1, 0);
	for (cu64 i = 0; i < n; i++) rstart[i + 1] = rstart[i] + sm_records(S, i);
	S.rstart = rstart.data();
	const cu64 R = rstart[n];
	std::vector<cu64> off(R + 1, 0);
	for (cu64 r = 0; r < R; r++) {
		SmCount o;
		sm_line(S, r, o);
		off[r + 1] = off[r] + o.n;
	}
	g_text.assign(off[R], '\0');
	for (cu64 r = 0; r < R; r++) {
		SmWrite o{&g_text[0] + off[r]};
		sm_line(S, r, o);
		if (o.o != &g_text[0] + off[r + 1]) return ~0ull;                     // a line must fill exactly its counted bytes
	}
	*text = g_text.data();
	return off[R];
}

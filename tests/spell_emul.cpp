// TEST INFRASTRUCTURE: runs the per-thread bodies of metagenomics_b200/csrc/ogb_spell.cuh -- the functions the spelling kernels call
// -- on the CPU in the launch order of ogb_graph_spell (csrc/ogb_device.cu), scans included, so that the logic of the device spelling
// is checked against the plain restatement (oracle/unitig_spell.py) where no GPU is present. The product never links or calls this
// file; the -m gpu tests check the kernels themselves.
//
// Build: g++ -O2 -std=c++17 -shared -fPIC -o tests/_build/libspell_emul.so tests/spell_emul.cpp
#include <cstring>
#include <vector>

#include "../include/ogb.h"
#include "../metagenomics_b200/csrc/ogb_spell.cuh"

// words / meta: the read store (meta[idx] = off << 16 | L); edges / items: the simplified graph. Writes the records and packed words
// of unitigs [0, all) of the selection; returns the number of records, or -1 when a buffer is too small.
extern "C" long long emul_spell(const cu64 *words, const cu64 *meta, uint32_t n_reads, const ogb_cedge *edges, uint64_t ne,
                                const ogb_clist_item *items, uint64_t ni, int canonical_only, ogb_unitig *rec, uint64_t rec_cap, cu64 *out,
                                uint64_t out_cap)
{
	(void)n_reads;
	SpellArgs A;
	A.words = words; A.meta = meta; A.uniform_len = 0; A.uniform_pw = 0; A.edges = edges; A.items = items;
	std::vector<cu32> sel(ne);
	std::vector<cu64> rank(ne + 1, 0), ipos(ni + 1, 0);
	for (cu64 i = 0; i < ne; i++) sel[i] = canonical_only ? (sp_canonical(edges, i) ? 1u : 0u) : 1u;
	for (cu64 i = 0; i < ne; i++) rank[i + 1] = rank[i] + sel[i];
	for (cu64 i = 0; i < ni; i++) ipos[i + 1] = ipos[i] + items[i].offset;
	A.ipos = ipos.data();
	const cu64 n_rec = rank[ne];
	if (n_rec > rec_cap) return -1;
	std::vector<cu32> nw(n_rec + 1, 0);
	for (cu64 i = ne; i-- > 0;) if (sel[i]) sp_record(A, i, rank[i], 0, n_rec, rec, nw.data());      // thread order must not matter
	std::vector<cu64> wpos(n_rec + 1, 0);
	for (cu64 u = 0; u < n_rec; u++) wpos[u + 1] = wpos[u] + nw[u];
	if (wpos[n_rec] > out_cap) return -1;
	A.rec = rec; A.n_rec = n_rec; A.wpos = wpos.data();
	for (cu64 w = wpos[n_rec]; w-- > 0;) out[w] = sp_word(A, w, rec);
	return (long long)n_rec;
}

// ogb_host.cpp -- host half of libogb.so: the Dataset stage that defines read IDs
// (filter -> canonical strand -> lexicographic sort -> dedupe, SURVEY.md 8(a1,a2)) and the seeded
// synthetic read generator. No CUDA in this file.
//
// Reference behaviour restated here (file:line relative to MetaGenomics/):
//   Dataset.cpp:110-193  readDataset      FASTA/FASTQ parsing, case folding, filter, canonical strand
//   Dataset.cpp:398-413  testRead         ACGT only, no base count >= (UINT64)(len*.8)
//   Dataset.cpp:197-202  sortReads        std::sort on the forward strings
//   Dataset.cpp:316-345  removeDupicateReads  frequency + ID = rank+1
//   Dataset.cpp:421-455  getReadFromString    binary search
// Unlike the reference (std::string per read, single thread) reads are 2-bit packed with an
// order-preserving code (A0 C1 G2 T3, MSB first) at parse time, so the sort compares 64-bit words
// and runs on all host threads.

#include "ogb_internal.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <string>
#include <thread>
#include <vector>

thread_local char g_ogb_err[512] = "";

void ogb_set_error(const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_ogb_err, sizeof g_ogb_err, fmt, ap);
	va_end(ap);
}

extern "C" int ogb_version(void) { return OGB_VERSION; }
extern "C" const char *ogb_last_error(void) { return g_ogb_err; }

namespace {

unsigned host_threads()
{
	unsigned t = std::thread::hardware_concurrency();
	if (t == 0) t = 1;
	if (t > 64) t = 64;
	const char *e = getenv("OGB_HOST_THREADS");
	if (e && atoi(e) > 0) t = (unsigned)atoi(e);
	return t;
}

template <class F> void parallel_for(uint64_t n, uint64_t grain, F f)
{
	unsigned nt = host_threads();
	if (n <= grain || nt == 1) { f(0, n); return; }
	std::atomic<uint64_t> next(0);
	auto body = [&]() {
		for (;;) {
			uint64_t lo = next.fetch_add(grain);
			if (lo >= n) break;
			f(lo, std::min(n, lo + grain));
		}
	};
	std::vector<std::thread> ts;
	for (unsigned t = 1; t < nt; t++) ts.emplace_back(body);
	body();
	for (auto &t : ts) t.join();
}

inline int base_code(unsigned char c)
{
	switch (c) {
	case 'A': return 0;
	case 'C': return 1;
	case 'G': return 2;
	case 'T': return 3;
	default: return -1;
	}
}

// Packs `len` upper-case bases into w[0..ceil(len/32)), forward and reverse complement.
inline void pack_both(const char *s, uint32_t len, uint64_t *fw, uint64_t *rc, uint32_t nw)
{
	for (uint32_t k = 0; k < nw; k++) fw[k] = rc[k] = 0;
	for (uint32_t i = 0; i < len; i++) {
		uint64_t c = (uint64_t)base_code((unsigned char)s[i]);
		fw[i >> 5] |= c << (62 - 2 * (i & 31));
		uint32_t r = len - 1 - i;
		rc[r >> 5] |= (3 - c) << (62 - 2 * (r & 31));
	}
}

}  // namespace

extern "C" int ogb_dataset_create(ogb_dataset **out)
{
	if (!out) { ogb_set_error("ogb_dataset_create: out is NULL"); return OGB_E_ARG; }
	*out = new (std::nothrow) ogb_dataset();
	if (!*out) { ogb_set_error("ogb_dataset_create: out of memory"); return OGB_E_NOMEM; }
	return OGB_OK;
}

extern "C" void ogb_dataset_destroy(ogb_dataset *ds) { if (ds && ds->fetch) ogb_dataset_forget_context(ds); delete ds; }

extern "C" int ogb_dataset_add_reads(ogb_dataset *ds, const char *bases, const uint64_t *offsets, uint64_t n)
{
	if (!ds || (n && (!bases || !offsets))) { ogb_set_error("ogb_dataset_add_reads: NULL argument"); return OGB_E_ARG; }
	if (ds->finalized) { ogb_set_error("ogb_dataset_add_reads: dataset already finalized"); return OGB_E_STATE; }
	if (n == 0) return OGB_OK;
	uint64_t base = ds->raw.size(), first = offsets[0];
	ds->raw.insert(ds->raw.end(), bases + first, bases + offsets[n]);
	for (uint64_t i = 1; i <= n; i++) {
		if (offsets[i] < offsets[i - 1]) { ogb_set_error("ogb_dataset_add_reads: offsets not monotone at %llu", (unsigned long long)i); return OGB_E_ARG; }
		ds->raw_offs.push_back(base + offsets[i] - first);
	}
	return OGB_OK;
}

extern "C" int ogb_dataset_add_file(ogb_dataset *ds, const char *path)
{
	if (!ds || !path) { ogb_set_error("ogb_dataset_add_file: NULL argument"); return OGB_E_ARG; }
	if (ds->finalized) { ogb_set_error("ogb_dataset_add_file: dataset already finalized"); return OGB_E_STATE; }
	std::ifstream f(path);
	if (!f) { ogb_set_error("Unable to open file: %s", path); return OGB_E_IO; }
	std::string line;
	if (!std::getline(f, line)) return OGB_OK;
	auto push = [&](const std::string &s) {
		ds->raw.insert(ds->raw.end(), s.begin(), s.end());
		ds->raw_offs.push_back(ds->raw.size());
	};
	auto chomp = [](std::string &s) { while (!s.empty() && (s.back() == '\r' || s.back() == '\n')) s.pop_back(); };
	if (line[0] == '>') {			// FASTA: header, then sequence lines up to the next '>'
		std::string seq;
		bool have = true;
		while (std::getline(f, line)) {
			if (!line.empty() && line[0] == '>') { push(seq); seq.clear(); have = true; continue; }
			chomp(line);
			seq += line;
		}
		if (have) push(seq);
	} else if (line[0] == '@') {	// FASTQ: 4 lines per record, sequence on the second
		for (;;) {
			std::string seq, plus, qual;
			if (!std::getline(f, seq)) break;
			std::getline(f, plus);
			std::getline(f, qual);
			chomp(seq);
			push(seq);
			if (!std::getline(f, line)) break;	// next '@' header
		}
	} else {
		ogb_set_error("Unknown input file format: %s", path);
		return OGB_E_IO;
	}
	return OGB_OK;
}

extern "C" int ogb_dataset_raw_reads(const ogb_dataset *ds, const char **bases, const uint64_t **offsets, uint64_t *n)
{
	if (!ds || !bases || !offsets || !n) { ogb_set_error("ogb_dataset_raw_reads: NULL argument"); return OGB_E_ARG; }
	if (ds->finalized) { ogb_set_error("ogb_dataset_raw_reads: the data set is finalized; its raw reads are gone"); return OGB_E_STATE; }
	*bases = ds->raw.data(); *offsets = ds->raw_offs.data(); *n = ds->raw_offs.size() - 1;
	return OGB_OK;
}

int ogb_dataset_filter(ogb_dataset *ds, uint32_t min_overlap, std::vector<uint64_t> &idx)
{
	if (!ds) { ogb_set_error("ogb_dataset_finalize: NULL dataset"); return OGB_E_ARG; }
	if (ds->finalized) { ogb_set_error("ogb_dataset_finalize: already finalized"); return OGB_E_STATE; }
	if (min_overlap < 2) { ogb_set_error("ogb_dataset_finalize: minOverlap must be >= 2"); return OGB_E_ARG; }
	ds->min_overlap = min_overlap;
	const uint64_t n_raw = ds->raw_offs.size() - 1;
	char *raw = ds->raw.data();
	const uint64_t *ro = ds->raw_offs.data();

	// case folding (Dataset.cpp:155-156) + filter (:158, testRead :398-413)
	std::vector<uint8_t> good(n_raw, 0);
	parallel_for(n_raw, 1 << 14, [&](uint64_t lo, uint64_t hi) {
		for (uint64_t i = lo; i < hi; i++) {
			uint64_t len = ro[i + 1] - ro[i];
			char *s = raw + ro[i];
			uint64_t cnt[4] = {0, 0, 0, 0};
			bool ok = len > min_overlap && len < 65536;
			for (uint64_t k = 0; ok && k < len; k++) {
				unsigned char c = (unsigned char)s[k];
				if (c >= 'a' && c <= 'z') { c = (unsigned char)(c - 32); s[k] = (char)c; }
				int b = base_code(c);
				if (b < 0) ok = false; else cnt[b]++;
			}
			if (ok) {
				uint64_t threshold = (uint64_t)(len * .8);	// same double arithmetic as :409
				if (cnt[0] >= threshold || cnt[1] >= threshold || cnt[2] >= threshold || cnt[3] >= threshold) ok = false;
			}
			good[i] = ok;
		}
	});
	idx.clear();
	idx.reserve(n_raw);
	uint64_t shortest = ~0ULL, longest = 0;
	for (uint64_t i = 0; i < n_raw; i++)
		if (good[i]) {
			idx.push_back(i);
			uint64_t len = ro[i + 1] - ro[i];
			shortest = std::min(shortest, len);
			longest = std::max(longest, len);
		}
	ds->n_good = idx.size();
	ds->shortest = shortest;
	ds->longest = longest;
	ds->finalized = true;
	ds->word_offs.assign(1, 0);
	if (idx.empty()) { ds->raw.clear(); ds->raw.shrink_to_fit(); }
	return OGB_OK;
}

extern "C" int ogb_dataset_finalize(ogb_dataset *ds, uint32_t min_overlap)
{
	std::vector<uint64_t> idx;
	int rc = ogb_dataset_filter(ds, min_overlap, idx);
	if (rc != OGB_OK) return rc;
	const uint64_t n_good = idx.size();
	if (n_good == 0) return OGB_OK;
	char *raw = ds->raw.data();
	const uint64_t *ro = ds->raw_offs.data();
	const uint64_t longest = ds->longest;

	// pass 2: pack forward + reverse complement, keep the smaller (:161-164; equal -> same string)
	const uint32_t W = (uint32_t)((longest + 31) / 32);
	std::vector<uint64_t> keys(n_good * (uint64_t)W);
	std::vector<uint16_t> klen(n_good);
	parallel_for(n_good, 1 << 13, [&](uint64_t lo, uint64_t hi) {
		std::vector<uint64_t> fw(W), rc(W);
		for (uint64_t g = lo; g < hi; g++) {
			uint64_t i = idx[g];
			uint32_t len = (uint32_t)(ro[i + 1] - ro[i]);
			uint32_t nw = (len + 31) / 32;
			pack_both(raw + ro[i], len, fw.data(), rc.data(), nw);
			bool use_fw = std::lexicographical_compare(fw.begin(), fw.begin() + nw, rc.begin(), rc.begin() + nw);
			uint64_t *dst = &keys[g * W];
			const uint64_t *src = use_fw ? fw.data() : rc.data();
			for (uint32_t k = 0; k < nw; k++) dst[k] = src[k];
			for (uint32_t k = nw; k < W; k++) dst[k] = 0;
			klen[g] = (uint16_t)len;
		}
	});
	ds->raw.clear(); ds->raw.shrink_to_fit();
	ds->raw_offs.clear(); ds->raw_offs.shrink_to_fit();

	// sort (:197-202). Padding is 'A' (0), the smallest base, so word order + length tiebreak is
	// exactly std::string operator< (a proper prefix sorts first).
	struct Ent { uint64_t w0; uint32_t g; };
	std::vector<Ent> ord(n_good);
	for (uint64_t g = 0; g < n_good; g++) ord[g] = Ent{keys[g * W], (uint32_t)g};
	auto less = [&](const Ent &a, const Ent &b) {
		if (a.w0 != b.w0) return a.w0 < b.w0;
		const uint64_t *x = &keys[(uint64_t)a.g * W], *y = &keys[(uint64_t)b.g * W];
		for (uint32_t k = 1; k < W; k++)
			if (x[k] != y[k]) return x[k] < y[k];
		return klen[a.g] < klen[b.g];
	};
	{
		unsigned nt = host_threads();
		unsigned parts = 1;
		while (parts * 2 <= nt && n_good / (parts * 2) >= (1u << 15)) parts *= 2;
		std::vector<uint64_t> cut(parts + 1);
		for (unsigned p = 0; p <= parts; p++) cut[p] = n_good * p / parts;
		{
			std::vector<std::thread> ts;
			for (unsigned p = 1; p < parts; p++) ts.emplace_back([&, p]() { std::sort(ord.begin() + cut[p], ord.begin() + cut[p + 1], less); });
			std::sort(ord.begin() + cut[0], ord.begin() + cut[1], less);
			for (auto &t : ts) t.join();
		}
		for (unsigned width = 1; width < parts; width *= 2) {
			std::vector<std::thread> ts;
			for (unsigned p = 0; p + width < parts; p += 2 * width) {
				uint64_t a = cut[p], m = cut[p + width], b = cut[std::min(parts, p + 2 * width)];
				ts.emplace_back([&, a, m, b]() { std::inplace_merge(ord.begin() + a, ord.begin() + m, ord.begin() + b, less); });
			}
			for (auto &t : ts) t.join();
		}
	}

	// dedupe + frequency + IDs (:316-345)
	std::vector<uint32_t> uniq;
	uniq.reserve(n_good);
	ds->freq.clear();
	for (uint64_t r = 0; r < n_good; r++) {
		uint32_t g = ord[r].g;
		bool same = false;
		if (!uniq.empty()) {
			uint32_t p = uniq.back();
			same = klen[p] == klen[g] && memcmp(&keys[(uint64_t)p * W], &keys[(uint64_t)g * W], W * 8) == 0;
		}
		if (same) ds->freq.back()++;
		else { uniq.push_back(g); ds->freq.push_back(1); }
	}
	const uint64_t nu = uniq.size();
	ds->lens.resize(nu);
	ds->word_offs.resize(nu + 1);
	uint64_t tot = 0;
	for (uint64_t i = 0; i < nu; i++) { ds->word_offs[i] = tot; ds->lens[i] = klen[uniq[i]]; tot += (klen[uniq[i]] + 31) / 32; }
	ds->word_offs[nu] = tot;
	ds->words.resize(tot);
	parallel_for(nu, 1 << 15, [&](uint64_t lo, uint64_t hi) {
		for (uint64_t i = lo; i < hi; i++) {
			uint32_t nw = (ds->lens[i] + 31) / 32;
			memcpy(&ds->words[ds->word_offs[i]], &keys[(uint64_t)uniq[i] * W], nw * 8);
		}
	});
	return OGB_OK;
}

extern "C" uint64_t ogb_dataset_n_reads(const ogb_dataset *ds) { return ds ? ds->n_good : 0; }
extern "C" uint64_t ogb_dataset_n_unique(const ogb_dataset *ds) { return ds ? ds->n_unique() : 0; }
extern "C" uint64_t ogb_dataset_shortest(const ogb_dataset *ds) { return ds ? ds->shortest : 0; }
extern "C" uint64_t ogb_dataset_longest(const ogb_dataset *ds) { return ds ? ds->longest : 0; }
extern "C" uint32_t ogb_dataset_min_overlap(const ogb_dataset *ds) { return ds ? ds->min_overlap : 0; }
extern "C" const uint64_t *ogb_dataset_words(const ogb_dataset *ds, uint64_t *n_words)
{
	if (!ds) return nullptr;
	if (ogb_dataset_ensure_words(ds) != OGB_OK) return nullptr;
	if (n_words) *n_words = ds->words.size();
	return ds->words.data();
}
extern "C" const uint64_t *ogb_dataset_word_offsets(const ogb_dataset *ds) { return ds ? ds->word_offs.data() : nullptr; }
extern "C" const uint16_t *ogb_dataset_lengths(const ogb_dataset *ds) { return ds ? ds->lens.data() : nullptr; }
extern "C" const uint32_t *ogb_dataset_frequencies(const ogb_dataset *ds) { return ds ? ds->freq.data() : nullptr; }

extern "C" int ogb_dataset_get_read(const ogb_dataset *ds, uint64_t id, int strand, char *out, uint32_t cap, uint32_t *len)
{
	if (!ds || !out) { ogb_set_error("ogb_dataset_get_read: NULL argument"); return OGB_E_ARG; }
	if (id < 1 || id > ds->n_unique()) { ogb_set_error("ID %llu out of bound.", (unsigned long long)id); return OGB_E_ARG; }
	uint32_t L = ds->lens[id - 1];
	if (len) *len = L;
	if (cap < L) { ogb_set_error("ogb_dataset_get_read: buffer too small"); return OGB_E_CAPACITY; }
	if (int rc = ogb_dataset_ensure_words(ds)) return rc;
	const uint64_t *w = &ds->words[ds->word_offs[id - 1]];
	static const char B[4] = {'A', 'C', 'G', 'T'};
	for (uint32_t i = 0; i < L; i++) {
		uint32_t c = (uint32_t)(w[i >> 5] >> (62 - 2 * (i & 31))) & 3;
		if (strand == 0) out[i] = B[c]; else out[L - 1 - i] = B[3 - c];
	}
	return OGB_OK;
}

extern "C" int ogb_dataset_find_read(const ogb_dataset *ds, const char *bases, uint32_t len, uint64_t *id)
{
	if (!ds || !bases || !id) { ogb_set_error("ogb_dataset_find_read: NULL argument"); return OGB_E_ARG; }
	*id = 0;
	if (len == 0 || len > 65535 || ds->n_unique() == 0) return OGB_OK;
	if (int rc = ogb_dataset_ensure_words(ds)) return rc;
	uint32_t nw = (len + 31) / 32;
	std::vector<uint64_t> fw(nw), rc(nw);
	std::string up(bases, bases + len);
	for (auto &c : up) { c = (char)toupper((unsigned char)c); if (base_code((unsigned char)c) < 0) return OGB_OK; }
	pack_both(up.data(), len, fw.data(), rc.data(), nw);
	const uint64_t *q = std::lexicographical_compare(fw.begin(), fw.end(), rc.begin(), rc.end()) ? fw.data() : rc.data();
	// three-way compare of the query against read i with std::string semantics
	auto cmp = [&](uint64_t i) {
		const uint64_t *w = &ds->words[ds->word_offs[i]];
		uint32_t L = ds->lens[i], mw = (std::min(L, len) + 31) / 32;
		for (uint32_t k = 0; k < mw; k++) {
			uint64_t a = w[k], b = q[k];
			if (k == mw - 1 && (std::min(L, len) & 31)) { uint64_t m = ~0ULL << (64 - 2 * (std::min(L, len) & 31)); a &= m; b &= m; }
			if (a != b) return a < b ? -1 : 1;
		}
		return L < len ? -1 : (L > len ? 1 : 0);
	};
	uint64_t lo = 0, hi = ds->n_unique();
	while (lo < hi) {
		uint64_t mid = (lo + hi) / 2;
		int c = cmp(mid);
		if (c == 0) { *id = mid + 1; return OGB_OK; }
		if (c < 0) lo = mid + 1; else hi = mid;
	}
	return OGB_OK;
}

// ------------------------------------------------------------------------------------------------
// Synthetic generator (splitmix64 seeding + xoshiro256**; per-read streams so the result does not
// depend on the number of host threads).
// ------------------------------------------------------------------------------------------------
namespace {

struct Rng {
	uint64_t s[4];
	static uint64_t splitmix(uint64_t &x)
	{
		uint64_t z = (x += 0x9e3779b97f4a7c15ULL);
		z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
		z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
		return z ^ (z >> 31);
	}
	explicit Rng(uint64_t seed) { for (int i = 0; i < 4; i++) s[i] = splitmix(seed); }
	static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
	uint64_t next()
	{
		uint64_t r = rotl(s[1] * 5, 7) * 9, t = s[1] << 17;
		s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45);
		return r;
	}
	uint64_t below(uint64_t n) { return (uint64_t)(((unsigned __int128)next() * n) >> 64); }
	double uniform() { return (next() >> 11) * (1.0 / 9007199254740992.0); }
	double normal()
	{
		double u1 = uniform(), u2 = uniform();
		if (u1 < 1e-300) u1 = 1e-300;
		return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
	}
};

inline char comp(char c) { return c == 'A' ? 'T' : c == 'C' ? 'G' : c == 'G' ? 'C' : 'A'; }
inline void copy_rc(const char *src, uint32_t len, char *dst) { for (uint32_t i = 0; i < len; i++) dst[len - 1 - i] = comp(src[i]); }

}  // namespace

extern "C" int ogb_synth_genome(uint64_t seed, uint64_t len, char *out)
{
	if (!out && len) { ogb_set_error("ogb_synth_genome: NULL output"); return OGB_E_ARG; }
	static const char B[4] = {'A', 'C', 'G', 'T'};
	const uint64_t chunk = 1 << 20;
	parallel_for((len + chunk - 1) / chunk, 1, [&](uint64_t lo, uint64_t hi) {
		for (uint64_t c = lo; c < hi; c++) {
			Rng r(seed * 0x2545f4914f6cdd1dULL + c);
			uint64_t e = std::min(len, (c + 1) * chunk);
			for (uint64_t i = c * chunk; i < e;) {
				uint64_t x = r.next();
				for (int k = 0; k < 32 && i < e; k++, i++) { out[i] = B[x & 3]; x >>= 2; }
			}
		}
	});
	return OGB_OK;
}

extern "C" int ogb_synth_reads(uint64_t seed, const char *genomes, const uint64_t *g_offsets, const double *weights,
                               uint32_t n_genomes, uint64_t n_reads, uint32_t len_min, uint32_t len_max, int paired,
                               double insert_mean, double insert_sd, char *out_bases, uint64_t out_cap,
                               uint64_t *out_offsets)
{
	if (!genomes || !g_offsets || !out_bases || !out_offsets || n_genomes == 0) { ogb_set_error("ogb_synth_reads: NULL argument"); return OGB_E_ARG; }
	if (len_min == 0 || len_min > len_max) { ogb_set_error("ogb_synth_reads: bad length range"); return OGB_E_ARG; }
	if (paired && (n_reads & 1)) { ogb_set_error("ogb_synth_reads: paired output needs an even read count"); return OGB_E_ARG; }
	std::vector<double> cum(n_genomes);
	double tot = 0;
	for (uint32_t g = 0; g < n_genomes; g++) {
		uint64_t gl = g_offsets[g + 1] - g_offsets[g];
		uint64_t need = paired ? (uint64_t)std::max<double>(2.0 * len_max, insert_mean + 6 * insert_sd) : len_max;
		if (gl < need) { ogb_set_error("ogb_synth_reads: genome %u shorter than a read/fragment", g); return OGB_E_ARG; }
		tot += (weights ? weights[g] : 1.0) * (double)gl;
		cum[g] = tot;
	}
	const uint64_t units = paired ? n_reads / 2 : n_reads;
	const uint64_t per = paired ? 2 : 1;
	// pass 1: lengths (first draws of each unit's stream)
	parallel_for(units, 1 << 15, [&](uint64_t lo, uint64_t hi) {
		for (uint64_t u = lo; u < hi; u++) {
			Rng r(seed * 0x9e3779b97f4a7c15ULL + u * 0xd1342543de82ef95ULL + 1);
			for (uint64_t k = 0; k < per; k++) out_offsets[u * per + k + 1] = len_min + r.below(len_max - len_min + 1);
		}
	});
	out_offsets[0] = 0;
	for (uint64_t i = 1; i <= n_reads; i++) out_offsets[i] += out_offsets[i - 1];
	if (out_offsets[n_reads] > out_cap) { ogb_set_error("ogb_synth_reads: output needs %llu bytes", (unsigned long long)out_offsets[n_reads]); return OGB_E_CAPACITY; }
	// pass 2: sequences
	parallel_for(units, 1 << 13, [&](uint64_t lo, uint64_t hi) {
		for (uint64_t u = lo; u < hi; u++) {
			Rng r(seed * 0x9e3779b97f4a7c15ULL + u * 0xd1342543de82ef95ULL + 1);
			uint32_t L[2];
			for (uint64_t k = 0; k < per; k++) L[k] = (uint32_t)(len_min + r.below(len_max - len_min + 1));
			double x = r.uniform() * tot;
			uint32_t g = (uint32_t)(std::lower_bound(cum.begin(), cum.end(), x) - cum.begin());
			if (g >= n_genomes) g = n_genomes - 1;
			const char *G = genomes + g_offsets[g];
			uint64_t gl = g_offsets[g + 1] - g_offsets[g];
			if (!paired) {
				uint64_t start = r.below(gl - L[0] + 1);
				char *dst = out_bases + out_offsets[u];
				if (r.next() & 1) memcpy(dst, G + start, L[0]); else copy_rc(G + start, L[0], dst);
			} else {
				uint64_t F = (uint64_t)llround(insert_mean + insert_sd * r.normal());
				uint64_t lo_f = std::max<uint64_t>(L[0], L[1]) * 2;
				if (F < lo_f) F = lo_f;
				if (F > gl) F = gl;
				uint64_t start = r.below(gl - F + 1);
				bool flip = r.next() & 1;
				char *d0 = out_bases + out_offsets[2 * u], *d1 = out_bases + out_offsets[2 * u + 1];
				if (!flip) { memcpy(d0, G + start, L[0]); copy_rc(G + start + F - L[1], L[1], d1); }
				else { copy_rc(G + start + F - L[0], L[0], d0); memcpy(d1, G + start, L[1]); }
			}
		}
	});
	return OGB_OK;
}

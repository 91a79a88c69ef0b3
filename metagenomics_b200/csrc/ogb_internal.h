// ogb_internal.h -- shared by the host and device halves of libogb.so.
#ifndef OGB_INTERNAL_H_
#define OGB_INTERNAL_H_

#include <cstdarg>
#include <cstdint>
#include <cstdlib>
#include <vector>

#include "../../include/ogb.h"

void ogb_set_error(const char *fmt, ...);

// Dataset (Dataset.h:17-62): raw reads until finalize, then the sorted unique reads, 2-bit packed.
struct ogb_dataset {
	std::vector<char> raw;
	std::vector<uint64_t> raw_offs{0};
	bool keep_names = false;              // ogb_dataset_keep_names: the sample files' read names, aligned with raw_offs
	std::vector<char> names;
	std::vector<uint64_t> name_offs{0};
	bool finalized = false;
	uint32_t min_overlap = 0;
	uint64_t n_good = 0, shortest = ~0ULL, longest = 0;
	std::vector<uint64_t> words;
	std::vector<uint64_t> word_offs;
	std::vector<uint16_t> lens;
	std::vector<uint32_t> freq;
	const void *resident_ctx = nullptr;   // context whose HBM already holds these reads (ogb_dataset_finalize_device)
	uint64_t resident_stamp = 0;
	// ogb_dataset_finalize_device leaves the tight packed words on the device until the host asks for them (they are the bulk of
	// the host views and most callers never look at them): fetch(ds) downloads them; pending_words counts them meanwhile
	int (*fetch)(ogb_dataset *) = nullptr;
	void *fetch_ctx = nullptr;
	uint64_t pending_words = 0;
	uint64_t n_unique() const { return lens.size(); }
};

// First half of the Dataset constructor, on the host: case folding + filter (Dataset.cpp:155-158, testRead :398-413).
// Fills idx with the raw indices of the reads that stay and sets n_good / shortest / longest / min_overlap / finalized.
int ogb_dataset_filter(ogb_dataset *ds, uint32_t min_overlap, std::vector<uint64_t> &idx);
// downloads the packed words a device finalize left behind (no-op otherwise)
inline int ogb_dataset_ensure_words(const ogb_dataset *ds) { ogb_dataset *d = const_cast<ogb_dataset *>(ds); return d->fetch ? d->fetch(d) : 0; }
void ogb_dataset_forget_context(ogb_dataset *ds);   // ogb_device.cu: the data set goes away before its context

#endif

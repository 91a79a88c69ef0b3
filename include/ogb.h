/*
 * ogb.h -- C ABI of the B200 overlap-graph builder (libogb.so).
 *
 * The reference (abiswas-odu/metagenomics) has no plugin / FFI interface; its boundary for the
 * overlap-graph build is the C++ class API used at one call site (MetaGenomics/main.cpp:33,45-47):
 *
 *     Dataset *dataSet = new Dataset(pairedEndFileNames, singleEndFileNames, minimumOverlapLength);
 *     HashTable *hashTable = new HashTable();
 *     hashTable->insertDataset(dataSet, minimumOverlapLength);
 *     overlapGraph = new OverlapGraph(hashTable);
 *
 * metagenomics_b200/host/ re-implements those classes (same names, signatures and post-conditions)
 * on top of the entry points below; INTEGRATION.md shows the binding. Every entry point cites the
 * reference interface it replaces (file:line relative to MetaGenomics/).
 *
 * Conventions: plain pointers and sizes only; every call returns 0 on success or a non-zero
 * OGB_E_* code (text via ogb_last_error(), thread local); nothing calls exit(); read IDs are
 * 1-based like the reference's (Dataset.cpp:335-341); all device work is CUDA for sm_100a -- there
 * is no CPU fallback: device entry points fail with OGB_E_CUDA when no GPU is usable.
 */
#ifndef OGB_H_
#define OGB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OGB_VERSION 210

enum {
	OGB_OK = 0,
	OGB_E_ARG = 1,      /* bad argument */
	OGB_E_CUDA = 2,     /* CUDA runtime / no device */
	OGB_E_NCCL = 3,     /* NCCL */
	OGB_E_STATE = 4,    /* call order (e.g. build before upload) */
	OGB_E_CAPACITY = 5, /* output buffer too small / internal capacity exceeded */
	OGB_E_IO = 6,       /* file could not be read */
	OGB_E_NOMEM = 7
};

typedef struct ogb_dataset ogb_dataset; /* host: filtered, canonical, sorted, unique reads */
typedef struct ogb_context ogb_context; /* device: one GPU (one rank) */

/* One directed overlap edge, the flat form of the reference's Edge record (Edge.h:17-44):
 * source / destination read IDs, overlapOrientation 0..3 and overlapOffset (UINT16 at creation,
 * OverlapGraph.cpp:407,410). */
typedef struct ogb_edge {
	uint32_t src;
	uint32_t dst;
	uint16_t offset;
	uint8_t orient;
	uint8_t reserved;
} ogb_edge; /* 12 bytes */

/* Kernel classes of ogb_stats.ms_kernel / n_kernel. */
enum {
	OGB_KC_HASH = 0,        /* K1  k_hash_insert */
	OGB_KC_WINDOW,          /* K3a k_window_part (overlap pass) */
	OGB_KC_PROBE,           /* K3b k_probe_parts (or the direct probe kernels) */
	OGB_KC_VERIFY,          /* K3c k_verify */
	OGB_KC_ROWS,            /*     k_rows_finish */
	OGB_KC_MARK1,           /* K5  k_mark_fast<1>: degree 1..32 */
	OGB_KC_MARK2,           /* K5  k_mark_fast<2>: degree 33..64 */
	OGB_KC_MARKANY,         /* K5  k_mark_any */
	OGB_KC_KEEP,            /* K6  k_keep + k_keep_big */
	OGB_KC_EMIT,            /* K6  scan + k_emit_small + k_emit */
	OGB_KC_CONTAIN_WINDOW,  /* K2  k_window_part (containment pass) */
	OGB_KC_CONTAIN_PROBE,   /* K2  probe */
	OGB_KC_CONTAIN_VERIFY,  /* K2  k_verify<CONTAIN> */
	OGB_KC_EXCH_INDEX,      /* several ranks: allgather of the index slices */
	OGB_KC_EXCH_ROWS,       /* C1: allgather of the adjacency rows */
	OGB_KC_EXCH_BITS,       /* C2: allgather of the ELIM bits */
	OGB_KC_EXCH_FINAL,      /* C3: allgather of the final edges */
	OGB_KC_PROBE_VERIFY,    /* K3b+c k_probe_verify: probe of chunk i and verification of chunk i-1 in one warp-specialised launch */
	OGB_KC_COUNT = 20
};

/* Counters and device timings of the last build (CUDA events on the context's stream). */
typedef struct ogb_stats {
	uint64_t n_reads;          /* unique reads resident on the device */
	uint64_t table_buckets;    /* index size in buckets */
	uint64_t table_bytes;
	uint64_t n_contained;      /* reads with superReadID != 0 */
	uint64_t contain_probes;   /* P_c  windows scanned by the containment pass (0 if skipped) */
	uint64_t contain_hits;     /* C_c  verified containment hits */
	uint64_t overlap_probes;   /* P_e  windows scanned by the overlap pass (this rank) */
	uint64_t probe_sectors;    /* index buckets (32 B sectors) actually loaded by the overlap pass */
	uint64_t candidates;       /* fingerprint matches sent to verification */
	uint64_t edges_pre;        /* E_pre  directed edges before reduction (global) */
	uint64_t edges_pre_local;  /* emitted by this rank */
	uint64_t pivot_entries;    /* T  adjacency entries scanned by active pivots (this rank) */
	uint64_t active_pivots;
	uint64_t edges_final;      /* E_final directed edges after reduction (global) */
	uint64_t nodes_final;      /* numberOfNodes (reads with >= 1 surviving edge) */
	uint64_t max_degree;       /* largest pre-reduction out-degree (this rank) */
	uint64_t overflow_reads;   /* heavy nodes of this rank (degree > slots per read: list kept in the extension area) */
	uint32_t kernel_launches;  /* kernels of this library launched by the last hash_build+build_graph */
	uint32_t probe_launches;   /* launches of the probe kernel (one per chunk of query reads) */
	uint32_t hash_partitions;  /* hash partitions of the index (ranks x partitions per rank) */
	uint32_t hash_build_attempts; /* 1 + retries of K1 after a partition filled up (skewed keys) */
	float ms_pack;             /* K0 */
	float ms_hash_build;       /* K1 */
	float ms_contain;          /* K2 (+ allreduce) */
	float ms_overlap;          /* K3 probe + verify (all chunks), degree scan, heavy-list placement */
	float ms_exchange_pre;     /* row headers + overflow entries (k_rows_finish) and, on several ranks, C1: allgather of the adjacency rows */
	float ms_mark;             /* K5 */
	float ms_reduce;           /* K6 (+C2/C3) */
	float ms_total;            /* hash_build + mark_contained + build_graph, device time */
	float ms_scan_kernel;      /* K3 alone: all probe + verify launches */
	float ms_probe_launch;     /* average duration of the probe of one chunk (the roofline kernel(s): k_window_part + k_probe_parts, or k_probe), measured in place */
	float ms_window_launch;    /* of which k_window_part (hash + filter + scatter to the partition queues); 0 on the direct path */
	float ms_kernel[OGB_KC_COUNT];     /* device time per kernel class (OGB_KC_*), summed over its launches of the last hash_build + mark_contained +
	                                    * build_graph: CUDA event pairs on the launching stream, recorded in place (kernels of the two K3 streams overlap) */
	uint32_t n_kernel[OGB_KC_COUNT];   /* launches (event pairs) behind ms_kernel */
} ogb_stats;

int ogb_version(void);
const char *ogb_last_error(void);

/* ----------------------------------------------------------------------------------------------
 * Host side: the Dataset stage that defines read IDs (adjacent to the hot path, SURVEY.md 8(a2)).
 * -------------------------------------------------------------------------------------------- */

/* Dataset::Dataset() (Dataset.cpp:24-33). */
int ogb_dataset_create(ogb_dataset **out);
void ogb_dataset_destroy(ogb_dataset *ds);

/* Dataset::readDataset (Dataset.cpp:110-193) for in-memory reads: n ASCII reads, read i =
 * bases[offsets[i] .. offsets[i+1]). Case is folded like :155-156. Reads are only collected here;
 * filtering happens in ogb_dataset_finalize because it needs minOverlap. */
int ogb_dataset_add_reads(ogb_dataset *ds, const char *bases, const uint64_t *offsets, uint64_t n);

/* Dataset::readDataset (Dataset.cpp:110-193) for a FASTA ('>') or FASTQ ('@') file; multi-line
 * FASTA records are joined (:145). */
int ogb_dataset_add_file(ogb_dataset *ds, const char *path);

/* The rest of Dataset::Dataset(pe, se, minOverlap) (Dataset.cpp:39-65): keep reads with
 * length > minOverlap made of ACGT only and with no base count >= (UINT64)(len*.8)
 * (:158, testRead :398-413); store the lexicographically smaller of read / reverse complement
 * (:161-164); sort lexicographically, shorter prefix first (sortReads :197-202); merge equal reads
 * counting frequency and assign ID = rank+1 (removeDupicateReads :316-345). */
int ogb_dataset_finalize(ogb_dataset *ds, uint32_t min_overlap);

/* The same on the GPU of `ctx` (SURVEY.md 8(f) rank 2), every step of it: the filter (k_ds_filter), canonical strand, a
 * hand-written stable LSD radix sort over the packed words (8-bit passes, bytes in which no two reads differ skipped), dedupe and
 * frequencies. Same post-conditions and host views as ogb_dataset_finalize (the packed words are downloaded when the host first asks
 * for them); in addition the packed reads stay in the context's HBM, so the ogb_reads_upload_dataset that follows
 * (HashTable::insertDataset) has nothing left to copy. On failure the raw reads are kept and ogb_dataset_finalize can still run. */
int ogb_dataset_finalize_device(ogb_dataset *ds, ogb_context *ctx, uint32_t min_overlap);

uint64_t ogb_dataset_n_reads(const ogb_dataset *ds);   /* Dataset::getNumberOfReads (:352): good reads */
uint64_t ogb_dataset_n_unique(const ogb_dataset *ds);  /* Dataset::getNumberOfUniqueReads (:361) */
uint64_t ogb_dataset_shortest(const ogb_dataset *ds);  /* Dataset::shortestReadLength (Dataset.h:36) */
uint64_t ogb_dataset_longest(const ogb_dataset *ds);   /* Dataset::longestReadLength  (Dataset.h:37) */
uint32_t ogb_dataset_min_overlap(const ogb_dataset *ds);

/* Packed form handed to the device: read id (1-based) occupies words
 * [word_offsets[id-1], word_offsets[id-1] + ceil(len/32)) of `words`; base k of the read sits in
 * bits 63-2*(k%32) .. 62-2*(k%32) of word k/32 (A=0 C=1 G=2 T=3, unused low bits zero). */
const uint64_t *ogb_dataset_words(const ogb_dataset *ds, uint64_t *n_words);
const uint64_t *ogb_dataset_word_offsets(const ogb_dataset *ds); /* n_unique + 1 entries */
const uint16_t *ogb_dataset_lengths(const ogb_dataset *ds);      /* n_unique entries (Read::getReadLength) */
const uint32_t *ogb_dataset_frequencies(const ogb_dataset *ds);  /* n_unique entries (Read::getFrequency) */

/* Read::getStringForward / getStringReverse (Read.h:58-59) of Dataset::getReadFromID(id)
 * (Dataset.cpp:482-492). strand 0 = forward, 1 = reverse complement. out holds >= len bytes. */
int ogb_dataset_get_read(const ogb_dataset *ds, uint64_t id, int strand, char *out, uint32_t cap, uint32_t *len);

/* Dataset::getReadFromString (Dataset.cpp:421-455): binary search of min(read, rc); *id = 0 if
 * the string is not in the dataset (the reference exits there). */
int ogb_dataset_find_read(const ogb_dataset *ds, const char *bases, uint32_t len, uint64_t *id);

/* The reads added to a data set that is not finalized, as added (no filter, no case folding): read i = (*bases)[(*offsets)[i] ..
 * (*offsets)[i+1]), *n reads. Views into the data set, valid until it changes. A finalized data set: OGB_E_STATE. Lets a caller read
 * sample files (ogb_dataset_add_file) for ogb_graph_map_reads. */
int ogb_dataset_raw_reads(const ogb_dataset *ds, const char **bases, const uint64_t **offsets, uint64_t *n);

/* ----------------------------------------------------------------------------------------------
 * Device side.
 * -------------------------------------------------------------------------------------------- */

/* One context per process and GPU. Single-GPU: rank 0 of 1. */
int ogb_context_create(ogb_context **out, int device);

/* Multi-GPU (one process per GPU): `nccl_uid` is the 128-byte ncclUniqueId made by
 * ogb_nccl_unique_id on rank 0 and distributed by the caller (torch.distributed store, MPI, ...). */
int ogb_nccl_unique_id(void *out128);
int ogb_context_create_dist(ogb_context **out, int device, int rank, int n_ranks, const void *nccl_uid);
void ogb_context_destroy(ogb_context *ctx);
int ogb_context_rank(const ogb_context *ctx, int *rank, int *n_ranks);

/* Read storage (Read::setRead + Read::reverseComplement, Read.cpp:75-82,115-127): copies the n
 * sorted unique reads to the device and runs K0, which 2-bit packs forward strands (ASCII variant)
 * and writes the reverse complements. IDs = index + 1. Replaces any previous upload. */
int ogb_reads_upload(ogb_context *ctx, const char *bases, const uint64_t *offsets, uint64_t n);
int ogb_reads_upload_packed(ogb_context *ctx, const uint64_t *words, const uint64_t *word_offsets,
                            const uint16_t *lengths, uint64_t n);
int ogb_reads_upload_dataset(ogb_context *ctx, const ogb_dataset *ds);
/* Several ranks, one read length: this rank passes only the reads of its own shard -- reads (per*rank, per*(rank+1)] of
 * the n_total sorted unique reads, per = ceil(n_total / n_ranks), ceil(read_len/32) tight words each -- and the packed
 * store is replicated by an allgather over NVLink instead of n_ranks full uploads over PCIe. Collective: every rank calls it. */
int ogb_reads_upload_packed_sharded(ogb_context *ctx, const uint64_t *shard_words, uint64_t n_total, uint32_t read_len);

/* HashTable::insertDataset(Dataset*, minOverlapLength) (HashTable.cpp:50-80): hashStringLength =
 * minOverlap-1 (:54); 4 keys per read -- prefix/suffix of forward and of reverse complement
 * (hashRead :88-104) -- inserted by K1 into an open-addressing table of 64-byte buckets (ten
 * fingerprint/value slots each), cut into L2-sized hash partitions; on several ranks every rank builds the partitions
 * it owns and the slices are allgathered. */
int ogb_hash_build(ogb_context *ctx, uint32_t min_overlap);

/* HashTable::getListOfReads(string) (HashTable.cpp:202-221) for n_keys keys of hashStringLength
 * bases each (keys concatenated, ASCII). Returns for key k the entries (id | orientation<<62,
 * HashTable.cpp:165) in out[out_offsets[k] .. out_offsets[k+1]), ascending id then orientation
 * (the reference's insertion order). out_offsets has n_keys+1 entries. */
int ogb_hash_lookup(ogb_context *ctx, const char *keys, uint64_t n_keys, uint64_t *out, uint64_t out_cap,
                    uint64_t *out_offsets);
uint64_t ogb_hash_string_length(const ogb_context *ctx); /* HashTable::getHashStringLength (HashTable.h:34) */
uint64_t ogb_hash_table_size(const ogb_context *ctx);    /* HashTable::getHashTableSize (HashTable.h:33): slots */

/* OverlapGraph::markContainedReads (OverlapGraph.cpp:225-290) with checkOverlapForContainedRead
 * (:302-340): K2. No-op when all reads have one length (:228). */
int ogb_mark_contained(ogb_context *ctx);
/* Read::superReadID (Read.h:50) for ids 0..n (entry 0 unused, = 0). */
int ogb_super_read_ids(ogb_context *ctx, uint64_t *out, uint64_t cap);

/* Dataset::storeMatePairInformation (Dataset.cpp:208-310; called at OverlapGraph.cpp:142, after markContainedReads) for a
 * batch: sequence i = bases[offsets[i] .. offsets[i+1]) as sequenced (ASCII; sequences 2k and 2k+1 are mates). For each:
 * the filter of :268 (length > minOverlap, testRead), getReadFromString (:421-455) as one verified index lookup, the
 * redirection of a contained read to its super read (:280-284) and the orientation bit -- 1 iff the sequence is a substring
 * of that read's forward strand (:291-292). out_id[i] = ID of the read that stands for sequence i (0: filtered out; a pair
 * is good when both are non-zero), out_orient[i] = the bit. Sequences longer than 960 bases are reported as 0 (host loop). */
int ogb_mate_lookup(ogb_context *ctx, const char *bases, const uint64_t *offsets, uint64_t n_seqs, uint32_t min_overlap,
                    uint32_t *out_id, uint8_t *out_orient);

/* OverlapGraph::buildOverlapGraphFromHashTable (OverlapGraph.cpp:107-210, up to `delete hashTable`)
 * minus markContainedReads/readMatePairsFromFile: insertAllEdgesOfRead + checkOverlap (K3, :354-383,
 * :529-565), the per-node order by offset (:563, produced on the fly by K5/K6), markTransitiveEdges (K5, :574-615),
 * removeTransitiveEdges (K6, :623-661) and, on several ranks, the edge exchanges. The result stays
 * on the device until ogb_graph_edges. keep_pre != 0 keeps the pre-reduction edge list readable. */
int ogb_build_graph(ogb_context *ctx, int keep_pre);

/* Number of directed edges in the graph: which = 0 post-reduction (OverlapGraph::getNumberOfEdges,
 * OverlapGraph.h:76), 1 pre-reduction (needs keep_pre). */
int ogb_graph_edge_count(ogb_context *ctx, int which, uint64_t *n);
/* Copies the edges, sorted by (src, offset, dst, orient), to host memory. */
int ogb_graph_edges(ogb_context *ctx, int which, ogb_edge *out, uint64_t cap);

/* The post-reduction edges whose source is in this rank's node range (same order; one rank: the whole list). */
int ogb_graph_edges_shard(ogb_context *ctx, ogb_edge *out, uint64_t cap, uint64_t *n_out);
/* Order-independent checksum of the edge list on the device: xor and sum (mod 2^64) over all edges of
 * mix(src*K1 ^ dst*K2 ^ offset*K3 ^ orient*K4), mix(x) = (x ^ x>>29) * K5, then ^ >>32 -- the figure the oracle's
 * full-size goldens carry (tests/golden/full_size.json), so a result of GBs can be checked without leaving HBM. */
int ogb_graph_checksum(ogb_context *ctx, int which, uint64_t *xor_out, uint64_t *sum_out);

/* ----------------------------------------------------------------------------------------------
 * Graph simplification: the fix-point that ends OverlapGraph::buildOverlapGraphFromHashTable,
 *     do { counter = contractCompositePaths(); counter += removeDeadEndNodes(); } while (counter > 0);
 * (OverlapGraph.cpp:211-215; contractCompositePaths :669-694, mergeEdges :702-752, mergeList :760-785,
 * removeDeadEndNodes :931-988), on the device, on the post-reduction edge list of this context.
 * -------------------------------------------------------------------------------------------- */

/* One directed edge of the simplified graph: an Edge record (Edge.h:17-44) whose listOfReads / listOfOverlapOffsets /
 * listOfOrientations are items[list_start .. list_start + count). twin = index of the reverse edge in the same array. */
typedef struct ogb_cedge {
	uint32_t src;
	uint32_t dst;
	uint64_t offset;     /* overlapOffset: UINT64 once edges are merged (Edge.h:25) */
	uint64_t list_start;
	uint32_t count;
	uint32_t twin;
	uint8_t orient;
	uint8_t reserved[3];
	uint32_t reserved2;
} ogb_cedge; /* 40 bytes */

/* One read inside a composite edge: read ID, its overlap offset from the previous read (UINT16) and its orientation
 * (1 forward, 0 reverse) -- the three parallel vectors of Edge.h:30-32. */
typedef struct ogb_clist_item {
	uint32_t read;
	uint16_t offset;
	uint8_t orient;
	uint8_t reserved;
} ogb_clist_item; /* 8 bytes */

typedef struct ogb_simplify_stats {
	uint64_t n_edges_in, n_edges_out, n_items;
	uint64_t merges, dead_ends;   /* sums of the reference's two counters over all iterations */
	uint32_t iterations;          /* of the do-while */
	uint32_t rounds;              /* launches pairs of the contraction sweeps (see csrc/ogb_contract.cuh) */
	uint32_t jumps;               /* pointer-jumping launches that ranked the read lists */
	uint32_t launches;
	float ms;                     /* device time of the whole stage = the four parts below */
	float ms_setup;               /* rows, entries, twin links */
	float ms_sweeps;              /* contraction rounds */
	float ms_dead_ends;
	float ms_lists;               /* survivors, scans, list ranking, output */
	uint32_t reserved;
} ogb_simplify_stats;

/* Runs the fix-point on the graph ogb_build_graph left on the device (every rank holds the whole post-reduction list, so this
 * is rank-local: no collective) and keeps the result on the device. The edge list of ogb_graph_edges stays as it was. */
int ogb_graph_simplify(ogb_context *ctx, ogb_simplify_stats *stats);
/* Copies the simplified graph to host memory: edges in (src, position in the source's original row) order, items as indexed
 * by list_start. Capacities in elements (ogb_simplify_stats.n_edges_out / n_items). */
int ogb_graph_composite_edges(ogb_context *ctx, ogb_cedge *edges, uint64_t edge_cap, ogb_clist_item *items, uint64_t item_cap);

/* ----------------------------------------------------------------------------------------------
 * Unitig sequences: OverlapGraph::getStringInEdge (OverlapGraph.cpp:2009) for the composite edges of the simplified graph, on the
 * device (csrc/ogb_spell.cuh). Edge e = (src, dst, orient, offset) with items k = 1..c stands for reads src, item reads, dst;
 * src is taken forward iff orient is 2 or 3, dst iff orient is 1 or 3, item k iff its orient is 1; they sit at P_0 = 0,
 * P_k = sum of the first k item offsets, P_{c+1} = offset. The sequence has offset + length(dst) bases, base p taken from the
 * read with the largest P_k <= p. Canonical unitigs are the edges saveGraphToFile writes (OverlapGraph.cpp:321-326): src < dst,
 * or src == dst and index < twin.
 * -------------------------------------------------------------------------------------------- */

/* One spelled unitig. The sequences are laid out word-aligned: unitig i occupies packed words [start/32, start/32 + ceil(length/32))
 * (2-bit, base p in bits 63-2(p%32) .. 62-2(p%32) of word p/32, A0 C1 G2 T3, unused bits zero), or bytes [start, start + length)
 * of the ASCII form (32 bytes per word; the bytes after a unitig's end up to its next word are padding). */
typedef struct ogb_unitig {
	uint32_t edge;        /* index into the ogb_graph_composite_edges order */
	uint32_t src;
	uint32_t dst;
	uint8_t orient;
	uint8_t reserved[3];
	uint64_t length;      /* bases */
	uint64_t start;       /* in bases of the word-aligned layout: a multiple of 32 */
} ogb_unitig; /* 32 bytes */

typedef struct ogb_spell_stats {
	uint64_t unitigs;     /* spelled by the last ogb_graph_spell */
	uint64_t bases;
	uint64_t words;       /* packed output words (ASCII: 32 bytes each) */
	uint32_t launches;
	float ms;             /* device time of ogb_graph_spell */
} ogb_spell_stats;

/* OverlapGraph::getStringInEdge (OverlapGraph.cpp:2009) for unitigs [first, first + count) of the selected edges (all, or the
 * canonical ones with canonical_only != 0) in edge order; count = UINT64_MAX: all from first on. Several ranks can split the
 * unitigs by range with no collective: every rank holds the whole simplified graph. The result stays on the device until the next
 * upload, build, simplify or spell. Needs ogb_graph_simplify on the reads still uploaded (OGB_E_STATE otherwise); first beyond the
 * number of selected edges is OGB_E_ARG. */
int ogb_graph_spell(ogb_context *ctx, int canonical_only, uint64_t first, uint64_t count, ogb_spell_stats *stats);
/* Copies the records of the last ogb_graph_spell and the sequences: packed words (out_cap in bytes >= 8 * words) or, ascii != 0,
 * ACGT bytes decoded on the device (out_cap >= 32 * words). OGB_E_CAPACITY names the sizes needed (ogb_spell_stats.unitigs /
 * words) when a buffer is too small. */
int ogb_graph_unitigs(ogb_context *ctx, ogb_unitig *recs, uint64_t rec_cap, void *out, uint64_t out_cap, int ascii);
/* Writes the unitigs of the last ogb_graph_spell as FASTA, one record per unitig in record order, the sequence on one line:
 *     >unitig_<i> src=<src> dst=<dst> orient=<o> reads=<c+2> length=<L>
 * (i = first + position in the range, c = reads inside the edge). Decoded on the device in bounded chunks staged through pinned
 * host memory. No unitigs: an empty file. OGB_E_IO when the file cannot be written. */
int ogb_graph_write_unitigs(ogb_context *ctx, const char *path);

/* ----------------------------------------------------------------------------------------------
 * Unitig coverage: per-base read depth of the unitigs of the last ogb_graph_spell, on the device (csrc/ogb_coverage.cuh).
 * With f(r) the read's frequency (the Dataset's dedupe count), the depth D[p] of base p of a unitig is the sum of f(r_k) over
 * its placements k (reads src, items, dst at P_k as above) with P_k <= p < P_k + length(r_k), plus f(x) for every contained read x
 * whose superReadID is one of those reads, over the interval x occupies in it: q = the smallest shift at which x's stored strand
 * occurs in the super read's forward strand, else the smallest at which its reverse complement does; the interval starts at
 * P_k + q (super read forward in the unitig) or P_k + length(super) - q - length(x) (reverse). A twin's profile is the reverse.
 * -------------------------------------------------------------------------------------------- */

typedef struct ogb_unitig_coverage {
	uint32_t edge;         /* as ogb_unitig.edge */
	uint32_t reads;        /* placements: reads inside the edge + 2 */
	uint32_t contained;    /* contained reads placed in the unitig */
	uint32_t depth_min;
	uint32_t depth_max;
	uint32_t reserved;
	uint64_t length;       /* as ogb_unitig.length / .start: the profile is depth[start .. start + length) */
	uint64_t start;
	uint64_t read_count;   /* sum of f over the placements and the contained reads placed */
	uint64_t depth_sum;    /* sum of D over the bases (= sum of f * length over the same reads) */
	uint64_t depth_sq_sum; /* sum of D^2, mod 2^64: exact while depth_max^2 * length < 2^64 */
} ogb_unitig_coverage; /* 64 bytes */

typedef struct ogb_coverage_stats {
	uint64_t unitigs;
	uint64_t bases;
	uint64_t placements;            /* reads of the unitigs, src and dst included */
	uint64_t contained_placements;  /* contained reads placed, over all unitigs */
	uint64_t unplaced;              /* contained reads found in neither strand of their super read: 0 on a graph K2 verified */
	uint32_t launches;
	float ms;                       /* device time of ogb_graph_coverage */
	float ms_locate;                /* upload of freq (from the caller's memory) and contained reads located in their super reads */
	float ms_depth;                 /* placements into the difference array, and its scan */
	float ms_reduce;                /* per-base profile and per-unitig sums */
	uint32_t reserved;
} ogb_coverage_stats; /* 64 bytes */

/* The coverage of the unitigs of the last ogb_graph_spell (the same range and selection). freq = the frequency of every uploaded
 * read by ID - 1 (n = the uploaded read count; anything else is OGB_E_ARG), copied to the device per call. The frequencies must
 * sum to less than 2^32, as the depth is kept in 32 bits: a larger sum is OGB_E_ARG, and the error names it (a Dataset's
 * frequencies sum to its kept raw reads, below 2^32). No spell on the current reads: OGB_E_STATE. A refused call leaves the
 * previous result as it was. The result stays on the device until the next upload, build, simplify or spell. Integers only:
 * two runs give the same bits. */
int ogb_graph_coverage(ogb_context *ctx, const uint32_t *freq, uint64_t n, ogb_coverage_stats *stats);
/* Copies the records of the last ogb_graph_coverage (rec_cap >= unitigs) and, when depth is not NULL, the u32 profile in the
 * spell's word-aligned layout (depth_cap in elements >= 32 * ogb_spell_stats.words; padding bases are 0). OGB_E_CAPACITY names
 * the sizes needed. */
int ogb_graph_unitig_coverage(ogb_context *ctx, ogb_unitig_coverage *recs, uint64_t rec_cap, uint32_t *depth, uint64_t depth_cap);
/* Writes the last ogb_graph_coverage as TSV: one '#' header line, then per unitig in record order
 *     unitig_<i> src dst length reads contained read_count mean_depth sd_depth min_depth max_depth
 * with i as in ogb_graph_write_unitigs (the names join with the FASTA), mean = depth_sum / length and
 * sd = sqrt(max(0, depth_sq_sum / length - mean^2)) in double, printed %.4f. OGB_E_IO when the file cannot be written. */
int ogb_graph_write_coverage(ogb_context *ctx, const char *path);

/* ----------------------------------------------------------------------------------------------
 * Sample mapping: per-sample read depth of the unitigs of the last ogb_graph_spell, on the device (csrc/ogb_map.cuh), for the
 * contig x sample depth tables metagenome binners take. A sample is a list of ASCII reads. A read is kept iff it passes the Dataset
 * filter for the build's minOverlap m (length > m and < 65536, ACGT only in either case, no base count >= (UINT64)(len*.8)). A
 * placement of a kept read s of length L is (u, p) with bases [p, p + L) of unitig u equal to s or to its reverse complement; a
 * read equal to its own reverse complement is tested on one strand only. Every placement adds 1 to the depth on [p, p + L). Raw reads
 * count one by one, and a read with several placements counts at each. Reads with indels or clipped alignments do not map.
 *
 * Substitutions (ogb_graph_map_reads_approx): with d = max_mismatches (0 <= d <= OGB_MAP_MAX_MISMATCHES) and K = min(32, m + 1), the
 * key length of the index, a kept read of length L is searched with d_r = min(d, floor(L / K) - 1) substitutions (pigeonhole needs
 * d_r + 1 disjoint K-mers in the read). With m = 50 (K = 32): 100 bp reads at most 2, 150 bp reads at most 3, reads shorter than 2K
 * exactly only. A candidate (u, p, strand) has bases [p, p + L) inside unitig u; its mismatch count H is the Hamming distance to the
 * read (strand 0) or its reverse complement (strand 1). The read's best stratum b is the least H over the candidates of both strands;
 * the read is mapped iff b <= d_r, and its placements are the distinct (u, p) with min(H_fw, H_rc) == b (a (u, p) reached on both
 * strands counts once). Ties all count, as for exact reads. d = 0 is the exact definition above, bit for bit; raising d never removes
 * a placement (a read mapped at b counts the same placements at every d >= b), so the depth at d2 >= d1 is >= that at d1 on every base.
 * -------------------------------------------------------------------------------------------- */

#define OGB_MAP_FILTERED 0xFFFFFFFFu /* hits[i] of a read the filter dropped */
#define OGB_MAP_UNPLACED 0xFF        /* mismatches[i] of a read that is filtered or not mapped */
#define OGB_MAP_MAX_MISMATCHES 8     /* the largest max_mismatches of ogb_graph_map_reads_approx */

typedef struct ogb_map_stats {
	uint64_t reads_in;
	uint64_t filtered;
	uint64_t mapped;          /* kept reads with >= 1 placement */
	uint64_t multi;           /* kept reads with >= 2 placements */
	uint64_t placements;
	uint64_t index_entries;   /* positions of the K-mer index over the unitigs, K = min(32, m + 1) */
	uint64_t index_buckets;
	uint32_t sample;          /* this sample's index among the samples mapped since the spell */
	uint32_t launches;
	float ms;                 /* device time of ogb_graph_map_reads = the four parts below */
	float ms_index;           /* index build; 0 when the index of an earlier sample was reused */
	float ms_upload;          /* reads to the device, filter, packing */
	float ms_map;             /* lookups, verification, difference array (and the hit counts to the host) */
	float ms_reduce;          /* scan, per-base profile and per-unitig sums */
	uint32_t reserved;
} ogb_map_stats; /* 88 bytes */

/* Maps one sample: n reads, read i = bases[offsets[i] .. offsets[i+1]) (ASCII), onto the unitigs of the last ogb_graph_spell (the
 * same range and selection), in bounded chunks of reads. Its records (ogb_unitig_coverage, one per unitig: reads = read_count = its
 * placements, contained = 0, depth sums, min and max as in ogb_graph_coverage) are appended to those of the samples mapped since the
 * spell, 64 B x unitigs per sample on the host; its u32 profile stays on the device until the next sample. hits (NULL or n entries):
 * the placements of every read, OGB_MAP_FILTERED for a read the filter dropped. The K-mer index is built by the first mapping after a
 * spell and kept for the later samples. n = 0 is a valid sample. No spell on the current reads: OGB_E_STATE; a layout of >= 2^32
 * bases: OGB_E_CAPACITY; NULL buffers with n > 0 or offsets that decrease: OGB_E_ARG. Integers only: two runs give the same bits.
 * An upload, build, simplify or spell drops the index and the samples. The coverage of ogb_graph_coverage is left as it is. */
int ogb_graph_map_reads(ogb_context *ctx, const char *bases, const uint64_t *offsets, uint64_t n, uint32_t *hits, ogb_map_stats *stats);
/* ogb_graph_map_reads with up to max_mismatches substitutions per read (the definition above); ogb_graph_map_reads is this call with
 * (0, hits, NULL). mismatches (NULL or n entries): every read's best stratum b, OGB_MAP_UNPLACED for a read that is filtered or not
 * mapped. hits and the counters of stats (mapped, multi, placements) count best-stratum placements. Samples mapped with different
 * max_mismatches share the index and append to the same list. max_mismatches > OGB_MAP_MAX_MISMATCHES: OGB_E_ARG; otherwise the
 * errors of ogb_graph_map_reads. */
int ogb_graph_map_reads_approx(ogb_context *ctx, const char *bases, const uint64_t *offsets, uint64_t n, uint32_t max_mismatches, uint32_t *hits,
                               uint8_t *mismatches, ogb_map_stats *stats);
/* Copies the records of sample `sample` (rec_cap >= unitigs) and, when depth is not NULL, its u32 profile in the spell's word-aligned
 * layout (depth_cap >= 32 * ogb_spell_stats.words) -- kept for the last sample only: depth must be NULL for any other. No samples:
 * OGB_E_STATE; a sample beyond the last, or depth for an earlier one: OGB_E_ARG; OGB_E_CAPACITY names the sizes needed. */
int ogb_graph_sample_coverage(ogb_context *ctx, uint32_t sample, ogb_unitig_coverage *recs, uint64_t rec_cap, uint32_t *depth, uint64_t depth_cap);
/* Writes the depth table of every sample since the spell in MetaBAT's layout (jgi_summarize_bam_contig_depths):
 *     contigName  contigLen  totalAvgDepth  <name_1>  <name_1>-var  ...
 * then per unitig, tab-separated: unitig_<i> (i as in ogb_graph_write_unitigs), its length, the sum of the means, and per sample the
 * mean depth_sum / length and the population variance max(0, depth_sq_sum / length - mean^2), in double, printed %.4f. No edge
 * trimming. names: one per sample (NULL: sample_<j>). No samples: OGB_E_STATE; a name with a tab or a newline: OGB_E_ARG; a file that
 * cannot be written: OGB_E_IO. */
int ogb_graph_write_depths(ogb_context *ctx, const char *path, const char *const *names);

int ogb_get_stats(ogb_context *ctx, ogb_stats *out);

/* Measurement helpers: CUDA events on the context's stream (the stream every kernel of this library
 * is launched on). ogb_timer_end synchronises and returns the elapsed device time. ogb_l2_flush
 * overwrites a scratch buffer of `bytes` (> L2) so that the next build starts cold. */
int ogb_timer_begin(ogb_context *ctx);
int ogb_timer_end(ogb_context *ctx, float *ms);
int ogb_l2_flush(ogb_context *ctx, size_t bytes);

/* Random-gather ceiling of this GPU's HBM (the "HBM random-access roofline" the probe / verify / mark kernels are
 * measured against): every thread keeps four independent, random, aligned loads of gather_bytes (32, 64 or 128) in flight
 * over a scratch buffer of buffer_bytes (a power of two; use the size of the structure the kernel gathers from -- beyond
 * ~256 MB the rate is bound by address translation, not by DRAM bandwidth). Returns useful GB/s = bytes requested / time. */
int ogb_gather_ceiling(ogb_context *ctx, size_t buffer_bytes, uint32_t gather_bytes, double *gb_per_s);

/* Pinned host memory for upload/download staging (released by ogb_free_host). */
int ogb_alloc_host(void **out, size_t bytes);
void ogb_free_host(void *p);

/* ----------------------------------------------------------------------------------------------
 * Synthetic read generator used by bench.py and the tests (seeded, host only). Not part of the
 * reference; SURVEY.md 8(d) defines the five configurations.
 * -------------------------------------------------------------------------------------------- */

/* Uniform i.i.d. ACGT genome of `len` bases. */
int ogb_synth_genome(uint64_t seed, uint64_t len, char *out);

/* Samples n_reads error-free reads from the concatenated genomes (genome g =
 * genomes[g_offsets[g] .. g_offsets[g+1]), picked with probability weights[g]*len). Read length is
 * uniform in [len_min, len_max]; strand flipped with p = 0.5. paired != 0: reads come in pairs
 * (2i, 2i+1), mate 2 = reverse complement of the far end of a fragment ~ N(insert_mean, insert_sd)
 * clipped to >= 2*len. Output: bases (concatenated) + offsets (n_reads + 1). */
int ogb_synth_reads(uint64_t seed, const char *genomes, const uint64_t *g_offsets, const double *weights,
                    uint32_t n_genomes, uint64_t n_reads, uint32_t len_min, uint32_t len_max, int paired,
                    double insert_mean, double insert_sd, char *out_bases, uint64_t out_cap,
                    uint64_t *out_offsets);

#ifdef __cplusplus
}
#endif
#endif /* OGB_H_ */

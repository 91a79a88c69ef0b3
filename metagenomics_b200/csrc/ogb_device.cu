// ogb_device.cu -- device half of libogb.so: context, HBM pools, kernel orchestration and the
// extern "C" entry points declared in include/ogb.h. One context = one GPU = one rank.
//
// Orchestration of one build (reference call sites in brackets):
//   ogb_reads_upload*   H2D + K0                         [Read::setRead, Read.cpp:75-82]
//   ogb_hash_build      K1                               [HashTable::insertDataset, HashTable.cpp:50-80]
//   ogb_mark_contained  K2 (+ allreduce-max)             [OverlapGraph::markContainedReads, OverlapGraph.cpp:225-290]
//   ogb_build_graph     K3 -> [C1] -> K5 -> [C2] -> K6 -> [C3]   [buildOverlapGraphFromHashTable, OverlapGraph.cpp:107-210]; C* only on several ranks
// All buffers are grow-only pools owned by the context, so a repeated build allocates nothing.

#include "ogb_internal.h"
#include "ogb_kernels.cuh"
#include "ogb_contract.cuh"
#include "ogb_spell.cuh"
#include "ogb_coverage.cuh"
#include "ogb_map.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <string>
#include <vector>

#define CUDA_TRY(x)                                                                                      \
	do {                                                                                                 \
		cudaError_t e_ = (x);                                                                            \
		if (e_ != cudaSuccess) {                                                                         \
			ogb_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #x); \
			return OGB_E_CUDA;                                                                           \
		}                                                                                                \
	} while (0)
#define OGB_TRY(x) do { int r_ = (x); if (r_ != OGB_OK) return r_; } while (0)

// ---- NCCL through dlopen: no link-time dependency, and inside a torch process the already loaded
// libnccl.so.2 (torch's bundled one) is reused instead of a second copy.
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { NCCL_UINT8 = 1, NCCL_UINT32 = 3, NCCL_UINT64 = 5 };   // ncclDataType_t values (nccl.h)
enum { NCCL_MAX = 2 };                                         // ncclRedOp_t
struct NcclApi {
	void *lib = nullptr;
	int (*GetUniqueId)(ncclUniqueId *) = nullptr;
	int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
	int (*CommDestroy)(ncclComm_t) = nullptr;
	int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*Send)(const void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*Recv)(void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*GroupStart)() = nullptr;
	int (*GroupEnd)() = nullptr;
	const char *(*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load()
{
	if (g_nccl.lib) return OGB_OK;
	void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
	if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
	if (!lib) { ogb_set_error("cannot load libnccl.so.2: %s", dlerror()); return OGB_E_NCCL; }
#define SYM(field, name) *(void **)(&g_nccl.field) = dlsym(lib, name); if (!g_nccl.field) { ogb_set_error("libnccl: missing %s", name); return OGB_E_NCCL; }
	SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy")
	SYM(AllGather, "ncclAllGather") SYM(AllReduce, "ncclAllReduce") SYM(Broadcast, "ncclBroadcast") SYM(Send, "ncclSend") SYM(Recv, "ncclRecv")
	SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd") SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
	g_nccl.lib = lib;
	return OGB_OK;
}
#define NCCL_TRY(x)                                                                                   \
	do {                                                                                              \
		int r_ = (x);                                                                                 \
		if (r_ != 0) { ogb_set_error("NCCL error %s at %s:%d", g_nccl.GetErrorString(r_), __FILE__, __LINE__); return OGB_E_NCCL; } \
	} while (0)

template <class T> struct Pool {
	T *p = nullptr;
	size_t cap = 0;   // elements
	int ensure(size_t need)
	{
		if (need <= cap) return OGB_OK;
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		cudaError_t e = cudaMalloc((void **)&p, need * sizeof(T));
		if (e != cudaSuccess) { ogb_set_error("cudaMalloc of %zu bytes failed: %s", need * sizeof(T), cudaGetErrorString(e)); return OGB_E_NOMEM; }
		cap = need;
		return OGB_OK;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// d_xchg layout (u64 words): per-rank verdict vectors, scratch
enum { OGB_MAX_RANKS = 64, XCHG_PER_RANK = 8, XCHG_SCRATCH = XCHG_PER_RANK * OGB_MAX_RANKS, XCHG_WORDS = XCHG_SCRATCH + 8 };


// Stream-ordered temporaries (cudaMallocAsync on the context's stream): the Dataset stage needs a dozen scratch arrays for
// a few milliseconds; plain cudaMalloc / cudaFree of them cost more than the kernels (measured: 80 ms + up to seconds).
template <class T> struct Tmp {
	T *p = nullptr;
	cudaStream_t st = nullptr;
	int ensure(size_t need, cudaStream_t stream)
	{
		if (p) return OGB_OK;
		st = stream;
		cudaError_t e = cudaMallocAsync((void **)&p, std::max<size_t>(need, 1) * sizeof(T), stream);
		if (e != cudaSuccess) { ogb_set_error("cudaMallocAsync of %zu bytes failed: %s", need * sizeof(T), cudaGetErrorString(e)); p = nullptr; return OGB_E_NOMEM; }
		return OGB_OK;
	}
	void release() { if (p) cudaFreeAsync(p, st); p = nullptr; }
};

enum { EV_BEGIN = 0, EV_PACK0, EV_PACK1, EV_HASH0, EV_HASH1, EV_CONT0, EV_CONT1, EV_OVL0, EV_OVL1, EV_XPRE1, EV_MARK1, EV_RED1, EV_K3A, EV_K3B, EV_T0, EV_T1, EV_CV1, EV_CV2, EV_MP0, EV_MP1, EV_MP2, EV_MP3, EV_MP4, EV_COUNT };

struct ogb_context {
	int device = 0, rank = 0, nranks = 1, sm_count = 148;
	cudaStream_t stream = nullptr;
	cudaStream_t stream2 = nullptr;   // verify kernels run here, overlapping the next chunk's probe
	cudaEvent_t ev_probe[2] = {}, ev_verify[2] = {};
	cudaEvent_t ev_pk[2 * 64] = {};   // timing pairs around the first 64 probe launches of a build
	cudaEvent_t ev_pm[64] = {};       // ... and between k_window_part and k_probe_parts
	u32 n_pk = 0;
	// per-kernel-class device times of a build (ogb_stats.ms_kernel): event pairs on the launching stream, read back at the end
	struct KEv { cudaEvent_t a = nullptr, b = nullptr; int cls = 0; };
	std::vector<KEv> kev;
	u32 n_kev = 0;
	ncclComm_t comm = nullptr;
	cudaEvent_t ev[EV_COUNT] = {};
	// packed reads
	Pool<u64> words, meta;
	Pool<u64> ds_words;              // tight packed words of the data set last finalized on this device (downloaded on demand)
	ogb_dataset *pending_ds = nullptr;   // ... whose host copy of them is still outstanding
	Pool<char> stage_bytes;          // upload staging (ASCII bases / tight words)
	Pool<u64> stage_offs;
	Pool<unsigned short> stage_lens;
	u32 n = 0, uniform_len = 0, uniform_pw = 0, min_len = 0, max_len = 0;
	bool have_reads = false;
	uint64_t reads_stamp = 0;        // changes with every upload (ogb_dataset::resident_stamp)
	// index
	Pool<u32> slots, summary;
	u32 nb = 0, h = 0, nparts = 1;
	bool use_summary = false;       // the per-bucket summary pays off once the index no longer fits L2
	bool have_table = false;
	// containment
	Pool<u64> sup;
	Pool<u32> contained;
	bool contain_done = false, any_contained = false;
	// graph
	Pool<u64> pos, sums, surv;       // surv: the (at most OGB_SURV) surviving edge words of every own node
	Pool<u64> cand, big;             // K5 -> K6: candidates per own node (edge word, twin bit address); record list of the nodes with more
	Pool<u32> cnt, cntc, scratch_keys;
	Pool<ogb_edge> fin, pre, fin_stage;
	// the adjacency: per-read slot regions, degrees, heavy lists (GraphView)
	Pool<u64> slots_e, ext;
	Pool<u32> deg;
	// what a node looks like to the others (pivot scans, twin verdicts): 128-byte rows by global read index, overflow
	// entries per rank segment, one ELIM bit per entry (GraphView); on several ranks each is allgathered
	Pool<u32> rows, more, more_own, ebits, hrows;   // more_own: this rank's overflow entries (one rank: the whole of `more`); hrows: heavy-row records
	u64 more_stride = 0, more_cap = 0;
	cudaStream_t xs = nullptr;       // several ranks: the rows of a finished chunk travel here while the next chunk is probed
	// ... as copy-engine pushes into the peers' row arrays (mapped with CUDA IPC): no SM of either side is involved, unlike NCCL
	// send / receive kernels, which would compete with the probe for the SMs during the whole of K3
	u32 *peer_rows[64] = {};
	const void *rows_shared = nullptr;   // the allocation the peers currently have mapped
	bool rows_dma = false;
	cudaEvent_t ev_rows[2] = {}, ev_xs = nullptr;
	// scan staging: candidate queue of one chunk, spill list of heavy nodes
	Pool<u32> cand_q, fill, ov_q;    // cand_q / cand_v hold two ping-pong queues of cand_cap entries
	Pool<u64> cand_v, ov_e;
	u64 cand_cap = 0;
	// partitioned probe (index beyond L2): per-partition window queues of one chunk
	Pool<u32> pq_b, pq_f, pq_q;
	u64 *d_pq_cursor = nullptr;
	bool partitioned = false, part_chunk_set = false;
	u64 pq_cap = 0;
	u32 pq_slack = 5;                // queue capacity = even share x pq_slack / 4 (5/4 at first; doubled when a skewed partition overflows)
	u64 *d_cursor = nullptr;         // the two candidate-queue cursors
	u64 *d_xchg = nullptr;           // small per-rank values exchanged with NCCL (XCHG_* layout)
	u32 slot_cap = 64;               // slots per read (adapted to the largest degree seen)
	u32 chunk_reads = 1u << 16;      // query reads per probe/verify launch pair
	int probe_blocks_per_sm = 0, verify_blocks_per_sm = 0;   // 0 = as many as fit
	Pool<char> flush;
	u64 n_final = 0, n_pre = 0;
	u64 fin_own_off = 0, fin_own_cnt = 0;   // this rank's node range inside the final list
	bool have_graph = false, have_pre = false;
	u64 *d_ctr = nullptr, *h_ctr = nullptr;
	u64 *d_tot = nullptr;            // [0] scan total of pre-reduction degrees, [1] of surviving edges
	// simplification (ogb_contract.cuh): CSR of entries, rope records, per-sweep work lists, the result
	Pool<CEntry> sE;
	Pool<CRec> s_rec;
	Pool<u32> s_rowptr, s_cp, s_info, s_list, s_keep, s_items, s_blocker;
	Pool<uint8_t> s_state, s_ready, s_flag;
	Pool<u64> s_epos, s_lpos, s_ctr;
	Pool<ogb_cedge> s_out;
	Pool<ogb_clist_item> s_out_items;
	bool have_simplified = false;
	uint64_t s_stamp = 0;            // reads_stamp of the reads the simplified graph was built on
	ogb_simplify_stats sst = {};
	// unitig sequences (ogb_spell.cuh): selection and item scans, records, packed words, ASCII scratch
	Pool<u32> sp_sel, sp_ioff, sp_nw;
	Pool<u64> sp_rank, sp_ipos, sp_wpos, sp_words;
	Pool<ogb_unitig> sp_rec;
	Pool<char> sp_ascii;
	bool have_spelled = false;
	u64 sp_first = 0;
	ogb_spell_stats spst = {};
	// unitig coverage (ogb_coverage.cuh): contained-read offsets and CSR, placement scan, difference array (then the profile), its scan
	Pool<u32> cv_freq, cv_q, cv_cnt, cv_clist, cv_np, cv_depth;
	Pool<u64> cv_cstart, cv_ppos, cv_scan;
	Pool<ogb_unitig_coverage> cv_rec;
	bool have_covered = false;
	ogb_coverage_stats cvst = {};
	// sample mapping (ogb_map.cuh): K-mer index over the spell's layout, one chunk's reads, difference array (then the profile) and
	// its scan; the records of every sample since the spell on the host
	Pool<u32> mp_cnt, mp_good, mp_khits, mp_hits, mp_diff;
	Pool<u64> mp_bstart, mp_ent, mp_roffs, mp_pos, mp_start, mp_meta, mp_words, mp_scan, mp_ctr;
	Pool<char> mp_raw;
	Pool<unsigned short> mp_len;
	Pool<ogb_unitig_coverage> mp_rec;
	bool mp_have_index = false;
	u32 mp_K = 0;
	u64 mp_buckets = 0, mp_entries = 0;
	std::vector<ogb_unitig_coverage> mp_samples;   // spst.unitigs records per sample
	u32 mp_n_samples = 0;
	bool mp_have_profile = false;                    // mp_diff holds the profile of the last sample
	// L2 persistence window on the bucket summary (l2_keep_summary)
	const void *l2_window_ptr = nullptr;
	size_t l2_window_bytes = 0;
	bool l2_refused = false;
	ogb_stats st = {};
	u32 launches = 0;

	ReadStore rs() const { ReadStore r; r.words = words.p; r.meta = uniform_len ? nullptr : meta.p; r.n = n; r.uniform_len = uniform_len; r.uniform_pw = uniform_pw; return r; }
	Table tb() const
	{
		Table t;
		t.slots = slots.p; t.summary = use_summary ? summary.p : nullptr; t.nb = nb; t.nparts = nparts; t.part_buckets = nb / nparts;
		t.sub = nparts / nranks; t.my_rank = rank; t.h = h; t.ctr = d_ctr;
		return t;
	}
	void shard(u32 &lo, u32 &hi) const
	{
		u64 per = ((u64)n + nranks - 1) / nranks;
		lo = (u32)std::min<u64>(n, per * rank);
		hi = (u32)std::min<u64>(n, per * (rank + 1));
	}
};

// Brackets one launch (or one NCCL call) of class `cls` on `st` with an event pair; at most OGB_KEV_MAX pairs per build.
enum { OGB_KEV_MAX = 4096 };
static int kev_begin(ogb_context *c, int cls, cudaStream_t st)
{
	if (c->n_kev >= OGB_KEV_MAX) return -1;
	if (c->n_kev >= c->kev.size()) {
		ogb_context::KEv e;
		if (cudaEventCreate(&e.a) != cudaSuccess || cudaEventCreate(&e.b) != cudaSuccess) { cudaGetLastError(); return -1; }
		c->kev.push_back(e);
	}
	const int i = (int)c->n_kev++;
	c->kev[i].cls = cls;
	cudaEventRecord(c->kev[i].a, st);
	return i;
}
static void kev_end(ogb_context *c, int i, cudaStream_t st) { if (i >= 0) cudaEventRecord(c->kev[i].b, st); }
// after a synchronisation: adds the pairs recorded since the last collection to st.ms_kernel / st.n_kernel
static void kev_collect(ogb_context *c)
{
	for (u32 i = 0; i < c->n_kev; i++) {
		float ms = 0;
		if (cudaEventElapsedTime(&ms, c->kev[i].a, c->kev[i].b) == cudaSuccess) { c->st.ms_kernel[c->kev[i].cls] += ms; c->st.n_kernel[c->kev[i].cls]++; }
		else cudaGetLastError();
	}
	c->n_kev = 0;
}
#define KEV(cls, stream, launch) do { const int kev_i_ = kev_begin(c, cls, stream); launch; kev_end(c, kev_i_, stream); } while (0)

static int fetch_words_cb(ogb_dataset *ds);

static int ctr_zero(ogb_context *c) { CUDA_TRY(cudaMemsetAsync(c->d_ctr, 0, CTR_COUNT * sizeof(u64), c->stream)); return OGB_OK; }
static int ctr_fetch(ogb_context *c)
{
	CUDA_TRY(cudaMemcpyAsync(c->h_ctr, c->d_ctr, CTR_COUNT * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}
static int grid_for(ogb_context *c, const void *kernel, int block)
{
	int per_sm = 1;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
	return c->sm_count * per_sm;
}
static float ev_ms(ogb_context *c, int a, int b) { float ms = 0; if (cudaEventElapsedTime(&ms, c->ev[a], c->ev[b]) != cudaSuccess) { cudaGetLastError(); return 0; } return ms; }

static int context_create_common(ogb_context **out, int device)
{
	if (!out) { ogb_set_error("ogb_context_create: out is NULL"); return OGB_E_ARG; }
	*out = nullptr;
	int count = 0;
	cudaError_t e = cudaGetDeviceCount(&count);
	if (e != cudaSuccess || count == 0) {
		ogb_set_error("no usable CUDA device (%s); libogb has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
		cudaGetLastError();
		return OGB_E_CUDA;
	}
	if (device < 0 || device >= count) { ogb_set_error("device %d out of range (%d devices)", device, count); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(device));
	ogb_context *c = new ogb_context();
	c->device = device;
	cudaDeviceProp prop;
	CUDA_TRY(cudaGetDeviceProperties(&prop, device));
	c->sm_count = prop.multiProcessorCount;
	// Experiment knob: OGB_L2_FETCH=32|64|128 sets cudaLimitMaxL2FetchGranularity (a hint).
	{
		const char *g = getenv("OGB_L2_FETCH");
		size_t gran = g ? (size_t)atoi(g) : 0;                              // measured: no effect on B200 (profiles/exp_r1_table.txt)
		if (gran == 32 || gran == 64 || gran == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran);
		cudaGetLastError();
	}
	CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	{
		// keep up to 2 GB of freed stream-ordered temporaries cached in the device's default pool (Dataset stage scratch)
		cudaMemPool_t pool;
		if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) { uint64_t keep = 2ull << 30; cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep); }
		cudaGetLastError();
	}
	for (int i = 0; i < EV_COUNT; i++) CUDA_TRY(cudaEventCreate(&c->ev[i]));
	for (int i = 0; i < 128; i++) CUDA_TRY(cudaEventCreate(&c->ev_pk[i]));
	for (int i = 0; i < 64; i++) CUDA_TRY(cudaEventCreate(&c->ev_pm[i]));
	CUDA_TRY(cudaMalloc((void **)&c->d_ctr, CTR_COUNT * sizeof(u64)));
	CUDA_TRY(cudaMalloc((void **)&c->d_tot, 2 * sizeof(u64)));
	CUDA_TRY(cudaMalloc((void **)&c->d_cursor, 2 * sizeof(u64)));
	CUDA_TRY(cudaMalloc((void **)&c->d_pq_cursor, OGB_MAXPART * sizeof(u64)));
	CUDA_TRY(cudaMalloc((void **)&c->d_xchg, XCHG_WORDS * sizeof(u64)));
	CUDA_TRY(cudaMemset(c->d_xchg, 0, XCHG_WORDS * sizeof(u64)));
	CUDA_TRY(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
	CUDA_TRY(cudaStreamCreateWithFlags(&c->xs, cudaStreamNonBlocking));
	for (int i = 0; i < 2; i++) CUDA_TRY(cudaEventCreateWithFlags(&c->ev_rows[i], cudaEventDisableTiming));
	CUDA_TRY(cudaEventCreateWithFlags(&c->ev_xs, cudaEventDisableTiming));
	for (int i = 0; i < 2; i++) { CUDA_TRY(cudaEventCreateWithFlags(&c->ev_probe[i], cudaEventDisableTiming)); CUDA_TRY(cudaEventCreateWithFlags(&c->ev_verify[i], cudaEventDisableTiming)); }
	CUDA_TRY(cudaMemset(c->d_tot, 0, 2 * sizeof(u64)));
	CUDA_TRY(cudaMallocHost((void **)&c->h_ctr, CTR_COUNT * sizeof(u64)));
	CUDA_TRY(cudaMemset(c->d_ctr, 0, CTR_COUNT * sizeof(u64)));
	*out = c;
	return OGB_OK;
}

extern "C" int ogb_context_create(ogb_context **out, int device) { return context_create_common(out, device); }

extern "C" int ogb_nccl_unique_id(void *out128)
{
	if (!out128) { ogb_set_error("ogb_nccl_unique_id: NULL output"); return OGB_E_ARG; }
	OGB_TRY(nccl_load());
	ncclUniqueId id;
	NCCL_TRY(g_nccl.GetUniqueId(&id));
	memcpy(out128, &id, sizeof id);
	return OGB_OK;
}

extern "C" int ogb_context_create_dist(ogb_context **out, int device, int rank, int n_ranks, const void *nccl_uid)
{
	if (n_ranks < 1 || rank < 0 || rank >= n_ranks) { ogb_set_error("ogb_context_create_dist: bad rank %d of %d", rank, n_ranks); return OGB_E_ARG; }
	if (n_ranks > OGB_MAX_RANKS || n_ranks > OGB_MAXPART) { ogb_set_error("ogb_context_create_dist: at most %d ranks", OGB_MAX_RANKS < OGB_MAXPART ? OGB_MAX_RANKS : OGB_MAXPART); return OGB_E_ARG; }
	OGB_TRY(context_create_common(out, device));
	ogb_context *c = *out;
	c->rank = rank; c->nranks = n_ranks;
	if (n_ranks > 1) {
		if (!nccl_uid) { ogb_set_error("ogb_context_create_dist: NULL nccl id"); return OGB_E_ARG; }
		OGB_TRY(nccl_load());
		ncclUniqueId id;
		memcpy(&id, nccl_uid, sizeof id);
		NCCL_TRY(g_nccl.CommInitRank(&c->comm, n_ranks, id, rank));
	}
	return OGB_OK;
}

extern "C" void ogb_context_destroy(ogb_context *c)
{
	if (!c) return;
	cudaSetDevice(c->device);
	cudaStreamSynchronize(c->stream);
	if (c->pending_ds) fetch_words_cb(c->pending_ds);                        // a data set still expects its packed words from this device
	if (c->l2_window_ptr) cudaCtxResetPersistingL2Cache();                   // hand the set-aside part of L2 back
	if (c->stream2) cudaStreamSynchronize(c->stream2);
	if (c->xs) cudaStreamSynchronize(c->xs);
	{
		bool mapped = false;
		for (int p = 0; p < 64; p++) if (c->peer_rows[p]) { cudaIpcCloseMemHandle(c->peer_rows[p]); c->peer_rows[p] = nullptr; mapped = true; }
		if (mapped && c->comm) {                                                // nobody frees an array a peer still has mapped
			g_nccl.AllReduce(c->d_xchg + XCHG_SCRATCH + 6, c->d_xchg + XCHG_SCRATCH + 6, 1, NCCL_UINT64, 2 /*ncclMax*/, c->comm, c->stream);
			cudaStreamSynchronize(c->stream);
		}
	}
	if (c->comm) g_nccl.CommDestroy(c->comm);
	c->words.release(); c->meta.release(); c->ds_words.release(); c->stage_bytes.release(); c->stage_offs.release(); c->stage_lens.release();
	c->slots.release(); c->summary.release(); c->sup.release(); c->contained.release(); c->pos.release();
	c->sums.release(); c->surv.release(); c->cand.release(); c->big.release(); c->cntc.release(); c->cnt.release();
	c->scratch_keys.release(); c->fin.release(); c->pre.release(); c->flush.release(); c->fin_stage.release();
	c->sE.release(); c->s_rec.release(); c->s_rowptr.release(); c->s_cp.release(); c->s_info.release(); c->s_list.release(); c->s_keep.release(); c->s_items.release(); c->s_blocker.release();
	c->s_state.release(); c->s_ready.release(); c->s_flag.release(); c->s_epos.release(); c->s_lpos.release(); c->s_ctr.release(); c->s_out.release(); c->s_out_items.release();
	c->sp_sel.release(); c->sp_ioff.release(); c->sp_nw.release(); c->sp_rank.release(); c->sp_ipos.release(); c->sp_wpos.release(); c->sp_words.release();
	c->sp_rec.release(); c->sp_ascii.release();
	c->cv_freq.release(); c->cv_q.release(); c->cv_cnt.release(); c->cv_clist.release(); c->cv_np.release(); c->cv_depth.release();
	c->cv_cstart.release(); c->cv_ppos.release(); c->cv_scan.release(); c->cv_rec.release();
	c->mp_cnt.release(); c->mp_good.release(); c->mp_khits.release(); c->mp_hits.release(); c->mp_diff.release(); c->mp_bstart.release(); c->mp_ent.release();
	c->mp_roffs.release(); c->mp_pos.release(); c->mp_start.release(); c->mp_meta.release(); c->mp_words.release(); c->mp_scan.release(); c->mp_ctr.release();
	c->mp_raw.release(); c->mp_len.release(); c->mp_rec.release();
	if (c->d_ctr) cudaFree(c->d_ctr);
	if (c->d_tot) cudaFree(c->d_tot);
	if (c->d_cursor) cudaFree(c->d_cursor);
	if (c->d_pq_cursor) cudaFree(c->d_pq_cursor);
	c->pq_b.release(); c->pq_f.release(); c->pq_q.release();
	if (c->d_xchg) cudaFree(c->d_xchg);
	c->cand_q.release(); c->deg.release(); c->fill.release(); c->ov_q.release();
	c->cand_v.release(); c->slots_e.release(); c->ext.release(); c->ov_e.release(); c->rows.release(); c->more.release(); c->more_own.release(); c->hrows.release(); c->ebits.release();
	if (c->h_ctr) cudaFreeHost(c->h_ctr);
	for (int i = 0; i < EV_COUNT; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
	for (int i = 0; i < 128; i++) if (c->ev_pk[i]) cudaEventDestroy(c->ev_pk[i]);
	for (int i = 0; i < 64; i++) if (c->ev_pm[i]) cudaEventDestroy(c->ev_pm[i]);
	for (auto &e : c->kev) { if (e.a) cudaEventDestroy(e.a); if (e.b) cudaEventDestroy(e.b); }
	for (int i = 0; i < 2; i++) { if (c->ev_probe[i]) cudaEventDestroy(c->ev_probe[i]); if (c->ev_verify[i]) cudaEventDestroy(c->ev_verify[i]); }
	for (int i = 0; i < 2; i++) if (c->ev_rows[i]) cudaEventDestroy(c->ev_rows[i]);
	if (c->ev_xs) cudaEventDestroy(c->ev_xs);
	if (c->xs) cudaStreamDestroy(c->xs);
	if (c->stream2) cudaStreamDestroy(c->stream2);
	if (c->stream) cudaStreamDestroy(c->stream);
	delete c;
}

extern "C" int ogb_context_rank(const ogb_context *c, int *rank, int *n_ranks)
{
	if (!c) { ogb_set_error("NULL context"); return OGB_E_ARG; }
	if (rank) *rank = c->rank;
	if (n_ranks) *n_ranks = c->nranks;
	return OGB_OK;
}

extern "C" int ogb_alloc_host(void **out, size_t bytes)
{
	if (!out) { ogb_set_error("ogb_alloc_host: NULL output"); return OGB_E_ARG; }
	cudaError_t e = cudaMallocHost(out, bytes ? bytes : 1);
	if (e != cudaSuccess) { ogb_set_error("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return OGB_E_CUDA; }
	return OGB_OK;
}
extern "C" void ogb_free_host(void *p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------------
// Read upload + K0
// ------------------------------------------------------------------------------------------------

// Decides the device layout from the lengths: uniform stride or per-read meta.
static int layout_reads(ogb_context *c, const std::vector<u32> &lens, u64 &total_words, std::vector<u64> &meta_host)
{
	u32 n = (u32)lens.size();
	u32 mn = 0xFFFFFFFFu, mx = 0;
	for (u32 i = 0; i < n; i++) { mn = std::min(mn, lens[i]); mx = std::max(mx, lens[i]); }
	c->n = n; c->min_len = n ? mn : 0; c->max_len = mx;
	if (n && mn == mx) {
		c->uniform_len = mx;
		c->uniform_pw = ((mx + 63) >> 6) << 1;
		total_words = (u64)n * 2 * c->uniform_pw;
		meta_host.clear();
	} else {
		c->uniform_len = 0; c->uniform_pw = 0;
		meta_host.resize(n);
		u64 off = 0;
		for (u32 i = 0; i < n; i++) {
			if (off >= (1ull << 47)) { ogb_set_error("read store too large"); return OGB_E_CAPACITY; }
			meta_host[i] = (off << 16) | lens[i];
			off += 2 * (u64)(((lens[i] + 63) >> 6) << 1);
		}
		total_words = off;
	}
	return OGB_OK;
}

static int upload_common(ogb_context *c, u64 total_words, const std::vector<u64> &meta_host)
{
	OGB_TRY(c->words.ensure(total_words + 8));          // +8: window extraction may touch two words past a strand
	CUDA_TRY(cudaMemsetAsync(c->words.p + total_words, 0, 8 * sizeof(u64), c->stream));
	if (!meta_host.empty()) {
		OGB_TRY(c->meta.ensure(meta_host.size()));
		CUDA_TRY(cudaMemcpyAsync(c->meta.p, meta_host.data(), meta_host.size() * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
	}
	c->slot_cap = 64;
	c->reads_stamp++;
	c->have_reads = true; c->have_table = false; c->contain_done = false; c->any_contained = false; c->have_graph = false; c->have_pre = false; c->have_spelled = false; c->have_covered = false;
	return OGB_OK;
}

extern "C" int ogb_reads_upload(ogb_context *c, const char *bases, const uint64_t *offsets, uint64_t n)
{
	if (!c || (n && (!bases || !offsets))) { ogb_set_error("ogb_reads_upload: NULL argument"); return OGB_E_ARG; }
	if (n >= (1ull << 30)) { ogb_set_error("ogb_reads_upload: at most 2^30-1 reads per context"); return OGB_E_CAPACITY; }
	CUDA_TRY(cudaSetDevice(c->device));
	std::vector<u32> lens(n);
	for (u64 i = 0; i < n; i++) {
		u64 L = offsets[i + 1] - offsets[i];
		if (L < 2 || L > 65535) { ogb_set_error("ogb_reads_upload: read %llu has length %llu (allowed 2..65535)", (unsigned long long)(i + 1), (unsigned long long)L); return OGB_E_ARG; }
		lens[i] = (u32)L;
	}
	u64 total_words = 0;
	std::vector<u64> meta_host;
	OGB_TRY(layout_reads(c, lens, total_words, meta_host));
	OGB_TRY(upload_common(c, total_words, meta_host));
	if (n == 0) return OGB_OK;
	u64 nbytes = offsets[n] - offsets[0];
	OGB_TRY(c->stage_bytes.ensure(nbytes));
	OGB_TRY(c->stage_offs.ensure(n + 1));
	std::vector<u64> rel(n + 1);
	for (u64 i = 0; i <= n; i++) rel[i] = offsets[i] - offsets[0];
	CUDA_TRY(cudaEventRecord(c->ev[EV_PACK0], c->stream));
	CUDA_TRY(cudaMemcpyAsync(c->stage_bytes.p, bases + offsets[0], nbytes, cudaMemcpyHostToDevice, c->stream));
	CUDA_TRY(cudaMemcpyAsync(c->stage_offs.p, rel.data(), (n + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
	u32 max_pw = ((c->max_len + 63) >> 6) << 1;
	u64 threads = (u64)n * max_pw;
	k_pack_ascii<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(c->stage_bytes.p, c->stage_offs.p, c->words.p,
	                                                                      c->uniform_len ? nullptr : c->meta.p, (u32)n, c->uniform_len, c->uniform_pw, max_pw);
	CUDA_TRY(cudaGetLastError());
	CUDA_TRY(cudaEventRecord(c->ev[EV_PACK1], c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	c->st.ms_pack = ev_ms(c, EV_PACK0, EV_PACK1);
	c->st.n_reads = n;
	return OGB_OK;
}

extern "C" int ogb_reads_upload_packed(ogb_context *c, const uint64_t *words, const uint64_t *word_offsets, const uint16_t *lengths, uint64_t n)
{
	if (!c || (n && (!words || !word_offsets || !lengths))) { ogb_set_error("ogb_reads_upload_packed: NULL argument"); return OGB_E_ARG; }
	if (n >= (1ull << 30)) { ogb_set_error("ogb_reads_upload_packed: at most 2^30-1 reads per context"); return OGB_E_CAPACITY; }
	CUDA_TRY(cudaSetDevice(c->device));
	uint16_t mn = 0xFFFF, mx = 0;
	for (u64 i = 0; i < n; i++) { mn = std::min(mn, lengths[i]); mx = std::max(mx, lengths[i]); }
	if (n && mn < 2) { ogb_set_error("ogb_reads_upload_packed: a read is shorter than 2"); return OGB_E_ARG; }
	u64 total_words = 0;
	std::vector<u64> meta_host;
	const u64 in_words = n ? word_offsets[n] - word_offsets[0] : 0;
	// one read length and a tight input: only the words travel, the kernel derives offsets and lengths
	const bool regular = n && mn == mx && in_words == n * (u64)((mx + 31) / 32);
	if (regular) {
		c->n = (u32)n; c->min_len = c->max_len = mx; c->uniform_len = mx; c->uniform_pw = ((mx + 63) >> 6) << 1;
		total_words = n * 2 * c->uniform_pw;
	} else {
		std::vector<u32> lens(n);
		for (u64 i = 0; i < n; i++) lens[i] = lengths[i];
		OGB_TRY(layout_reads(c, lens, total_words, meta_host));
	}
	OGB_TRY(upload_common(c, total_words, meta_host));
	if (n == 0) return OGB_OK;
	OGB_TRY(c->stage_bytes.ensure(in_words * sizeof(u64)));
	std::vector<u64> rel;
	const u64 *offs_src = (const u64 *)word_offsets;
	if (!regular) {
		OGB_TRY(c->stage_offs.ensure(n + 1));
		OGB_TRY(c->stage_lens.ensure(n));
		if (word_offsets[0] != 0) { rel.resize(n + 1); for (u64 i = 0; i <= n; i++) rel[i] = word_offsets[i] - word_offsets[0]; offs_src = rel.data(); }
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_PACK0], c->stream));
	CUDA_TRY(cudaMemcpyAsync(c->stage_bytes.p, words + word_offsets[0], in_words * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
	if (!regular) {
		CUDA_TRY(cudaMemcpyAsync(c->stage_offs.p, offs_src, (n + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		CUDA_TRY(cudaMemcpyAsync(c->stage_lens.p, lengths, n * sizeof(uint16_t), cudaMemcpyHostToDevice, c->stream));
	}
	u32 max_pw = ((c->max_len + 63) >> 6) << 1;
	u64 threads = (u64)n * max_pw;
	k_pack_words<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>((const u64 *)c->stage_bytes.p, regular ? nullptr : c->stage_offs.p,
	                                                                      regular ? nullptr : c->stage_lens.p, c->words.p,
	                                                                      c->uniform_len ? nullptr : c->meta.p, (u32)n, c->uniform_len, c->uniform_pw, max_pw);
	CUDA_TRY(cudaGetLastError());
	CUDA_TRY(cudaEventRecord(c->ev[EV_PACK1], c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	c->st.ms_pack = ev_ms(c, EV_PACK0, EV_PACK1);
	c->st.n_reads = n;
	return OGB_OK;
}

extern "C" int ogb_reads_upload_dataset(ogb_context *c, const ogb_dataset *ds)
{
	if (!c || !ds) { ogb_set_error("ogb_reads_upload_dataset: NULL argument"); return OGB_E_ARG; }
	if (ds->resident_ctx == c && ds->resident_stamp == c->reads_stamp && c->have_reads) return OGB_OK;   // ogb_dataset_finalize_device left them in HBM
	uint64_t nw = 0;
	const uint64_t *w = ogb_dataset_words(ds, &nw);
	return ogb_reads_upload_packed(c, w, ogb_dataset_word_offsets(ds), ogb_dataset_lengths(ds), ogb_dataset_n_unique(ds));
}

// Several ranks, one read length: every rank uploads only the reads of its own shard (tight forward words) over PCIe,
// K0 packs them into its segment of the read store and one in-place allgather over NVLink replicates the store --
// instead of G copies of the whole read set crossing PCIe at once.
extern "C" int ogb_reads_upload_packed_sharded(ogb_context *c, const uint64_t *shard_words, uint64_t n_total, uint32_t read_len)
{
	if (!c || (n_total && !shard_words)) { ogb_set_error("ogb_reads_upload_packed_sharded: NULL argument"); return OGB_E_ARG; }
	if (n_total >= (1ull << 30)) { ogb_set_error("ogb_reads_upload_packed_sharded: at most 2^30-1 reads per context"); return OGB_E_CAPACITY; }
	if (read_len < 2 || read_len > 65535) { ogb_set_error("ogb_reads_upload_packed_sharded: read length %u (allowed 2..65535)", read_len); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	const int G = c->nranks;
	c->n = (u32)n_total; c->min_len = c->max_len = read_len; c->uniform_len = read_len; c->uniform_pw = ((read_len + 63) >> 6) << 1;
	const u64 per = (n_total + G - 1) / G, stride = 2ull * c->uniform_pw, nw = (read_len + 31) / 32;
	const u64 total_words = per * G * stride;                               // the last rank's segment is padded to the common size
	std::vector<u64> none;
	OGB_TRY(upload_common(c, total_words, none));
	if (n_total == 0) return OGB_OK;
	u32 lo, hi;
	c->shard(lo, hi);
	const u64 nloc = hi - lo;
	OGB_TRY(c->stage_bytes.ensure(std::max<u64>(nloc * nw, 1) * sizeof(u64)));
	CUDA_TRY(cudaEventRecord(c->ev[EV_PACK0], c->stream));
	if (nloc) {
		CUDA_TRY(cudaMemcpyAsync(c->stage_bytes.p, shard_words, nloc * nw * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		const u64 threads = nloc * c->uniform_pw;
		k_pack_words<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>((const u64 *)c->stage_bytes.p, nullptr, nullptr, c->words.p + (u64)lo * stride, nullptr,
		                                                                      (u32)nloc, c->uniform_len, c->uniform_pw, c->uniform_pw);
		CUDA_TRY(cudaGetLastError());
	}
	if (G > 1) NCCL_TRY(g_nccl.AllGather(c->words.p + per * stride * c->rank, c->words.p, per * stride, NCCL_UINT64, c->comm, c->stream));
	CUDA_TRY(cudaEventRecord(c->ev[EV_PACK1], c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	c->st.ms_pack = ev_ms(c, EV_PACK0, EV_PACK1);
	c->st.n_reads = n_total;
	return OGB_OK;
}

static int exclusive_scan(ogb_context *c, const u32 *cnt, u32 n, u64 *out, u64 *d_total, u64 *d_max = nullptr, u64 *d_more = nullptr);

// ------------------------------------------------------------------------------------------------
// Dataset stage on the device
// ------------------------------------------------------------------------------------------------
// the packed words a device finalize left in c->ds_words reach the host vectors now (ogb_dataset::fetch)
static int fetch_words_cb(ogb_dataset *ds)
{
	ogb_context *c = (ogb_context *)ds->fetch_ctx;
	ds->fetch = nullptr; ds->fetch_ctx = nullptr;
	if (!c) return OGB_OK;
	if (c->pending_ds == ds) c->pending_ds = nullptr;
	CUDA_TRY(cudaSetDevice(c->device));
	ds->words.resize(ds->pending_words);
	if (ds->pending_words) {
		CUDA_TRY(cudaMemcpyAsync(ds->words.data(), c->ds_words.p, ds->pending_words * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
	}
	ds->pending_words = 0;
	return OGB_OK;
}
void ogb_dataset_forget_context(ogb_dataset *ds)
{
	ogb_context *c = (ogb_context *)ds->fetch_ctx;
	if (c && c->pending_ds == ds) c->pending_ds = nullptr;
	ds->fetch = nullptr; ds->fetch_ctx = nullptr;
}

// One 8-bit pass of the radix sort over n (key, value) pairs: histogram, scan, stable scatter (ogb_kernels.cuh).
static int radix_pass(ogb_context *c, const u64 *key, const u32 *val, u64 *key_out, u32 *val_out, u32 n, u32 shift, u32 *d_hist, u64 *d_offs)
{
	const u32 nblk = (n + OGB_RS_TILE - 1) / OGB_RS_TILE;
	k_rs_hist<<<nblk, 256, 0, c->stream>>>(key, n, shift, d_hist, nblk);
	OGB_TRY(exclusive_scan(c, d_hist, 256 * nblk, d_offs, c->d_tot));
	k_rs_scatter<<<nblk, 256, 0, c->stream>>>(key, val, key_out, val_out, n, shift, d_offs, nblk);
	CUDA_TRY(cudaGetLastError());
	return OGB_OK;
}

extern "C" int ogb_dataset_finalize_device(ogb_dataset *ds, ogb_context *c, uint32_t min_overlap)
{
	if (!c || !ds) { ogb_set_error("ogb_dataset_finalize_device: NULL argument"); return OGB_E_ARG; }
	if (ds->finalized) { ogb_set_error("ogb_dataset_finalize: already finalized"); return OGB_E_STATE; }
	if (min_overlap < 2) { ogb_set_error("ogb_dataset_finalize: minOverlap must be >= 2"); return OGB_E_ARG; }
	const bool dbg = getenv("OGB_DBG_TIMING") != nullptr;
	auto t_last = std::chrono::steady_clock::now();
	auto lap = [&](const char *what) {
		if (!dbg) return;
		cudaStreamSynchronize(c->stream);
		auto now = std::chrono::steady_clock::now();
		fprintf(stderr, "[finalize_device] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
		t_last = now;
	};
	const u64 n_raw64 = ds->raw_offs.size() - 1;
	if (n_raw64 >= (1ull << 31)) { ogb_set_error("ogb_dataset_finalize_device: at most 2^31-1 raw reads per call"); return OGB_E_CAPACITY; }
	CUDA_TRY(cudaSetDevice(c->device));
	if (c->pending_ds) OGB_TRY(fetch_words_cb(c->pending_ds));               // the previous data set's words are about to be overwritten
	const u32 n_raw = (u32)n_raw64;
	ds->min_overlap = min_overlap;

	Tmp<char> d_raw;
	Tmp<u64> d_roffs, d_start, d_rows, d_key, d_key2, d_pos, d_woff, d_offs;
	Tmp<unsigned short> d_len, d_ulen;
	Tmp<u32> d_good, d_perm, d_perm2, d_head, d_usrc, d_unw, d_ustart, d_freq, d_hist;
	auto release = [&]() {
		d_raw.release(); d_roffs.release(); d_start.release(); d_rows.release(); d_key.release(); d_key2.release(); d_pos.release(); d_woff.release(); d_offs.release();
		d_len.release(); d_ulen.release(); d_good.release(); d_perm.release(); d_perm2.release(); d_head.release(); d_usrc.release(); d_unw.release();
		d_ustart.release(); d_freq.release(); d_hist.release();
	};
	// (pinning the raw bases with cudaHostRegister for the one upload was measured: 58 ms against 16 ms for the pageable copy of 150 MB)
	auto run = [&]() -> int {
		// ---- filter on the device (Dataset.cpp:155-158, :398-413): every raw read is uploaded, the good ones are compacted
		OGB_TRY(d_raw.ensure(ds->raw.size() + 1, c->stream)); OGB_TRY(d_roffs.ensure((u64)n_raw + 1, c->stream));
		OGB_TRY(d_good.ensure((u64)n_raw + 1, c->stream)); OGB_TRY(d_pos.ensure((u64)n_raw + 1, c->stream));
		if (!ds->raw.empty()) CUDA_TRY(cudaMemcpyAsync(d_raw.p, ds->raw.data(), ds->raw.size(), cudaMemcpyHostToDevice, c->stream));
		CUDA_TRY(cudaMemcpyAsync(d_roffs.p, ds->raw_offs.data(), ((size_t)n_raw + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		lap("alloc + H2D of the raw reads");
		u64 stat[2] = {~0ull, 0};
		CUDA_TRY(cudaMemcpyAsync(c->d_xchg + XCHG_SCRATCH, stat, sizeof stat, cudaMemcpyHostToDevice, c->stream));
		if (n_raw) k_ds_filter<<<(n_raw + 127) / 128, 128, 0, c->stream>>>(d_raw.p, d_roffs.p, n_raw, min_overlap, d_good.p, c->d_xchg + XCHG_SCRATCH);
		CUDA_TRY(cudaGetLastError());
		OGB_TRY(exclusive_scan(c, d_good.p, n_raw, d_pos.p, c->d_tot));
		u64 n64 = 0;
		CUDA_TRY(cudaMemcpyAsync(&n64, c->d_tot, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaMemcpyAsync(stat, c->d_xchg + XCHG_SCRATCH, sizeof stat, cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		lap("filter kernel + scan");
		ds->n_good = n64; ds->shortest = n64 ? stat[0] : ~0ULL; ds->longest = n64 ? stat[1] : 0;
		ds->finalized = true;
		ds->word_offs.assign(1, 0); ds->words.clear(); ds->lens.clear(); ds->freq.clear();
		if (n64 == 0) return OGB_OK;
		if (n64 >= (1ull << 30)) { ogb_set_error("ogb_dataset_finalize_device: at most 2^30-1 reads per context"); return OGB_E_CAPACITY; }
		const u32 n = (u32)n64, W = (u32)((ds->longest + 31) / 32);
		OGB_TRY(d_start.ensure(n, c->stream)); OGB_TRY(d_len.ensure(n, c->stream)); OGB_TRY(d_rows.ensure((u64)n * W, c->stream));
		OGB_TRY(d_key.ensure(n, c->stream)); OGB_TRY(d_key2.ensure(n, c->stream)); OGB_TRY(d_perm.ensure(n, c->stream)); OGB_TRY(d_perm2.ensure(n, c->stream)); OGB_TRY(d_head.ensure(n, c->stream));
		const u32 nblk = (n + OGB_RS_TILE - 1) / OGB_RS_TILE;
		OGB_TRY(d_hist.ensure(256ull * nblk, c->stream)); OGB_TRY(d_offs.ensure(256ull * nblk + 1, c->stream));
		k_ds_compact<<<(n_raw + 255) / 256, 256, 0, c->stream>>>(d_good.p, d_pos.p, d_roffs.p, n_raw, d_start.p, d_len.p);
		const unsigned g256 = (n + 255) / 256;
		k_ds_canon<<<(n + 127) / 128, 128, 0, c->stream>>>(d_raw.p, d_start.p, d_len.p, d_rows.p, n, W);
		k_ds_iota<<<g256, 256, 0, c->stream>>>(d_perm.p, n);
		CUDA_TRY(cudaGetLastError());
		lap("compact + canonical strand");
		// ---- LSD radix sort: length first (least significant), then the words from last to first; every pass is stable.
		// Bytes in which no two keys differ (zero padding, equal lengths, shared high bits) need no pass.
		u32 *pa = d_perm.p, *pb = d_perm2.p;
		u64 *ka = d_key.p, *kb = d_key2.p;
		u32 passes = 0;
		for (int word = (int)W; word >= 0; word--) {
			k_ds_key<<<g256, 256, 0, c->stream>>>(d_rows.p, d_len.p, pa, ka, n, W, (u32)word);
			u64 oa[2] = {0, ~0ull};
			CUDA_TRY(cudaMemcpyAsync(c->d_xchg + XCHG_SCRATCH, oa, sizeof oa, cudaMemcpyHostToDevice, c->stream));
			k_rs_orand<<<c->sm_count * 4, 256, 0, c->stream>>>(ka, n, c->d_xchg + XCHG_SCRATCH);
			CUDA_TRY(cudaMemcpyAsync(oa, c->d_xchg + XCHG_SCRATCH, sizeof oa, cudaMemcpyDeviceToHost, c->stream));
			CUDA_TRY(cudaStreamSynchronize(c->stream));
			const u64 varying = oa[0] ^ oa[1];
			for (u32 shift = 0; shift < 64; shift += 8) {
				if (!((varying >> shift) & 255u)) continue;
				OGB_TRY(radix_pass(c, ka, pa, kb, pb, n, shift, d_hist.p, d_offs.p));
				std::swap(ka, kb); std::swap(pa, pb);
				passes++;
			}
		}
		if (dbg) fprintf(stderr, "[finalize_device] %u radix passes\n", passes);
		lap("radix sort passes");
		// ---- dedupe: heads -> unique index, run lengths = frequencies
		OGB_TRY(d_pos.ensure((u64)n + 1, c->stream));
		k_ds_heads<<<g256, 256, 0, c->stream>>>(d_rows.p, d_len.p, pa, d_head.p, n, W);
		CUDA_TRY(cudaGetLastError());
		OGB_TRY(exclusive_scan(c, d_head.p, n, d_pos.p, c->d_tot));
		u64 nu64 = 0;
		CUDA_TRY(cudaMemcpyAsync(&nu64, c->d_tot, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		const u32 nu = (u32)nu64;
		OGB_TRY(d_usrc.ensure(nu, c->stream)); OGB_TRY(d_ulen.ensure(nu, c->stream)); OGB_TRY(d_unw.ensure(nu, c->stream)); OGB_TRY(d_ustart.ensure(nu, c->stream)); OGB_TRY(d_freq.ensure(nu, c->stream)); OGB_TRY(d_woff.ensure((u64)nu + 1, c->stream));
		k_ds_unique<<<g256, 256, 0, c->stream>>>(d_head.p, d_pos.p, pa, d_len.p, d_usrc.p, d_ulen.p, d_unw.p, d_ustart.p, n);
		CUDA_TRY(cudaGetLastError());
		OGB_TRY(exclusive_scan(c, d_unw.p, nu, d_woff.p, c->d_tot));
		u64 total_in = 0;
		CUDA_TRY(cudaMemcpyAsync(&total_in, c->d_tot, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		CUDA_TRY(cudaMemcpyAsync(d_woff.p + nu, c->d_tot, sizeof(u64), cudaMemcpyDeviceToDevice, c->stream));
		OGB_TRY(c->ds_words.ensure(total_in + 4));
		k_ds_emit<<<(nu + 255) / 256, 256, 0, c->stream>>>(d_rows.p, d_usrc.p, d_unw.p, d_ustart.p, d_woff.p, d_freq.p, c->ds_words.p, nu, n, W);
		CUDA_TRY(cudaGetLastError());
		lap("dedupe + emit");
		// ---- host views: lengths, frequencies and word offsets now (small); the packed words stay on the device until somebody
		// asks for them (ogb_dataset::fetch) -- they are two thirds of the bytes and the reads are already where the build needs them
		ds->lens.resize(nu); ds->freq.resize(nu); ds->word_offs.resize((size_t)nu + 1);
		CUDA_TRY(cudaMemcpyAsync(ds->lens.data(), d_ulen.p, nu * sizeof(unsigned short), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaMemcpyAsync(ds->freq.data(), d_freq.p, nu * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaMemcpyAsync(ds->word_offs.data(), d_woff.p, ((size_t)nu + 1) * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		ds->pending_words = total_in; ds->fetch = fetch_words_cb; ds->fetch_ctx = c; c->pending_ds = ds;
		lap("D2H of the small host views");
		// ... and the read store of the context is filled straight from the device copy (K0), no second upload
		u64 total_words = 0;
		std::vector<u64> meta_host;
		std::vector<u32> lens32(ds->lens.begin(), ds->lens.end());
		OGB_TRY(layout_reads(c, lens32, total_words, meta_host));
		OGB_TRY(upload_common(c, total_words, meta_host));
		const u32 max_pw = ((c->max_len + 63) >> 6) << 1;
		const u64 threads = (u64)nu * max_pw;
		CUDA_TRY(cudaEventRecord(c->ev[EV_PACK0], c->stream));
		k_pack_words<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(c->ds_words.p, d_woff.p, d_ulen.p, c->words.p, c->uniform_len ? nullptr : c->meta.p,
		                                                                      nu, c->uniform_len, c->uniform_pw, max_pw);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaEventRecord(c->ev[EV_PACK1], c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		c->st.ms_pack = ev_ms(c, EV_PACK0, EV_PACK1);
		c->st.n_reads = nu;
		ds->resident_ctx = c; ds->resident_stamp = c->reads_stamp;
		lap("layout + K0");
		return OGB_OK;
	};
	const int rc = run();
	cudaStreamSynchronize(c->stream);
	release();
	lap("cudaFree");
	if (rc != OGB_OK) {
		// leave the dataset as it was before the call: the raw reads stay, so the caller can still run ogb_dataset_finalize on the host
		ds->finalized = false;
		ds->lens.clear(); ds->freq.clear(); ds->word_offs.clear(); ds->words.clear();
		ds->resident_ctx = nullptr;
		if (c->pending_ds == ds) c->pending_ds = nullptr;
		ds->fetch = nullptr; ds->fetch_ctx = nullptr; ds->pending_words = 0;
		return rc;
	}
	ds->raw.clear(); ds->raw.shrink_to_fit();
	ds->raw_offs.clear(); ds->raw_offs.shrink_to_fit();
	lap("free raw");
	return rc;
}

// ------------------------------------------------------------------------------------------------
// K1
// ------------------------------------------------------------------------------------------------
// The per-bucket summary is the one structure of K3 every window reads at random and that is small enough for L2 (4 bytes per
// bucket: 34 MB at config 3), but the streams of the kernels around it (window queues, buckets, partner strands) keep evicting it:
// k_window_part alone read 0.53 GB from DRAM per launch for a 34 MB array. An access-policy window on the scan stream makes its
// sectors persisting in a set-aside part of L2 (hit ratio = what fits): 0.06 GB per launch, K3 17.1 -> 15.7 ms at config 3.
// The window is open while K2 / K3 run only, and closing it also resets the persisting lines and takes the set-aside back: with
// the set-aside left in place K1 of the next build went from 1.8 to 2.3 ms (4.3 -> 10.4 ms with a 69 MB summary), and neither
// closing the window alone nor resetting the lines gives that back (profiles/r2/exp_l2_persist.txt). It is a hint: if the runtime
// refuses any of the calls the context goes on without it. OGB_L2_PERSIST=0 turns it off.
static int l2_keep_summary(ogb_context *c, bool enable)
{
	static int max_persist = -1, max_window = 0;
	if (c->l2_refused) return OGB_OK;
	if (max_persist < 0) {
		cudaDeviceProp prop;
		CUDA_TRY(cudaGetDeviceProperties(&prop, c->device));
		max_persist = prop.persistingL2CacheMaxSize; max_window = prop.accessPolicyMaxWindowSize;
	}
	const char *e = getenv("OGB_L2_PERSIST");
	const bool on = enable && c->use_summary && max_persist > 0 && max_window > 0 && !(e && atoi(e) == 0);
	const size_t bytes = on ? (size_t)c->nb * sizeof(u32) : 0, window = std::min<size_t>(bytes, (size_t)max_window);
	const size_t set_aside = std::min<size_t>(window, (size_t)max_persist);
	if (c->l2_window_ptr == (on ? (const void *)c->summary.p : nullptr) && c->l2_window_bytes == window) return OGB_OK;   // already so
	cudaStreamAttrValue attr;
	memset(&attr, 0, sizeof attr);
	bool ok = true;
	if (on) {
		ok = cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside) == cudaSuccess;
		attr.accessPolicyWindow.base_ptr = c->summary.p;
		attr.accessPolicyWindow.num_bytes = window;
		attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)set_aside / (double)std::max<size_t>(window, 1));
		attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
		attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
	}
	else { attr.accessPolicyWindow.num_bytes = 0; attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal; attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal; }
	ok = ok && cudaStreamSetAttribute(c->stream, cudaStreamAttributeAccessPolicyWindow, &attr) == cudaSuccess;
	if (!on && c->l2_window_ptr) ok = ok && cudaCtxResetPersistingL2Cache() == cudaSuccess && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0) == cudaSuccess;
	if (!ok) {                                                               // not an error of the build: go on with a plain L2
		cudaGetLastError();
		memset(&attr, 0, sizeof attr);
		attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal; attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
		cudaStreamSetAttribute(c->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
		cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0);
		cudaGetLastError();
		c->l2_refused = true; c->l2_window_ptr = nullptr; c->l2_window_bytes = 0;
		return OGB_OK;
	}
	c->l2_window_ptr = on ? c->summary.p : nullptr; c->l2_window_bytes = window;
	return OGB_OK;
}

extern "C" int ogb_hash_build(ogb_context *c, uint32_t min_overlap)
{
	if (!c) { ogb_set_error("NULL context"); return OGB_E_ARG; }
	if (!c->have_reads) { ogb_set_error("ogb_hash_build: upload reads first"); return OGB_E_STATE; }
	if (min_overlap < 2) { ogb_set_error("ogb_hash_build: minOverlap must be >= 2"); return OGB_E_ARG; }
	if (c->n && c->min_len <= min_overlap) { ogb_set_error("ogb_hash_build: every read must be longer than minOverlap (Dataset.cpp:158); shortest is %u", c->min_len); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	OGB_TRY(l2_keep_summary(c, false));                                     // K1 runs without the window (see l2_keep_summary)
	c->h = min_overlap - 1;                                                 // HashTable.cpp:54
	// The reference sizes the table at the first listed prime > 8N+1 slots (HashTable.cpp:56), i.e.
	// load factor <= 0.5 for its 4N entries. Here: N buckets of 10 slots (64 B per read, load 0.4).
	double buckets_per_read = 1.0;
	{
		const char *lf = getenv("OGB_TABLE_BUCKETS_PER_READ");
		if (lf && atof(lf) >= 0.5) buckets_per_read = atof(lf);
	}
	{
		// The per-bucket summary (4 B per bucket) lets the probe drop the windows that cannot have an entry before
		// the bucket fetch and compact the rest (PendQueue); OGB_SUMMARY=0 turns it off (experiment knob).
		const char *e = getenv("OGB_SUMMARY");
		c->use_summary = e ? atoi(e) != 0 : true;
	}
	{
		// Probe through per-partition window queues (k_window_part + k_probe_parts) whenever the summary exists: measured
		// faster than the direct kernel even with an L2-resident index (config 2: K3 2.21 -> 1.91 ms), and the only way to keep
		// the bucket fetches in L2 beyond it (config 3: 24.7 -> 18.2 ms). OGB_PARTITIONED=0: direct path (experiment knob).
		const char *e = getenv("OGB_PARTITIONED");
		c->partitioned = e ? atoi(e) != 0 : true;
	}
	c->launches = 0;
	c->n_kev = 0;
	memset(c->st.ms_kernel, 0, sizeof c->st.ms_kernel); memset(c->st.n_kernel, 0, sizeof c->st.n_kernel);
	CUDA_TRY(cudaEventRecord(c->ev[EV_HASH0], c->stream));
	// One hash partition per rank: every rank inserts only the keys of its own partition (a slice of
	// nb/G buckets that stays L2- and TLB-friendly), then the slices are allgathered. A replicated build
	// of the whole table cost 3.8 ms at 8 ranks (TLB-bound inserts into 664 MB).
	// Partitions per rank: 1 up to 192 MB of slice; beyond that the slice is cut into pieces of <= 160 MB, the
	// unit the partitioned probe (k_window_part / k_probe_parts) works through at a time.
	// A partition is chosen by the key's first 16 bases alone and linear probing wraps inside it, so a skewed read set can
	// fill one up (K1 raises CTR_TABLE_FULL after a whole lap; a key queue that overflows raises it to 2): the build is then repeated with half as many partitions per
	// rank and, once there is one per rank, with twice the buckets -- a collective decision, all ranks see the same flag.
	u64 sub_limit = OGB_MAXPART / c->nranks, nb = 0;
	bool k1_direct = false;
	for (int attempt = 0;; attempt++) {
		if (attempt == 12) { ogb_set_error("ogb_hash_build: a hash partition kept filling up (%u partitions, %.1f buckets per read)", c->nparts, buckets_per_read); return OGB_E_CAPACITY; }
		nb = std::max<u64>((u64)(buckets_per_read * c->n) + 1, 512);
		{
			const u64 slice_bytes = nb * OGB_BWORDS * sizeof(u32) / c->nranks;
			// measured (profiles/r2/exp_partitions.txt): the optimum is ~140-180 MB per partition at 0.55, 0.6 and 1.1 GB of index --
			// what a partition buys is translation reach and full queue tiles, not L2 residency (46 MB partitions: +7 %)
			u64 sub = slice_bytes > (192ull << 20) ? (slice_bytes + (160ull << 20) - 1) / (160ull << 20) : 1;
			const char *e = getenv("OGB_SUB_PARTITIONS");                        // experiment knob
			if (e && atoi(e) >= 1) sub = (u64)atoi(e);
			sub = std::max<u64>(1, std::min<u64>(sub, sub_limit));
			c->nparts = (u32)(c->nranks * sub);
		}
		nb = (nb + c->nparts - 1) / c->nparts * c->nparts;
		if (nb >= (1ull << 32)) { ogb_set_error("index too large"); return OGB_E_CAPACITY; }
		c->nb = (u32)nb;
		OGB_TRY(c->slots.ensure(nb * OGB_BWORDS));
		if (c->use_summary) OGB_TRY(c->summary.ensure(nb));
		{
			// only this rank's slice is cleared and filled; the allgather below overwrites the others
			const u64 pb = nb / c->nranks;
			CUDA_TRY(cudaMemsetAsync(c->slots.p + pb * OGB_BWORDS * c->rank, 0, pb * OGB_BWORDS * sizeof(u32), c->stream));
			if (c->use_summary) CUDA_TRY(cudaMemsetAsync(c->summary.p + pb * c->rank, 0, pb * sizeof(u32), c->stream));
		}
		CUDA_TRY(cudaMemsetAsync(c->d_ctr + CTR_TABLE_FULL, 0, sizeof(u64), c->stream));
		if (c->n) {
			u64 threads = (u64)c->n * 4;
			// Several partitions per rank (index beyond L2): the keys go through per-partition queues and are inserted one
			// L2-resident partition at a time. A skewed set that overflows a queue (checked below) is rebuilt by the direct kernel.
			const u32 sub = c->nparts / c->nranks;
			const char *eq = getenv("OGB_K1_QUEUES");                            // experiment knob: 0 = always the direct kernel
			const bool queued = sub > 1 && !k1_direct && !(eq && atoi(eq) == 0);
			if (queued) {
				const u64 qcap = threads / c->nparts * 5 / 4 + 4096;             // 25 % slack over an even split of the 4N keys over the partitions
				OGB_TRY(c->pq_b.ensure(qcap * sub)); OGB_TRY(c->pq_f.ensure(qcap * sub)); OGB_TRY(c->pq_q.ensure(qcap * sub));
				KeyQueue kq;
				kq.b = c->pq_b.p; kq.f = c->pq_f.p; kq.v = c->pq_q.p; kq.cursor = c->d_pq_cursor; kq.cap = qcap;
				kq.nparts = c->nparts; kq.first = (u32)c->rank * sub; kq.count = sub;
				CUDA_TRY(cudaMemsetAsync(c->d_pq_cursor, 0, OGB_MAXPART * sizeof(u64), c->stream));
				const u64 tiles = (threads + 256 * OGB_KPT - 1) / (256 * OGB_KPT);
				const int ke = kev_begin(c, OGB_KC_HASH, c->stream);
				k_key_part<<<(unsigned)std::min<u64>(grid_for(c, (const void *)k_key_part, 256), tiles), 256, 0, c->stream>>>(c->rs(), c->tb(), kq);
				k_insert_parts<<<grid_for(c, (const void *)k_insert_parts, 256), 256, 0, c->stream>>>(c->tb(), kq);
				kev_end(c, ke, c->stream);
				CUDA_TRY(cudaGetLastError());
				c->launches += 2;
			}
			if (!queued) {
				KEV(OGB_KC_HASH, c->stream, (k_hash_insert<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(c->rs(), c->tb())));
				CUDA_TRY(cudaGetLastError());
				c->launches++;
			}
		}
		// the verdict travels with the slices: on several ranks it is max-reduced first (tiny), then every rank decides alike
		u64 full = 0;
		if (c->nranks > 1) NCCL_TRY(g_nccl.AllReduce(c->d_ctr + CTR_TABLE_FULL, c->d_ctr + CTR_TABLE_FULL, 1, NCCL_UINT64, NCCL_MAX, c->comm, c->stream));
		CUDA_TRY(cudaMemcpyAsync(c->h_ctr + CTR_TABLE_FULL, c->d_ctr + CTR_TABLE_FULL, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		if (c->nranks > 1) {
			const u64 pb = nb / c->nranks;
			const int ke = kev_begin(c, OGB_KC_EXCH_INDEX, c->stream);
			NCCL_TRY(g_nccl.AllGather(c->slots.p + pb * OGB_BWORDS * c->rank, c->slots.p, pb * OGB_BWORDS, NCCL_UINT32, c->comm, c->stream));
			if (c->use_summary) NCCL_TRY(g_nccl.AllGather(c->summary.p + pb * c->rank, c->summary.p, pb, NCCL_UINT32, c->comm, c->stream));
			kev_end(c, ke, c->stream);
		}
		CUDA_TRY(cudaEventRecord(c->ev[EV_HASH1], c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		kev_collect(c);
		full = c->h_ctr[CTR_TABLE_FULL];
		c->st.hash_build_attempts = (uint32_t)attempt + 1;
		if (!full) break;
		if (full >= 2 && !k1_direct) { k1_direct = true; continue; }         // a key queue overflowed: same geometry, direct kernel
		if (c->nparts > (u32)c->nranks) sub_limit = std::max<u64>(1, c->nparts / c->nranks / 2);
		else buckets_per_read *= 2;
	}
	OGB_TRY(l2_keep_summary(c, true));
	c->st.ms_hash_build = ev_ms(c, EV_HASH0, EV_HASH1);
	c->st.table_buckets = nb;
	c->st.hash_partitions = c->nparts;
	c->st.table_bytes = nb * OGB_BWORDS * sizeof(u32);
	c->part_chunk_set = false; c->pq_slack = 5;
	if (!c->partitioned && c->chunk_reads > (1u << 16)) c->chunk_reads = 1u << 16;
	c->have_table = true; c->contain_done = false; c->any_contained = false; c->have_graph = false;
	c->st.ms_contain = 0; c->st.n_contained = 0; c->st.contain_probes = 0; c->st.contain_hits = 0;
	return OGB_OK;
}

extern "C" uint64_t ogb_hash_string_length(const ogb_context *c) { return c ? c->h : 0; }
extern "C" uint64_t ogb_hash_table_size(const ogb_context *c) { return c ? (uint64_t)c->nb * OGB_SLOTS : 0; }

extern "C" int ogb_hash_lookup(ogb_context *c, const char *keys, uint64_t n_keys, uint64_t *out, uint64_t out_cap, uint64_t *out_offsets)
{
	if (!c || !out_offsets || (n_keys && !keys)) { ogb_set_error("ogb_hash_lookup: NULL argument"); return OGB_E_ARG; }
	if (!c->have_table) { ogb_set_error("ogb_hash_lookup: build the hash table first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	const u32 h = c->h, kw = (h + 31) / 32;
	out_offsets[0] = 0;
	if (n_keys == 0) return OGB_OK;
	std::vector<u64> packed(n_keys * (kw + 2) + 4, 0);
	for (u64 k = 0; k < n_keys; k++)
		for (u32 i = 0; i < h; i++) {
			u64 code;
			switch (keys[k * h + i]) {
			case 'A': case 'a': code = 0; break;
			case 'C': case 'c': code = 1; break;
			case 'G': case 'g': code = 2; break;
			case 'T': case 't': code = 3; break;
			default: ogb_set_error("ogb_hash_lookup: key %llu is not ACGT", (unsigned long long)k); return OGB_E_ARG;
			}
			packed[k * (kw + 2) + (i >> 5)] |= code << (62 - 2 * (i & 31));
		}
	Pool<u64> d_keys, d_pos, d_out;
	Pool<u32> d_cnt;
	int rc = OGB_OK;
	std::vector<u32> cnt(n_keys);
	std::vector<u64> pos(n_keys + 1, 0);
	auto run = [&]() -> int {
		OGB_TRY(d_keys.ensure(packed.size())); OGB_TRY(d_cnt.ensure(n_keys)); OGB_TRY(d_pos.ensure(n_keys + 1));
		CUDA_TRY(cudaMemcpyAsync(d_keys.p, packed.data(), packed.size() * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		unsigned grid = (unsigned)((n_keys + 127) / 128);
		k_lookup<<<grid, 128, 0, c->stream>>>(c->rs(), c->tb(), d_keys.p, kw, n_keys, d_cnt.p, nullptr, nullptr, 0);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaMemcpyAsync(cnt.data(), d_cnt.p, n_keys * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		for (u64 k = 0; k < n_keys; k++) pos[k + 1] = pos[k] + cnt[k];
		for (u64 k = 0; k <= n_keys; k++) out_offsets[k] = pos[k];
		if (pos[n_keys] > out_cap || (pos[n_keys] && !out)) { ogb_set_error("ogb_hash_lookup: output needs %llu entries", (unsigned long long)pos[n_keys]); return OGB_E_CAPACITY; }
		if (pos[n_keys] == 0) return OGB_OK;
		OGB_TRY(d_out.ensure(pos[n_keys]));
		CUDA_TRY(cudaMemcpyAsync(d_pos.p, pos.data(), (n_keys + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		k_lookup<<<grid, 128, 0, c->stream>>>(c->rs(), c->tb(), d_keys.p, kw, n_keys, d_cnt.p, d_pos.p, d_out.p, 1);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaMemcpyAsync(out, d_out.p, pos[n_keys] * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		// the reference's bucket order is insertion order: ascending id, then orientation
		for (u64 k = 0; k < n_keys; k++)
			std::sort(out + pos[k], out + pos[k + 1], [](u64 a, u64 b) {
				u64 ia = a & 0x3FFFFFFFFFFFFFFFull, ib = b & 0x3FFFFFFFFFFFFFFFull;
				return ia != ib ? ia < ib : (a >> 62) < (b >> 62);
			});
		return OGB_OK;
	};
	rc = run();
	d_keys.release(); d_pos.release(); d_out.release(); d_cnt.release();
	return rc;
}

// ------------------------------------------------------------------------------------------------
// K2
// ------------------------------------------------------------------------------------------------
static ScanArgs scan_args(ogb_context *c, u32 lo, u32 hi)
{
	ScanArgs a;
	a.R = c->rs(); a.T = c->tb(); a.lo = lo; a.hi = hi;
	a.contained = c->any_contained ? c->contained.p : nullptr;
	a.cand_q = c->cand_q.p; a.cand_v = c->cand_v.p; a.cand_cap = c->cand_cap; a.cand_cursor = c->d_cursor;
	a.sup = c->sup.p; a.slots_e = c->slots_e.p; a.slot_lo = lo; a.cap = c->slot_cap; a.deg = c->deg.p;
	a.ov_q = c->ov_q.p; a.ov_e = c->ov_e.p; a.ov_cap = c->ov_q.cap; a.ctr = c->d_ctr; a.prefetch = 1;
	return a;
}

static GraphView graph_view(const ogb_context *c, u32 lo);

// (Re)maps every rank's row array into the others (collective; the array is (re)allocated at the same moment on all ranks
// because its size depends on the read count and the rank count only). On any failure the exchange falls back to NCCL.
static int share_rows(ogb_context *c)
{
	const int G = c->nranks;
	if (G == 1 || c->rows_shared == (const void *)c->rows.p) return OGB_OK;
	for (int p = 0; p < G; p++) if (c->peer_rows[p]) { cudaIpcCloseMemHandle(c->peer_rows[p]); c->peer_rows[p] = nullptr; }
	c->rows_dma = false;
	c->rows_shared = c->rows.p;
	const char *e = getenv("OGB_ROWS_NCCL");
	u64 ok = !(e && atoi(e) != 0);
	cudaIpcMemHandle_t mine;
	memset(&mine, 0, sizeof mine);
	if (ok && cudaIpcGetMemHandle(&mine, c->rows.p) != cudaSuccess) { cudaGetLastError(); ok = 0; }
	// handles (64 bytes) + an "I can" flag travel through a small device buffer
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
	const size_t rec = 72;
	Pool<unsigned char> buf;
	OGB_TRY(buf.ensure(rec * G));
	std::vector<unsigned char> host(rec * G, 0);
	memcpy(host.data() + rec * c->rank, &mine, 64);
	memcpy(host.data() + rec * c->rank + 64, &ok, 8);
	CUDA_TRY(cudaMemcpyAsync(buf.p + rec * c->rank, host.data() + rec * c->rank, rec, cudaMemcpyHostToDevice, c->stream));
	NCCL_TRY(g_nccl.AllGather(buf.p + rec * c->rank, buf.p, rec, NCCL_UINT8, c->comm, c->stream));
	CUDA_TRY(cudaMemcpyAsync(host.data(), buf.p, rec * G, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	buf.release();
	bool all = true;
	for (int p = 0; p < G; p++) { u64 f; memcpy(&f, host.data() + rec * p + 64, 8); all = all && f != 0; }
	u64 opened = all;
	if (all)
		for (int p = 0; p < G && opened; p++) {
			if (p == c->rank) continue;
			cudaIpcMemHandle_t h;
			memcpy(&h, host.data() + rec * p, 64);
			void *ptr = nullptr;
			if (cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); opened = 0; break; }
			c->peer_rows[p] = (u32 *)ptr;
		}
	// everybody must have every mapping, or nobody pushes (a rank that pushes while its peer expects an NCCL receive would hang it)
	CUDA_TRY(cudaMemcpyAsync(c->d_xchg + XCHG_SCRATCH + 6, &opened, sizeof(u64), cudaMemcpyHostToDevice, c->stream));
	NCCL_TRY(g_nccl.AllReduce(c->d_xchg + XCHG_SCRATCH + 6, c->d_xchg + XCHG_SCRATCH + 6, 1, NCCL_UINT64, 3 /*ncclMin*/, c->comm, c->stream));
	CUDA_TRY(cudaMemcpyAsync(&opened, c->d_xchg + XCHG_SCRATCH + 6, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	c->rows_dma = opened != 0;
	if (!c->rows_dma) for (int p = 0; p < G; p++) if (c->peer_rows[p]) { cudaIpcCloseMemHandle(c->peer_rows[p]); c->peer_rows[p] = nullptr; }
	return OGB_OK;
}

// Several ranks: chunk `ci` of every rank's rows (reads [lo_r + ci*chunk, lo_r + (ci+1)*chunk) of rank r) goes to every other
// rank, as one group of point-to-point sends / receives on the exchange stream. Every rank calls this for the same chunk
// grid; a rank whose chunk is empty only receives.
static int exchange_chunk_rows(ogb_context *c, u32 ci, cudaStream_t st)
{
	const int G = c->nranks;
	const u64 per = ((u64)c->n + G - 1) / G;
	auto range = [&](int r, u64 &a, u64 &b) {
		const u64 lo = std::min<u64>(c->n, per * r), hi = std::min<u64>(c->n, per * (r + 1));
		a = std::min(hi, lo + (u64)ci * c->chunk_reads); b = std::min(hi, a + c->chunk_reads);
	};
	u64 ma, mb;
	range(c->rank, ma, mb);
	if (c->rows_dma) {
		// push: one device-to-device copy per peer into its mapped row array (copy engines over NVLink). The peers learn that the
		// rows have landed from the next collective on the main stream (the verdict allgather of ogb_build_graph), which every rank
		// enqueues behind its own pushes.
		for (int k = 1; k < G && mb > ma; k++) {
			const int p = (c->rank + k) % G;
			CUDA_TRY(cudaMemcpyAsync(c->peer_rows[p] + ma * OGB_ROW_W, c->rows.p + ma * OGB_ROW_W, (mb - ma) * OGB_ROW_W * sizeof(u32), cudaMemcpyDeviceToDevice, st));
		}
		return OGB_OK;
	}
	NCCL_TRY(g_nccl.GroupStart());
	for (int p = 0; p < G; p++) {
		if (p == c->rank) continue;
		u64 pa, pb;
		range(p, pa, pb);
		if (mb > ma) NCCL_TRY(g_nccl.Send(c->rows.p + ma * OGB_ROW_W, (mb - ma) * OGB_ROW_W, NCCL_UINT32, p, c->comm, st));
		if (pb > pa) NCCL_TRY(g_nccl.Recv(c->rows.p + pa * OGB_ROW_W, (pb - pa) * OGB_ROW_W, NCCL_UINT32, p, c->comm, st));
	}
	NCCL_TRY(g_nccl.GroupEnd());
	return OGB_OK;
}

// k_probe + k_verify over [lo,hi) in chunks of c->chunk_reads reads, so that the candidate queue of a
// chunk (and the partner strands its probe prefetched) stay L2-resident. The probe of chunk i+1 runs
// on the main stream while the verify of chunk i runs on stream2 (ping-pong queues): the former is
// issue-bound, the latter latency-bound, so they share the SMs well and the launch tails overlap.
// Nothing here synchronises with the host.
template <int MODE> static int scan_chunks(ogb_context *c, u32 lo, u32 hi)
{
	// Partitioned probe over larger chunks (k_window_part + k_probe_parts). Mixed read lengths: the windows are laid out
	// with the stride of the longest read.
	const bool part_mode = c->partitioned && hi > lo;
	const u32 nwin_u = (c->uniform_len ? c->uniform_len : c->max_len) - c->h - 1;
	{
		const char *e = getenv("OGB_CHUNK_READS");                           // experiment knob
		if (e && atoll(e) >= 256 && !part_mode) c->chunk_reads = (u32)std::min<long long>(atoll(e), 1ll << 16);
	}
	if (part_mode) {
		if (!c->part_chunk_set) { const char *e = getenv("OGB_CHUNK_READS"); c->chunk_reads = e && atoll(e) >= 256 ? (u32)std::min<long long>(atoll(e), 1ll << 23) : 3u << 17; c->part_chunk_set = true; }   // 384 k reads per chunk (flat optimum 256 k .. 512 k, profiles/r2/exp_chunk_table.txt)
		c->chunk_reads = (u32)std::max<u64>(256, std::min<u64>(c->chunk_reads, (64ull << 20) / std::max<u32>(nwin_u, 1)));   // <= 64 M windows per chunk (reads up to ~300 bp: the full 256 k reads)
		const u64 pcap = std::min<u64>(c->chunk_reads, hi - lo) * nwin_u / c->nparts * std::min<u64>(c->pq_slack, 4ull * c->nparts) / 4 + 4096;   // a quarter of slack over a perfectly even split at first
		OGB_TRY(c->pq_b.ensure(pcap * c->nparts)); OGB_TRY(c->pq_f.ensure(pcap * c->nparts)); OGB_TRY(c->pq_q.ensure(pcap * c->nparts));
		c->pq_cap = pcap;
	} else
	if (c->chunk_reads > (1u << 16)) c->chunk_reads = 1u << 16;             // k_probe_uniform indexes windows with 32 bits
	{
		// candidate queues (two, ping-pong): ~25 candidates per read at 30x coverage; an overflow halves the chunk and retries
		const u64 want = part_mode ? std::max<u64>(32ull << 20, (u64)c->chunk_reads * 40) : 8ull << 20;
		if (c->cand_cap < want) { OGB_TRY(c->cand_q.ensure(2 * want)); OGB_TRY(c->cand_v.ensure(2 * want)); c->cand_cap = want; }
	}
	int gp = grid_for(c, (const void *)k_probe<MODE>, 256), gv = grid_for(c, (const void *)k_verify<MODE>, 256);
	int gu = grid_for(c, (const void *)k_probe_uniform<MODE>, 256);
	{
		// probe (issue-bound) and verify (latency-bound) of neighbouring chunks are meant to be co-resident:
		// cap the resident blocks per SM of each so that neither grid fills the machine alone
		const char *ep = getenv("OGB_PROBE_BLOCKS_PER_SM"), *ev = getenv("OGB_VERIFY_BLOCKS_PER_SM");
		const int bp = ep ? atoi(ep) : c->probe_blocks_per_sm, bv = ev ? atoi(ev) : c->verify_blocks_per_sm;
		if (bp > 0) { gp = std::min(gp, c->sm_count * bp); gu = std::min(gu, c->sm_count * bp); }
		if (bv > 0) gv = std::min(gv, c->sm_count * bv);
	}
	const bool overlap_streams = getenv("OGB_ONE_STREAM") == nullptr;
	cudaStream_t sv = overlap_streams ? c->stream2 : c->stream;
	ScanArgs a = scan_args(c, lo, hi);
	u32 i = 0;
	// several ranks (overlap pass): every rank walks the same chunk grid -- ceil(reads per rank / chunk) chunks -- so that the row
	// exchanges pair up; the chunks a shorter last shard does not have are empty here
	const bool xchg = MODE == MODE_OVERLAP && c->nranks > 1;
	const u64 per_rank = ((u64)c->n + c->nranks - 1) / c->nranks;
	const u32 n_chunks = (u32)(((xchg ? per_rank : (u64)(hi - lo)) + c->chunk_reads - 1) / c->chunk_reads);
	const GraphView gv_rows = graph_view(c, lo);
	const int g_rows = grid_for(c, (const void *)k_rows_finish<false>, 256);
	// Fused schedule (experiment knob OGB_FUSED=1; the default is the two-stream schedule below): one stream, and from the second
	// chunk on the probe of chunk i and the verification of chunk i-1 are ONE warp-specialised launch (k_probe_verify), so that the
	// two share every SM instead of taking turns. Measured SLOWER (config 3: K3 21.8 ms against 17.2 ms; a fused launch 0.70 ms against
	// 0.30 + 0.30 ms apart): both kernels wait for the same thing -- random accesses beyond the translation reach -- and co-residency
	// only makes their working sets compete (profiles/r2/exp_fused.txt).
	const bool fused = part_mode && getenv("OGB_FUSED") && atoi(getenv("OGB_FUSED")) == 1;
	bool have_prev = false;
	ScanArgs a_prev = a;
	u32 prev_i = 0;
	// rows of a verified chunk on the third stream (+ their exchange on several ranks)
	auto finish_chunk = [&](const ScanArgs &av, u32 ci, cudaStream_t after) -> int {
		if (MODE != MODE_OVERLAP) return OGB_OK;
		CUDA_TRY(cudaEventRecord(c->ev_rows[ci & 1], after));
		CUDA_TRY(cudaStreamWaitEvent(c->xs, c->ev_rows[ci & 1], 0));
		KEV(OGB_KC_ROWS, c->xs, (k_rows_finish<false><<<std::min<int>(g_rows, (int)((av.hi - av.lo + 255) / 256)), 256, 0, c->xs>>>(gv_rows, av.lo, av.hi, c->more_own.p, c->more_cap, c->d_ctr, nullptr, 0)));
		c->launches++;
		if (xchg) {
			const int ke = kev_begin(c, OGB_KC_EXCH_ROWS, c->xs);
			OGB_TRY(exchange_chunk_rows(c, ci, c->xs));
			kev_end(c, ke, c->xs);
		}
		return OGB_OK;
	};
	auto flush_prev = [&]() -> int {                                          // the last verified-later chunk: its verify runs alone
		if (!have_prev) return OGB_OK;
		KEV(MODE == MODE_OVERLAP ? OGB_KC_VERIFY : OGB_KC_CONTAIN_VERIFY, c->stream, (k_verify<MODE><<<gv, 256, 0, c->stream>>>(a_prev)));
		c->launches++;
		have_prev = false;
		return finish_chunk(a_prev, prev_i, c->stream);
	};
	for (; i < n_chunks; i++) {
		const u64 b0 = (u64)lo + (u64)i * c->chunk_reads;
		const int q = i & 1;
		if (b0 >= hi) {                                                        // no reads of this rank in the chunk: only its part of the exchange
			if (fused) OGB_TRY(flush_prev());
			if (xchg) { const int ke = kev_begin(c, OGB_KC_EXCH_ROWS, c->xs); OGB_TRY(exchange_chunk_rows(c, i, c->xs)); kev_end(c, ke, c->xs); }
			continue;
		}
		if (fused) {
			a.lo = (u32)b0; a.hi = (u32)std::min<u64>(hi, b0 + c->chunk_reads);
			a.cand_q = c->cand_q.p + q * c->cand_cap; a.cand_v = c->cand_v.p + q * c->cand_cap; a.cand_cursor = c->d_cursor + q;
			a.prefetch = 0;
			CUDA_TRY(cudaMemsetAsync(a.cand_cursor, 0, sizeof(u64), c->stream));
			CUDA_TRY(cudaMemsetAsync(c->d_pq_cursor, 0, OGB_MAXPART * sizeof(u64), c->stream));
			PartQueue pq;
			pq.b = c->pq_b.p; pq.f = c->pq_f.p; pq.q = c->pq_q.p; pq.cursor = c->d_pq_cursor; pq.cap = c->pq_cap; pq.nparts = c->nparts;
			const u32 nreads = a.hi - a.lo;
			const u64 tiles = ((u64)nreads * nwin_u + 256 * OGB_WPT - 1) / (256 * OGB_WPT);
			const bool uni = c->uniform_len && !a.contained;
			const int gw = grid_for(c, uni ? (const void *)k_window_part<MODE, true> : (const void *)k_window_part<MODE, false>, 256);
			const int kc = MODE == MODE_OVERLAP ? 0 : OGB_KC_CONTAIN_WINDOW - OGB_KC_WINDOW;
			const bool timed = MODE == MODE_OVERLAP && i < 64;
			if (timed) CUDA_TRY(cudaEventRecord(c->ev_pk[2 * i], c->stream));
			if (uni) KEV(OGB_KC_WINDOW + kc, c->stream, (k_window_part<MODE, true><<<(unsigned)std::min<u64>(gw, tiles), 256, 0, c->stream>>>(a, nwin_u, ~0ull / nwin_u + 1, pq)));
			else KEV(OGB_KC_WINDOW + kc, c->stream, (k_window_part<MODE, false><<<(unsigned)std::min<u64>(gw, tiles), 256, 0, c->stream>>>(a, nwin_u, ~0ull / nwin_u + 1, pq)));
			if (timed) CUDA_TRY(cudaEventRecord(c->ev_pm[i], c->stream));
			if (have_prev) {
				KEV(MODE == MODE_OVERLAP ? OGB_KC_PROBE_VERIFY : OGB_KC_CONTAIN_PROBE, c->stream,
				    (k_probe_verify<MODE><<<grid_for(c, (const void *)k_probe_verify<MODE>, 256), 256, 0, c->stream>>>(a, pq, a_prev)));
				OGB_TRY(finish_chunk(a_prev, prev_i, c->stream));
			} else
				KEV(OGB_KC_PROBE + kc, c->stream, (k_probe_parts<MODE><<<grid_for(c, (const void *)k_probe_parts<MODE>, 256), 256, 0, c->stream>>>(a, pq)));
			if (timed) { CUDA_TRY(cudaEventRecord(c->ev_pk[2 * i + 1], c->stream)); c->n_pk = i + 1; }
			c->launches += 2;
			have_prev = true; a_prev = a; prev_i = i;
			continue;
		}
		a.lo = (u32)b0; a.hi = (u32)std::min<u64>(hi, b0 + c->chunk_reads);
		a.cand_q = c->cand_q.p + q * c->cand_cap; a.cand_v = c->cand_v.p + q * c->cand_cap; a.cand_cursor = c->d_cursor + q;
		if (overlap_streams && i >= 2) CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_verify[q], 0));   // queue q is free again
		CUDA_TRY(cudaMemsetAsync(a.cand_cursor, 0, sizeof(u64), c->stream));
		const u32 warps = a.hi - a.lo;
		const bool timed = MODE == MODE_OVERLAP && i < 64;
		if (timed) CUDA_TRY(cudaEventRecord(c->ev_pk[2 * i], c->stream));
		if (part_mode) {
			PartQueue pq;
			pq.b = c->pq_b.p; pq.f = c->pq_f.p; pq.q = c->pq_q.p; pq.cursor = c->d_pq_cursor; pq.cap = c->pq_cap; pq.nparts = c->nparts;
			a.prefetch = 0;
			CUDA_TRY(cudaMemsetAsync(c->d_pq_cursor, 0, OGB_MAXPART * sizeof(u64), c->stream));
			const u64 tiles = ((u64)warps * nwin_u + 256 * OGB_WPT - 1) / (256 * OGB_WPT);
			const bool uni = c->uniform_len && !a.contained;
			const int gw = grid_for(c, uni ? (const void *)k_window_part<MODE, true> : (const void *)k_window_part<MODE, false>, 256), gb = grid_for(c, (const void *)k_probe_parts<MODE>, 256);
			const int kc = MODE == MODE_OVERLAP ? 0 : OGB_KC_CONTAIN_WINDOW - OGB_KC_WINDOW;
			if (uni) KEV(OGB_KC_WINDOW + kc, c->stream, (k_window_part<MODE, true><<<(unsigned)std::min<u64>(gw, tiles), 256, 0, c->stream>>>(a, nwin_u, ~0ull / nwin_u + 1, pq)));
			else KEV(OGB_KC_WINDOW + kc, c->stream, (k_window_part<MODE, false><<<(unsigned)std::min<u64>(gw, tiles), 256, 0, c->stream>>>(a, nwin_u, ~0ull / nwin_u + 1, pq)));
			if (timed) CUDA_TRY(cudaEventRecord(c->ev_pm[i], c->stream));
			KEV(OGB_KC_PROBE + kc, c->stream, (k_probe_parts<MODE><<<gb, 256, 0, c->stream>>>(a, pq)));
			c->launches++;
		} else if (c->uniform_len && !a.contained) {
			const u32 nwin = c->uniform_len - c->h - 1;
			const u64 rounds = ((u64)warps * nwin + 31) / 32;
			KEV(MODE == MODE_OVERLAP ? OGB_KC_PROBE : OGB_KC_CONTAIN_PROBE, c->stream, (k_probe_uniform<MODE><<<(unsigned)std::min<u64>(gu, (rounds * 32 + 255) / 256), 256, 0, c->stream>>>(a, nwin, ~0ull / nwin + 1)));
		} else
			KEV(MODE == MODE_OVERLAP ? OGB_KC_PROBE : OGB_KC_CONTAIN_PROBE, c->stream, (k_probe<MODE><<<(unsigned)std::min<u64>(gp, ((u64)warps * 32 + 255) / 256), 256, 0, c->stream>>>(a)));
		if (timed) { CUDA_TRY(cudaEventRecord(c->ev_pk[2 * i + 1], c->stream)); c->n_pk = i + 1; }
		if (overlap_streams) {
			CUDA_TRY(cudaEventRecord(c->ev_probe[q], c->stream));
			CUDA_TRY(cudaStreamWaitEvent(sv, c->ev_probe[q], 0));
		}
		KEV(MODE == MODE_OVERLAP ? OGB_KC_VERIFY : OGB_KC_CONTAIN_VERIFY, sv, (k_verify<MODE><<<gv, 256, 0, sv>>>(a)));
		if (MODE == MODE_OVERLAP) {
			// rows of the chunk's nodes right behind their verification (slot regions still in L2), on the third stream so that the
			// next verify does not queue behind them; nodes with more edges than slots wait for the heavy pass after K3. Several
			// ranks: the finished rows leave on the same stream.
			CUDA_TRY(cudaEventRecord(c->ev_rows[q], sv));
			CUDA_TRY(cudaStreamWaitEvent(c->xs, c->ev_rows[q], 0));
			KEV(OGB_KC_ROWS, c->xs, (k_rows_finish<false><<<std::min<int>(g_rows, (int)((a.hi - a.lo + 255) / 256)), 256, 0, c->xs>>>(gv_rows, a.lo, a.hi, c->more_own.p, c->more_cap, c->d_ctr, nullptr, 0)));
			c->launches++;
			if (xchg) {
				const int ke = kev_begin(c, OGB_KC_EXCH_ROWS, c->xs);
				OGB_TRY(exchange_chunk_rows(c, i, c->xs));
				kev_end(c, ke, c->xs);
			}
		}
		if (overlap_streams) CUDA_TRY(cudaEventRecord(c->ev_verify[q], sv));
		c->launches += 2;
	}
	if (fused) OGB_TRY(flush_prev());
	if (overlap_streams && !fused)                                           // the main stream continues after every verify
		for (int q = 0; q < 2 && q < (int)i; q++) CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_verify[q], 0));
	if (MODE == MODE_OVERLAP) { CUDA_TRY(cudaEventRecord(c->ev_xs, c->xs)); CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_xs, 0)); }
	CUDA_TRY(cudaGetLastError());
	return OGB_OK;
}

extern "C" int ogb_mark_contained(ogb_context *c)
{
	if (!c) { ogb_set_error("NULL context"); return OGB_E_ARG; }
	if (!c->have_table) { ogb_set_error("ogb_mark_contained: build the hash table first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	OGB_TRY(l2_keep_summary(c, true));
	c->contain_done = true; c->any_contained = false; c->have_graph = false;
	c->st.n_contained = 0; c->st.contain_probes = 0; c->st.contain_hits = 0; c->st.ms_contain = 0;
	OGB_TRY(c->sup.ensure((size_t)c->n + 1));
	CUDA_TRY(cudaMemsetAsync(c->sup.p, 0, ((size_t)c->n + 1) * sizeof(u64), c->stream));
	if (c->n == 0 || c->min_len == c->max_len) { CUDA_TRY(cudaStreamSynchronize(c->stream)); return OGB_OK; }   // OverlapGraph.cpp:228
	OGB_TRY(c->contained.ensure(((size_t)c->n + 31) / 32 + 1));
	u32 lo, hi;
	c->shard(lo, hi);
	CUDA_TRY(cudaEventRecord(c->ev[EV_CONT0], c->stream));
	for (int attempt = 0;; attempt++) {
		if (attempt == 12) { ogb_set_error("ogb_mark_contained: candidate queue kept overflowing"); return OGB_E_CAPACITY; }
		OGB_TRY(ctr_zero(c));
		CUDA_TRY(cudaMemsetAsync(c->sup.p, 0, ((size_t)c->n + 1) * sizeof(u64), c->stream));
		bool saved = c->any_contained;
		c->any_contained = false;
		int rc = scan_chunks<MODE_CONTAIN>(c, lo, hi);
		c->any_contained = saved;
		OGB_TRY(rc);
		OGB_TRY(ctr_fetch(c));
		if (c->h_ctr[CTR_CAND_MAX] > c->cand_cap) { c->chunk_reads = std::max<u32>(256, c->chunk_reads / 2); continue; }
		break;
	}
	c->st.contain_probes = c->h_ctr[CTR_PROBES];
	c->st.contain_hits = c->h_ctr[CTR_CONTAIN_HITS];
	OGB_TRY(ctr_zero(c));
	if (c->nranks > 1) NCCL_TRY(g_nccl.AllReduce(c->sup.p, c->sup.p, c->n, NCCL_UINT64, NCCL_MAX, c->comm, c->stream));   // C0
	k_contained_bitmap<<<(c->n + 255) / 256, 256, 0, c->stream>>>(c->sup.p, c->n, c->contained.p, c->d_ctr);
	CUDA_TRY(cudaGetLastError());
	c->launches++;
	CUDA_TRY(cudaEventRecord(c->ev[EV_CONT1], c->stream));
	OGB_TRY(ctr_fetch(c));
	kev_collect(c);
	c->st.ms_contain = ev_ms(c, EV_CONT0, EV_CONT1);
	c->st.n_contained = c->h_ctr[CTR_N_CONTAINED];
	c->any_contained = c->st.n_contained > 0;
	return OGB_OK;
}

extern "C" int ogb_super_read_ids(ogb_context *c, uint64_t *out, uint64_t cap)
{
	if (!c || !out) { ogb_set_error("ogb_super_read_ids: NULL argument"); return OGB_E_ARG; }
	if (cap < (uint64_t)c->n + 1) { ogb_set_error("ogb_super_read_ids: need %u entries", c->n + 1); return OGB_E_CAPACITY; }
	out[0] = 0;
	if (!c->contain_done || c->n == 0) { for (u32 i = 1; i <= c->n; i++) out[i] = 0; return OGB_OK; }
	CUDA_TRY(cudaSetDevice(c->device));
	CUDA_TRY(cudaMemcpyAsync(out + 1, c->sup.p, (size_t)c->n * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	for (u32 i = 1; i <= c->n; i++) out[i] = out[i] ? (uint64_t)(0xFFFFFFFFu - (u32)(out[i] & 0xFFFFFFFFull)) + 1 : 0;   // idx -> id
	return OGB_OK;
}

// ------------------------------------------------------------------------------------------------
// K3..K6
// ------------------------------------------------------------------------------------------------
static int exclusive_scan(ogb_context *c, const u32 *cnt, u32 n, u64 *out, u64 *d_total, u64 *d_max, u64 *d_more)
{
	u32 nblocks = (n + OGB_SCAN_ITEMS - 1) / OGB_SCAN_ITEMS;
	if (nblocks == 0) nblocks = 1;
	OGB_TRY(c->sums.ensure(nblocks + 1));
	k_scan_sums<<<nblocks, 256, 0, c->stream>>>(cnt, n, c->sums.p, d_max, d_more);
	k_scan_top<<<1, 1024, 0, c->stream>>>(c->sums.p, nblocks, d_total);
	k_scan_apply<<<nblocks, 256, 0, c->stream>>>(cnt, n, c->sums.p, out);
	CUDA_TRY(cudaGetLastError());
	c->launches += 3;
	return OGB_OK;
}

static GraphView graph_view(const ogb_context *c, u32 lo)
{
	GraphView g;
	const u64 per = ((u64)c->n + c->nranks - 1) / c->nranks;
	g.slots = c->slots_e.p; g.deg = c->deg.p; g.ext = c->ext.p; g.lo = lo; g.cap = c->slot_cap;
	g.rows = c->rows.p; g.more = c->nranks > 1 ? c->more.p : c->more_own.p; g.ebits = c->ebits.p;
	g.more_stride = c->more_stride; g.nrows = per * c->nranks;
	g.per_magic = c->nranks > 1 && per > 1 ? ~0ull / per + 1 : 0;          // exact floor(v / per) for 32-bit v (Lemire); per == 1: see rank_of
	g.my_rank = (u32)c->rank;
	return g;
}

// Allgather of per-rank segments of `count[r]` records each: every rank has written its own segment at
// stage + stride*rank; one in-place ncclAllGather at the common stride, then the segments are copied
// down into the contiguous list `out`.
template <class T> static int gather_segments(ogb_context *c, Pool<T> &stage, u64 stride, const std::vector<u64> &count, T *out)
{
	const int G = c->nranks;
	if (stride) NCCL_TRY(g_nccl.AllGather(stage.p + stride * c->rank, stage.p, stride * sizeof(T), NCCL_UINT8, c->comm, c->stream));
	u64 at = 0;
	for (int r = 0; r < G; r++) {
		if (count[r]) CUDA_TRY(cudaMemcpyAsync(out + at, stage.p + stride * r, count[r] * sizeof(T), cudaMemcpyDeviceToDevice, c->stream));
		at += count[r];
	}
	return OGB_OK;
}

extern "C" int ogb_build_graph(ogb_context *c, int keep_pre)
{
	if (!c) { ogb_set_error("NULL context"); return OGB_E_ARG; }
	if (!c->have_table) { ogb_set_error("ogb_build_graph: build the hash table first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	OGB_TRY(l2_keep_summary(c, true));                                      // (a second build on the same index: the first one closed the window)
	// buildOverlapGraphFromHashTable always marks contained reads first (OverlapGraph.cpp:140)
	if (!c->contain_done) OGB_TRY(ogb_mark_contained(c));
	c->have_graph = false; c->have_pre = false; c->have_simplified = false; c->have_spelled = false; c->have_covered = false; c->n_final = 0; c->n_pre = 0;
	const u32 n = c->n;
	if (n == 0) { c->have_graph = true; c->have_pre = keep_pre != 0; c->st.edges_pre = c->st.edges_pre_local = c->st.edges_final = c->st.nodes_final = 0; return OGB_OK; }
	u32 lo, hi;
	c->shard(lo, hi);
	const int G = c->nranks;
	const u64 per = ((u64)n + G - 1) / G;
	const u32 nloc = hi - lo;
	{
		const char *e = getenv("OGB_SLOT_CAP");                              // experiment knob: fixed slots per read
		if (e && atoi(e) >= 8 && atoi(e) <= 256) c->slot_cap = (u32)atoi(e);
	}
	OGB_TRY(c->cnt.ensure(per + 1));
	OGB_TRY(c->cntc.ensure(per + 1));
	OGB_TRY(c->pos.ensure(per + 1));
	OGB_TRY(c->fill.ensure(per + 1));
	OGB_TRY(c->surv.ensure((per + 1) * OGB_SURV));
	OGB_TRY(c->cand.ensure((per + 1) * OGB_SURV * 2));
	if (G > 1 && per * G * OGB_ROW_W + 64 > c->rows.cap && c->rows_shared) {
		// the array is about to be reallocated (on every rank: same size rule): the peers' mappings of the old one go first
		for (int p = 0; p < G; p++) if (c->peer_rows[p]) { cudaIpcCloseMemHandle(c->peer_rows[p]); c->peer_rows[p] = nullptr; }
		c->rows_dma = false; c->rows_shared = nullptr;
		NCCL_TRY(g_nccl.AllReduce(c->d_xchg + XCHG_SCRATCH + 6, c->d_xchg + XCHG_SCRATCH + 6, 1, NCCL_UINT64, 2 /*ncclMax*/, c->comm, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
	}
	OGB_TRY(c->rows.ensure(per * G * OGB_ROW_W + 64));
	OGB_TRY(share_rows(c));
	if (c->ov_q.cap == 0) { OGB_TRY(c->ov_q.ensure(1 << 20)); OGB_TRY(c->ov_e.ensure(1 << 20)); }

	// ---- K3 (probe + verify in chunks) into the slot regions and the adjacency rows; retried with larger pools when a
	// capacity was exceeded. Every decision below derives from values all ranks share.
	CUDA_TRY(cudaEventRecord(c->ev[EV_OVL0], c->stream));
	u64 local_edges = 0, exact_edges = 0, more_need = 0, heavy_max = 0;
	std::vector<u64> seg_cnt(G, 0), hrow_cnt(G, 0);
	for (int attempt = 0;; attempt++) {
		if (attempt == 16) { ogb_set_error("ogb_build_graph: staging pools kept overflowing"); return OGB_E_CAPACITY; }
		OGB_TRY(c->slots_e.ensure(per * c->slot_cap + 64));
		OGB_TRY(c->deg.ensure((size_t)n + 1));
		OGB_TRY(c->ext.ensure(1 << 16));
		if (c->more_cap == 0) c->more_cap = per * 8 + 1024;                  // entries beyond the rows; grows with the need (same value on every rank)
		OGB_TRY(c->more_own.ensure((c->more_cap + 1023) & ~1023ull));      // rounded like the exchange stride: never reallocated after K3 has filled it
		OGB_TRY(ctr_zero(c));
		if (nloc) CUDA_TRY(cudaMemsetAsync(c->deg.p + lo, 0, (size_t)nloc * sizeof(u32), c->stream));
		CUDA_TRY(cudaEventRecord(c->ev[EV_K3A], c->stream));
		OGB_TRY(scan_chunks<MODE_OVERLAP>(c, lo, hi));
		CUDA_TRY(cudaEventRecord(c->ev[EV_K3B], c->stream));
		// edge count, largest degree, entries beyond the 30 a row holds, positions for keep_pre
		OGB_TRY(exclusive_scan(c, c->deg.p + lo, nloc, c->pos.p, c->d_tot, c->d_ctr + CTR_MAX_DEGREE, c->d_ctr + CTR_MORE_NEED));
		CUDA_TRY(cudaMemcpyAsync(&local_edges, c->d_tot, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		OGB_TRY(ctr_fetch(c));
		const u64 n_over = c->h_ctr[CTR_OVERFLOW], n_heavy = c->h_ctr[CTR_BIG_NODES];
		// [0] candidate queue overflowed, [1] spilled edges, [2] largest degree, [3] edges of this rank, [4] words its heavy lists need,
		// [5] a window queue overflowed, [6] entries of this rank beyond the rows, [7] its heavy nodes
		u64 verdict[XCHG_PER_RANK] = {c->h_ctr[CTR_CAND_MAX] > c->cand_cap, n_over, c->h_ctr[CTR_MAX_DEGREE], local_edges, n_over + n_heavy * c->slot_cap, c->h_ctr[CTR_PQ_OVERFLOW] != 0, c->h_ctr[CTR_MORE_NEED], n_heavy};
		more_need = verdict[6]; heavy_max = n_heavy;
		seg_cnt[0] = local_edges; exact_edges = local_edges;
		hrow_cnt.assign(G, 0); hrow_cnt[0] = n_heavy;
		if (G > 1) {
			// one small allgather carries the retry verdicts and the per-rank edge counts
			CUDA_TRY(cudaMemcpyAsync(c->d_xchg + XCHG_PER_RANK * c->rank, verdict, sizeof verdict, cudaMemcpyHostToDevice, c->stream));
			NCCL_TRY(g_nccl.AllGather(c->d_xchg + XCHG_PER_RANK * c->rank, c->d_xchg, XCHG_PER_RANK, NCCL_UINT64, c->comm, c->stream));
			std::vector<u64> all((size_t)XCHG_PER_RANK * G);
			CUDA_TRY(cudaMemcpyAsync(all.data(), c->d_xchg, all.size() * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
			CUDA_TRY(cudaStreamSynchronize(c->stream));
			exact_edges = 0;
			for (int r = 0; r < G; r++) {
				const u64 *v = &all[(size_t)XCHG_PER_RANK * r];
				verdict[0] = std::max(verdict[0], v[0]); verdict[1] = std::max(verdict[1], v[1]); verdict[2] = std::max(verdict[2], v[2]); verdict[5] = std::max(verdict[5], v[5]);
				more_need = std::max(more_need, v[6]); heavy_max = std::max(heavy_max, v[7]);
				seg_cnt[r] = v[3]; exact_edges += v[3]; hrow_cnt[r] = v[7];
			}
		}
		if (verdict[5]) { c->pq_slack *= 2; continue; }                      // a partition's window queue overflowed (skewed keys): more slack, up to everything in one partition
		if (more_need > c->more_cap) { c->more_cap = more_need + more_need / 8 + 1024; continue; }   // the overflow segment was too small for some rank
		if (verdict[0]) { c->chunk_reads = std::max<u32>(256, c->chunk_reads / 2); continue; }
		if (verdict[1] > c->ov_q.cap) {                                      // many heavy nodes: more slots per read, bigger spill list
			if (c->slot_cap < 256) c->slot_cap *= 2;
			else { OGB_TRY(c->ov_q.ensure(verdict[1] + verdict[1] / 8 + 1024)); OGB_TRY(c->ov_e.ensure(verdict[1] + verdict[1] / 8 + 1024)); }
			continue;
		}
		c->st.max_degree = verdict[2];
		c->st.overflow_reads = n_heavy;
		if (verdict[1]) {                                                    // repeats: some rank has nodes with more than slot_cap edges
			OGB_TRY(c->ext.ensure(n_over + n_heavy * c->slot_cap + 64));
			if (n_over) {
				k_heavy_move<<<(nloc + 255) / 256, 256, 0, c->stream>>>(c->slots_e.p, c->deg.p, lo, hi, c->slot_cap, c->ext.p, c->ext.cap, c->fill.p, c->d_ctr);
				k_heavy_place<<<(unsigned)((n_over + 255) / 256), 256, 0, c->stream>>>(c->ov_q.p, c->ov_e.p, n_over, c->slots_e.p, lo, c->slot_cap, c->ext.p, c->fill.p);
				CUDA_TRY(cudaGetLastError());
				c->launches += 2;
			}
		}
		break;
	}
	c->st.overlap_probes = c->h_ctr[CTR_PROBES];
	c->st.probe_sectors = c->h_ctr[CTR_SECTORS];
	c->st.candidates = c->h_ctr[CTR_CANDIDATES];
	c->st.edges_pre_local = local_edges;
	c->st.edges_pre = exact_edges;
	c->n_pre = exact_edges;
	CUDA_TRY(cudaEventRecord(c->ev[EV_OVL1], c->stream));
	OGB_TRY(l2_keep_summary(c, false));                                     // K3 is over: the launches from here on see a plain L2

	// ---- rows of the heavy nodes (their lists are complete only now), then what is left of C1 on several ranks: the heavy
	// rows as (node, row) records and the overflow segments at a common stride. The rows of all other nodes were built and
	// sent chunk by chunk behind k_verify (scan_chunks).
	if (more_need >= (1ull << 32) - 2048) { ogb_set_error("ogb_build_graph: adjacency overflow area too large"); return OGB_E_CAPACITY; }
	c->more_stride = G > 1 ? std::max<u64>(1024, (more_need + 1023) & ~1023ull) : ((c->more_cap + 1023) & ~1023ull);
	if (G > 1) OGB_TRY(c->more.ensure(c->more_stride * G));                  // more_own already holds >= more_stride entries (more_need <= more_cap)
	const u64 nrows = per * G, obit_words = c->more_stride / 32;          // overflow bits: one word-aligned segment per rank
	OGB_TRY(c->ebits.ensure(nrows + obit_words * G + 2));
	CUDA_TRY(cudaMemsetAsync(c->ebits.p + nrows + obit_words * c->rank, 0, obit_words * sizeof(u32), c->stream));
	if (heavy_max) {
		const u64 hstride = heavy_max;
		if (G > 1) OGB_TRY(c->hrows.ensure(hstride * G * OGB_HROW_W));
		u32 *my_h = G > 1 ? c->hrows.p + hstride * c->rank * OGB_HROW_W : nullptr;
		if (nloc && hrow_cnt[c->rank])
			KEV(OGB_KC_ROWS, c->stream, (k_rows_finish<true><<<grid_for(c, (const void *)k_rows_finish<true>, 256), 256, 0, c->stream>>>(graph_view(c, lo), lo, hi, c->more_own.p, c->more_cap, c->d_ctr, my_h, hstride)));
		CUDA_TRY(cudaGetLastError());
		c->launches++;
		if (G > 1) {
			const int ke = kev_begin(c, OGB_KC_EXCH_ROWS, c->stream);
			NCCL_TRY(g_nccl.AllGather(c->hrows.p + hstride * c->rank * OGB_HROW_W, c->hrows.p, hstride * OGB_HROW_W, NCCL_UINT32, c->comm, c->stream));
			kev_end(c, ke, c->stream);
			OGB_TRY(c->sums.ensure(G + 8));
			CUDA_TRY(cudaMemcpyAsync(c->sums.p, hrow_cnt.data(), (size_t)G * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
			k_scatter_hrows<<<c->sm_count, 256, 0, c->stream>>>(c->hrows.p, hstride, c->sums.p, (u32)G, (u32)c->rank, c->rows.p);
			CUDA_TRY(cudaGetLastError());
			c->launches++;
		}
	}
	if (G > 1 && more_need) {
		const int ke = kev_begin(c, OGB_KC_EXCH_ROWS, c->stream);
		NCCL_TRY(g_nccl.AllGather(c->more_own.p, c->more.p, c->more_stride, NCCL_UINT32, c->comm, c->stream));
		kev_end(c, ke, c->stream);
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_XPRE1], c->stream));

	const u32 cap_now = c->slot_cap;
	const int g_emit = grid_for(c, (const void *)k_emit<false>, OGB_WARPS * 32);
	if (keep_pre) {
		// the pre-reduction list as records, in node order (positions = the degree scan above)
		OGB_TRY(c->pre.ensure(std::max<u64>(exact_edges, 1)));
		if (G == 1) {
			k_emit<true><<<g_emit, OGB_WARPS * 32, 0, c->stream>>>(c->slots_e.p, c->ext.p, c->deg.p, nullptr, c->pos.p, c->pre.p, lo, hi, cap_now, 0, 0);
			CUDA_TRY(cudaGetLastError());
		} else {
			u64 stride = 0;
			for (int r = 0; r < G; r++) stride = std::max(stride, seg_cnt[r]);
			stride = (stride + 63) & ~63ull;
			OGB_TRY(c->fin_stage.ensure(std::max<u64>(stride * G, 1)));
			k_emit<true><<<g_emit, OGB_WARPS * 32, 0, c->stream>>>(c->slots_e.p, c->ext.p, c->deg.p, nullptr, c->pos.p, c->fin_stage.p, lo, hi, cap_now, stride * c->rank, 0);
			CUDA_TRY(cudaGetLastError());
			OGB_TRY(gather_segments(c, c->fin_stage, stride, seg_cnt, c->pre.p));
		}
		c->have_pre = true;
	}

	// ---- K5
	MarkArgs m;
	m.G = graph_view(c, lo);
	m.hi = hi; m.cnt = c->cnt.p; m.cntc = c->cntc.p; m.cand = c->cand.p;
	OGB_TRY(c->big.ensure((local_edges + 1) * 3));                          // every edge a candidate of an overfull node: cannot overflow
	m.big = c->big.p; m.big_cap = local_edges + 1;
	if (c->scratch_keys.cap == 0) OGB_TRY(c->scratch_keys.ensure(1 << 20));
	for (int attempt = 0;; attempt++) {
		if (attempt == 4) { ogb_set_error("ogb_build_graph: neighbour-set scratch kept overflowing"); return OGB_E_CAPACITY; }
		OGB_TRY(ctr_zero(c));
		m.scratch_keys = c->scratch_keys.p; m.scratch_cap = c->scratch_keys.cap; m.ctr = c->d_ctr;
		// degree 1..32, 33..64 (edges in registers), the rest (and the few nodes the fast kernels hand over)
		KEV(OGB_KC_MARK1, c->stream, (k_mark_fast<1><<<grid_for(c, (const void *)k_mark_fast<1>, OGB_WARPS * 32), OGB_WARPS * 32, 0, c->stream>>>(m)));
		if (c->st.max_degree > 32) KEV(OGB_KC_MARK2, c->stream, (k_mark_fast<2><<<grid_for(c, (const void *)k_mark_fast<2>, OGB_WARPS * 32), OGB_WARPS * 32, 0, c->stream>>>(m)));
		c->launches += c->st.max_degree > 32 ? 2 : 1;
		KEV(OGB_KC_MARKANY, c->stream, (k_mark_any<<<grid_for(c, (const void *)k_mark_any, OGB_WARPS * 32), OGB_WARPS * 32, 0, c->stream>>>(m)));
		CUDA_TRY(cudaGetLastError());
		c->launches++;
		if (c->st.max_degree * 2 <= OGB_SETCAP) break;                      // no node can have used the scratch pool
		OGB_TRY(ctr_fetch(c));
		if (c->h_ctr[CTR_SCRATCH_FAIL] == 0) break;
		u64 need = c->h_ctr[CTR_SCRATCH_CURSOR] + 1024;                     // a rerun repeats the same verdicts: the bits already set stay valid
		OGB_TRY(c->scratch_keys.ensure(need));
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_MARK1], c->stream));
	if (G > 1) {                                                             // C2: one ELIM bit per entry
		const int ke = kev_begin(c, OGB_KC_EXCH_BITS, c->stream);
		NCCL_TRY(g_nccl.AllGather(c->ebits.p + per * c->rank, c->ebits.p, per, NCCL_UINT32, c->comm, c->stream));
		if (more_need) NCCL_TRY(g_nccl.AllGather(c->ebits.p + nrows + obit_words * c->rank, c->ebits.p + nrows, obit_words, NCCL_UINT32, c->comm, c->stream));
		kev_end(c, ke, c->stream);
	}

	// ---- K6
	const int ke_keep = kev_begin(c, OGB_KC_KEEP, c->stream);
	if (nloc) k_keep<<<(nloc + 255) / 256, 256, 0, c->stream>>>(m, c->surv.p);
	k_keep_big<<<c->sm_count, 256, 0, c->stream>>>(m);
	kev_end(c, ke_keep, c->stream);
	const int ke_emit = kev_begin(c, OGB_KC_EMIT, c->stream);
	CUDA_TRY(cudaGetLastError());
	c->launches += 2;
	OGB_TRY(exclusive_scan(c, c->cnt.p, nloc, c->pos.p, c->d_tot + 1));
	if (G == 1) {
		OGB_TRY(c->fin.ensure(std::max<u64>(exact_edges, 1)));               // E_final <= E_pre: no sync needed to size it
		if (nloc) k_emit_small<<<(nloc + 255) / 256, 256, 0, c->stream>>>(c->surv.p, c->cnt.p, c->cntc.p, c->pos.p, c->fin.p, lo, hi, 0);
		k_emit<false><<<g_emit, OGB_WARPS * 32, 0, c->stream>>>(c->slots_e.p, c->ext.p, c->deg.p, c->cntc.p, c->pos.p, c->fin.p, lo, hi, cap_now, 0, OGB_SURV);
		CUDA_TRY(cudaGetLastError());
		kev_end(c, ke_emit, c->stream);
		c->launches += 2;
		u64 tot = 0;
		CUDA_TRY(cudaMemcpyAsync(&tot, c->d_tot + 1, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		OGB_TRY(ctr_fetch(c));
		c->n_final = tot; c->fin_own_off = 0; c->fin_own_cnt = tot;
	} else {
		// C3: the final edges of every rank's node range (the exchange north_star names). Segment sizes
		// travel first (one word per rank); the segments are emitted at a common stride so that the
		// exchange is one ncclAllGather, then copied down into the contiguous, globally sorted list.
		std::vector<u64> fin_cnt(G, 0), all(G, 0);
		CUDA_TRY(cudaMemcpyAsync(c->d_xchg + c->rank, c->d_tot + 1, sizeof(u64), cudaMemcpyDeviceToDevice, c->stream));
		NCCL_TRY(g_nccl.AllGather(c->d_xchg + c->rank, c->d_xchg, 1, NCCL_UINT64, c->comm, c->stream));
		CUDA_TRY(cudaMemcpyAsync(fin_cnt.data(), c->d_xchg, (size_t)G * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		u64 stride = 0, total = 0;
		for (int r = 0; r < G; r++) { stride = std::max(stride, fin_cnt[r]); total += fin_cnt[r]; }
		stride = (stride + 63) & ~63ull;
		c->n_final = total; c->fin_own_off = 0; for (int r = 0; r < c->rank; r++) c->fin_own_off += fin_cnt[r]; c->fin_own_cnt = fin_cnt[c->rank];
		OGB_TRY(c->fin_stage.ensure(std::max<u64>(stride * G, 1)));
		OGB_TRY(c->fin.ensure(std::max<u64>(total, 1)));
		if (nloc) k_emit_small<<<(nloc + 255) / 256, 256, 0, c->stream>>>(c->surv.p, c->cnt.p, c->cntc.p, c->pos.p, c->fin_stage.p, lo, hi, stride * c->rank);
		k_emit<false><<<g_emit, OGB_WARPS * 32, 0, c->stream>>>(c->slots_e.p, c->ext.p, c->deg.p, c->cntc.p, c->pos.p, c->fin_stage.p, lo, hi, cap_now, stride * c->rank, OGB_SURV);
		CUDA_TRY(cudaGetLastError());
		kev_end(c, ke_emit, c->stream);
		c->launches += 2;
		const int ke_fin = kev_begin(c, OGB_KC_EXCH_FINAL, c->stream);
		OGB_TRY(gather_segments(c, c->fin_stage, stride, fin_cnt, c->fin.p));
		kev_end(c, ke_fin, c->stream);
		NCCL_TRY(g_nccl.AllReduce(c->d_ctr + CTR_NODES_FINAL, c->d_xchg + XCHG_SCRATCH + 2, 1, NCCL_UINT64, 0 /*ncclSum*/, c->comm, c->stream));
		OGB_TRY(ctr_fetch(c));
		CUDA_TRY(cudaMemcpyAsync(&c->h_ctr[CTR_NODES_FINAL], c->d_xchg + XCHG_SCRATCH + 2, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_RED1], c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	kev_collect(c);
	if (c->h_ctr[CTR_ASYMMETRIC]) { ogb_set_error("ogb_build_graph: %llu edges without a twin (internal error)", (unsigned long long)c->h_ctr[CTR_ASYMMETRIC]); return OGB_E_STATE; }
	// next build on these reads: slots sized to the largest degree seen (a collective value: same decision on every rank)
	{
		u32 want = (u32)std::min<u64>(256, std::max<u64>(32, (c->st.max_degree * 5 / 4 + 7) / 8 * 8));
		if (want < c->slot_cap) c->slot_cap = want;
	}
	c->st.pivot_entries = c->h_ctr[CTR_PIVOT_ENTRIES];
	c->st.active_pivots = c->h_ctr[CTR_ACTIVE_PIVOTS];
	c->st.edges_final = c->n_final;
	c->st.nodes_final = c->h_ctr[CTR_NODES_FINAL];
	c->st.ms_overlap = ev_ms(c, EV_OVL0, EV_OVL1);
	c->st.ms_scan_kernel = ev_ms(c, EV_K3A, EV_K3B);
	{
		float sum = 0;
		for (u32 i = 0; i < c->n_pk; i++) { float ms = 0; if (cudaEventElapsedTime(&ms, c->ev_pk[2 * i], c->ev_pk[2 * i + 1]) == cudaSuccess) sum += ms; else cudaGetLastError(); }
		c->st.ms_probe_launch = c->n_pk ? sum / c->n_pk : 0;
		float wsum = 0;
		if (c->partitioned)
			for (u32 i = 0; i < c->n_pk; i++) { float ms = 0; if (cudaEventElapsedTime(&ms, c->ev_pk[2 * i], c->ev_pm[i]) == cudaSuccess) wsum += ms; else cudaGetLastError(); }
		c->st.ms_window_launch = c->n_pk ? wsum / c->n_pk : 0;
		c->st.probe_launches = (nloc + c->chunk_reads - 1) / c->chunk_reads;
	}
	c->st.ms_exchange_pre = ev_ms(c, EV_OVL1, EV_XPRE1);
	c->st.ms_mark = ev_ms(c, EV_XPRE1, EV_MARK1);
	c->st.ms_reduce = ev_ms(c, EV_MARK1, EV_RED1);
	c->st.ms_total = c->st.ms_hash_build + c->st.ms_contain + ev_ms(c, EV_OVL0, EV_RED1);
	c->st.kernel_launches = c->launches;
	c->have_graph = true;
	return OGB_OK;
}

extern "C" int ogb_graph_edge_count(ogb_context *c, int which, uint64_t *n)
{
	if (!c || !n) { ogb_set_error("ogb_graph_edge_count: NULL argument"); return OGB_E_ARG; }
	if (!c->have_graph) { ogb_set_error("ogb_graph_edge_count: build the graph first"); return OGB_E_STATE; }
	if (which == 1 && !c->have_pre) { ogb_set_error("ogb_graph_edge_count: pre-reduction edges were not kept"); return OGB_E_STATE; }
	*n = which ? c->n_pre : c->n_final;
	return OGB_OK;
}

extern "C" int ogb_graph_edges(ogb_context *c, int which, ogb_edge *out, uint64_t cap)
{
	uint64_t n = 0;
	OGB_TRY(ogb_graph_edge_count(c, which, &n));
	if (n == 0) return OGB_OK;
	if (!out || cap < n) { ogb_set_error("ogb_graph_edges: need room for %llu edges", (unsigned long long)n); return OGB_E_CAPACITY; }
	CUDA_TRY(cudaSetDevice(c->device));
	CUDA_TRY(cudaMemcpyAsync(out, which ? c->pre.p : c->fin.p, n * sizeof(ogb_edge), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

// The final edges whose source lies in this rank's node range (one rank: all of them): what a rank hands back to its
// host when the ranks' hosts each continue with their own part.
extern "C" int ogb_graph_edges_shard(ogb_context *c, ogb_edge *out, uint64_t cap, uint64_t *n_out)
{
	if (!c || !n_out) { ogb_set_error("ogb_graph_edges_shard: NULL argument"); return OGB_E_ARG; }
	if (!c->have_graph) { ogb_set_error("ogb_graph_edges_shard: build the graph first"); return OGB_E_STATE; }
	*n_out = c->fin_own_cnt;
	if (c->fin_own_cnt == 0) return OGB_OK;
	if (!out || cap < c->fin_own_cnt) { ogb_set_error("ogb_graph_edges_shard: need room for %llu edges", (unsigned long long)c->fin_own_cnt); return OGB_E_CAPACITY; }
	CUDA_TRY(cudaSetDevice(c->device));
	CUDA_TRY(cudaMemcpyAsync(out, c->fin.p + c->fin_own_off, c->fin_own_cnt * sizeof(ogb_edge), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

extern "C" int ogb_graph_checksum(ogb_context *c, int which, uint64_t *xor_out, uint64_t *sum_out)
{
	uint64_t n = 0;
	OGB_TRY(ogb_graph_edge_count(c, which, &n));
	if (!xor_out || !sum_out) { ogb_set_error("ogb_graph_checksum: NULL argument"); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	CUDA_TRY(cudaMemsetAsync(c->d_xchg + XCHG_SCRATCH + 4, 0, 2 * sizeof(u64), c->stream));
	if (n) k_edge_checksum<<<c->sm_count * 8, 256, 0, c->stream>>>(which ? c->pre.p : c->fin.p, n, c->d_xchg + XCHG_SCRATCH + 4);
	CUDA_TRY(cudaGetLastError());
	u64 h[2] = {0, 0};
	CUDA_TRY(cudaMemcpyAsync(h, c->d_xchg + XCHG_SCRATCH + 4, sizeof h, cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	*xor_out = h[0]; *sum_out = h[1];
	return OGB_OK;
}

// ------------------------------------------------------------------------------------------------
// Simplification (OverlapGraph.cpp:211-215): see ogb_contract.cuh for the formulation.
// ------------------------------------------------------------------------------------------------
static int read_u64(ogb_context *c, const u64 *d, u64 *h, u32 n)
{
	CUDA_TRY(cudaMemcpyAsync(h, d, n * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

extern "C" int ogb_graph_simplify(ogb_context *c, ogb_simplify_stats *stats)
{
	if (!c) { ogb_set_error("ogb_graph_simplify: NULL context"); return OGB_E_ARG; }
	if (!c->have_graph) { ogb_set_error("ogb_graph_simplify: build the graph first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	const u64 ne = c->n_final;
	const u32 n = c->n;
	if (ne >= (1ull << 31) || n >= (1u << 30)) { ogb_set_error("ogb_graph_simplify: %llu edges / %u reads exceed the 31-bit entry and record indices", (unsigned long long)ne, n); return OGB_E_CAPACITY; }
	c->have_simplified = false; c->have_spelled = false; c->have_covered = false;
	ogb_simplify_stats st = {};
	st.n_edges_in = ne;
	const u64 nrec = 2 * ((u64)n + 1);
	OGB_TRY(c->sE.ensure(std::max<u64>(ne, 1))); OGB_TRY(c->s_rec.ensure(nrec)); OGB_TRY(c->s_info.ensure(nrec)); OGB_TRY(c->s_cp.ensure(nrec));
	OGB_TRY(c->s_rowptr.ensure((u64)n + 2)); OGB_TRY(c->s_list.ensure(2 * ((u64)n + 1))); OGB_TRY(c->s_keep.ensure(std::max<u64>(ne, 1))); OGB_TRY(c->s_items.ensure(std::max<u64>(ne, 1)));
	OGB_TRY(c->s_state.ensure((u64)n + 1)); OGB_TRY(c->s_ready.ensure((u64)n + 1)); OGB_TRY(c->s_flag.ensure((u64)n + 2)); OGB_TRY(c->s_blocker.ensure((u64)n + 1));
	OGB_TRY(c->s_epos.ensure(ne + 1)); OGB_TRY(c->s_lpos.ensure(ne + 1)); OGB_TRY(c->s_ctr.ensure(16));
	CGraph G;
	G.E = c->sE.p; G.rowptr = c->s_rowptr.p; G.n = n; G.n_entries = ne; G.rec = c->s_rec.p; G.rec_info = c->s_info.p; G.state = c->s_state.p; G.cp = c->s_cp.p;
	G.meta = c->uniform_len ? nullptr : c->meta.p; G.uniform_len = c->uniform_len; G.blocker = c->s_blocker.p;
	// counters (u64): [0] merges, [1] dead ends, [2] twin / ranking errors, [3] largest list, [4] unfinished ropes, [5] total edges, [6] total items; [8], [9]: the two list cursors (u32)
	u64 *ctr = c->s_ctr.p;
	u32 *cursor = reinterpret_cast<u32 *>(ctr + 8);
	const int grid_max = c->sm_count * 8;
	auto grid = [&](u64 items) { return (unsigned)std::max<u64>(1, std::min<u64>((items + 255) / 256, (u64)grid_max)); };
	CUDA_TRY(cudaEventRecord(c->ev[EV_T0], c->stream));
	CUDA_TRY(cudaMemsetAsync(ctr, 0, 16 * sizeof(u64), c->stream));
	CUDA_TRY(cudaMemsetAsync(c->s_rowptr.p, 0, ((u64)n + 2) * sizeof(u32), c->stream));
	CUDA_TRY(cudaMemsetAsync(c->s_state.p, 0, (u64)n + 1, c->stream));
	k_c_records<<<grid(nrec), 256, 0, c->stream>>>(G);
	st.launches++;
	if (ne) {
		k_c_rowptr<<<grid(ne), 256, 0, c->stream>>>(c->fin.p, ne, n, c->s_rowptr.p);
		k_c_entries<<<grid(ne), 256, 0, c->stream>>>(c->fin.p, G);
		k_c_twins<<<grid(ne), 256, 0, c->stream>>>(c->fin.p, G, ctr + 2);
		st.launches += 3;
	}
	CUDA_TRY(cudaGetLastError());
	u64 h[8];
	OGB_TRY(read_u64(c, ctr, h, 8));
	if (h[2]) { ogb_set_error("ogb_graph_simplify: %llu edges without a twin", (unsigned long long)h[2]); return OGB_E_STATE; }
	u32 *list[2] = {c->s_list.p, c->s_list.p + ((u64)n + 1)};
	cudaEvent_t *tev = c->ev_pk;                                                 // free outside a build: [0] set-up done, then 3 per iteration
	const u32 timed_iterations = 40;
	CUDA_TRY(cudaEventRecord(tev[0], c->stream));
	for (;;) {
		if (ne == 0) break;
		const u32 it = st.iterations++;
		if (it < timed_iterations) CUDA_TRY(cudaEventRecord(tev[1 + 3 * it], c->stream));
		CUDA_TRY(cudaMemsetAsync(ctr, 0, 2 * sizeof(u64), c->stream));
		CUDA_TRY(cudaMemsetAsync(cursor, 0, 2 * sizeof(u32), c->stream));
		k_c_candidates<<<grid(n), 256, 0, c->stream>>>(G, list[0], cursor);
		st.launches++;
		u32 hc[2] = {0, 0};
		CUDA_TRY(cudaMemcpyAsync(hc, cursor, sizeof hc, cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		u32 bound = hc[0];                                                       // what the host knows: an upper bound of the work list's length
		int cur = 0;
		while (bound) {
			// the list's length lives on the device, so a few rounds are queued per host round trip (the list shrinks by ~20 % per round:
			// the grids stay sized for `bound`); a round with an empty list is two empty launches
			const int batch = bound > (1u << 20) ? 2 : (bound > (1u << 16) ? 4 : 8);
			for (int r = 0; r < batch; r++) {
				CUDA_TRY(cudaMemsetAsync(cursor + (cur ^ 1), 0, sizeof(u32), c->stream));
				k_c_ready<<<grid(bound), 256, 0, c->stream>>>(G, list[cur], cursor + cur, c->s_ready.p);
				k_c_turns<<<grid(bound), 256, 0, c->stream>>>(G, list[cur], cursor + cur, c->s_ready.p, list[cur ^ 1], cursor + (cur ^ 1), ctr);
				st.launches += 2; st.rounds++;
				cur ^= 1;
			}
			CUDA_TRY(cudaGetLastError());
			CUDA_TRY(cudaMemcpyAsync(hc, cursor, sizeof hc, cudaMemcpyDeviceToHost, c->stream));
			CUDA_TRY(cudaStreamSynchronize(c->stream));
			if (hc[cur] >= bound) { ogb_set_error("ogb_graph_simplify: contraction rounds made no progress (%u nodes pending)", bound); return OGB_E_STATE; }
			bound = hc[cur];
		}
		if (it < timed_iterations) CUDA_TRY(cudaEventRecord(tev[2 + 3 * it], c->stream));
		k_c_dead_ends<<<grid(n), 256, 0, c->stream>>>(G, c->s_flag.p, ctr);
		k_c_dead_remove<<<grid(n), 256, 0, c->stream>>>(G, c->s_flag.p);
		CUDA_TRY(cudaGetLastError());
		st.launches += 2;
		if (it < timed_iterations) CUDA_TRY(cudaEventRecord(tev[3 + 3 * it], c->stream));
		OGB_TRY(read_u64(c, ctr, h, 2));
		st.merges += h[0]; st.dead_ends += h[1];
		if (h[0] + h[1] == 0) break;                                             // while (counter > 0)  (:215)
	}
	// result: surviving entries in row order, list positions, ropes ranked and written
	u64 n_out = 0, n_items = 0;
	if (ne) {
		k_c_survivors<<<grid(ne), 256, 0, c->stream>>>(G, c->s_keep.p, c->s_items.p, ctr + 3);
		st.launches++;
		OGB_TRY(exclusive_scan(c, c->s_keep.p, (u32)ne, c->s_epos.p, ctr + 5, nullptr, nullptr));
		OGB_TRY(exclusive_scan(c, c->s_items.p, (u32)ne, c->s_lpos.p, ctr + 6, nullptr, nullptr));
		st.launches += 6;
		OGB_TRY(read_u64(c, ctr, h, 8));
		n_out = h[5]; n_items = h[6];
		for (u64 unfinished = n_items ? 1 : 0; unfinished;) {
			if (st.jumps > 40) { ogb_set_error("ogb_graph_simplify: list ranking did not finish"); return OGB_E_STATE; }
			CUDA_TRY(cudaMemsetAsync(ctr + 4, 0, sizeof(u64), c->stream));
			k_c_jump<<<grid(nrec), 256, 0, c->stream>>>(G, ctr + 4);
			CUDA_TRY(cudaGetLastError());
			st.launches++; st.jumps++;
			OGB_TRY(read_u64(c, ctr + 4, &unfinished, 1));
		}
		OGB_TRY(c->s_out.ensure(std::max<u64>(n_out, 1))); OGB_TRY(c->s_out_items.ensure(std::max<u64>(n_items, 1)));
		k_c_emit_edges<<<grid(n), 256, 0, c->stream>>>(G, c->s_keep.p, c->s_epos.p, c->s_lpos.p, c->s_out.p);
		if (n_items) k_c_emit_items<<<grid(nrec), 256, 0, c->stream>>>(G, c->s_lpos.p, c->s_out_items.p, ctr + 2);      // no items: no rope was ranked
		CUDA_TRY(cudaGetLastError());
		st.launches += 2;
		OGB_TRY(read_u64(c, ctr, h, 8));
		if (h[2]) { ogb_set_error("ogb_graph_simplify: %llu list records left unranked", (unsigned long long)h[2]); return OGB_E_STATE; }
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_T1], c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaEventElapsedTime(&st.ms, c->ev[EV_T0], c->ev[EV_T1]));
	CUDA_TRY(cudaEventElapsedTime(&st.ms_setup, c->ev[EV_T0], tev[0]));
	for (u32 it = 0; it < std::min(st.iterations, timed_iterations); it++) {
		float a = 0, b = 0;
		CUDA_TRY(cudaEventElapsedTime(&a, tev[1 + 3 * it], tev[2 + 3 * it]));
		CUDA_TRY(cudaEventElapsedTime(&b, tev[2 + 3 * it], tev[3 + 3 * it]));
		st.ms_sweeps += a; st.ms_dead_ends += b;
	}
	st.ms_lists = st.ms - st.ms_setup - st.ms_sweeps - st.ms_dead_ends;
	st.n_edges_out = n_out; st.n_items = n_items;
	c->sst = st; c->have_simplified = true; c->s_stamp = c->reads_stamp;
	if (stats) *stats = st;
	return OGB_OK;
}

extern "C" int ogb_graph_composite_edges(ogb_context *c, ogb_cedge *edges, uint64_t edge_cap, ogb_clist_item *items, uint64_t item_cap)
{
	if (!c) { ogb_set_error("ogb_graph_composite_edges: NULL context"); return OGB_E_ARG; }
	if (!c->have_simplified) { ogb_set_error("ogb_graph_composite_edges: run ogb_graph_simplify first"); return OGB_E_STATE; }
	const u64 ne = c->sst.n_edges_out, ni = c->sst.n_items;
	if ((ne && (!edges || edge_cap < ne)) || (ni && (!items || item_cap < ni))) {
		ogb_set_error("ogb_graph_composite_edges: need room for %llu edges and %llu list items", (unsigned long long)ne, (unsigned long long)ni);
		return OGB_E_CAPACITY;
	}
	CUDA_TRY(cudaSetDevice(c->device));
	if (ne) CUDA_TRY(cudaMemcpyAsync(edges, c->s_out.p, ne * sizeof(ogb_cedge), cudaMemcpyDeviceToHost, c->stream));
	if (ni) CUDA_TRY(cudaMemcpyAsync(items, c->s_out_items.p, ni * sizeof(ogb_clist_item), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

// ------------------------------------------------------------------------------------------------
// Unitig sequences (OverlapGraph::getStringInEdge, OverlapGraph.cpp:2009): see ogb_spell.cuh.
// ------------------------------------------------------------------------------------------------
static SpellArgs spell_args(const ogb_context *c)
{
	SpellArgs A;
	A.words = c->words.p; A.meta = c->uniform_len ? nullptr : c->meta.p; A.uniform_len = c->uniform_len; A.uniform_pw = c->uniform_pw;
	A.edges = c->s_out.p; A.items = c->s_out_items.p; A.ipos = c->sp_ipos.p; A.rec = c->sp_rec.p; A.n_rec = c->spst.unitigs; A.wpos = c->sp_wpos.p;
	return A;
}

extern "C" int ogb_graph_spell(ogb_context *c, int canonical_only, uint64_t first, uint64_t count, ogb_spell_stats *stats)
{
	if (!c) { ogb_set_error("ogb_graph_spell: NULL context"); return OGB_E_ARG; }
	if (!c->have_simplified || c->s_stamp != c->reads_stamp) { ogb_set_error("ogb_graph_spell: run ogb_graph_simplify on the uploaded reads first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	c->have_spelled = false; c->have_covered = false;
	c->mp_have_index = false; c->mp_samples.clear(); c->mp_n_samples = 0; c->mp_have_profile = false;
	const u64 ne = c->sst.n_edges_out, ni = c->sst.n_items, cap = std::min<u64>(count, ne);
	ogb_spell_stats st = {};
	const int grid_max = c->sm_count * 8;
	auto grid = [&](u64 items) { return (unsigned)std::max<u64>(1, std::min<u64>((items + 255) / 256, (u64)grid_max)); };
	OGB_TRY(c->sp_sel.ensure(std::max<u64>(ne, 1))); OGB_TRY(c->sp_rank.ensure(ne + 1));
	OGB_TRY(c->sp_ioff.ensure(std::max<u64>(ni, 1))); OGB_TRY(c->sp_ipos.ensure(ni + 1));
	OGB_TRY(c->sp_rec.ensure(std::max<u64>(cap, 1))); OGB_TRY(c->sp_nw.ensure(std::max<u64>(cap, 1))); OGB_TRY(c->sp_wpos.ensure(cap + 1));
	OGB_TRY(c->s_ctr.ensure(16));
	u64 *ctr = c->s_ctr.p;
	CUDA_TRY(cudaEventRecord(c->ev[EV_T0], c->stream));
	CUDA_TRY(cudaMemsetAsync(ctr, 0, 2 * sizeof(u64), c->stream));                // [0] selected edges, [1] bases
	CUDA_TRY(cudaMemsetAsync(c->sp_ipos.p + ni, 0, sizeof(u64), c->stream));
	CUDA_TRY(cudaMemsetAsync(c->sp_wpos.p + cap, 0, sizeof(u64), c->stream));
	SpellArgs A = spell_args(c);
	if (ne) {
		k_sp_select<<<grid(ne), 256, 0, c->stream>>>(c->s_out.p, ne, canonical_only, c->sp_sel.p);
		st.launches++;
		OGB_TRY(exclusive_scan(c, c->sp_sel.p, (u32)ne, c->sp_rank.p, ctr, nullptr, nullptr));
		st.launches += 3;
	}
	if (ni) {
		k_sp_item_offsets<<<grid(ni), 256, 0, c->stream>>>(c->s_out_items.p, ni, c->sp_ioff.p);
		st.launches++;
		OGB_TRY(exclusive_scan(c, c->sp_ioff.p, (u32)ni, c->sp_ipos.p, c->sp_ipos.p + ni, nullptr, nullptr));
		st.launches += 3;
	}
	if (cap) {
		CUDA_TRY(cudaMemsetAsync(c->sp_nw.p, 0, cap * sizeof(u32), c->stream));       // the range may end before cap records
		k_sp_records<<<grid(ne), 256, 0, c->stream>>>(A, ne, c->sp_sel.p, c->sp_rank.p, first, cap, c->sp_rec.p, c->sp_nw.p, ctr + 1);
		st.launches++;
		OGB_TRY(exclusive_scan(c, c->sp_nw.p, (u32)cap, c->sp_wpos.p, c->sp_wpos.p + cap, nullptr, nullptr));
		st.launches += 3;
	}
	CUDA_TRY(cudaGetLastError());
	u64 h[3] = {0, 0, 0};
	CUDA_TRY(cudaMemcpyAsync(h, ctr, 2 * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaMemcpyAsync(h + 2, c->sp_wpos.p + cap, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	const u64 n_sel = h[0];
	if (first > n_sel) { ogb_set_error("ogb_graph_spell: first unitig %llu beyond the %llu selected", (unsigned long long)first, (unsigned long long)n_sel); return OGB_E_ARG; }
	st.unitigs = std::min<u64>(cap, n_sel - first);
	st.bases = h[1]; st.words = h[2];
	c->spst = st;
	OGB_TRY(c->sp_words.ensure(st.words + 1));                                    // + one zero word: sp_extract32 reads word w + 1 (ogb_map.cuh)
	CUDA_TRY(cudaMemsetAsync(c->sp_words.p + st.words, 0, sizeof(u64), c->stream));
	if (st.words) {
		A = spell_args(c);
		k_spell_words<<<grid(st.words), 256, 0, c->stream>>>(A, st.words, c->sp_rec.p, c->sp_words.p);
		CUDA_TRY(cudaGetLastError());
		st.launches++;
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_T1], c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	CUDA_TRY(cudaEventElapsedTime(&st.ms, c->ev[EV_T0], c->ev[EV_T1]));
	c->spst = st;
	c->sp_first = first;
	c->have_spelled = true;
	if (stats) *stats = c->spst;
	return OGB_OK;
}

extern "C" int ogb_graph_unitigs(ogb_context *c, ogb_unitig *recs, uint64_t rec_cap, void *out, uint64_t out_cap, int ascii)
{
	if (!c) { ogb_set_error("ogb_graph_unitigs: NULL context"); return OGB_E_ARG; }
	if (!c->have_spelled) { ogb_set_error("ogb_graph_unitigs: run ogb_graph_spell first"); return OGB_E_STATE; }
	const u64 nu = c->spst.unitigs, nw = c->spst.words, bytes = nw * (ascii ? 32 : 8);
	if ((nu && (!recs || rec_cap < nu)) || (bytes && (!out || out_cap < bytes))) {
		ogb_set_error("ogb_graph_unitigs: need room for %llu records and %llu bytes (%llu words%s)", (unsigned long long)nu, (unsigned long long)bytes,
		              (unsigned long long)nw, ascii ? " x 32 ASCII bytes" : "");
		return OGB_E_CAPACITY;
	}
	CUDA_TRY(cudaSetDevice(c->device));
	if (nu) CUDA_TRY(cudaMemcpyAsync(recs, c->sp_rec.p, nu * sizeof(ogb_unitig), cudaMemcpyDeviceToHost, c->stream));
	if (nw && !ascii) CUDA_TRY(cudaMemcpyAsync(out, c->sp_words.p, bytes, cudaMemcpyDeviceToHost, c->stream));
	if (nw && ascii) {
		OGB_TRY(c->sp_ascii.ensure(bytes));
		k_spell_ascii<<<(unsigned)std::min<u64>((nw + 255) / 256, (u64)c->sm_count * 8), 256, 0, c->stream>>>(c->sp_words.p, 0, nw, c->sp_ascii.p);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaMemcpyAsync(out, c->sp_ascii.p, bytes, cudaMemcpyDeviceToHost, c->stream));
	}
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

// The FASTA writer: chunks of OGB_SPELL_CHUNK words are decoded on the device and staged through pinned memory; a record's header is
// written when its first base arrives, so a unitig longer than a chunk spans several.
enum { OGB_SPELL_CHUNK = 1 << 20 };   // 32 MB of ASCII per chunk
extern "C" int ogb_graph_write_unitigs(ogb_context *c, const char *path)
{
	if (!c || !path) { ogb_set_error("ogb_graph_write_unitigs: NULL argument"); return OGB_E_ARG; }
	if (!c->have_spelled) { ogb_set_error("ogb_graph_write_unitigs: run ogb_graph_spell first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	const u64 nu = c->spst.unitigs, nw = c->spst.words, ne = c->sst.n_edges_out;
	std::vector<ogb_unitig> rec(nu);
	std::vector<ogb_cedge> edges(nu ? ne : 0);                                 // for the read counts of the headers
	if (nu) {
		CUDA_TRY(cudaMemcpyAsync(rec.data(), c->sp_rec.p, nu * sizeof(ogb_unitig), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaMemcpyAsync(edges.data(), c->s_out.p, ne * sizeof(ogb_cedge), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
	}
	FILE *f = fopen(path, "wb");
	if (!f) { ogb_set_error("ogb_graph_write_unitigs: cannot open %s for writing", path); return OGB_E_IO; }
	char *stage = nullptr;
	int rc = OGB_OK;
	auto body = [&]() -> int {
		if (!nw) return OGB_OK;
		const u64 chunk = std::min<u64>(nw, OGB_SPELL_CHUNK);
		OGB_TRY(c->sp_ascii.ensure(chunk * 32));
		CUDA_TRY(cudaMallocHost((void **)&stage, chunk * 32));
		u64 r = 0;                                                               // record whose bases come next
		for (u64 w0 = 0; w0 < nw; w0 += chunk) {
			const u64 w1 = std::min(nw, w0 + chunk);
			k_spell_ascii<<<(unsigned)std::min<u64>((w1 - w0 + 255) / 256, (u64)c->sm_count * 8), 256, 0, c->stream>>>(c->sp_words.p, w0, w1, c->sp_ascii.p);
			CUDA_TRY(cudaGetLastError());
			CUDA_TRY(cudaMemcpyAsync(stage, c->sp_ascii.p, (w1 - w0) * 32, cudaMemcpyDeviceToHost, c->stream));
			CUDA_TRY(cudaStreamSynchronize(c->stream));
			const u64 b0 = 32 * w0, b1 = 32 * w1;                                // bases of the word-aligned layout in the stage
			for (; r < nu && rec[r].start < b1; r++) {
				const ogb_unitig &u = rec[r];
				const u64 a = std::max<u64>(u.start, b0), b = std::min<u64>(u.start + u.length, b1);
				if (a == u.start) fprintf(f, ">unitig_%llu src=%u dst=%u orient=%u reads=%u length=%llu\n", (unsigned long long)(c->sp_first + r), u.src, u.dst,
				                           (unsigned)u.orient, edges[u.edge].count + 2, (unsigned long long)u.length);
				if (b > a && fwrite(stage + (a - b0), 1, b - a, f) != b - a) { ogb_set_error("ogb_graph_write_unitigs: write to %s failed", path); return OGB_E_IO; }
				if (u.start + u.length > b1) break;                              // continues in the next chunk
				fputc('\n', f);
			}
		}
		return OGB_OK;
	};
	rc = body();
	if (stage) cudaFreeHost(stage);
	if (fclose(f) != 0 && rc == OGB_OK) { ogb_set_error("ogb_graph_write_unitigs: closing %s failed", path); rc = OGB_E_IO; }
	return rc;
}

// ------------------------------------------------------------------------------------------------
// Unitig coverage: see ogb_coverage.cuh.
// ------------------------------------------------------------------------------------------------
extern "C" int ogb_graph_coverage(ogb_context *c, const uint32_t *freq, uint64_t n, ogb_coverage_stats *stats)
{
	if (!c) { ogb_set_error("ogb_graph_coverage: NULL context"); return OGB_E_ARG; }
	if (!c->have_spelled) { ogb_set_error("ogb_graph_coverage: run ogb_graph_spell on the uploaded reads first"); return OGB_E_STATE; }
	if (n != c->n || (n && !freq)) { ogb_set_error("ogb_graph_coverage: need the frequencies of the %u uploaded reads (got %llu)", c->n, (unsigned long long)(freq ? n : 0)); return OGB_E_ARG; }
	const u64 nu = c->spst.unitigs, nw = c->spst.words, nb = 32 * nw + 1, ni = c->sst.n_items;
	if (nb >= (1ull << 32)) { ogb_set_error("ogb_graph_coverage: %llu bases of layout exceed the 32-bit scan", (unsigned long long)nb); return OGB_E_CAPACITY; }
	CUDA_TRY(cudaSetDevice(c->device));
	c->have_covered = false;
	const u32 nr = c->n;
	const bool locate = c->any_contained && nr;
	ogb_coverage_stats st = {};
	st.unitigs = nu; st.bases = c->spst.bases;
	const int grid_max = c->sm_count * 8;
	auto grid = [&](u64 items) { return (unsigned)std::max<u64>(1, std::min<u64>((items + 255) / 256, (u64)grid_max)); };
	OGB_TRY(c->cv_freq.ensure(std::max<u32>(nr, 1))); OGB_TRY(c->cv_rec.ensure(std::max<u64>(nu, 1))); OGB_TRY(c->cv_np.ensure(std::max<u64>(nu, 1)));
	OGB_TRY(c->cv_ppos.ensure(nu + 1)); OGB_TRY(c->cv_depth.ensure(nb)); OGB_TRY(c->cv_scan.ensure(nb)); OGB_TRY(c->s_ctr.ensure(16));
	if (locate) { OGB_TRY(c->cv_q.ensure(nr)); OGB_TRY(c->cv_cnt.ensure(nr)); OGB_TRY(c->cv_cstart.ensure((u64)nr + 1)); OGB_TRY(c->cv_clist.ensure(nr)); }
	u64 *ctr = c->s_ctr.p;                                                        // [0] unplaced, [1] contained placements, [2] scan total
	CovArgs A;
	A.S = spell_args(c); A.ppos = c->cv_ppos.p; A.freq = c->cv_freq.p;
	A.sup = locate ? c->sup.p : nullptr; A.q = locate ? c->cv_q.p : nullptr; A.cstart = locate ? c->cv_cstart.p : nullptr; A.clist = locate ? c->cv_clist.p : nullptr;
	CUDA_TRY(cudaEventRecord(c->ev[EV_T0], c->stream));
	CUDA_TRY(cudaMemsetAsync(ctr, 0, 3 * sizeof(u64), c->stream));
	if (nr) CUDA_TRY(cudaMemcpyAsync(c->cv_freq.p, freq, (size_t)nr * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
	if (locate) {
		CUDA_TRY(cudaMemsetAsync(c->cv_cnt.p, 0, (size_t)nr * sizeof(u32), c->stream));
		k_cov_locate<<<grid(nr), 256, 0, c->stream>>>(A, nr, c->cv_q.p, c->cv_cnt.p, ctr);
		OGB_TRY(exclusive_scan(c, c->cv_cnt.p, nr, c->cv_cstart.p, c->cv_cstart.p + nr, nullptr, nullptr));
		CUDA_TRY(cudaMemsetAsync(c->cv_cnt.p, 0, (size_t)nr * sizeof(u32), c->stream));          // now the fill cursors
		k_cov_scatter<<<grid(nr), 256, 0, c->stream>>>(c->sup.p, c->cv_q.p, nr, c->cv_cstart.p, c->cv_cnt.p, c->cv_clist.p);
		st.launches += 5;
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_CV1], c->stream));
	CUDA_TRY(cudaMemsetAsync(c->cv_depth.p, 0, nb * sizeof(u32), c->stream));   // the difference array until the scan
	CUDA_TRY(cudaMemsetAsync(c->cv_ppos.p + nu, 0, sizeof(u64), c->stream));
	if (nu) {
		k_cov_init<<<grid(nu), 256, 0, c->stream>>>(c->sp_rec.p, c->s_out.p, nu, c->cv_rec.p, c->cv_np.p);
		OGB_TRY(exclusive_scan(c, c->cv_np.p, (u32)nu, c->cv_ppos.p, c->cv_ppos.p + nu, nullptr, nullptr));
		k_cov_place<<<grid(ni + 2 * nu), 256, 0, c->stream>>>(A, c->cv_ppos.p + nu, c->cv_depth.p, c->cv_rec.p, ctr + 1);
		OGB_TRY(exclusive_scan(c, c->cv_depth.p, (u32)nb, c->cv_scan.p, ctr + 2, nullptr, nullptr));
		st.launches += 8;
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_CV2], c->stream));
	if (nw) {
		k_cov_reduce<<<grid(nw), 256, 0, c->stream>>>(c->cv_scan.p, c->sp_wpos.p, nu, nw, c->cv_depth.p, c->cv_rec.p);
		st.launches++;
	}
	CUDA_TRY(cudaGetLastError());
	CUDA_TRY(cudaEventRecord(c->ev[EV_T1], c->stream));
	u64 h[3] = {0, 0, 0};
	CUDA_TRY(cudaMemcpyAsync(h, ctr, 2 * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaMemcpyAsync(h + 2, c->cv_ppos.p + nu, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	st.unplaced = h[0]; st.contained_placements = h[1]; st.placements = h[2];
	st.ms = ev_ms(c, EV_T0, EV_T1); st.ms_locate = ev_ms(c, EV_T0, EV_CV1); st.ms_depth = ev_ms(c, EV_CV1, EV_CV2); st.ms_reduce = ev_ms(c, EV_CV2, EV_T1);
	c->cvst = st;
	c->have_covered = true;
	if (stats) *stats = st;
	return OGB_OK;
}

extern "C" int ogb_graph_unitig_coverage(ogb_context *c, ogb_unitig_coverage *recs, uint64_t rec_cap, uint32_t *depth, uint64_t depth_cap)
{
	if (!c) { ogb_set_error("ogb_graph_unitig_coverage: NULL context"); return OGB_E_ARG; }
	if (!c->have_covered) { ogb_set_error("ogb_graph_unitig_coverage: run ogb_graph_coverage first"); return OGB_E_STATE; }
	const u64 nu = c->cvst.unitigs, nd = 32 * c->spst.words;
	if ((nu && (!recs || rec_cap < nu)) || (depth && depth_cap < nd)) {
		ogb_set_error("ogb_graph_unitig_coverage: need room for %llu records and %llu depth entries", (unsigned long long)nu, (unsigned long long)nd);
		return OGB_E_CAPACITY;
	}
	CUDA_TRY(cudaSetDevice(c->device));
	if (nu) CUDA_TRY(cudaMemcpyAsync(recs, c->cv_rec.p, nu * sizeof(ogb_unitig_coverage), cudaMemcpyDeviceToHost, c->stream));
	if (depth && nd) CUDA_TRY(cudaMemcpyAsync(depth, c->cv_depth.p, nd * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

extern "C" int ogb_graph_write_coverage(ogb_context *c, const char *path)
{
	if (!c || !path) { ogb_set_error("ogb_graph_write_coverage: NULL argument"); return OGB_E_ARG; }
	if (!c->have_covered) { ogb_set_error("ogb_graph_write_coverage: run ogb_graph_coverage first"); return OGB_E_STATE; }
	CUDA_TRY(cudaSetDevice(c->device));
	const u64 nu = c->cvst.unitigs;
	std::vector<ogb_unitig_coverage> cov(nu);
	std::vector<ogb_unitig> rec(nu);                                           // src, dst
	if (nu) {
		CUDA_TRY(cudaMemcpyAsync(cov.data(), c->cv_rec.p, nu * sizeof(ogb_unitig_coverage), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaMemcpyAsync(rec.data(), c->sp_rec.p, nu * sizeof(ogb_unitig), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
	}
	FILE *f = fopen(path, "wb");
	if (!f) { ogb_set_error("ogb_graph_write_coverage: cannot open %s for writing", path); return OGB_E_IO; }
	fprintf(f, "#name\tsrc\tdst\tlength\treads\tcontained\tread_count\tmean_depth\tsd_depth\tmin_depth\tmax_depth\n");
	for (u64 r = 0; r < nu; r++) {
		const ogb_unitig_coverage &v = cov[r];
		const double len = (double)v.length, mean = (double)v.depth_sum / len;
		const double sd = std::sqrt(std::max(0.0, (double)v.depth_sq_sum / len - mean * mean));
		fprintf(f, "unitig_%llu\t%u\t%u\t%llu\t%u\t%u\t%llu\t%.4f\t%.4f\t%u\t%u\n", (unsigned long long)(c->sp_first + r), rec[r].src, rec[r].dst,
		        (unsigned long long)v.length, v.reads, v.contained, (unsigned long long)v.read_count, mean, sd, v.depth_min, v.depth_max);
	}
	if (ferror(f)) { fclose(f); ogb_set_error("ogb_graph_write_coverage: write to %s failed", path); return OGB_E_IO; }
	if (fclose(f) != 0) { ogb_set_error("ogb_graph_write_coverage: closing %s failed", path); return OGB_E_IO; }
	return OGB_OK;
}

// ------------------------------------------------------------------------------------------------
// Sample mapping: see ogb_map.cuh.
// ------------------------------------------------------------------------------------------------
// Reads per chunk, and bytes per chunk (a bound for long reads): what the sample stage holds on the device at a time
enum { OGB_MAP_CHUNK_READS = 1 << 22 };
static const u64 OGB_MAP_CHUNK_BYTES = 1ull << 30;

static MapArgs map_args(const ogb_context *c)
{
	MapArgs A;
	A.layout = c->sp_words.p; A.wpos = c->sp_wpos.p; A.rec = c->sp_rec.p; A.n_rec = c->spst.unitigs;
	A.K = c->mp_K; A.bmask = c->mp_buckets - 1; A.bstart = c->mp_bstart.p; A.ent = c->mp_ent.p;
	A.rwords = c->mp_words.p; A.rmeta = c->mp_meta.p;
	return A;
}

extern "C" int ogb_graph_map_reads(ogb_context *c, const char *bases, const uint64_t *offsets, uint64_t n, uint32_t *hits, ogb_map_stats *stats)
{
	if (!c) { ogb_set_error("ogb_graph_map_reads: NULL context"); return OGB_E_ARG; }
	if (!c->have_spelled) { ogb_set_error("ogb_graph_map_reads: run ogb_graph_spell on the uploaded reads first"); return OGB_E_STATE; }
	const u64 nu = c->spst.unitigs, nw = c->spst.words, nb = 32 * nw + 1;
	if (nb >= (1ull << 32)) { ogb_set_error("ogb_graph_map_reads: %llu bases of layout exceed the 32-bit positions", (unsigned long long)nb); return OGB_E_CAPACITY; }
	if (n && (!bases || !offsets)) { ogb_set_error("ogb_graph_map_reads: NULL reads"); return OGB_E_ARG; }
	for (u64 i = 0; i < n; i++)
		if (offsets[i + 1] < offsets[i]) { ogb_set_error("ogb_graph_map_reads: offsets decrease at read %llu", (unsigned long long)i); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	c->mp_have_profile = false;
	const u32 m = c->h + 1;
	ogb_map_stats st = {};
	st.reads_in = n; st.sample = c->mp_n_samples;
	const int grid_max = c->sm_count * 8;
	auto grid = [&](u64 items) { return (unsigned)std::max<u64>(1, std::min<u64>((items + 255) / 256, (u64)grid_max)); };
	OGB_TRY(c->mp_ctr.ensure(8)); OGB_TRY(c->mp_rec.ensure(std::max<u64>(nu, 1))); OGB_TRY(c->mp_diff.ensure(nb)); OGB_TRY(c->mp_scan.ensure(nb));
	u64 *ctr = c->mp_ctr.p;                                                       // [0] mapped, [1] multi, [2] placements, [3..4] filter stat, [5] kept, [6] scan total
	CUDA_TRY(cudaEventRecord(c->ev[EV_T0], c->stream));
	// ---- index over the layout, once per spell
	const bool build_index = !c->mp_have_index;
	if (build_index) {
		c->mp_K = std::min<u32>(32, m + 1);
		c->mp_buckets = mp_buckets(c->spst.bases);
		OGB_TRY(c->mp_cnt.ensure(c->mp_buckets)); OGB_TRY(c->mp_bstart.ensure(c->mp_buckets + 1)); OGB_TRY(c->mp_ent.ensure(std::max<u64>(c->spst.bases, 1)));
		CUDA_TRY(cudaMemsetAsync(c->mp_cnt.p, 0, c->mp_buckets * sizeof(u32), c->stream));
		MapArgs A = map_args(c);
		if (nw) k_map_count<<<grid(nw), 256, 0, c->stream>>>(A, nw, c->mp_cnt.p);
		OGB_TRY(exclusive_scan(c, c->mp_cnt.p, (u32)c->mp_buckets, c->mp_bstart.p, c->mp_bstart.p + c->mp_buckets, nullptr, nullptr));
		CUDA_TRY(cudaMemsetAsync(c->mp_cnt.p, 0, c->mp_buckets * sizeof(u32), c->stream));      // now the fill cursors
		if (nw) k_map_fill<<<grid(nw), 256, 0, c->stream>>>(A, nw, c->mp_cnt.p, c->mp_ent.p);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaMemcpyAsync(&c->mp_entries, c->mp_bstart.p + c->mp_buckets, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		st.launches += nw ? 5 : 3;
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_MP0], c->stream));
	CUDA_TRY(cudaMemsetAsync(ctr, 0, 8 * sizeof(u64), c->stream));
	CUDA_TRY(cudaMemsetAsync(c->mp_diff.p, 0, nb * sizeof(u32), c->stream));     // the difference array until the scan
	if (nu) { k_cov_init<<<grid(nu), 256, 0, c->stream>>>(c->sp_rec.p, c->s_out.p, nu, c->mp_rec.p, nullptr); st.launches++; }
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	c->mp_have_index = true;
	// ---- the sample, chunk by chunk
	for (u64 c0 = 0; c0 < n;) {
		u64 c1 = c0 + 1;
		while (c1 < n && c1 - c0 < OGB_MAP_CHUNK_READS && offsets[c1 + 1] - offsets[c0] <= OGB_MAP_CHUNK_BYTES) c1++;
		const u32 nc = (u32)(c1 - c0);
		const u64 nbytes = offsets[c1] - offsets[c0];
		std::vector<u64> rel(nc + 1);
		for (u32 i = 0; i <= nc; i++) rel[i] = offsets[c0 + i] - offsets[c0];
		OGB_TRY(c->mp_raw.ensure(nbytes + 1)); OGB_TRY(c->mp_roffs.ensure(nc + 1)); OGB_TRY(c->mp_good.ensure(nc)); OGB_TRY(c->mp_pos.ensure(nc));
		OGB_TRY(c->mp_start.ensure(nc)); OGB_TRY(c->mp_len.ensure(nc)); OGB_TRY(c->mp_khits.ensure(nc)); OGB_TRY(c->mp_meta.ensure(nc + 1));
		CUDA_TRY(cudaEventRecord(c->ev[EV_MP1], c->stream));
		CUDA_TRY(cudaMemcpyAsync(c->mp_raw.p, bases + offsets[c0], nbytes, cudaMemcpyHostToDevice, c->stream));
		CUDA_TRY(cudaMemcpyAsync(c->mp_roffs.p, rel.data(), (nc + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		const u64 stat[2] = {~0ull, 0};
		CUDA_TRY(cudaMemcpyAsync(ctr + 3, stat, sizeof stat, cudaMemcpyHostToDevice, c->stream));
		k_ds_filter<<<(nc + 127) / 128, 128, 0, c->stream>>>(c->mp_raw.p, c->mp_roffs.p, nc, m, c->mp_good.p, ctr + 3);
		OGB_TRY(exclusive_scan(c, c->mp_good.p, nc, c->mp_pos.p, ctr + 5));
		u64 h[3];
		CUDA_TRY(cudaMemcpyAsync(h, ctr + 3, 3 * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		const u32 kept = (u32)h[2], max_pw = kept ? ((u32)(h[1] + 63) >> 6) << 1 : 0;
		st.filtered += nc - kept;
		st.launches += 4;
		if (kept) {
			// the chunk's read store: 2 pw words per read <= 4 (nbytes / 64 + kept), + the words a strand's last extract may touch
			OGB_TRY(c->mp_words.ensure(4 * (nbytes / 64 + kept) + 8));
			k_ds_compact<<<(nc + 255) / 256, 256, 0, c->stream>>>(c->mp_good.p, c->mp_pos.p, c->mp_roffs.p, nc, c->mp_start.p, c->mp_len.p);
			k_map_geom<<<grid(kept), 256, 0, c->stream>>>(c->mp_len.p, kept, c->mp_khits.p);                 // (khits: scratch until k_map_reads)
			OGB_TRY(exclusive_scan(c, c->mp_khits.p, kept, c->mp_meta.p, c->mp_meta.p + kept));
			k_map_meta<<<grid(kept), 256, 0, c->stream>>>(c->mp_len.p, kept, c->mp_meta.p);
			k_pack_ascii<<<(unsigned)(((u64)kept * max_pw + 255) / 256), 256, 0, c->stream>>>(c->mp_raw.p, c->mp_start.p, c->mp_words.p, c->mp_meta.p, kept, 0, 0, max_pw);
			st.launches += 7;
		}
		CUDA_TRY(cudaEventRecord(c->ev[EV_MP2], c->stream));
		if (kept) {
			k_map_reads<<<grid(kept), 256, 0, c->stream>>>(map_args(c), kept, c->mp_diff.p, c->mp_rec.p, c->mp_khits.p, ctr);
			st.launches++;
		}
		if (hits) {
			OGB_TRY(c->mp_hits.ensure(nc));
			k_map_hits<<<grid(nc), 256, 0, c->stream>>>(c->mp_good.p, c->mp_pos.p, c->mp_khits.p, nc, c->mp_hits.p);
			CUDA_TRY(cudaMemcpyAsync(hits + c0, c->mp_hits.p, (size_t)nc * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
			st.launches++;
		}
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaEventRecord(c->ev[EV_MP3], c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		st.ms_upload += ev_ms(c, EV_MP1, EV_MP2); st.ms_map += ev_ms(c, EV_MP2, EV_MP3);
		c0 = c1;
	}
	// ---- depth
	CUDA_TRY(cudaEventRecord(c->ev[EV_MP4], c->stream));
	if (nu) {
		OGB_TRY(exclusive_scan(c, c->mp_diff.p, (u32)nb, c->mp_scan.p, ctr + 6, nullptr, nullptr));
		k_cov_reduce<<<grid(nw), 256, 0, c->stream>>>(c->mp_scan.p, c->sp_wpos.p, nu, nw, c->mp_diff.p, c->mp_rec.p);
		CUDA_TRY(cudaGetLastError());
		st.launches += 4;
	}
	CUDA_TRY(cudaEventRecord(c->ev[EV_T1], c->stream));
	const size_t old = c->mp_samples.size();
	c->mp_samples.resize(old + nu);
	if (nu) CUDA_TRY(cudaMemcpyAsync(c->mp_samples.data() + old, c->mp_rec.p, nu * sizeof(ogb_unitig_coverage), cudaMemcpyDeviceToHost, c->stream));
	u64 h[3];
	CUDA_TRY(cudaMemcpyAsync(h, ctr, 3 * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
	const cudaError_t e = cudaStreamSynchronize(c->stream);
	if (e != cudaSuccess) { c->mp_samples.resize(old); CUDA_TRY(e); }
	st.mapped = h[0]; st.multi = h[1]; st.placements = h[2];
	st.index_entries = c->mp_entries; st.index_buckets = c->mp_buckets;
	st.ms = ev_ms(c, EV_T0, EV_T1); st.ms_index = build_index ? ev_ms(c, EV_T0, EV_MP0) : 0.f; st.ms_reduce = ev_ms(c, EV_MP4, EV_T1);
	c->mp_n_samples++;
	c->mp_have_profile = true;
	if (stats) *stats = st;
	return OGB_OK;
}

extern "C" int ogb_graph_sample_coverage(ogb_context *c, uint32_t sample, ogb_unitig_coverage *recs, uint64_t rec_cap, uint32_t *depth, uint64_t depth_cap)
{
	if (!c) { ogb_set_error("ogb_graph_sample_coverage: NULL context"); return OGB_E_ARG; }
	if (!c->have_spelled || !c->mp_n_samples) { ogb_set_error("ogb_graph_sample_coverage: no sample mapped since the last ogb_graph_spell"); return OGB_E_STATE; }
	if (sample >= c->mp_n_samples) { ogb_set_error("ogb_graph_sample_coverage: sample %u of %u", sample, c->mp_n_samples); return OGB_E_ARG; }
	if (depth && (sample + 1 != c->mp_n_samples || !c->mp_have_profile)) { ogb_set_error("ogb_graph_sample_coverage: the profile is kept for the last sample only"); return OGB_E_ARG; }
	const u64 nu = c->spst.unitigs, nd = 32 * c->spst.words;
	if ((nu && (!recs || rec_cap < nu)) || (depth && depth_cap < nd)) {
		ogb_set_error("ogb_graph_sample_coverage: need room for %llu records and %llu depth entries", (unsigned long long)nu, (unsigned long long)nd);
		return OGB_E_CAPACITY;
	}
	if (nu) memcpy(recs, c->mp_samples.data() + (size_t)sample * nu, nu * sizeof(ogb_unitig_coverage));
	if (depth && nd) {
		CUDA_TRY(cudaSetDevice(c->device));
		CUDA_TRY(cudaMemcpyAsync(depth, c->mp_diff.p, nd * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
	}
	return OGB_OK;
}

extern "C" int ogb_graph_write_depths(ogb_context *c, const char *path, const char *const *names)
{
	if (!c || !path) { ogb_set_error("ogb_graph_write_depths: NULL argument"); return OGB_E_ARG; }
	if (!c->have_spelled || !c->mp_n_samples) { ogb_set_error("ogb_graph_write_depths: no sample mapped since the last ogb_graph_spell"); return OGB_E_STATE; }
	const u32 ns = c->mp_n_samples;
	std::vector<std::string> nm(ns);
	for (u32 j = 0; j < ns; j++) {
		if (!names) { nm[j] = "sample_" + std::to_string(j); continue; }
		if (!names[j] || strpbrk(names[j], "\t\n\r")) { ogb_set_error("ogb_graph_write_depths: sample name %u is NULL or holds a tab or a newline", j); return OGB_E_ARG; }
		nm[j] = names[j];
	}
	const u64 nu = c->spst.unitigs;
	FILE *f = fopen(path, "wb");
	if (!f) { ogb_set_error("ogb_graph_write_depths: cannot open %s for writing", path); return OGB_E_IO; }
	fprintf(f, "contigName\tcontigLen\ttotalAvgDepth");
	for (u32 j = 0; j < ns; j++) fprintf(f, "\t%s\t%s-var", nm[j].c_str(), nm[j].c_str());
	fputc('\n', f);
	std::vector<double> mean(ns), var(ns);
	for (u64 r = 0; r < nu; r++) {
		const double len = (double)c->mp_samples[r].length;
		double total = 0;
		for (u32 j = 0; j < ns; j++) {
			const ogb_unitig_coverage &v = c->mp_samples[(size_t)j * nu + r];
			mean[j] = (double)v.depth_sum / len;
			var[j] = std::max(0.0, (double)v.depth_sq_sum / len - mean[j] * mean[j]);
			total += mean[j];
		}
		fprintf(f, "unitig_%llu\t%llu\t%.4f", (unsigned long long)(c->sp_first + r), (unsigned long long)c->mp_samples[r].length, total);
		for (u32 j = 0; j < ns; j++) fprintf(f, "\t%.4f\t%.4f", mean[j], var[j]);
		fputc('\n', f);
	}
	if (ferror(f)) { fclose(f); ogb_set_error("ogb_graph_write_depths: write to %s failed", path); return OGB_E_IO; }
	if (fclose(f) != 0) { ogb_set_error("ogb_graph_write_depths: closing %s failed", path); return OGB_E_IO; }
	return OGB_OK;
}

extern "C" int ogb_get_stats(ogb_context *c, ogb_stats *out)
{
	if (!c || !out) { ogb_set_error("ogb_get_stats: NULL argument"); return OGB_E_ARG; }
	*out = c->st;
	return OGB_OK;
}

extern "C" int ogb_timer_begin(ogb_context *c)
{
	if (!c) { ogb_set_error("NULL context"); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	CUDA_TRY(cudaEventRecord(c->ev[EV_T0], c->stream));
	return OGB_OK;
}

extern "C" int ogb_timer_end(ogb_context *c, float *ms)
{
	if (!c || !ms) { ogb_set_error("ogb_timer_end: NULL argument"); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	CUDA_TRY(cudaEventRecord(c->ev[EV_T1], c->stream));
	CUDA_TRY(cudaEventSynchronize(c->ev[EV_T1]));
	CUDA_TRY(cudaEventElapsedTime(ms, c->ev[EV_T0], c->ev[EV_T1]));
	return OGB_OK;
}

extern "C" int ogb_l2_flush(ogb_context *c, size_t bytes)
{
	if (!c) { ogb_set_error("NULL context"); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	OGB_TRY(c->flush.ensure(bytes));
	CUDA_TRY(cudaMemsetAsync(c->flush.p, 0x5a, bytes, c->stream));
	CUDA_TRY(cudaStreamSynchronize(c->stream));
	return OGB_OK;
}

extern "C" int ogb_gather_ceiling(ogb_context *c, size_t buffer_bytes, uint32_t gather_bytes, double *gb_per_s)
{
	if (!c || !gb_per_s) { ogb_set_error("ogb_gather_ceiling: NULL argument"); return OGB_E_ARG; }
	if (gather_bytes != 32 && gather_bytes != 64 && gather_bytes != 128) { ogb_set_error("ogb_gather_ceiling: gather_bytes must be 32, 64 or 128"); return OGB_E_ARG; }
	if (buffer_bytes < (1u << 20) || (buffer_bytes & (buffer_bytes - 1))) { ogb_set_error("ogb_gather_ceiling: buffer_bytes must be a power of two >= 1 MiB"); return OGB_E_ARG; }
	CUDA_TRY(cudaSetDevice(c->device));
	OGB_TRY(c->flush.ensure(buffer_bytes));
	CUDA_TRY(cudaMemsetAsync(c->flush.p, 1, buffer_bytes, c->stream));
	const u64 nblocks = buffer_bytes / gather_bytes;
	const u32 per_thread = 256;
	const int grid = c->sm_count * 8;
	float best = 1e30f;
	for (int rep = 0; rep < 4; rep++) {
		CUDA_TRY(cudaEventRecord(c->ev[EV_T0], c->stream));
		if (gather_bytes == 32) k_gather_ceiling<32><<<grid, 256, 0, c->stream>>>((const u64 *)c->flush.p, nblocks, per_thread, c->d_tot);
		else if (gather_bytes == 64) k_gather_ceiling<64><<<grid, 256, 0, c->stream>>>((const u64 *)c->flush.p, nblocks, per_thread, c->d_tot);
		else k_gather_ceiling<128><<<grid, 256, 0, c->stream>>>((const u64 *)c->flush.p, nblocks, per_thread, c->d_tot);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaEventRecord(c->ev[EV_T1], c->stream));
		CUDA_TRY(cudaEventSynchronize(c->ev[EV_T1]));
		float ms = 0;
		CUDA_TRY(cudaEventElapsedTime(&ms, c->ev[EV_T0], c->ev[EV_T1]));
		if (rep && ms < best) best = ms;                                      // the first run warms the TLBs
	}
	*gb_per_s = (double)grid * 256 * per_thread * gather_bytes / (best * 1e-3) / 1e9;
	return OGB_OK;
}

// Dataset::storeMatePairInformation for a batch of sequences (see k_mate_lookup). Needs the reads, the index and the
// containment marks of the same context (the reference calls it at OverlapGraph.cpp:142, between markContainedReads and the
// edge build, for that reason).
extern "C" int ogb_mate_lookup(ogb_context *c, const char *bases, const uint64_t *offsets, uint64_t n_seqs, uint32_t min_overlap, uint32_t *out_id, uint8_t *out_orient)
{
	if (!c || (n_seqs && (!bases || !offsets || !out_id || !out_orient))) { ogb_set_error("ogb_mate_lookup: NULL argument"); return OGB_E_ARG; }
	if (!c->have_table || !c->contain_done) { ogb_set_error("ogb_mate_lookup: build the hash table and mark contained reads first"); return OGB_E_STATE; }
	if (n_seqs == 0) return OGB_OK;
	CUDA_TRY(cudaSetDevice(c->device));
	const u64 nbytes = offsets[n_seqs] - offsets[0];
	Tmp<char> d_bases;
	Tmp<u64> d_offs;
	Tmp<u32> d_id;
	Tmp<unsigned char> d_or;
	std::vector<u64> rel;
	const u64 *offs_src = (const u64 *)offsets;
	if (offsets[0] != 0) { rel.resize(n_seqs + 1); for (u64 i = 0; i <= n_seqs; i++) rel[i] = offsets[i] - offsets[0]; offs_src = rel.data(); }
	auto run = [&]() -> int {
		OGB_TRY(d_bases.ensure(nbytes + 1, c->stream)); OGB_TRY(d_offs.ensure(n_seqs + 1, c->stream));
		OGB_TRY(d_id.ensure(n_seqs, c->stream)); OGB_TRY(d_or.ensure(n_seqs, c->stream));
		CUDA_TRY(cudaMemcpyAsync(d_bases.p, bases + offsets[0], nbytes, cudaMemcpyHostToDevice, c->stream));
		CUDA_TRY(cudaMemcpyAsync(d_offs.p, offs_src, (n_seqs + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
		k_mate_lookup<<<(unsigned)((n_seqs + 127) / 128), 128, 0, c->stream>>>(c->rs(), c->tb(), c->any_contained ? c->sup.p : nullptr, d_bases.p, d_offs.p, n_seqs, min_overlap, d_id.p, d_or.p);
		CUDA_TRY(cudaGetLastError());
		CUDA_TRY(cudaMemcpyAsync(out_id, d_id.p, n_seqs * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaMemcpyAsync(out_orient, d_or.p, n_seqs, cudaMemcpyDeviceToHost, c->stream));
		CUDA_TRY(cudaStreamSynchronize(c->stream));
		return OGB_OK;
	};
	const int rc = run();
	d_bases.release(); d_offs.release(); d_id.release(); d_or.release();
	return rc;
}

#!/usr/bin/env python
"""bench.py -- overlap-graph build throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 3] [--scale 1.0] [--dump-outputs DIR]

Workload: BASELINE.json configs[2] (config 3: 20-genome mock metagenome, 10 M x 100 bp reads, minOverlap 50) -- the
largest configuration one GPU holds; N GPUs build config 3 at N times the genomes and reads (weak scaling, N x 10 M reads).
configs 1, 2, 4, 5 are parity-test cases (tests/test_gpu_full_size.py, tests/test_multi_gpu.py), selectable with --config.

A *step* is one pass of the hot path with the packed reads already resident in HBM: K1 hash build -> K2 containment
(skipped for one read length, like the reference) -> K3 window scan + verification -> adjacency rows -> K5 transitive
marking -> K6 twin verdicts + compaction (+ the NCCL exchanges on N > 1). `value` = unique reads / device time of a step
(CUDA events on the library's stream, mean of K steps, max over ranks), L2 flushed between steps. `e2e` is the same
metric through the public C ABI with HOST buffers: H2D of the packed reads from pinned memory (N > 1: every rank its own
shard, replicated over NVLink) + build + D2H of the final edges (N > 1: every rank its own node range), every step.
`parity` compares the result of the timed configuration -- counters and an order-independent checksum of the final edge
set -- with the oracle's golden in tests/golden/full_size.json. `roofline` is the dominant kernel of the step, measured
live with CUDA event pairs around every launch; `kernels` has every kernel class; `roofline_step` the whole step against
SURVEY.md 8(d)'s algorithmic bytes. `cpu_baseline` times the reference's own CPU implementation (oracle/_ref/ref_overlap,
the unmodified reference) on a bounded sample.

--impl reference runs that CPU implementation as the measured arm (rank 0 only; this arm never imports the package or
maps libogb.so: the sample is generated with numpy and the reference runs as a subprocess).

--dump-outputs DIR writes what the last timed step computed, as a caller of the build receives it, to DIR/<name>.npy (rank 0,
float64, < 64 MB in all): edges.npy (k, 4) [src, dst, offset, orient] rows of the final edge list in its canonical order (all
rows, or a seeded sample of 2^20 row positions in ascending order), super_read_ids.npy (superReadID of reads 1..n, or a seeded
sample of 2^21 of them), edge_checksum.npy (the device's order-independent [xor, sum] over every final edge, each 64-bit word
as four 16-bit limbs, low first) and counts.npy [unique reads, pre-reduction edges, final edges, nodes, contained reads].
The inputs are seeded: the same arguments give the same inputs on every run, so two builds can be compared file by file.
The bench reads the tree as __graft_entry__.build() left it and writes nothing there.
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True        # the tree may be read-only: no __pycache__ next to the modules imported below
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "overlap_graph_build_reads_per_sec"
UNIT = "reads/s"
SECTOR = 32           # bytes per probed window (SURVEY.md 8(d): S)
EDGE_BYTES = 8        # device edge word; SURVEY.md's B_e = 16 is used for roofline_step
CPU_SAMPLE_SCALE = {1: 1.0, 2: 0.12, 3: 0.015, 4: 0.004, 5: 0.08}   # bounded sample: ~5-30 s of the single-core reference
NAMES = {1: "config1: 100 kb genome, 10k x 100 bp, minOverlap 40",
         2: "config2: 5 Mb genome, 30x, 1.5M x 100 bp paired-end, minOverlap 50",
         3: "config3: 20 genomes log-normal abundance, 10M x 100 bp, minOverlap 50",
         4: "config4: 200 genomes, 50M x 150 bp, minOverlap 60",
         5: "config5: containment/duplication stress, mixed 75-250 bp, 20% duplicate+contained, minOverlap 50"}
MIN_OVERLAP = {1: 40, 2: 50, 3: 50, 4: 60, 5: 50}


def workload_name(cfg_id, scale, n_gpus):
    return NAMES[cfg_id] + (f" x{n_gpus} (weak scaling: {n_gpus}x genomes and reads)" if n_gpus > 1 else "") + (f" [scale {scale}]" if scale != 1.0 else "")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md): a thread polling NVML every 2 ms
    (the timed region of this bench lasts well under a second -- `nvidia-smi -lms` would not produce a line in time)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, device):
        self.sm, self.mask, self.h, self.nv, self.run, self.mx = [], 0, None, None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _reasons(self):
        for name in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            f = getattr(self.nv, name, None)
            if f is not None:
                try:
                    return int(f(self.h))
                except Exception:
                    pass
        return 0

    def _poll(self):
        while self.run:
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.mask |= self._reasons()
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.h is None:
            return
        self.run = True
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self.run = False
        self.t.join(timeout=2)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                "reasons": sorted(v for k, v in self.REASONS.items() if self.mask & k), "samples": len(self.sm)}


# ------------------------------------------------------------------------------------------------------------------
# Reference arm / cpu_baseline: the unmodified reference on a bounded sample of the workload
# ------------------------------------------------------------------------------------------------------------------
_COMP = np.zeros(256, dtype=np.uint8)
for _a, _c in zip(b"ACGT", b"TGCA"):
    _COMP[_a] = _c


def numpy_sample(cfg_id, scale, seed=None):
    """A sample of configuration cfg_id at `scale` (genome lengths and read counts scaled together: the coverage -- hence
    degree, hit rate and bytes per read -- stays that of the named configuration), generated with numpy only: the same
    read model as metagenomics_b200/synth.py (uniform random genomes, uniform read starts, strand flipped with p = 0.5,
    error-free; config 2 paired with inserts ~ N(300, 30); configs 3/4 log-normal abundance; config 5 mixed lengths with
    20 % derived reads). Returns (list of uint8 read arrays or an (n, L) uint8 matrix, paired)."""
    rng = np.random.default_rng(1000 + cfg_id if seed is None else seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)

    def genome(n):
        return acgt[rng.integers(0, 4, int(n))]

    def uniform_reads(gs, weights, n, L):
        glen = np.array([len(g) for g in gs], dtype=np.float64)
        p = weights * glen
        which = rng.choice(len(gs), size=n, p=p / p.sum())
        out = np.empty((n, L), dtype=np.uint8)
        for gi, g in enumerate(gs):
            idx = np.nonzero(which == gi)[0]
            if len(idx) == 0:
                continue
            st = rng.integers(0, len(g) - L + 1, len(idx))
            out[idx] = g[st[:, None] + np.arange(L)[None, :]]
        flip = rng.integers(0, 2, n).astype(bool)
        out[flip] = _COMP[out[flip][:, ::-1]]
        return out

    s = float(scale)
    if cfg_id == 1:
        return uniform_reads([genome(max(2000, 100_000 * s))], np.ones(1), max(100, int(10_000 * s)), 100), False
    if cfg_id == 2:
        g = genome(max(4000, 5_000_000 * s))
        pairs = max(100, int(750_000 * s))
        ins = np.maximum(rng.normal(300.0, 30.0, pairs), 200.0).astype(np.int64)
        st = (rng.random(pairs) * (len(g) - ins)).astype(np.int64)
        ar = np.arange(100)[None, :]
        r1 = g[st[:, None] + ar]
        r2 = _COMP[g[(st + ins - 100)[:, None] + ar][:, ::-1]]
        flip = rng.integers(0, 2, pairs).astype(bool)
        a = np.where(flip[:, None], r2, r1)
        b = np.where(flip[:, None], r1, r2)
        out = np.empty((2 * pairs, 100), dtype=np.uint8)
        out[0::2], out[1::2] = a, b
        return out, True
    if cfg_id in (3, 4):
        ng, lo, hi, n, L = (20, 1e6, 5e6, 10_000_000, 100) if cfg_id == 3 else (200, 1e6, 8e6, 50_000_000, 150)
        lens = np.maximum((rng.uniform(lo, hi, ng) * s).astype(np.int64), 2000)
        w = np.exp(rng.normal(0.0, 1.0, ng))
        return uniform_reads([genome(l) for l in lens], w, max(1000, int(n * s)), L), False
    if cfg_id == 5:
        g = genome(max(4000, 20_000_000 * s))
        n_primary = max(200, int(1_600_000 * s))
        lens = rng.integers(75, 251, n_primary)
        st = (rng.random(n_primary) * (len(g) - lens)).astype(np.int64)
        reads = []
        for a, l in zip(st.tolist(), lens.tolist()):
            r = g[a:a + l]
            reads.append(_COMP[r[::-1]] if rng.integers(0, 2) else r)
        for i, src in enumerate(rng.integers(0, n_primary, n_primary // 4).tolist()):
            r = reads[src]
            if i % 2 == 1 and len(r) > 75:
                ln = int(rng.integers(75, len(r)))
                a = int(rng.integers(0, len(r) - ln + 1))
                r = r[a:a + ln]
            reads.append(_COMP[r[::-1]] if rng.integers(0, 2) else r)
        return reads, False
    raise ValueError("config 1..5")


def write_fasta(path, reads):
    with open(path, "wb") as f:
        for i, r in enumerate(reads):
            f.write(b">r%d\n" % i)
            f.write(memoryview(np.ascontiguousarray(r)))
            f.write(b"\n")


def cpu_reference(cfg_id, steps, warmup, scale=None):
    """Times the reference's own CPU implementation (unmodified, a subprocess of oracle/_ref/ref_overlap; the lean oracle
    port on all host threads when the reference binary did not travel) on a bounded sample of the workload.
    Returns (reads_per_s, info dict). Never imports metagenomics_b200 / maps libogb.so."""
    from oracle_lib import REF_BIN, have_reference, run_reference
    sc = scale if scale is not None else CPU_SAMPLE_SCALE[cfg_id]
    reads, paired = numpy_sample(cfg_id, sc)
    n_raw = len(reads)
    sample = f"{NAMES[cfg_id]} at scale {sc} ({n_raw} raw reads, same coverage; generated with numpy, same read model)"
    times, n_unique, e_final = [], 0, 0
    host_cores = os.cpu_count() or 1
    if have_reference():
        with tempfile.TemporaryDirectory() as td:
            fa = os.path.join(td, "sample.fa")
            write_fasta(fa, reads)
            for i in range(warmup + steps):
                d, t, _ = run_reference([fa], MIN_OVERLAP[cfg_id], paired=paired)
                if i >= warmup:
                    times.append(t["t_insert_s"] + t["t_build_s"])     # insertDataset + build to :210, mate-pair I/O excluded
                n_unique, e_final = d["n"], len(d["edges"])
        kind, cores, how = "reference", 1, f"{os.path.relpath(REF_BIN, ROOT)} (unmodified reference, single-threaded like the original) on 1 of {host_cores} host cores"
    else:
        from oracle_lib import LeanOracle
        if isinstance(reads, np.ndarray):
            bases = reads.reshape(-1)
            offs = np.arange(0, (n_raw + 1) * reads.shape[1], reads.shape[1], dtype=np.uint64)
        else:
            bases = np.concatenate(reads)
            offs = np.zeros(n_raw + 1, dtype=np.uint64)
            offs[1:] = np.cumsum([len(r) for r in reads], dtype=np.uint64)
        cores = host_cores
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            orc = LeanOracle(bases, offs, MIN_OVERLAP[cfg_id], threads=cores).run()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
            n_unique, e_final = orc.n, orc.counters()["E_final"]
        kind, how = "port", f"oracle/lean_oracle.cpp (CPU restatement) on {cores} host threads"
    t = float(np.mean(times))
    return n_unique / t, dict(kind=kind, cores=cores, host_cores=host_cores, sample=sample, how=how, seconds_per_step=t, n_unique=n_unique,
                              edges_final=e_final, edges_per_s=e_final / t)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    v, info = cpu_reference(args.config, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": info["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": workload_name(args.config, args.scale, world), "min_overlap": MIN_OVERLAP[args.config], "sample": info["sample"]},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": info["cores"], "host_cores": info["host_cores"], "kind": info["kind"],
                             "sample": info["sample"], "how": info["how"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "edges_per_sec": info["edges_per_s"], "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def golden_for(cfg_id, scale):
    p = os.path.join(ROOT, "tests", "golden", "full_size.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        for g in json.load(f):
            if g["config"] == cfg_id and abs(g["scale"] - scale) < 1e-9:
                return g
    return None


DUMP_SEED = 20250601
DUMP_EDGE_ROWS = 1 << 20      # 32 MiB of float64 edge rows
DUMP_READS = 1 << 21          # 16 MiB of float64 superReadIDs


def seeded_positions(n, cap):
    """All of 0..n-1, or `cap` of them drawn with a fixed seed (the same positions for the same n), ascending."""
    if n <= cap:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=cap, replace=False))


def u64_limbs(words):
    """64-bit words -> float64 16-bit limbs (low first): exact in float64."""
    return np.array([(int(w) >> s) & 0xFFFF for w in words for s in (0, 16, 32, 48)], dtype=np.float64)


def dump_outputs(out_dir, L, ctx, n_unique, st):
    """What the last timed step left on the device, downloaded as a caller of the C ABI receives it (see the module docstring)."""
    from metagenomics_b200._lib import check
    from metagenomics_b200.api import EDGE_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    n = C.c_uint64()
    check(L.ogb_graph_edge_count(ctx._h, 0, C.byref(n)))
    edges = np.zeros(n.value, dtype=EDGE_DTYPE)
    check(L.ogb_graph_edges(ctx._h, 0, edges.ctypes.data, n.value))
    rows = edges[seeded_positions(len(edges), DUMP_EDGE_ROWS)]
    np.save(os.path.join(out_dir, "edges.npy"), np.stack([rows[k].astype(np.float64) for k in ("src", "dst", "offset", "orient")], axis=1))
    del edges, rows
    sup = np.zeros(n_unique + 1, dtype=np.uint64)
    check(L.ogb_super_read_ids(ctx._h, sup.ctypes.data, n_unique + 1))
    np.save(os.path.join(out_dir, "super_read_ids.npy"), sup[1:][seeded_positions(n_unique, DUMP_READS)].astype(np.float64))
    gx, gs = C.c_uint64(), C.c_uint64()
    check(L.ogb_graph_checksum(ctx._h, 0, C.byref(gx), C.byref(gs)))
    np.save(os.path.join(out_dir, "edge_checksum.npy"), u64_limbs([gx.value, gs.value]))
    np.save(os.path.join(out_dir, "counts.npy"),
            np.array([n_unique, st["edges_pre"], n.value, st["nodes_final"], st["n_contained"]], dtype=np.float64))


def next_pow2(x):
    p = 1 << 20
    while p < x:
        p <<= 1
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="scale of the configuration per GPU (weak scaling multiplies it by the GPU count)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (see above)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    args.warmup = max(args.warmup, 3)         # timing rule: at least three warm-up steps

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the overlap-graph build has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from metagenomics_b200 import Context, Dataset, nccl_unique_id
    from metagenomics_b200._lib import check, lib
    from metagenomics_b200.api import EDGE_DTYPE
    from metagenomics_b200.dist import shard_bounds

    uid = None
    if world > 1:
        box = [nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
    ctx = Context(local_rank, rank, world, uid)
    L = lib()

    # ---- setup (untimed): synthetic reads -> host Dataset stage (filter, canonical strand, sort, dedupe) on rank 0; the
    # packed result reaches the other ranks' hosts through /dev/shm (one generation + sort instead of N)
    total_scale = args.scale * world
    wname = workload_name(args.config, args.scale, world)
    m = MIN_OVERLAP[args.config]
    shm = f"/dev/shm/ogb_bench_{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if world > 1 else os.getpid()}"
    t_dataset = t_dataset_dev = None
    meta = None
    if rank == 0:
        from metagenomics_b200 import synth
        cfg = synth.config(args.config, scale=total_scale)
        assert cfg["name"] == NAMES[args.config] and cfg["min_overlap"] == m
        t0 = time.perf_counter()
        ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=m)
        t_dataset = time.perf_counter() - t0
        if world == 1 and args.config != 3:
            # the same stage with canonical strand / sort / dedupe on the GPU (second call: CUDA modules and pools warm), for the record
            for _ in range(2):
                t0 = time.perf_counter()
                dsd = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=m, device=ctx)
                t_dataset_dev = time.perf_counter() - t0
            assert dsd.getNumberOfUniqueReads() == ds.getNumberOfUniqueReads()
            del dsd
        words, woffs, lens = ds.packed()
        raw_reads = len(cfg["offsets"]) - 1
        del cfg
        uniform = len(lens) > 0 and int(lens.min()) == int(lens.max())
        meta = dict(n=len(lens), uniform=bool(uniform), L=int(lens[0]) if uniform else 0, raw=raw_reads)
        if world > 1:
            np.save(shm + "_words.npy", words)
            if not uniform:
                np.save(shm + "_woffs.npy", woffs)
                np.save(shm + "_lens.npy", lens)
    if world > 1:
        box = [meta]
        dist.broadcast_object_list(box, src=0)
        meta = box[0]
        if rank != 0:
            words = np.load(shm + "_words.npy", mmap_mode="r")
            woffs = np.load(shm + "_woffs.npy", mmap_mode="r") if not meta["uniform"] else None
            lens = np.load(shm + "_lens.npy", mmap_mode="r") if not meta["uniform"] else None
    n_unique, uniform, read_len = meta["n"], meta["uniform"], meta["L"]
    s_lo, s_hi = shard_bounds(n_unique, rank, world)
    sharded = uniform                      # one read length: only the words travel (every rank its own shard; one rank: all of them)
    nw = (read_len + 31) // 32 if uniform else 0

    # pinned host staging for the uploads (the value arm uploads once, the e2e arm every step)
    def pinned(arr):
        p = C.c_void_p()
        check(L.ogb_alloc_host(C.byref(p), max(arr.nbytes, 1)))
        if arr.nbytes:
            C.memmove(p, np.ascontiguousarray(arr).ctypes.data, arr.nbytes)
        return p
    if sharded:
        mine = np.ascontiguousarray(words[s_lo * nw:s_hi * nw])
        p_words, p_offs, p_lens = pinned(mine), None, None
        h2d = mine.nbytes
    else:
        if uniform and world == 1:
            woffs_a, lens_a = woffs, lens
        else:
            woffs_a, lens_a = np.ascontiguousarray(woffs), np.ascontiguousarray(lens)
        p_words, p_offs, p_lens = pinned(np.ascontiguousarray(words)), pinned(woffs_a), pinned(lens_a)
        h2d = words.nbytes + (0 if uniform else woffs_a.nbytes + lens_a.nbytes)
    if world > 1:
        dist.barrier()
        if rank == 0:
            for suffix in ("_words.npy", "_woffs.npy", "_lens.npy"):
                if os.path.exists(shm + suffix):
                    os.remove(shm + suffix)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def upload():
        if sharded:
            check(L.ogb_reads_upload_packed_sharded(ctx._h, p_words, n_unique, read_len))
        else:
            check(L.ogb_reads_upload_packed(ctx._h, p_words, p_offs, p_lens, n_unique))

    def build():
        check(L.ogb_hash_build(ctx._h, m))
        check(L.ogb_mark_contained(ctx._h))
        check(L.ogb_build_graph(ctx._h, 0))

    upload()
    build()                                   # sizes every pool; later steps allocate nothing
    st = ctx.stats()
    n_final = st["edges_final"]
    p_edges = C.c_void_p()
    edge_cap = max(n_final, 1)                # a rank's own range never exceeds the whole list
    check(L.ogb_alloc_host(C.byref(p_edges), edge_cap * EDGE_DTYPE.itemsize))
    FLUSH = 512 << 20

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            check(L.ogb_l2_flush(ctx._h, FLUSH))
            fn()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        per, wall0 = [], time.perf_counter()
        for _ in range(steps):
            check(L.ogb_l2_flush(ctx._h, FLUSH))      # untimed: the step starts with a cold L2
            barrier()
            ms = C.c_float()
            check(L.ogb_timer_begin(ctx._h))
            fn()
            check(L.ogb_timer_end(ctx._h, C.byref(ms)))
            per.append(ms.value)
        barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.stop() if rank == 0 else None
        t = torch.tensor(per, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks, per step
        return t.cpu().numpy(), wall, clocks

    # ---- value: device-resident inputs
    per_step, wall, clocks = timed(build, args.steps, args.warmup)
    st = ctx.stats()
    ms_step = float(per_step.mean())
    value = n_unique / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, L, ctx, n_unique, st)

    # ---- parity of the timed configuration: counters + checksum of the final edge set against the oracle's golden
    gx, gs = C.c_uint64(), C.c_uint64()
    check(L.ogb_graph_checksum(ctx._h, 0, C.byref(gx), C.byref(gs)))
    sums = torch.tensor([st["pivot_entries"], st["overlap_probes"], st["candidates"], st["active_pivots"], st["contain_probes"], st["contain_hits"]],
                        dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(sums)
    T_all, P_all, C_all, piv_all, Pc_all, Cc_all = (int(x) for x in sums.cpu())
    gold = golden_for(args.config, total_scale)
    parity, parity_detail = "no golden", {}
    if gold is not None:
        got = dict(n_unique=n_unique, E_pre=st["edges_pre"], E_final=n_final, nodes=st["nodes_final"], T=T_all, contained=st["n_contained"],
                   checksum=[gx.value, gs.value])
        bad = [k for k, v in got.items() if gold.get(k) != v]
        parity = "ok" if not bad else "MISMATCH"
        parity_detail = {"golden": f"tests/golden/full_size.json config {args.config} @ scale {total_scale} (oracle: {gold.get('oracle', 'port')})",
                         "checked": sorted(got), "mismatch": bad, "checksum": "device (ogb_graph_checksum)"}
        if rank == 0 and n_final <= 40_000_000:
            # cross-check of the device checksum: the same figure from the downloaded edge list, in numpy
            from oracle_lib import edge_checksum
            from metagenomics_b200 import edges_as_tuples
            check(L.ogb_graph_edges(ctx._h, 0, p_edges, n_final))
            host = np.ctypeslib.as_array(C.cast(p_edges, C.POINTER(C.c_uint8)), shape=(n_final * 12,)).view(EDGE_DTYPE)
            if edge_checksum(edges_as_tuples(host)) != [gx.value, gs.value]:
                parity, parity_detail["mismatch"] = "MISMATCH", bad + ["device checksum != host checksum"]
            parity_detail["checksum"] = "device (ogb_graph_checksum) == numpy over the downloaded list"

    # ---- e2e: host buffers in, host edge list out, through the C ABI
    d2h_box = [0]

    def e2e_step():
        upload()
        build()
        n = C.c_uint64()
        check(L.ogb_graph_edges_shard(ctx._h, p_edges, edge_cap, C.byref(n)))
        d2h_box[0] = n.value * EDGE_DTYPE.itemsize
    e2e_steps, _, _ = timed(e2e_step, max(2, args.steps // 2 + 1), 3)
    e2e_ms = float(e2e_steps.mean())
    xfer = torch.tensor([h2d, d2h_box[0]], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(xfer)
    h2d_all, d2h_all = (int(x) for x in xfer.cpu())

    # ---- the stage after the timed path (OverlapGraph.cpp:211-215: contraction + dead-end removal to the fix-point), on the graph
    # the last step left on the device. Not part of the metric (BASELINE's path ends at :210); reported beside it. One rank only.
    simplify = None
    if world == 1:
        from metagenomics_b200._lib import SimplifyStats
        try:
            ss = SimplifyStats()
            times = []
            for _ in range(3):
                check(L.ogb_graph_simplify(ctx._h, C.byref(ss)))
                times.append(ss.ms)
            simplify = dict(ss.as_dict(), ms=min(times[1:]), ms_runs=[round(float(x), 3) for x in times],
                            what="ogb_graph_simplify on the final graph of the last step, device time (CUDA events), result left on the device")
            if gold is not None and "simplified" in gold:
                # parity of the stage: counters of the fix-point and the checksum over every composite edge with its lists, against the
                # golden of the sequential restatement (oracle/contract_seq.cpp via tests/golden/make_simplified_full_size.py)
                from contract_lib import simplified_checksum
                from metagenomics_b200.api import CEDGE_DTYPE, CITEM_DTYPE
                ce, ci = np.zeros(ss.n_edges_out, dtype=CEDGE_DTYPE), np.zeros(ss.n_items, dtype=CITEM_DTYPE)
                check(L.ogb_graph_composite_edges(ctx._h, ce.ctypes.data, len(ce), ci.ctypes.data, len(ci)))
                w = gold["simplified"]
                same = ((ss.n_edges_out, ss.n_items, ss.merges, ss.dead_ends, ss.iterations) == (w["n_edges"], w["n_items"], w["merges"], w["dead_ends"], w["iterations"])
                        and simplified_checksum(ce, ci) == w["checksum"])
                simplify["parity"] = "ok" if same else "MISMATCH"
            else:
                simplify["parity"] = "no golden"
        except Exception as e:                                   # auxiliary stage: reported, never fatal for the bench line
            simplify = {"error": str(e)}

    peak, peak_src = measured_peaks()
    if rank == 0:
        # ---- per-kernel-class roofline (rank 0; event pairs around every launch, recorded during the last timed step)
        W = 16 * ((read_len + 63) // 64) if uniform else int(np.mean([16 * ((int(l) + 63) // 64) for l in lens[:: max(1, len(lens) // 4096)]]))
        nloc = s_hi - s_lo
        E, T, P, Cn, Fo = st["edges_pre_local"], st["pivot_entries"], st["overlap_probes"], st["candidates"], d2h_box[0] // 12
        alg = {   # algorithmic bytes per step of this rank, device record sizes (DESIGN.md section 4)
            "hash_insert": (2 * W * n_unique + 4 * n_unique * SECTOR) / world,
            "window_part": W * nloc + 4 * P,                 # own query strands streamed once + one summary word per window
            "probe_parts": SECTOR * P,                       # SURVEY 8(d): one sector per probed window
            "verify": Cn * 12 + E * (W + EDGE_BYTES),        # candidate record + partner strand per verified hit + edge word
            "rows_finish": E * (EDGE_BYTES + 4),
            "mark_fast1": None, "mark_fast2": None, "mark_any": None,   # split below
            "keep": 2 * st["active_pivots"] * 8 + st["active_pivots"] * 4,
            "emit": Fo * 12 + nloc * 8,
            # K2 (mixed read lengths only): the same scan over every window of every read, candidates = containment hits + fingerprint collisions
            "contain_window": W * nloc + 4 * st["contain_probes"],
            "contain_probe": SECTOR * st["contain_probes"],
            "contain_verify": st["contain_hits"] * (W + 12),
        }
        k = st["kernels"]
        # fused schedule: chunk i's probe and chunk i-1's verification are one launch (k_probe_verify); only the first probe and the
        # last verify run alone -- the probe / verify bytes are apportioned by launches
        nf = k.get("probe_verify", {}).get("launches", 0)
        npb, nvf = k.get("probe_parts", {}).get("launches", 0), k.get("verify", {}).get("launches", 0)
        if nf:
            probe_b, verify_b = alg["probe_parts"], alg["verify"]
            alg["probe_parts"] = probe_b * npb / (npb + nf)
            alg["verify"] = verify_b * nvf / (nvf + nf)
            alg["probe_verify"] = probe_b * nf / (npb + nf) + verify_b * nf / (nvf + nf)
        mark_ms = sum(k[c]["ms"] for c in ("mark_fast1", "mark_fast2", "mark_any") if c in k)
        mark_alg = E * EDGE_BYTES + T * 4                    # own lists (8-byte words) + pivot rows (4-byte entries)
        ktable = {}
        for name, v in k.items():
            a = alg.get(name)
            if name.startswith("mark_"):
                a = mark_alg * v["ms"] / mark_ms if mark_ms else None   # one figure for K5, apportioned by time
            row = {"ms_per_step": v["ms"], "launches_per_step": v["launches"], "share_of_step": v["ms"] / ms_step if ms_step else None}
            if a:
                row.update({"algorithmic_bytes_per_step": a, "achieved_gbs": a / (v["ms"] * 1e-3) / 1e9, "frac": a / (v["ms"] * 1e-3) / 1e9 / peak})
            ktable[name] = row
        compute = {n_: r for n_, r in ktable.items() if not n_.startswith("exch_")}
        dom = max(compute, key=lambda n_: compute[n_]["ms_per_step"]) if compute else None
        # random-gather ceilings of this GPU, measured now: the structure sizes of this workload, the gather sizes of the kernels
        ceil = {}
        for label, size, gb in (("read_store_32B", st["n_reads"] * 2 * W, 32), ("index_64B", st["table_bytes"], 64), ("rows_128B", st["n_reads"] * 128, 128)):
            v = C.c_double()
            check(L.ogb_gather_ceiling(ctx._h, min(next_pow2(size), 8 << 30), gb, C.byref(v)))
            ceil[label] = {"buffer_bytes": min(next_pow2(size), 8 << 30), "gather_bytes": gb, "useful_gbs": v.value}
        gather_of = {"verify": ("read_store_32B", E * W), "probe_parts": ("index_64B", st["probe_sectors"] * 64),
                     "probe_verify": ("read_store_32B", (E * W + st["probe_sectors"] * 64) * (nf / max(1, nvf + nf))), "mark_fast1": ("rows_128B", None),
                     "mark_fast2": ("rows_128B", None), "mark_any": ("rows_128B", None)}
        traffic = None
        tp = os.path.join(ROOT, "profiles", "kernel_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            if tj.get("workload") == f"config{args.config}@{args.scale}x{world}":
                traffic = tj.get("dram_bytes_per_launch")
        roofline = None
        if dom:
            r = ktable[dom]
            per_launch = r.get("algorithmic_bytes_per_step", 0) / max(1, r["launches_per_step"])
            ms_launch = r["ms_per_step"] / max(1, r["launches_per_step"])
            roofline = {"kernel": dom, "bound": "hbm", "achieved": r.get("achieved_gbs"), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                        "frac": r.get("frac"), "traffic": traffic.get(dom) if traffic else None, "algorithmic_bytes_per_launch": per_launch,
                        "kernel_ms": ms_launch, "launches_per_step": r["launches_per_step"], "share_of_step": r["share_of_step"],
                        "how": "CUDA event pairs around every launch on the launching stream, inside the timed region (last step)"}
            if dom in gather_of:
                label, gbytes = gather_of[dom]
                if gbytes is None:
                    gbytes = T * 4 * r["ms_per_step"] / mark_ms if mark_ms else 0     # K5: the pivot rows are the random part
                roofline["random_gather"] = {"ceiling": ceil[label], "gathered_bytes_per_step": gbytes,
                                             "achieved_gbs": gbytes / (r["ms_per_step"] * 1e-3) / 1e9,
                                             "frac_random_gather": gbytes / (r["ms_per_step"] * 1e-3) / 1e9 / ceil[label]["useful_gbs"]}
                roofline["frac_random_gather"] = roofline["random_gather"]["frac_random_gather"]
        # whole step against SURVEY.md 8(d)'s formula (S = 32, B_e = 16, W = padded strand), counters of this run, all ranks
        Wsum = W * n_unique
        bytes_alg = (2 * Wsum + 4 * n_unique * SECTOR + Pc_all * SECTOR + P_all * SECTOR + (Cc_all + st["edges_pre"]) * W + st["edges_pre"] * 16
                     + (st["edges_pre"] + T_all) * 16 + st["edges_pre"] / 8 + n_final * 16)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": wname, "min_overlap": m, "raw_reads": meta["raw"], "unique_reads": n_unique,
                       "l2": "flushed between steps (512 MiB write, untimed)", "parallelism": f"query-read shards x{world}, replicated reads and index",
                       "timing": "CUDA events on the library stream per step; max over ranks; mean of steps",
                       "weak_scaling_base": NAMES[args.config] + (f" [scale {args.scale}]" if args.scale != 1.0 else "") + " per GPU"},
            "parity": parity, "parity_detail": parity_detail,
            "edges_per_sec": n_final / (ms_step * 1e-3), "edges_pre_per_sec": st["edges_pre"] / (ms_step * 1e-3),
            "edges_final": n_final, "edges_pre": st["edges_pre"],
            "e2e": {"value": n_unique / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all,
                    "per_rank": {"h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_box[0]},
                    "what": ("every rank uploads its shard of the packed reads from pinned memory (replicated over NVLink) and downloads the final edges of its node range"
                             if sharded else "packed reads from pinned memory in, final edge list out"),
                    "per_step_ms": [round(float(x), 3) for x in e2e_steps]},
            "per_step_ms": [round(float(x), 3) for x in per_step],
            "gpu_launches": int(st["kernel_launches"]) * args.steps,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_step": {"bound": "hbm", "algorithmic_bytes": bytes_alg, "formula": "SURVEY.md 8(d): S = 32 B, B_e = 16 B, W = padded strand; counters of this run",
                              "achieved": bytes_alg / (ms_step * 1e-3) / 1e9, "peak": peak * world, "unit": "GB/s", "frac": bytes_alg / (ms_step * 1e-3) / 1e9 / (peak * world)},
            "kernels": ktable,
            "simplify": simplify,
            "gather_ceilings": ceil,
            "phases_ms": {k_: st[k_] for k_ in ("ms_hash_build", "ms_contain", "ms_overlap", "ms_scan_kernel", "ms_exchange_pre", "ms_mark", "ms_reduce", "ms_total")},
            "stats": {k_: st[k_] for k_ in ("table_bytes", "hash_partitions", "overlap_probes", "probe_sectors", "candidates", "pivot_entries", "active_pivots",
                                            "max_degree", "overflow_reads", "n_contained", "nodes_final")},
            "setup_s": {"dataset_sort_dedupe": t_dataset, "dataset_sort_dedupe_device": t_dataset_dev}, "wall_s_timed_region": wall,
        }
        if not args.no_cpu_baseline and world == 1:
            v, info = cpu_reference(args.config, 1, 0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": info["cores"], "host_cores": info["host_cores"], "kind": info["kind"],
                                    "sample": info["sample"], "how": info["how"], "seconds": info["seconds_per_step"], "edges_per_sec": info["edges_per_s"]}
        print(json.dumps(line), flush=True)

    for p in (p_words, p_offs, p_lens, p_edges):
        if p is not None:
            L.ogb_free_host(p)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Sample mapping with up to d substitutions per read (ogb_graph_map_reads_approx).

CPU: the restatement (tests/map_approx_lib.py: map_sample_approx) against a brute force over every (u, p) and, at d = 0, against
map_sample; the per-thread bodies of csrc/ogb_map.cuh run on the CPU (tests/map_approx_emul.cpp) against the restatement for d = 0..3
on the fixtures, the adversarial sets and paired_mixed, with samples of substituted reads; the refusals without a GPU.
GPU: d = 0 against ogb_graph_map_reads byte for byte; the kernels against the restatement for d = 1..3 on both selections and unitig
ranges; additivity over samples mapped with mixed d; config 3 at full size with a 0.5 % error sample (monotone in d); abundance of
three samples with 1 % substitutions against the synthetic truth; the driver's --mismatches; error paths."""
import collections
import ctypes as C
import glob
import math
import os
import subprocess

import numpy as np
import pytest

import datasets
from contract_lib import build_emul
from map_approx_lib import map_sample_approx
from map_lib import COUNTERS, decode_words, filter_sample, index_figures, join_reads, sm, split_reads, unitig_seqs
from oracle_lib import Oracle
from unitig_lib import build_spell_emul, reads_ascii, store_layout, us

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
FIXTURES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
EXE = os.path.join(ROOT, "metagenomics_b200", "host", "ogb_overlap")
UNPLACED = 0xFF
ACGT = b"ACGT"


# ---------------------------------------------------------------- helpers


def substitute_read(rng, r, k, where=None):
    """r with k distinct positions (drawn from `where`, default all) each replaced by one of the other three bases"""
    r = bytearray(r)
    cand = np.arange(len(r)) if where is None else np.asarray(where)
    for p in rng.choice(cand, min(k, len(cand)), replace=False).tolist():
        r[p] = ACGT[(ACGT.index(r[p]) + int(rng.integers(1, 4))) % 4]
    return bytes(r)


def pieces(seqs, rng, n, lengths, strand=True):
    """n exact windows of the unitigs (either strand when `strand`), lengths drawn from `lengths`"""
    out = []
    for _ in range(n):
        L = int(rng.choice(lengths))
        ok = [s for s in seqs if len(s) >= L]
        if not ok:
            continue
        s = ok[int(rng.integers(0, len(ok)))]
        a = int(rng.integers(0, len(s) - L + 1))
        r = s[a:a + L]
        out.append(sm.rc(r) if strand and rng.integers(0, 2) else r)
    return out


def substituted_sample(seqs, m, d, seed):
    """Windows of the unitigs with 0 .. d + 1 substitutions anywhere; with 1 .. d inside the first K bases only (so only a later
    seed finds the read); reads shorter than 2K with one substitution (d_r = 0); near-palindromic windows (rc within 2d of the
    window) with 0 .. d substitutions."""
    K = min(32, m + 1)
    rng = np.random.default_rng(seed)
    long_L = [L for L in (2 * K, 2 * K + 7, 3 * K, 4 * K + 3, 150) if L > m]
    out = [substitute_read(rng, r, int(rng.integers(0, d + 2))) for r in pieces(seqs, rng, 60, long_L)]
    out += [substitute_read(rng, r, int(rng.integers(1, max(d, 1) + 1)), where=range(K)) for r in pieces(seqs, rng, 20, long_L)]
    short = [L for L in range(m + 1, 2 * K) if L > m] or [m + 1]
    out += [substitute_read(rng, r, 1) for r in pieces(seqs, rng, 15, short)]
    for L in sorted({2 * K, 2 * K + 1}):
        for s in seqs:
            if len(s) < L:
                continue
            a = np.frombuffer(s, np.uint8)
            w = np.lib.stride_tricks.sliding_window_view(a, L)
            c = np.frombuffer(sm.rc(s), np.uint8)[::-1]                    # complement, position for position
            wr = np.lib.stride_tricks.sliding_window_view(c, L)[:, ::-1]   # rc of every window
            near = np.flatnonzero((w != wr).sum(axis=1) <= 2 * max(d, 1))
            for p in near[:4].tolist():
                out.append(substitute_read(rng, s[p:p + L], int(rng.integers(0, d + 1))))
    return out


def brute_force(seqs, reads, m, d):
    """(hits, mismatches, placed) over every (u, p) of every unitig and both strands"""
    K = min(32, m + 1)
    hits = np.zeros(len(reads), np.uint32)
    mis = np.full(len(reads), UNPLACED, np.uint8)
    placed = []
    arrs = [np.frombuffer(s, np.uint8) for s in seqs]
    for i, r in enumerate(reads):
        s = sm.kept(r, m)
        if s is None:
            hits[i] = sm.FILTERED
            continue
        L = len(s)
        dr = min(d, L // K - 1)
        t0, t1 = np.frombuffer(s, np.uint8), np.frombuffer(sm.rc(s), np.uint8)
        H = []
        for u, a in enumerate(arrs):
            if len(a) < L:
                continue
            w = np.lib.stride_tricks.sliding_window_view(a, L)
            h = np.minimum((w != t0).sum(axis=1), (w != t1).sum(axis=1))
            H += [(int(x), u, p) for p, x in enumerate(h.tolist())]
        b = min((x for x, _, _ in H), default=dr + 1)
        if b > dr:
            continue
        pl = sorted((u, p) for x, u, p in H if x == b)
        hits[i], mis[i] = len(pl), b
        placed += [(u, p, L, i) for u, p in pl]
    return hits, mis, placed


def build_approx_emul():
    """Compiles tests/map_approx_emul.cpp and returns emul(words, recs, reads, m, d) -> (records, depth, hits, mismatches, counters)
    with hits and mismatches per raw read (the filter is sample_map.kept, the read store unitig_lib.store_layout)."""
    from map_lib import HERE as H
    out = os.path.join(H, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libmap_approx_emul.so")
    src = os.path.join(H, "map_approx_emul.cpp")
    hdrs = [os.path.join(ROOT, "metagenomics_b200", "csrc", h) for h in ("ogb_map.cuh", "ogb_coverage.cuh", "ogb_spell.cuh")] + [os.path.join(ROOT, "include", "ogb.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in [src] + hdrs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.emul_map_approx.restype = None
    lib.emul_map_approx.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]

    def emul(words, recs, reads, m, d):
        from metagenomics_b200.api import COVERAGE_DTYPE
        ks = [sm.kept(bytes(r), m) for r in reads]
        kept = [s for s in ks if s is not None]
        L = np.array([len(s) for s in kept], np.int64)
        starts = np.concatenate([[0], np.cumsum(L)])[:-1].astype(np.int64)
        fw = np.frombuffer(b"".join(kept), np.uint8).copy() if kept else np.zeros(0, np.uint8)
        rwords, rmeta = store_layout(fw, starts, L)
        rmeta = np.ascontiguousarray(rmeta if len(rmeta) else np.zeros(1, np.uint64), np.uint64)
        words = np.ascontiguousarray(words, np.uint64)
        recs = np.ascontiguousarray(recs)
        n = len(kept)
        out = np.zeros(max(len(recs), 1), COVERAGE_DTYPE)
        depth = np.zeros(max(32 * len(words), 1), np.uint32)
        kh = np.zeros(max(n, 1), np.uint32)
        kb = np.zeros(max(n, 1), np.uint8)
        ctr = np.zeros(5, np.uint64)
        lib.emul_map_approx(words.ctypes.data, len(words), recs.ctypes.data, len(recs), rwords.ctypes.data, rmeta.ctypes.data, n, m, d,
                            out.ctypes.data, depth.ctypes.data, kh.ctypes.data, kb.ctypes.data, ctr.ctypes.data)
        hits = np.full(len(reads), sm.FILTERED, np.uint32)
        mis = np.full(len(reads), UNPLACED, np.uint8)
        idx = [i for i, s in enumerate(ks) if s is not None]
        hits[idx], mis[idx] = kh[:n], kb[:n]
        counters = dict(filtered=len(reads) - n, mapped=int(ctr[0]), multi=int(ctr[1]), placements=int(ctr[2]), index_entries=int(ctr[3]),
                        index_buckets=int(ctr[4]))
        return out[:len(recs)].copy(), depth[:32 * len(words)].copy(), hits, mis, counters
    return emul


def check_approx(want, recs, depth, hits, mis, counters, srecs, m, seqs):
    """device / emulated mapping == map_sample_approx: records, profile in the word-aligned layout, hits, strata, counters"""
    from coverage_lib import check_records, padded_profile
    check_records(recs, want, srecs)
    assert np.array_equal(depth.astype(np.int64), padded_profile(want, srecs))
    assert np.array_equal(hits, want["hits"])
    assert np.array_equal(mis, want["mismatches"])
    entries, buckets = index_figures(seqs, m)
    got = {k: int(counters[k]) for k in COUNTERS}
    assert got == dict(filtered=want["filtered"], mapped=want["mapped"], multi=want["multi"], placements=want["placements"],
                       index_entries=entries, index_buckets=buckets), got


def fixture(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    if "c_edges" not in g.files:
        pytest.skip("fixture predates the contracted dump")
    return g, dict(name=name, bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"]))


def spelled(cfg, edges, items, spell_emul, canon):
    """(packed layout, records, unitig sequences) of one selection, spelled by the spell body on the CPU"""
    from metagenomics_b200 import Dataset
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=int(cfg["min_overlap"]))
    fw, st, L = reads_ascii(ds)
    words, meta = store_layout(fw, st, L)
    srecs, packed = spell_emul(words, meta, len(L), edges, items, canon)
    return packed, srecs, decode_words(packed, srecs)


def adversarial_graphs(contract):
    for cfg in datasets.adversarial() + [datasets.paired_mixed()]:
        o = Oracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run_all(Oracle.THREE_PHASE, threads=8)
        edges, items, _ = contract(o.edges(), o.read_info()["len"])
        yield cfg, edges, items


@pytest.fixture(scope="module")
def emul():
    return build_emul(), build_spell_emul(), build_approx_emul()


# ---------------------------------------------------------------- CPU


def test_restatement_against_brute_force(emul):
    """map_sample_approx == a brute force over every (u, p) for d = 0..3 on the adversarial sets (tandem repeats, palindromes, K < 32),
    cut to a few thousand bases of unitigs, with 0 .. d + 1 substitutions per read; at d = 0 it is map_sample field for field."""
    contract, spell_emul, _ = emul
    for cfg, edges, items in adversarial_graphs(contract):
        m = cfg["min_overlap"]
        _, _, seqs = spelled(cfg, edges, items, spell_emul, True)
        small, tot = [], 0
        for s in sorted(seqs, key=len, reverse=True):
            if tot < 4000:
                small.append(s)
                tot += len(s)
        for d in range(4):
            reads = substituted_sample(small, m, d, seed=70 + d)[:70]
            want = map_sample_approx(small, reads, m, d)
            hits, mis, placed = brute_force(small, reads, m, d)
            assert np.array_equal(want["hits"], hits) and np.array_equal(want["mismatches"], mis), (cfg.get("name"), d)
            assert want["placed"] == placed
            if d == 0:
                exact = sm.map_sample(small, reads, m)
                for k, v in exact.items():
                    assert (v == want[k]) if not isinstance(v, np.ndarray) else np.array_equal(v, want[k]), k


def check_body(cfg, edges, items, spell_emul, approx, extra=()):
    m = cfg["min_overlap"]
    raw = split_reads(cfg["bases"], cfg["offsets"])
    for canon in (True, False):
        packed, srecs, seqs = spelled(cfg, edges, items, spell_emul, canon)
        for d in range(4):
            rng = np.random.default_rng(d)
            noisy = [substitute_read(rng, sm.kept(r, m), int(rng.integers(0, d + 2))) if sm.kept(r, m) else r for r in raw[:300]]
            for reads in [noisy, filter_sample(seqs, m)[:120], substituted_sample(seqs, m, d, seed=10 + d)] + [s(seqs) for s in extra]:
                want = map_sample_approx(seqs, reads, m, d)
                recs, depth, hits, mis, ctr = approx(packed, srecs, reads, m, d)
                check_approx(want, recs, depth, hits, mis, ctr, srecs, m, seqs)


@pytest.mark.parametrize("name", FIXTURES)
def test_kernel_body_matches_restatement_on_fixtures(name, emul):
    contract, spell_emul, approx = emul
    g, cfg = fixture(name)
    edges, items, _ = contract(g["edges"], g["len"])
    check_body(cfg, edges, items, spell_emul, approx)


def test_kernel_body_matches_restatement_on_adversarial_sets(emul):
    """tandem repeats: many candidates per seed and ties; palindromes: the strand rule; the m 20 / 24 sets: K < 32, so seeds are
    extracted across words; samples of 0 and 1 reads."""
    contract, spell_emul, approx = emul
    for cfg, edges, items in adversarial_graphs(contract):
        check_body(cfg, edges, items, spell_emul, approx, extra=(lambda s: [], lambda s: [s[0]] if s else [b"ACGT"]))


def test_monotone_in_d_on_a_fixture(emul):
    """raising d never removes a placement: a read mapped at b has the same hits at every d >= b, and the profile only grows"""
    contract, spell_emul, _ = emul
    g, cfg = fixture(FIXTURES[0])
    edges, items, _ = contract(g["edges"], g["len"])
    _, _, seqs = spelled(cfg, edges, items, spell_emul, True)
    m = cfg["min_overlap"]
    reads = substituted_sample(seqs, m, 3, seed=5)
    prev = None
    for d in range(5):
        got = map_sample_approx(seqs, reads, m, d)
        if prev is not None:
            assert (got["depth"] >= prev["depth"]).all()
            was = prev["mismatches"] != UNPLACED
            assert np.array_equal(got["hits"][was], prev["hits"][was]) and np.array_equal(got["mismatches"][was], prev["mismatches"][was])
        prev = got


def test_entry_point_fails_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from metagenomics_b200._lib import MapStats, lib
    st = MapStats()
    b, o = join_reads([b"ACGT" * 20])
    mis = np.zeros(1, np.uint8)
    assert lib().ogb_graph_map_reads_approx(None, b.ctypes.data, o.ctypes.data, 1, 2, None, mis.ctypes.data, C.byref(st)) == 1
    assert lib().ogb_graph_map_reads_approx(None, b.ctypes.data, o.ctypes.data, 1, 9, None, None, C.byref(st)) == 1


def test_binding_and_constants():
    from metagenomics_b200._lib import OGB_MAP_MAX_MISMATCHES, OGB_MAP_UNPLACED, PROTOTYPES
    assert "ogb_graph_map_reads_approx" in PROTOTYPES and OGB_MAP_UNPLACED == UNPLACED and OGB_MAP_MAX_MISMATCHES == 8
    hdr = open(os.path.join(ROOT, "include", "ogb.h")).read()
    assert "#define OGB_MAP_UNPLACED 0xFF " in hdr and "#define OGB_MAP_MAX_MISMATCHES 8 " in hdr


@pytest.mark.parametrize("args", [["--mismatches", "2"], ["--depths", "d.tsv", "--mismatches", "2"],
                                  ["-s", "--samples", "1", "x.fa", "--depths", "d.tsv", "--mismatches", "2"],
                                  ["--samples", "1", "x.fa", "--depths", "d.tsv", "--mismatches", "9"],
                                  ["--samples", "1", "x.fa", "--depths", "d.tsv", "--mismatches", "x"]])
def test_driver_refuses_mismatches_without_samples(tmp_path, args):
    r = subprocess.run([EXE, "-l", "50", "-se", "1", str(tmp_path / "in.fa"), "-f", str(tmp_path / "p")] + args, cwd=tmp_path,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and ("--mismatches" in r.stderr or "--samples" in r.stderr), r.stderr
    assert not (tmp_path / "d.tsv").exists()


# ---------------------------------------------------------------- GPU


def device_graph(ctx, cfg):
    from metagenomics_b200 import Dataset, HashTable, OverlapGraph
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
    ht = HashTable(ctx)
    ht.insertDataset(ds, cfg["min_overlap"])
    return ds, OverlapGraph(ht)


def gpu_sets():
    fx = []
    for name in FIXTURES:
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        fx.append(dict(name=name, bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"])))
    return fx + datasets.adversarial() + [datasets.paired_mixed()]


@pytest.mark.gpu
def test_d0_reproduces_exact_mapping():
    """ogb_graph_map_reads_approx(..., 0, ...) == ogb_graph_map_reads: records, profiles and hits byte for byte"""
    from metagenomics_b200 import Context
    ctx = Context(0)
    try:
        for cfg in gpu_sets():
            _, og = device_graph(ctx, cfg)
            og.simplify()
            for canon in (True, False):
                srecs, ascii = og.unitigs(canonical=canon)
                seqs = unitig_seqs(srecs, ascii)
                raw = split_reads(cfg["bases"], cfg["offsets"])
                rng = np.random.default_rng(3)
                for reads in (raw, [substitute_read(rng, sm.kept(r, cfg["min_overlap"]), 1) if sm.kept(r, cfg["min_overlap"]) else r for r in raw], filter_sample(seqs, cfg["min_overlap"])):
                    r0, s0, h0 = og.map_reads(reads, hits=True)
                    p0 = og.sample_depth()[1]
                    r1, s1, h1, b1 = og.map_reads(reads, hits=True, max_mismatches=0, strata=True)
                    p1 = og.sample_depth()[1]
                    assert r0.tobytes() == r1.tobytes() and p0.tobytes() == p1.tobytes() and h0.tobytes() == h1.tobytes()
                    same = lambda st: {k: v for k, v in st.items() if not k.startswith("ms") and k not in ("sample", "launches")}   # noqa: E731
                    assert same(s0) == same(s1)                               # (the first mapping of a spell also builds the index)
                    assert np.array_equal(b1 == 0, (h1 > 0) & (h1 != sm.FILTERED)) and np.all((b1 == 0) | (b1 == UNPLACED))
    finally:
        ctx.close()


def check_device(og, cfg, reads, d, first=0, count=None, canonical=True):
    m = cfg["min_overlap"]
    srecs, ascii = og.unitigs(canonical=canonical, first=first, count=count)
    seqs = unitig_seqs(srecs, ascii)
    recs, st, hits, mis = og.map_reads(reads, hits=True, max_mismatches=d, strata=True)
    _, depth = og.sample_depth()
    want = map_sample_approx(seqs, reads, m, d)
    check_approx(want, recs, depth, hits, mis, st, srecs, m, seqs)
    assert st["reads_in"] == len(reads)


@pytest.mark.gpu
def test_device_matches_restatement():
    from metagenomics_b200 import Context
    from metagenomics_b200.dist import unitig_range
    ctx = Context(0)
    try:
        for cfg in gpu_sets():
            _, og = device_graph(ctx, cfg)
            edges, _, _ = og.simplify()
            m = cfg["min_overlap"]
            raw = split_reads(cfg["bases"], cfg["offsets"])
            for canon in (True, False):
                srecs, ascii = og.unitigs(canonical=canon)
                seqs = unitig_seqs(srecs, ascii)
                for d in (1, 2, 3):
                    rng = np.random.default_rng(d)
                    noisy = [substitute_read(rng, sm.kept(r, m), int(rng.integers(0, d + 2))) if sm.kept(r, m) else r for r in raw[:400]]
                    for reads in (noisy, substituted_sample(seqs, m, d, seed=20 + d), [], noisy[:1]):
                        check_device(og, cfg, reads, d, canonical=canon)
                    for world in (2, 3):
                        for r in range(world):
                            f, n = unitig_range(edges, r, world, canon)
                            check_device(og, cfg, noisy, d, first=f, count=n, canonical=canon)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_samples_with_mixed_d_add_up_and_repeat():
    """A at d = 2, B at d = 1, then A || B mapped as A at d = 2 and B at d = 1 ... as the concatenation of two calls; then A || B at
    d = 2 equals A at 2 plus B at 2. Mapping again gives the same bytes; every sample lands in the one depth table."""
    from metagenomics_b200 import Context, synth
    ctx = Context(0)
    try:
        cfg = synth.config(5, scale=0.002)
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        b = synth.substitute(9, cfg["bases"], 0.01)
        raw = split_reads(b, cfg["offsets"])
        A, B = raw[:len(raw) // 3], raw[len(raw) // 3:]
        rA, _, hA, mA = og.map_reads(A, hits=True, max_mismatches=2, strata=True)
        pA = og.sample_depth()[1].astype(np.int64)
        rB1, _ = og.map_reads(B, max_mismatches=1)
        rB, _, hB, mB = og.map_reads(B, hits=True, max_mismatches=2, strata=True)
        pB = og.sample_depth()[1].astype(np.int64)
        rAB, st, hAB, mAB = og.map_reads(A + B, hits=True, max_mismatches=2, strata=True)
        pAB = og.sample_depth()[1]
        assert st["sample"] == 3 and st["ms_index"] == 0.0
        assert np.array_equal(pAB.astype(np.int64), pA + pB) and np.array_equal(hAB, np.concatenate([hA, hB])) and np.array_equal(mAB, np.concatenate([mA, mB]))
        for k in ("reads", "read_count", "depth_sum"):
            assert np.array_equal(rAB[k].astype(np.int64), rA[k].astype(np.int64) + rB[k]), k
        assert (rB["depth_sum"] >= rB1["depth_sum"]).all() and int(rB["reads"].sum()) >= int(rB1["reads"].sum())
        again, _, h2, m2 = og.map_reads(A + B, hits=True, max_mismatches=2, strata=True)
        assert again.tobytes() == rAB.tobytes() and np.array_equal(og.sample_depth()[1], pAB) and np.array_equal(h2, hAB) and np.array_equal(m2, mAB)
        assert og.sample_depth(1)[0].tobytes() == rB1.tobytes()
        assert int(((mA > 0) & (mA != UNPLACED)).sum()) > 0
    finally:
        ctx.close()


@pytest.mark.gpu
def test_config3_full_size_with_errors():
    """Config 3 at full size; its 10 M reads with 0.5 % substitutions as the sample (three chunks), at d = 0 and d = 2: the profile at
    d = 2 is >= the one at d = 0 on every base, and a read exact at d = 2 has the hits it has at d = 0."""
    from metagenomics_b200 import Context, synth
    cfg = synth.config(3)
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        b = synth.substitute(31, cfg["bases"], 0.005)
        o = cfg["offsets"]
        n = len(o) - 1
        r0, s0, h0, m0 = og.map_reads(bases=b, offsets=o, hits=True, strata=True)
        p0 = og.sample_depth()[1]
        r2, s2, h2, m2 = og.map_reads(bases=b, offsets=o, hits=True, max_mismatches=2, strata=True)
        p2 = og.sample_depth()[1]
        assert n > 2 * (1 << 22) and s2["reads_in"] == n
        assert (p2 >= p0).all() and (r2["depth_sum"] >= r0["depth_sum"]).all()
        ex = m2 == 0
        assert np.array_equal(h2[ex], h0[ex]) and np.array_equal(ex, m0 == 0)
        assert s2["mapped"] > s0["mapped"] and s2["mapped"] == int((m2 != UNPLACED).sum())
        fr = {d: s["mapped"] / (n - s["filtered"]) for d, s in ((0, s0), (2, s2))}
        print(f"config 3, 0.5 % substitutions: mapped fraction d=0 {fr[0]:.4f} d=2 {fr[2]:.4f} (strata at d=2: "
              f"{np.bincount(m2[m2 != UNPLACED], minlength=3).tolist()}); ms_map d=0 {s0['ms_map']:.1f} d=2 {s2['ms_map']:.1f}")
    finally:
        ctx.close()


@pytest.mark.gpu
def test_abundance_against_truth_with_errors_config3():
    """As test_abundance_against_truth_config3, with 1 % substitutions per base: the interior mean of every genome with
    lambda_g P >= 10 and enough interior bases is within 5 % of lambda_g P, P = P(Binom(100, 0.01) <= d_r) the share of reads with at
    most d_r = d substitutions -- 0.366 at d = 0, 0.921 at d = 2 (100 bp reads, m = 50: d_r = min(d, 2))."""
    from metagenomics_b200 import Context, synth
    MIN_INTERIOR = 50_000
    scale = 0.1
    cfg = synth.config(3, scale=scale)
    gs, _ = synth._metagenome(3, 20, 1e6, 5e6, scale)
    lens = np.array([len(g) for g in gs], np.float64)
    fwd = [g.tobytes() for g in gs]
    rcs = [us.rc_bytes(g) for g in fwd]
    known = {}

    def assign(s):
        if s not in known:
            hits = [i for i in range(len(gs)) if s in fwd[i] or s in rcs[i]]
            known[s] = hits[0] if len(hits) == 1 else None
        return known[s]

    def P(d):
        return sum(math.comb(100, k) * 0.01 ** k * 0.99 ** (100 - k) for k in range(min(d, 2) + 1))

    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        srecs, seqs = og.unitigs()
        checked = collections.Counter()
        for s in range(3):
            w = np.exp(np.random.default_rng(100 + s).normal(0.0, 1.0, len(gs)))
            N = 3_000_000
            b, o = synth.sample_reads(100 + s, gs, N, 100, weights=w)
            b = synth.substitute(200 + s, b, 0.01)
            for d in (0, 2):
                recs, st = og.map_reads(bases=b, offsets=o, max_mismatches=d)
                _, depth = og.sample_depth()
                lam = N * 100 * w / (w * lens).sum() * P(d)
                tot, n = collections.Counter(), collections.Counter()
                for r in recs:
                    L, a = int(r["length"]), int(r["start"])
                    key = assign(seqs[a:a + L].tobytes()) if L >= 1000 else None
                    if key is not None:
                        tot[key] += int(depth[a + 100:a + L - 100].astype(np.int64).sum())
                        n[key] += L - 200
                ratios = {g: tot[g] / n[g] / lam[g] for g in n if lam[g] >= 10 and n[g] >= MIN_INTERIOR}
                print(f"sample {s} d={d} (P = {P(d):.4f}, mapped {st['mapped'] / max(1, st['reads_in'] - st['filtered']):.4f}): interior mean / "
                      f"expected per genome:", {g: round(v, 4) for g, v in ratios.items()})
                assert ratios and all(abs(v - 1) <= 0.05 for v in ratios.values()), (d, ratios)
                checked[d] += len(ratios)
        assert checked[0] >= 3 and checked[2] >= 3, checked
    finally:
        ctx.close()


@pytest.mark.gpu
def test_driver_mismatches_writes_what_the_api_writes(tmp_path):
    from metagenomics_b200 import Context, synth
    cfg = synth.config(5, scale=0.002)
    fa = str(tmp_path / "in.fa")
    synth.write_fasta(fa, cfg["bases"], cfg["offsets"])
    gs = [synth.genome(5, max(4000, int(20_000_000 * 0.002)))]
    s1, s2 = str(tmp_path / "a.fa"), str(tmp_path / "b.fq")
    b1, o1 = synth.sample_reads(21, gs, 3000, 100)
    synth.write_fasta(s1, synth.substitute(1, b1, 0.01), o1)
    b2, o2 = synth.sample_reads(22, gs, 6000, 75, 150)
    b2 = synth.substitute(2, b2, 0.01)
    with open(s2, "wb") as f:
        for i in range(len(o2) - 1):
            r = b2[int(o2[i]):int(o2[i + 1])].tobytes()
            f.write(b"@q%d\n%s\n+\n%s\n" % (i, r, b"I" * len(r)))
    m = str(cfg["min_overlap"])
    run = lambda tag, extra: subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / tag), "--samples", "2", s1, s2,  # noqa: E731
                                             "--depths", str(tmp_path / (tag + ".tsv"))] + extra, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    exact, approx = run("x", []), run("y", ["--mismatches", "2"])
    assert exact.returncode == 0 and approx.returncode == 0, exact.stdout + approx.stdout
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        og.map_file(s1, max_mismatches=2)
        og.map_file(s2, max_mismatches=2)
        og.write_depths(str(tmp_path / "api2.tsv"), names=["a.fa", "b.fq"])
        og.spell()
        og.map_file(s1)
        og.map_file(s2)
        og.write_depths(str(tmp_path / "api0.tsv"), names=["a.fa", "b.fq"])
    finally:
        ctx.close()
    assert open(tmp_path / "api2.tsv", "rb").read() == open(tmp_path / "y.tsv", "rb").read()
    assert open(tmp_path / "api0.tsv", "rb").read() == open(tmp_path / "x.tsv", "rb").read()
    assert open(tmp_path / "x.tsv", "rb").read() != open(tmp_path / "y.tsv", "rb").read()
    lx, ly = exact.stdout.strip().split("\n"), approx.stdout.strip().split("\n")
    assert [x.split(" device ms")[0] for x in lx if not x.startswith("map: ")] == [x.split(" device ms")[0] for x in ly if not x.startswith("map: ")]


@pytest.mark.gpu
def test_error_paths():
    from metagenomics_b200 import Context, OgbError, synth
    from metagenomics_b200._lib import MapStats, lib
    ctx = Context(0)
    try:
        cfg = synth.config(5, scale=0.002)
        _, og = device_graph(ctx, cfg)
        st = MapStats()
        b, o = join_reads(split_reads(cfg["bases"], cfg["offsets"])[:100])
        mis = np.zeros(100, np.uint8)
        mp = lambda n, d, mm: lib().ogb_graph_map_reads_approx(ctx._h, b.ctypes.data, o.ctypes.data, n, d, None, mm, C.byref(st))   # noqa: E731
        assert mp(100, 2, mis.ctypes.data) == 4                          # OGB_E_STATE: no spell yet
        og.simplify()
        og.spell()
        assert mp(100, 9, mis.ctypes.data) == 1 and "max_mismatches" in lib().ogb_last_error().decode()
        assert mp(0, 2, mis.ctypes.data) == 0 and st.reads_in == 0 and st.sample == 0
        assert mp(100, 8, mis.ctypes.data) == 0 and st.sample == 1 and st.mapped > 0 and int((mis != UNPLACED).sum()) == st.mapped
        with pytest.raises(OgbError) as e:
            og.map_reads(bases=b, offsets=o, max_mismatches=9)
        assert e.value.code == 1
    finally:
        ctx.close()

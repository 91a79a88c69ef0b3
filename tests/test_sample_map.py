"""Per-sample read depth of the unitigs (ogb_graph_map_reads / ogb_graph_sample_coverage / ogb_graph_write_depths).

CPU: the restatement (oracle/sample_map.py) on the reference's contracted fixtures with each fixture's own raw reads as the sample
-- its depth is at least the coverage depth (oracle/unitig_coverage.py) on every base, and the difference is exactly the profile of
the occurrences outside the coverage placements -- and the per-thread bodies of csrc/ogb_map.cuh, run on the CPU
(tests/map_emul.cpp), against the restatement; the ABI and the driver's refusals.
GPU: the kernels through the C ABI and the Python API against the restatement, additivity over samples, the coverage result left
alone, config 3 at full size against its own coverage, abundance against the known truth of three samples, error paths and the
driver's --samples / --depths."""
import collections
import ctypes as C
import glob
import os
import subprocess

import numpy as np
import pytest

import datasets
from contract_lib import build_emul
from coverage_lib import cv
from map_lib import (build_map_emul, check_against, decode_words, filter_sample, join_reads, sm, split_reads, unitig_seqs)
from oracle_lib import Oracle
from unitig_lib import build_spell_emul, reads_ascii, store_layout, us

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
FIXTURES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
EXE = os.path.join(ROOT, "metagenomics_b200", "host", "ogb_overlap")


def fixture(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    if "c_edges" not in g.files:
        pytest.skip("fixture predates the contracted dump")
    return g, dict(name=name, bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"]))


def host_reads(cfg):
    from metagenomics_b200 import Dataset
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=int(cfg["min_overlap"]))
    return ds, reads_ascii(ds)


# ---------------------------------------------------------------- CPU


@pytest.mark.parametrize("name", FIXTURES)
def test_map_depth_bounds_coverage_depth_on_fixtures(name):
    """Sample = the fixture's raw reads. Every coverage placement (a list read at P_k, a contained read at its shift, f times) is an
    exact occurrence of f raw reads, so D_map >= D_cov; what is left over is the profile of the other occurrences, named here."""
    g, cfg = fixture(name)
    m = cfg["min_overlap"]
    _, (fw, st, L) = host_reads(cfg)
    freq, sup = g["freq"].astype(np.int64), g["sup"].astype(np.int64)
    q = cv.locate(fw, st, L, sup)
    ce, ls, cl = g["c_edges"].astype(np.int64), g["c_list_start"].astype(np.int64), g["c_lists"].astype(np.int64)
    args = (ce[:, 0], ce[:, 1], ce[:, 2], ce[:, 4], ls[:-1], ls[1:] - ls[:-1], cl[:, 0], cl[:, 1], cl[:, 2])
    cov = cv.coverage_all(fw, st, L, freq, sup, *args, q=q)
    flat, s0, sl = us.spell_all(fw, st, L, *args)
    seqs = [flat[a:a + n].tobytes() for a, n in zip(s0, sl)]
    raw = split_reads(cfg["bases"], cfg["offsets"])
    got = sm.map_sample(seqs, raw, m)
    assert np.array_equal(got["length"], cov["length"])
    extra = got["depth"] - cov["depth"]
    assert (extra >= 0).all(), name
    # the coverage placements as a multiset of (unitig, position, length), f each ...
    f6 = collections.Counter()
    for i, (s, d, o, _, off) in enumerate(ce.tolist()):
        it = cl[ls[i]:ls[i + 1]]
        for r, fwd, P in us._pieces(s, d, o, off, it[:, 0], it[:, 1], it[:, 2]):
            Lr = int(L[r - 1])
            f6[(i, P, Lr)] += int(freq[r - 1])
            for x in np.flatnonzero(sup == r):
                Lx = int(L[x])
                f6[(i, P + int(q[x]) if fwd else P + Lr - int(q[x]) - Lx, Lx)] += int(freq[x])
    # ... are contained in the mapping's, and the rest is exactly the difference of the profiles
    mp = collections.Counter((u, p, n) for u, p, n, _ in got["placed"])
    assert all(mp[k] >= v for k, v in f6.items()), name
    rest = mp - f6
    diff = np.zeros(len(extra) + 1, np.int64)
    for (u, p, n), c in rest.items():
        diff[cov["start"][u] + p] += c
        diff[cov["start"][u] + p + n] -= c
    assert np.array_equal(np.cumsum(diff[:-1]), extra), name
    culprits = sorted({i for u, p, n, i in got["placed"] if (u, p, n) in rest})
    print(f"{name}: {int((extra > 0).sum())} of {len(extra)} bases above the coverage depth, from {len(culprits)} raw reads "
          f"{[raw[i].decode()[:40] for i in culprits[:5]]}")
    if not rest:
        assert np.array_equal(got["depth"], cov["depth"])


@pytest.fixture(scope="module")
def emul():
    return build_emul(), build_spell_emul(), build_map_emul()


def check_body(cfg, edges, items, spell_emul, map_emul, extra_samples=()):
    _, (fw, st, L) = host_reads(cfg)
    words, meta = store_layout(fw, st, L)
    m = cfg["min_overlap"]
    for canon in (True, False):
        srecs, packed = spell_emul(words, meta, len(L), edges, items, canon)
        seqs = decode_words(packed, srecs)
        samples = [split_reads(cfg["bases"], cfg["offsets"]), filter_sample(seqs, m)] + [s(seqs) for s in extra_samples]
        for reads in samples:
            b, o = join_reads(reads)
            want = sm.map_sample(seqs, reads, m)
            recs, depth, hits, ctr = map_emul(packed, srecs, b, o, m)
            check_against(want, recs, depth, hits, ctr, srecs, m, seqs)


@pytest.mark.parametrize("name", FIXTURES)
def test_kernel_body_matches_restatement_on_fixtures(name, emul):
    contract, spell_emul, map_emul = emul
    g, cfg = fixture(name)
    edges, items, _ = contract(g["edges"], g["len"])
    check_body(cfg, edges, items, spell_emul, map_emul)


def test_kernel_body_matches_restatement_on_adversarial_sets(emul):
    """tandem repeats: many entries per bucket and many placements per read; palindromes: the one-strand rule; the m 20 / 24 sets:
    K < 32; samples of 0 and 1 reads."""
    contract, spell_emul, map_emul = emul
    for cfg in datasets.adversarial() + [datasets.paired_mixed()]:
        o = Oracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run_all(Oracle.THREE_PHASE, threads=8)
        info = o.read_info()
        edges, items, _ = contract(o.edges(), info["len"])
        check_body(cfg, edges, items, spell_emul, map_emul, extra_samples=(lambda s: [], lambda s: [s[0]] if s else [b"ACGT"]))


def test_layout_and_binding():
    from metagenomics_b200._lib import PROTOTYPES, MapStats
    assert C.sizeof(MapStats) == 88 and MapStats.sample.offset == 56 and MapStats.launches.offset == 60
    assert MapStats.ms.offset == 64 and MapStats.ms_reduce.offset == 80 and MapStats.index_buckets.offset == 48
    for n in ("ogb_graph_map_reads", "ogb_graph_sample_coverage", "ogb_graph_write_depths", "ogb_dataset_raw_reads"):
        assert n in PROTOTYPES
    hdr = open(os.path.join(ROOT, "include", "ogb.h")).read()
    assert "#define OGB_MAP_FILTERED 0xFFFFFFFFu" in hdr and "ogb_map_stats; /* 88 bytes */" in hdr


def test_entry_points_fail_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from metagenomics_b200._lib import MapStats, lib
    st = MapStats()
    b, o = join_reads([b"ACGT" * 20])
    assert lib().ogb_graph_map_reads(None, b.ctypes.data, o.ctypes.data, 1, None, C.byref(st)) == 1
    assert lib().ogb_graph_sample_coverage(None, 0, None, 0, None, 0) == 1
    assert lib().ogb_graph_write_depths(None, b"/nonexistent", None) == 1


def test_raw_reads_of_a_data_set(tmp_path):
    from metagenomics_b200._lib import lib
    fa = tmp_path / "s.fq"
    fa.write_text("@a\nACGTacgtNN\n+\nIIIIIIIIII\n@b\nTTTT\n+\nIIII\n")
    ds = C.c_void_p()
    assert lib().ogb_dataset_create(C.byref(ds)) == 0
    try:
        assert lib().ogb_dataset_add_file(ds, str(fa).encode()) == 0
        bp, op, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
        assert lib().ogb_dataset_raw_reads(ds, C.byref(bp), C.byref(op), C.byref(n)) == 0
        offs = np.ctypeslib.as_array(C.cast(op, C.POINTER(C.c_uint64)), shape=(n.value + 1,))
        assert n.value == 2 and list(offs) == [0, 10, 14] and C.string_at(bp, 14) == b"ACGTacgtNNTTTT"
        assert lib().ogb_dataset_raw_reads(ds, None, C.byref(op), C.byref(n)) == 1
        assert lib().ogb_dataset_finalize(ds, 2) == 0
        assert lib().ogb_dataset_raw_reads(ds, C.byref(bp), C.byref(op), C.byref(n)) == 4
    finally:
        lib().ogb_dataset_destroy(ds)


@pytest.mark.parametrize("args,what", [(["-s", "--samples", "1", "x.fa", "--depths", "d.tsv"], "-s"), (["--depths", "d.tsv"], "--samples"),
                                       (["--samples", "1", "x.fa"], "--depths")])
def test_driver_refuses_incomplete_or_resumed_sample_mapping(tmp_path, args, what):
    r = subprocess.run([EXE, "-l", "50", "-se", "1", str(tmp_path / "in.fa"), "-f", str(tmp_path / "p")] + args, cwd=tmp_path,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--samples" in r.stderr and "--depths" in r.stderr, (what, r.stderr)
    assert not (tmp_path / "d.tsv").exists()


# ---------------------------------------------------------------- GPU


def device_graph(ctx, cfg):
    from metagenomics_b200 import Dataset, HashTable, OverlapGraph
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
    ht = HashTable(ctx)
    ht.insertDataset(ds, cfg["min_overlap"])
    og = OverlapGraph(ht)
    return ds, og


def gpu_sets():
    fx = []
    for name in FIXTURES:
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        fx.append(dict(name=name, bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"])))
    return fx + datasets.adversarial() + [datasets.paired_mixed()]


def check_device(og, cfg, reads, first=0, count=None, canonical=True):
    """spells the range, maps `reads` and compares records, profile, hits and counters with the restatement"""
    m = cfg["min_overlap"]
    srecs, ascii = og.unitigs(canonical=canonical, first=first, count=count)
    seqs = unitig_seqs(srecs, ascii)
    b, o = join_reads(reads)
    recs, st, hits = og.map_reads(bases=b, offsets=o, hits=True)
    _, depth = og.sample_depth()
    want = sm.map_sample(seqs, reads, m)
    check_against(want, recs, depth, hits, st, srecs, m, seqs)
    assert st["reads_in"] == len(reads) and st["sample"] == 0
    return recs, depth, hits


@pytest.mark.gpu
def test_device_matches_restatement():
    from metagenomics_b200 import Context
    from metagenomics_b200.dist import unitig_range
    ctx = Context(0)
    try:
        for cfg in gpu_sets():
            _, og = device_graph(ctx, cfg)
            edges, _, _ = og.simplify()
            raw = split_reads(cfg["bases"], cfg["offsets"])
            for canon in (True, False):
                check_device(og, cfg, raw, canonical=canon)
                srecs, ascii = og.unitigs(canonical=canon)
                seqs = unitig_seqs(srecs, ascii)
                for reads in (filter_sample(seqs, cfg["min_overlap"]), [], raw[:1]):
                    check_device(og, cfg, reads, canonical=canon)
                for world in (2, 3):
                    for r in range(world):
                        f, n = unitig_range(edges, r, world, canon)
                        check_device(og, cfg, raw, first=f, count=n, canonical=canon)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_samples_add_up_and_repeat():
    """Map A, then B, then A || B as one sample: profiles and sums add exactly, hits concatenate; mapping A || B again gives the same
    bytes. The coverage of the same spell, copied after the mapping, equals the copy taken before."""
    from metagenomics_b200 import Context, synth
    from metagenomics_b200._lib import check, lib
    from metagenomics_b200.api import COVERAGE_DTYPE
    ctx = Context(0)
    try:
        cfg = synth.config(5, scale=0.002)
        _, og = device_graph(ctx, cfg)
        og.simplify()
        cov, cdepth = og.depth()                                          # spell + coverage
        raw = split_reads(cfg["bases"], cfg["offsets"])
        A, B = raw[:len(raw) // 3], raw[len(raw) // 3:]
        rA, _, hA = og.map_reads(A, hits=True)
        _, pA = og.sample_depth()
        rB, _, hB = og.map_reads(B, hits=True)
        _, pB = og.sample_depth()
        rAB, stAB, hAB = og.map_reads(A + B, hits=True)
        _, pAB = og.sample_depth()
        assert stAB["sample"] == 2 and stAB["ms_index"] == 0.0
        assert np.array_equal(pAB.astype(np.int64), pA.astype(np.int64) + pB) and np.array_equal(hAB, np.concatenate([hA, hB]))
        for k in ("reads", "read_count", "depth_sum"):
            assert np.array_equal(rAB[k].astype(np.int64), rA[k].astype(np.int64) + rB[k]), k
        again, _, h2 = og.map_reads(A + B, hits=True)
        assert again.tobytes() == rAB.tobytes() and np.array_equal(og.sample_depth()[1], pAB) and np.array_equal(h2, hAB)
        assert og.sample_depth(0)[0].tobytes() == rA.tobytes() and og.sample_depth(0)[1] is None
        recs = np.zeros(len(cov), COVERAGE_DTYPE)
        depth = np.zeros(len(cdepth), np.uint32)
        check(lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), depth.ctypes.data, len(depth)))
        assert recs.tobytes() == cov.tobytes() and np.array_equal(depth, cdepth)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_config3_full_size_own_reads():
    """Config 3 at full size with its own 10 M raw reads as the sample (three chunks): D_map >= the coverage depth on every base, and
    the three thirds mapped as samples of their own add up to the whole."""
    from metagenomics_b200 import Context, synth
    cfg = synth.config(3)
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        cov, dcov = og.depth()
        b, o = cfg["bases"], cfg["offsets"]
        recs, st = og.map_reads(bases=b, offsets=o)
        _, dmap = og.sample_depth()
        assert st["reads_in"] == len(o) - 1 and st["placements"] >= st["mapped"] > 0
        assert (dmap >= dcov).all()
        print(f"config 3: {int((dmap != dcov).sum())} of {int(cov['length'].sum())} bases map deeper than their coverage; "
              f"{st['multi']} reads with >= 2 placements; ms {st['ms']:.1f} (index {st['ms_index']:.1f}, upload {st['ms_upload']:.1f}, "
              f"map {st['ms_map']:.1f}, reduce {st['ms_reduce']:.1f})")
        del dcov
        n = len(o) - 1
        cuts = [0, n // 3, 2 * n // 3, n]
        total = np.zeros(len(dmap), np.int64)
        sums = np.zeros(len(recs), np.int64)
        for a, z in zip(cuts[:-1], cuts[1:]):
            r, _ = og.map_reads(bases=b, offsets=o[a:z + 1])
            total += og.sample_depth()[1]
            sums += r["depth_sum"].astype(np.int64)
        assert np.array_equal(total, dmap) and np.array_equal(sums, recs["depth_sum"].astype(np.int64))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_abundance_against_truth_config3():
    """Assemble config 3 x 0.1, then map three further samples of the same genomes, each with its own seeded log-normal weights
    w_s. Genome g gets a read with probability w_sg len_g / sum_h w_sh len_h, so its expected depth in sample s is
    N_s 100 w_sg / sum_h w_sh len_h. Every genome at >= 10x in a sample is within 5 % of it (interior bases) when the assembly gives it
    at least MIN_INTERIOR bases of interior: over fewer, the mean of a Poisson depth of ~10x correlated over 100-base reads has a
    standard deviation of several percent by itself (a genome the assembly sample covered thinly ends up in short unitigs)."""
    from metagenomics_b200 import Context, synth
    MIN_INTERIOR = 50_000
    scale = 0.1
    cfg = synth.config(3, scale=scale)
    gs, _ = synth._metagenome(3, 20, 1e6, 5e6, scale)
    lens = np.array([len(g) for g in gs], np.float64)
    fwd = [g.tobytes() for g in gs]
    rcs = [us.rc_bytes(g) for g in fwd]

    known = {}

    def assign(s):                                                  # the same unitigs for every sample: search each once
        if s not in known:
            hits = [i for i in range(len(gs)) if s in fwd[i] or s in rcs[i]]
            known[s] = hits[0] if len(hits) == 1 else None
        return known[s]

    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        og.simplify()
        srecs, seqs = og.unitigs()
        checked = 0
        for s in range(3):
            w = np.exp(np.random.default_rng(100 + s).normal(0.0, 1.0, len(gs)))
            N = 1_000_000
            b, o = synth.sample_reads(100 + s, gs, N, 100, weights=w)
            recs, st = og.map_reads(bases=b, offsets=o)
            _, depth = og.sample_depth()
            lam = N * 100 * w / (w * lens).sum()
            tot, n = collections.Counter(), collections.Counter()        # the pattern of test_coverage.interior_means, with the base counts
            for r in recs:
                L, a = int(r["length"]), int(r["start"])
                key = assign(seqs[a:a + L].tobytes()) if L >= 1000 else None
                if key is not None:
                    tot[key] += int(depth[a + 100:a + L - 100].astype(np.int64).sum())
                    n[key] += L - 200
            ratios = {g: tot[g] / n[g] / lam[g] for g in n if lam[g] >= 10 and n[g] >= MIN_INTERIOR}
            print(f"sample {s}: interior mean / expected per genome (>= 10x, >= {MIN_INTERIOR} interior bases):", {g: round(v, 4) for g, v in ratios.items()},
                  "left out (interior bases, ratio):", {g: (n[g], round(tot[g] / n[g] / lam[g], 4)) for g in n if lam[g] >= 10 and n[g] < MIN_INTERIOR},
                  "not assembled:", [g for g in range(len(gs)) if lam[g] >= 10 and g not in n])
            assert ratios and all(abs(v - 1) <= 0.05 for v in ratios.values()), ratios
            checked += len(ratios)
        assert checked >= 3
    finally:
        ctx.close()


@pytest.mark.gpu
def test_error_paths():
    from metagenomics_b200 import Context, OgbError, synth
    from metagenomics_b200._lib import MapStats, lib
    from metagenomics_b200.api import COVERAGE_DTYPE
    ctx = Context(0)
    try:
        cfg = synth.config(5, scale=0.002)
        _, og = device_graph(ctx, cfg)
        st = MapStats()
        b, o = join_reads(split_reads(cfg["bases"], cfg["offsets"])[:100])
        mp = lambda bb, oo, n: lib().ogb_graph_map_reads(ctx._h, bb, oo, n, None, C.byref(st))   # noqa: E731
        assert mp(b.ctypes.data, o.ctypes.data, 100) == 4                 # OGB_E_STATE: no spell yet
        og.simplify()
        sp = og.spell()
        assert lib().ogb_graph_sample_coverage(ctx._h, 0, None, 0, None, 0) == 4      # no sample yet
        assert lib().ogb_graph_write_depths(ctx._h, b"/tmp/never.tsv", None) == 4
        assert mp(None, o.ctypes.data, 100) == 1 and mp(b.ctypes.data, None, 100) == 1
        bad = o.copy()
        bad[50] = bad[49] - 1
        assert mp(b.ctypes.data, bad.ctypes.data, 100) == 1
        assert mp(None, None, 0) == 0 and st.reads_in == 0 and st.placements == 0 and st.sample == 0
        assert mp(b.ctypes.data, o.ctypes.data, 100) == 0 and st.sample == 1 and st.mapped > 0 and st.ms_index == 0.0
        recs = np.zeros(sp["unitigs"], COVERAGE_DTYPE)
        depth = np.zeros(32 * sp["words"], np.uint32)
        sc = lambda j, r, d, dc: lib().ogb_graph_sample_coverage(ctx._h, j, r.ctypes.data, len(r), d, dc)   # noqa: E731
        assert sc(2, recs, None, 0) == 1                                  # beyond the last sample
        assert sc(0, recs, depth.ctypes.data, len(depth)) == 1            # the profile of an earlier sample
        rc = sc(1, recs, depth.ctypes.data, len(depth) - 1)
        msg = lib().ogb_last_error().decode()
        assert rc == 5 and f"{sp['unitigs']} records" in msg and f"{32 * sp['words']} depth entries" in msg
        assert sc(1, recs[:-1], None, 0) == 5
        assert sc(1, recs, depth.ctypes.data, len(depth)) == 0 and int(recs["reads"].sum()) == st.placements
        names = (C.c_char_p * 2)(b"a", b"b\tc")
        assert lib().ogb_graph_write_depths(ctx._h, b"/tmp/never.tsv", names) == 1
        assert lib().ogb_graph_write_depths(ctx._h, b"/nonexistent/dir/d.tsv", None) == 6
        og.spell()                                                        # a new spell drops the samples
        assert sc(0, recs, None, 0) == 4
        og.map_reads(bases=b, offsets=o)
        og.buildOverlapGraphFromHashTable()                               # and so does a rebuild
        assert sc(0, recs, None, 0) == 4
        with pytest.raises(OgbError) as e:
            og.map_reads(bases=b, offsets=o)
        assert e.value.code == 4
    finally:
        ctx.close()


@pytest.mark.gpu
def test_driver_writes_what_the_api_writes(tmp_path):
    from metagenomics_b200 import Context, synth
    cfg = synth.config(5, scale=0.002)
    fa = str(tmp_path / "in.fa")
    synth.write_fasta(fa, cfg["bases"], cfg["offsets"])
    gs = [synth.genome(5, max(4000, int(20_000_000 * 0.002)))]
    s1, s2 = str(tmp_path / "s1.fa"), str(tmp_path / "deep.fq")
    b1, o1 = synth.sample_reads(21, gs, 3000, 100)
    synth.write_fasta(s1, b1, o1)
    b2, o2 = synth.sample_reads(22, gs, 6000, 75, 150)
    with open(s2, "wb") as f:
        for i in range(len(o2) - 1):
            r = b2[int(o2[i]):int(o2[i + 1])].tobytes()
            f.write(b"@q%d\n%s\n+\n%s\n" % (i, r, b"I" * len(r)))
    m = str(cfg["min_overlap"])
    base = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "a"), "--unitigs", str(tmp_path / "a.fa")],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    drv = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "b"), "--unitigs", str(tmp_path / "b.fa"), "--samples", "2", s1, s2,
                          "--depths", str(tmp_path / "drv.tsv")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert base.returncode == 0 and drv.returncode == 0, base.stdout + drv.stdout
    assert open(tmp_path / "a.unitig", "rb").read() == open(tmp_path / "b.unitig", "rb").read()
    assert open(tmp_path / "a.fa", "rb").read() == open(tmp_path / "b.fa", "rb").read()
    lb, ld = base.stdout.strip().split("\n"), drv.stdout.strip().split("\n")
    assert len(ld) == len(lb) + 2 and [x.split(" device ms")[0] for x in ld if not x.startswith("map: ")] == [x.split(" device ms")[0] for x in lb]
    assert [x.split()[1] for x in ld if x.startswith("map: ")] == ["s1.fa", "deep.fq"]
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        r1, _ = og.map_file(s1)
        r2, _ = og.map_file(s2)
        og.write_depths(str(tmp_path / "api.tsv"), names=["s1.fa", "deep.fq"])
        assert open(tmp_path / "api.tsv", "rb").read() == open(tmp_path / "drv.tsv", "rb").read()
        lines = open(tmp_path / "api.tsv").read().split("\n")
        assert lines[0] == "contigName\tcontigLen\ttotalAvgDepth\ts1.fa\ts1.fa-var\tdeep.fq\tdeep.fq-var" and lines[-1] == ""
        assert len(lines) == len(r1) + 2
        for i, line in enumerate(lines[1:-1]):
            f = line.split("\t")
            L = int(r1[i]["length"])
            m1, m2 = int(r1[i]["depth_sum"]) / L, int(r2[i]["depth_sum"]) / L
            assert f[0] == f"unitig_{i}" and f[1] == str(L) and float(f[2]) == pytest.approx(m1 + m2, abs=1e-4)
            assert f[3] == f"{m1:.4f}" and f[5] == f"{m2:.4f}" and float(f[4]) >= 0 and float(f[6]) >= 0
    finally:
        ctx.close()

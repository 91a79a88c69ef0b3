"""Per-base read depth and abundance of the unitigs (ogb_graph_coverage / ogb_graph_unitig_coverage / ogb_graph_write_coverage).

CPU: the restatement (oracle/unitig_coverage.py) on the reference's own contracted graphs of the fixtures -- depth_sum is the sum
of f * L over the placed reads, every base is covered, every contained read is found in its super read, the twin's profile is the
reverse -- and the per-thread bodies of csrc/ogb_coverage.cuh, run on the CPU (tests/coverage_emul.cpp), against the restatement.
GPU: the kernels through the C ABI and the Python API, ranges, error paths, the driver's --coverage, abundance against the known
truth of configs 3 and 5, and the full-size goldens (tests/golden/coverage_full_size.json, tests/golden/make_coverage_full_size.py)."""
import ctypes as C
import glob
import json
import os
import subprocess

import numpy as np
import pytest

import datasets
from contract_lib import build_emul
from coverage_lib import build_coverage_emul, check_records, cover_graph, cv, padded_profile, sup_packed
from oracle_lib import Oracle
from unitig_lib import build_spell_emul, canonical_mask, reads_ascii, store_layout, us

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
FIXTURES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
EXE = os.path.join(ROOT, "metagenomics_b200", "host", "ogb_overlap")


def host_reads(cfg):
    from metagenomics_b200 import Dataset
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=int(cfg["min_overlap"]))
    return ds, reads_ascii(ds)


def fixture(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    if "c_edges" not in g.files:
        pytest.skip("fixture predates the contracted dump")
    return g, dict(name=name, bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"]))


# ---------------------------------------------------------------- CPU


@pytest.mark.parametrize("name", FIXTURES)
def test_restatement_on_the_reference_graph(name):
    g, cfg = fixture(name)
    ds, (fw, st, L) = host_reads(cfg)
    assert np.array_equal(L, g["len"].astype(np.int64)) and np.array_equal(ds.frequencies(), g["freq"])
    freq, sup = g["freq"].astype(np.int64), g["sup"].astype(np.int64)
    q = cv.locate(fw, st, L, sup)
    assert (q[sup > 0] >= 0).all() and (q[sup == 0] == -2).all()      # unplaced == 0
    ce, ls, cl = g["c_edges"].astype(np.int64), g["c_list_start"].astype(np.int64), g["c_lists"].astype(np.int64)
    cov = cv.coverage_all(fw, st, L, freq, sup, ce[:, 0], ce[:, 1], ce[:, 2], ce[:, 4], ls[:-1], ls[1:] - ls[:-1], cl[:, 0], cl[:, 1], cl[:, 2], q=q)
    assert cov["unplaced"] == 0
    profiles = {}
    for i, (s, d, o, _, off) in enumerate(ce.tolist()):
        it = cl[ls[i]:ls[i + 1]]
        D, nc = cv.profile(fw, st, L, freq, sup, q, s, d, o, off, it[:, 0], it[:, 1], it[:, 2])
        a = int(cov["start"][i])
        assert np.array_equal(cov["depth"][a:a + len(D)], D) and cov["contained"][i] == nc, (name, i)   # the vectorised form is the definition
        assert (D >= 1).all(), (name, i)
        reads = [r for r, _, _ in us._pieces(s, d, o, off, it[:, 0], it[:, 1], it[:, 2])]
        placed = reads + [x + 1 for r in reads for x in np.flatnonzero(sup == r)]
        assert int(D.sum()) == sum(int(freq[r - 1]) * int(L[r - 1]) for r in placed) == int(cov["depth_sum"][i])
        assert int(cov["read_count"][i]) == sum(int(freq[r - 1]) for r in placed)
        profiles.setdefault((s, d), []).append(D.tobytes())
    for (s, d), ps in profiles.items():                                # the twin's profile is the reverse, per end-point pair
        assert sorted(ps) == sorted(np.frombuffer(p, np.int64)[::-1].tobytes() for p in profiles[(d, s)]), (name, s, d)
    if name == "paired_mixed":
        assert (sup > 0).mean() > 0.5 and cov["contained"].sum() > 0


@pytest.fixture(scope="module")
def emul():
    return build_emul(), build_spell_emul(), build_coverage_emul()


def check_body(cfg, edges, items, freq, sup_ids, spell_emul, cover_emul):
    _, (fw, st, L) = host_reads(cfg)
    words, meta = store_layout(fw, st, L)
    sup = sup_packed(sup_ids, L)
    q = cv.locate(fw, st, L, sup_ids)
    for canon in (True, False):
        sel = canonical_mask(edges) if canon else np.ones(len(edges), bool)
        srecs, _ = spell_emul(words, meta, len(L), edges, items, canon)
        recs, depth, unplaced, ncp = cover_emul(words, meta, edges, items, srecs, freq, sup)
        want = cover_graph(fw, st, L, freq, sup_ids, edges, items, sel, q=q)
        assert unplaced == want["unplaced"] == 0 and ncp == int(want["contained"].sum())
        check_records(recs, want, srecs)
        assert np.array_equal(depth.astype(np.int64), padded_profile(want, srecs)), cfg.get("name")
    return want


@pytest.mark.parametrize("name", FIXTURES)
def test_kernel_body_matches_restatement_on_fixtures(name, emul):
    contract, spell_emul, cover_emul = emul
    g, cfg = fixture(name)
    edges, items, _ = contract(g["edges"], g["len"])
    check_body(cfg, edges, items, g["freq"], g["sup"], spell_emul, cover_emul)


def test_kernel_body_matches_restatement_on_adversarial_sets(emul):
    """tandem repeats: many occurrences of a contained read in its super read (the smallest shift counts); palindromes: both
    strands match at one shift (the stored strand counts)."""
    contract, spell_emul, cover_emul = emul
    n_contained = 0
    for cfg in datasets.adversarial() + [datasets.paired_mixed()]:
        o = Oracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run_all(Oracle.THREE_PHASE, threads=8)
        info = o.read_info()
        edges, items, _ = contract(o.edges(), info["len"])
        want = check_body(cfg, edges, items, info["freq"], info["sup"], spell_emul, cover_emul)
        n_contained += int(want["contained"].sum())
    assert n_contained > 0


def test_layout_and_binding():
    from metagenomics_b200._lib import PROTOTYPES, CoverageStats
    from metagenomics_b200.api import COVERAGE_DTYPE
    assert COVERAGE_DTYPE.itemsize == 64 and COVERAGE_DTYPE.fields["length"][1] == 24 and COVERAGE_DTYPE.fields["depth_sq_sum"][1] == 56
    assert COVERAGE_DTYPE.fields["depth_min"][1] == 12 and COVERAGE_DTYPE.fields["read_count"][1] == 40
    assert C.sizeof(CoverageStats) == 64 and CoverageStats.launches.offset == 40 and CoverageStats.ms.offset == 44
    assert CoverageStats.ms_reduce.offset == 56
    for n in ("ogb_graph_coverage", "ogb_graph_unitig_coverage", "ogb_graph_write_coverage"):
        assert n in PROTOTYPES


def test_entry_points_fail_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from metagenomics_b200._lib import CoverageStats, lib
    st = CoverageStats()
    f = np.ones(4, np.uint32)
    assert lib().ogb_graph_coverage(None, f.ctypes.data, 4, C.byref(st)) == 1
    assert lib().ogb_graph_unitig_coverage(None, None, 0, None, 0) == 1
    assert lib().ogb_graph_write_coverage(None, b"/nonexistent") == 1


def test_driver_refuses_coverage_on_resume(tmp_path):
    r = subprocess.run([EXE, "-l", "50", "-se", "1", str(tmp_path / "in.fa"), "-f", str(tmp_path / "p"), "-s", "--coverage", str(tmp_path / "c.tsv")],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--coverage" in r.stderr
    assert not (tmp_path / "c.tsv").exists()


# ---------------------------------------------------------------- GPU


def device_graph(ctx, cfg):
    from metagenomics_b200 import Dataset, HashTable, OverlapGraph
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
    ht = HashTable(ctx)
    ht.insertDataset(ds, cfg["min_overlap"])
    og = OverlapGraph(ht)
    return ds, og


def gpu_sets():
    from metagenomics_b200 import synth
    fx = []
    for name in FIXTURES:
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        fx.append(dict(name=name, bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"])))
    return fx + datasets.adversarial() + [datasets.paired_mixed(), synth.config(2, scale=0.01), synth.config(3, scale=0.002)]


@pytest.mark.gpu
def test_device_matches_restatement():
    from metagenomics_b200 import Context
    ctx = Context(0)
    try:
        for cfg in gpu_sets():
            ds, og = device_graph(ctx, cfg)
            edges, items, _ = og.simplify()
            fw, st, L = reads_ascii(ds)
            sup = og.superReadIDs()[1:]
            freq = ds.frequencies()
            q = cv.locate(fw, st, L, sup)
            for canon in (True, False):
                sel = canonical_mask(edges) if canon else np.ones(len(edges), bool)
                want = cover_graph(fw, st, L, freq, sup, edges, items, sel, q=q)
                srecs, _ = og.unitigs(canonical=canon, ascii=False)
                recs, depth = og.depth(canonical=canon)
                check_records(recs, want, srecs)
                assert np.array_equal(depth.astype(np.int64), padded_profile(want, srecs)), cfg["name"]
                recs2, cst = og.coverage(canonical=canon)                 # a second run gives the same bits
                assert recs2.tobytes() == recs.tobytes()
                assert cst["unplaced"] == 0 and cst["unitigs"] == len(recs) and cst["bases"] == int(recs["length"].sum())
                assert cst["placements"] == int(recs["reads"].sum()) and cst["contained_placements"] == int(recs["contained"].sum())
    finally:
        ctx.close()


@pytest.mark.gpu
def test_ranges_concatenate_to_the_whole():
    from metagenomics_b200 import Context, synth
    from metagenomics_b200.dist import unitig_range
    """config 3 has many unitigs to split; config 5 (one genome, few unitigs, so some ranks get an empty range) has contained reads."""
    ctx = Context(0)
    try:
        for k, min_unitigs in ((3, 4), (5, 1)):
            ds, og = device_graph(ctx, synth.config(k, scale=0.004))
            edges, _, _ = og.simplify()
            fields = [n for n in og.coverage()[0].dtype.names if n != "start"]
            for canon in (True, False):
                recs, depth = og.depth(canonical=canon)
                assert len(recs) >= min_unitigs
                if k == 5:
                    assert recs["contained"].sum() > 0
                for world in (2, 3, 7):
                    parts = [og.depth(canonical=canon, first=f, count=n) for f, n in (unitig_range(edges, r, world, canon) for r in range(world))]
                    got = np.concatenate([p[0] for p in parts])
                    assert np.array_equal(got[fields], recs[fields])
                    assert np.array_equal(np.concatenate([p[1] for p in parts]), depth)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_error_paths():
    from metagenomics_b200 import Context, OgbError, synth
    from metagenomics_b200._lib import CoverageStats, lib
    from metagenomics_b200.api import COVERAGE_DTYPE
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, synth.config(5, scale=0.002))
        freq = ds.frequencies()
        st = CoverageStats()
        assert lib().ogb_graph_coverage(ctx._h, freq.ctypes.data, len(freq), C.byref(st)) == 4      # OGB_E_STATE: no spell yet
        og.simplify()
        sp = og.spell()
        assert lib().ogb_graph_coverage(ctx._h, freq.ctypes.data, len(freq) - 1, C.byref(st)) == 1  # OGB_E_ARG: wrong n
        assert lib().ogb_graph_coverage(ctx._h, None, len(freq), C.byref(st)) == 1
        assert lib().ogb_graph_coverage(ctx._h, freq.ctypes.data, len(freq), C.byref(st)) == 0
        assert st.unitigs == sp["unitigs"] > 0 and st.unplaced == 0 and st.contained_placements > 0
        recs = np.zeros(st.unitigs, COVERAGE_DTYPE)
        small = np.zeros(32 * sp["words"] - 1, np.uint32)
        rc = lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), small.ctypes.data, len(small))
        msg = lib().ogb_last_error().decode()
        assert rc == 5 and f"{st.unitigs} records" in msg and f"{32 * sp['words']} depth entries" in msg
        assert lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs) - 1, None, 0) == 5
        assert lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), None, 0) == 0
        og.spell()                                                      # a new spell invalidates the coverage
        assert lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), None, 0) == 4
        og.coverage()
        og.buildOverlapGraphFromHashTable()                             # and so does a rebuild
        assert lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), None, 0) == 4
        with pytest.raises(OgbError) as e:
            og.coverage()
        assert e.value.code == 4
    finally:
        ctx.close()


@pytest.mark.gpu
def test_driver_writes_what_the_api_writes(tmp_path):
    from metagenomics_b200 import Context, synth
    cfg = synth.config(5, scale=0.002)
    fa = str(tmp_path / "in.fa")
    synth.write_fasta(fa, cfg["bases"], cfg["offsets"])
    m = str(cfg["min_overlap"])
    base = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "a"), "--unitigs", str(tmp_path / "a.fa")],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    cov = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "b"), "--unitigs", str(tmp_path / "b.fa"), "--coverage", str(tmp_path / "drv.tsv")],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    only = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "c"), "--coverage", str(tmp_path / "only.tsv")],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert base.returncode == 0 and cov.returncode == 0 and only.returncode == 0, base.stdout + cov.stdout + only.stdout
    # --coverage leaves the .unitig file and the FASTA as they are, and adds one report line
    assert open(tmp_path / "a.unitig", "rb").read() == open(tmp_path / "b.unitig", "rb").read() == open(tmp_path / "c.unitig", "rb").read()
    assert open(tmp_path / "a.fa", "rb").read() == open(tmp_path / "b.fa", "rb").read()
    lb, lc = base.stdout.strip().split("\n"), cov.stdout.strip().split("\n")
    assert len(lc) == len(lb) + 1 and lc[0].split(" device ms")[0] == lb[0].split(" device ms")[0]
    assert sum(x.startswith("coverage: ") for x in lc) == 1 and sum(x.startswith("coverage: ") for x in only.stdout.split("\n")) == 1
    assert open(tmp_path / "drv.tsv", "rb").read() == open(tmp_path / "only.tsv", "rb").read()
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        og.simplify()
        og.write_coverage(str(tmp_path / "api.tsv"))
        assert open(tmp_path / "api.tsv", "rb").read() == open(tmp_path / "drv.tsv", "rb").read()
        recs, _ = og.coverage()
        srecs, _ = og.unitigs()
        lines = open(tmp_path / "api.tsv").read().split("\n")
        assert lines[0].startswith("#") and lines[-1] == "" and len(lines) == len(recs) + 2
        for i, line in enumerate(lines[1:-1]):
            f = line.split("\t")
            r, s = recs[i], srecs[i]
            mean = int(r["depth_sum"]) / int(r["length"])
            sd = max(0.0, int(r["depth_sq_sum"]) / int(r["length"]) - mean * mean) ** 0.5
            assert f == [f"unitig_{i}", str(s["src"]), str(s["dst"]), str(r["length"]), str(r["reads"]), str(r["contained"]), str(r["read_count"]),
                         f"{mean:.4f}", f"{sd:.4f}", str(r["depth_min"]), str(r["depth_max"])]
    finally:
        ctx.close()


def interior_means(recs, depth, seqs, longest, assign):
    """length-weighted interior mean depth per key: bases at least `longest` from either end of unitigs of >= 1 kb, each unitig
    mapped to a key by assign(sequence) (None: skipped)."""
    tot, n = {}, {}
    for r in recs:
        L, a = int(r["length"]), int(r["start"])
        if L < 1000:
            continue
        key = assign(seqs[a:a + L].tobytes())
        if key is None:
            continue
        d = depth[a + longest:a + L - longest].astype(np.int64)
        tot[key] = tot.get(key, 0) + int(d.sum())
        n[key] = n.get(key, 0) + len(d)
    return {k: tot[k] / n[k] for k in tot if n[k]}


@pytest.mark.gpu
def test_abundance_config3():
    """Config 3 x 0.1: 20 genomes, log-normal weights w_g; genome g gets reads with probability w_g len_g / sum_h w_h len_h, so its
    expected depth is N 100 w_g / sum_h w_h len_h. Every genome at >= 10x is within 5 % of it."""
    from metagenomics_b200 import Context, synth
    scale = 0.1
    cfg = synth.config(3, scale=scale)
    gs, w = synth._metagenome(3, 20, 1e6, 5e6, scale)
    N = len(cfg["offsets"]) - 1
    lens = np.array([len(g) for g in gs], np.float64)
    lam = N * 100 * w / (w * lens).sum()
    fwd = [g.tobytes() for g in gs]
    rcs = [us.rc_bytes(g) for g in fwd]

    def assign(s):
        hits = [i for i in range(len(gs)) if s in fwd[i] or s in rcs[i]]
        return hits[0] if len(hits) == 1 else None

    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        og.simplify()
        recs, depth = og.depth()
        _, seqs = og.unitigs()
        got = interior_means(recs, depth, seqs, int(ds.longestReadLength), assign)
        ratios = {g: got.get(g, 0.0) / lam[g] for g in range(len(gs)) if lam[g] >= 10}
        print("config 3 x 0.1: interior mean / expected per genome (>= 10x):", {g: round(v, 4) for g, v in ratios.items()})
        assert ratios and all(abs(v - 1) <= 0.05 for v in ratios.values()), ratios
    finally:
        ctx.close()


@pytest.mark.gpu
def test_abundance_config5():
    """Config 5 x 0.1: one genome; total raw bases / genome length is the expected depth, duplicates and contained reads
    included (without the contained reads the interior mean falls short of it)."""
    from metagenomics_b200 import Context, synth
    scale = 0.1
    cfg = synth.config(5, scale=scale)
    glen = max(4000, int(20_000_000 * scale))
    g = synth.genome(5, glen).tobytes()
    grc = us.rc_bytes(g)
    lam = int(cfg["offsets"][-1]) / glen
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        og.simplify()
        recs, depth = og.depth()
        _, seqs = og.unitigs()
        got = interior_means(recs, depth, seqs, int(ds.longestReadLength), lambda s: 0 if (s in g or s in grc) else None)
        ratio = got[0] / lam
        print(f"config 5 x 0.1: interior mean {got[0]:.3f} / expected {lam:.3f} = {ratio:.4f}")
        assert abs(ratio - 1) <= 0.05, ratio
    finally:
        ctx.close()


FULL = json.load(open(os.path.join(GOLDEN, "coverage_full_size.json")))


@pytest.mark.gpu
@pytest.mark.parametrize("gold", FULL, ids=[f"config{g['config']}@{g['scale']}" for g in FULL])
def test_full_size_matches_golden(gold):
    from metagenomics_b200 import Context, synth
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_coverage_full_size", os.path.join(GOLDEN, "make_coverage_full_size.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    cfg = synth.config(gold["config"], scale=gold["scale"])
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        assert ds.getNumberOfUniqueReads() == gold["n_unique"]
        og.simplify()
        recs, depth = og.depth()
        srecs, _ = og.unitigs(ascii=False)
        _, st = og.coverage()
        assert st["unplaced"] == 0
        cov = {k: recs[k] for k in ("reads", "contained", "read_count", "depth_sum", "depth_sq_sum", "depth_min", "depth_max", "length", "start")}
        cov["depth"] = depth
        got = mk.figures(srecs["src"].astype(np.int64), srecs["dst"].astype(np.int64), cov, both_halves=False)
        want = {k: v for k, v in gold.items() if k not in ("config", "scale", "n_unique", "unplaced")}
        assert got == want
    finally:
        ctx.close()

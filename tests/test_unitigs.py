"""Unitig sequences of the simplified graph (ogb_graph_spell / ogb_graph_unitigs / ogb_graph_write_unitigs; the reference's
getStringInEdge, OverlapGraph.cpp:2009).

CPU: the plain restatement (oracle/unitig_spell.py) on the reference's own contracted graphs of the fixtures -- every read of every list
is the substring at its position, the length is offset + L[dst], the twin spells the reverse complement -- and the per-word body of
csrc/ogb_spell.cuh, run on the CPU (tests/spell_emul.cpp), against the restatement on the fixtures and the adversarial sets (m < 31
included). GPU: the kernels through the C ABI, the Python API, the driver's --unitigs, the assembly property on config 2 and the
full-size goldens (tests/golden/unitigs_full_size.json, tests/golden/make_unitigs_full_size.py)."""
import ctypes as C
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import datasets
from contract_lib import build_emul
from oracle_lib import Oracle
from unitig_lib import build_spell_emul, canonical_mask, reads_ascii, spell_graph, store_layout, us

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
    return g, dict(bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"]))


# ---------------------------------------------------------------- CPU


@pytest.mark.parametrize("name", FIXTURES)
def test_restatement_on_the_reference_graph(name):
    g, cfg = fixture(name)
    _, (fw, st, L) = host_reads(cfg)
    assert np.array_equal(L, g["len"].astype(np.int64))
    ce, ls, cl = g["c_edges"].astype(np.int64), g["c_list_start"].astype(np.int64), g["c_lists"].astype(np.int64)
    seqs = {}
    for i, (s, d, o, _, off) in enumerate(ce.tolist()):
        it = cl[ls[i]:ls[i + 1]]
        S = us.spell(fw, st, L, s, d, o, off, it[:, 0], it[:, 1], it[:, 2])
        assert len(S) == off + L[d - 1]
        for r, f, p in us._pieces(s, d, o, off, it[:, 0], it[:, 1], it[:, 2]):
            read = us.oriented(fw, st, L, r, f)
            assert S[p:p + len(read)] == read, (name, i, r)
        seqs.setdefault((s, d), []).append(S)
    for (s, d), ss in seqs.items():                                  # S(twin(e)) == rc(S(e)), as multisets per end-point pair
        assert sorted(ss) == sorted(us.rc_bytes(x) for x in seqs[(d, s)]), (name, s, d)
    flat, starts, lens = us.spell_all(fw, st, L, ce[:, 0], ce[:, 1], ce[:, 2], ce[:, 4], ls[:-1], ls[1:] - ls[:-1], cl[:, 0], cl[:, 1], cl[:, 2])
    for i, (s, d, o, _, off) in enumerate(ce.tolist()):             # the vectorised form is the same definition
        it = cl[ls[i]:ls[i + 1]]
        assert flat[starts[i]:starts[i] + lens[i]].tobytes() == us.spell(fw, st, L, s, d, o, off, it[:, 0], it[:, 1], it[:, 2])


@pytest.fixture(scope="module")
def emul():
    return build_emul(), build_spell_emul()


def simplified(cfg, contract):
    o = Oracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run_all(Oracle.THREE_PHASE, threads=8)
    edges, items, _ = contract(o.edges(), o.read_info()["len"])
    return edges, items


def check_body(cfg, edges, items, spell_emul):
    _, (fw, st, L) = host_reads(cfg)
    words, meta = store_layout(fw, st, L)
    for canon in (True, False):
        sel = canonical_mask(edges) if canon else np.ones(len(edges), bool)
        recs, got = spell_emul(words, meta, len(L), edges, items, canon)
        assert np.array_equal(recs["edge"], np.flatnonzero(sel))
        flat, starts, lens = spell_graph(fw, st, L, edges, items, sel)
        assert np.array_equal(recs["length"], lens) and np.array_equal(recs["src"], edges["src"][sel]) and np.array_equal(recs["orient"], edges["orient"][sel])
        want, wstart = us.pack(flat, starts, lens)
        assert np.array_equal(recs["start"], 32 * wstart)
        assert np.array_equal(got, want), cfg.get("name")


@pytest.mark.parametrize("name", FIXTURES)
def test_kernel_body_matches_restatement_on_fixtures(name, emul):
    contract, spell_emul = emul
    g, cfg = fixture(name)
    edges, items, _ = contract(g["edges"], g["len"])
    check_body(cfg, edges, items, spell_emul)


def test_kernel_body_matches_restatement_on_adversarial_sets(emul):
    """tandem (m 24) and palindromes (m 20) take the loop over several reads per word."""
    contract, spell_emul = emul
    sets = datasets.adversarial() + [datasets.paired_mixed()]
    assert min(c["min_overlap"] for c in sets) < 31
    for cfg in sets:
        edges, items = simplified(cfg, contract)
        check_body(cfg, edges, items, spell_emul)


def test_layout_and_binding():
    from metagenomics_b200._lib import PROTOTYPES, SpellStats
    from metagenomics_b200.api import UNITIG_DTYPE
    assert UNITIG_DTYPE.itemsize == 32 and UNITIG_DTYPE.fields["orient"][1] == 12 and UNITIG_DTYPE.fields["length"][1] == 16
    assert UNITIG_DTYPE.fields["start"][1] == 24
    assert C.sizeof(SpellStats) == 32 and SpellStats.launches.offset == 24 and SpellStats.ms.offset == 28
    for n in ("ogb_graph_spell", "ogb_graph_unitigs", "ogb_graph_write_unitigs"):
        assert n in PROTOTYPES


def test_entry_points_fail_without_gpu():
    """No GPU: no context can be made (OGB_E_CUDA), and the new entry points refuse a missing one instead of touching memory."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from metagenomics_b200 import Context, OgbError
    from metagenomics_b200._lib import SpellStats, lib
    with pytest.raises(OgbError) as e:
        Context(0)
    assert e.value.code == 2
    st = SpellStats()
    assert lib().ogb_graph_spell(None, 1, 0, 2**64 - 1, C.byref(st)) == 1
    assert lib().ogb_graph_unitigs(None, None, 0, None, 0, 1) == 1
    assert lib().ogb_graph_write_unitigs(None, b"/nonexistent") == 1


def test_driver_refuses_unitigs_on_resume(tmp_path):
    r = subprocess.run([EXE, "-l", "50", "-se", "1", str(tmp_path / "in.fa"), "-f", str(tmp_path / "p"), "-s", "--unitigs", str(tmp_path / "u.fa")],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--unitigs" in r.stderr
    assert not (tmp_path / "u.fa").exists()


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
            for canon in (True, False):
                sel = canonical_mask(edges) if canon else np.ones(len(edges), bool)
                flat, starts, lens = spell_graph(fw, st, L, edges, items, sel)
                recs, seq = og.unitigs(canonical=canon, ascii=True)
                assert np.array_equal(recs["edge"], np.flatnonzero(sel)) and np.array_equal(recs["length"], lens), cfg["name"]
                assert np.array_equal(recs["src"], edges["src"][sel]) and np.array_equal(recs["dst"], edges["dst"][sel])
                assert np.array_equal(recs["orient"], edges["orient"][sel])
                idx = np.repeat(recs["start"].astype(np.int64), lens) + (np.arange(int(lens.sum())) - np.repeat(starts, lens))
                assert np.array_equal(seq[idx], flat), cfg["name"]
                recs2, words = og.unitigs(canonical=canon, ascii=False)
                want, wstart = us.pack(flat, starts, lens)
                assert np.array_equal(recs2, recs) and np.array_equal(recs["start"], 32 * wstart)
                assert np.array_equal(words, want), cfg["name"]
    finally:
        ctx.close()


@pytest.mark.gpu
def test_ranges_concatenate_to_the_whole():
    from metagenomics_b200 import Context, synth
    from metagenomics_b200.dist import unitig_range
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, synth.config(3, scale=0.004))
        edges, _, _ = og.simplify()
        for canon in (True, False):
            recs, words = og.unitigs(canonical=canon, ascii=False)
            assert len(recs) > 3
            for world in (2, 3, 7):
                parts = [og.unitigs(canonical=canon, ascii=False, first=f, count=n) for f, n in (unitig_range(edges, r, world, canon) for r in range(world))]
                got_r = np.concatenate([p[0] for p in parts])
                assert np.array_equal(got_r[["edge", "src", "dst", "orient", "length"]], recs[["edge", "src", "dst", "orient", "length"]])
                assert np.array_equal(np.concatenate([p[1] for p in parts]), words)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_error_paths():
    from metagenomics_b200 import Context, OgbError, synth
    from metagenomics_b200._lib import lib
    from metagenomics_b200.api import UNITIG_DTYPE
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, synth.config(1, scale=0.2))
        with pytest.raises(OgbError) as e:
            og.spell()
        assert e.value.code == 4                                     # OGB_E_STATE: no simplified graph yet
        og.simplify()
        st = og.spell()
        assert st["unitigs"] > 0 and st["words"] > 0 and st["bases"] > 0
        recs = np.zeros(st["unitigs"], UNITIG_DTYPE)
        small = np.zeros(st["words"] - 1, np.uint64)
        rc = lib().ogb_graph_unitigs(ctx._h, recs.ctypes.data, len(recs), small.ctypes.data, small.nbytes, 0)
        msg = lib().ogb_last_error().decode()
        assert rc == 5 and f"{st['unitigs']} records" in msg and f"{8 * st['words']} bytes" in msg
        rc = lib().ogb_graph_unitigs(ctx._h, recs.ctypes.data, len(recs) - 1, small.ctypes.data, 8 * st["words"], 0)
        assert rc == 5
        with pytest.raises(OgbError) as e:
            og.spell(first=st["unitigs"] + 1)
        assert e.value.code == 1
        assert og.spell(first=st["unitigs"])["unitigs"] == 0
        og.buildOverlapGraphFromHashTable()                           # a new build invalidates the spelled unitigs
        rc = lib().ogb_graph_unitigs(ctx._h, recs.ctypes.data, len(recs), small.ctypes.data, small.nbytes, 0)
        assert rc == 4
    finally:
        ctx.close()


def read_fasta(path):
    lines = open(path, "rb").read().split(b"\n")
    assert lines[-1] == b""
    return list(zip(lines[0:-1:2], lines[1:-1:2]))


@pytest.mark.gpu
def test_driver_writes_what_the_api_writes(tmp_path):
    from metagenomics_b200 import Context, synth
    g = np.load(os.path.join(GOLDEN, "palindromes.npz"))
    cfg = dict(bases=g["bases"], offsets=g["offsets"], min_overlap=int(g["min_overlap"]))
    fa = str(tmp_path / "in.fa")
    synth.write_fasta(fa, g["bases"], g["offsets"])
    m = str(cfg["min_overlap"])
    base = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "a")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    uni = subprocess.run([EXE, "-l", m, "-se", "1", fa, "-f", str(tmp_path / "b"), "--unitigs", str(tmp_path / "drv.fa")],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert base.returncode == 0 and uni.returncode == 0, base.stdout + uni.stdout
    # without --unitigs: the same .unitig file and the same report line as before (its timings aside), and nothing more
    assert open(tmp_path / "a.unitig", "rb").read() == open(tmp_path / "b.unitig", "rb").read()
    lb, lu = base.stdout.strip().split("\n"), uni.stdout.strip().split("\n")
    assert len(lb) == 1 and lb[0].split(" device ms")[0] == lu[0].split(" device ms")[0] and lu[1].startswith("unitigs: ")
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        edges, items, _ = og.simplify()
        st = og.write_unitigs(str(tmp_path / "api.fa"))
        assert open(tmp_path / "api.fa", "rb").read() == open(tmp_path / "drv.fa", "rb").read()
        recs, seq = og.unitigs()
        fw, s0, L = reads_ascii(ds)
        flat, starts, lens = spell_graph(fw, s0, L, edges, items, canonical_mask(edges))
        got = read_fasta(tmp_path / "api.fa")
        assert len(got) == st["unitigs"] == len(recs)
        for i, (h, s) in enumerate(got):
            r = recs[i]
            e = edges[r["edge"]]
            assert h == b">unitig_%d src=%d dst=%d orient=%d reads=%d length=%d" % (i, r["src"], r["dst"], r["orient"], e["count"] + 2, r["length"])
            assert s == flat[starts[i]:starts[i] + lens[i]].tobytes()
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [0.1, 1.0])
def test_canonical_unitigs_are_genome_substrings(scale):
    """Config 2 samples one genome, synth.genome(2, 5 Mb x scale), without errors: every canonical unitig is a substring of it or
    of its reverse complement. The covered fraction is printed, not asserted."""
    from metagenomics_b200 import Context, synth
    cfg = synth.config(2, scale=scale)
    genome = synth.genome(2, max(4000, int(5_000_000 * scale))).tobytes()
    grc = us.rc_bytes(genome)
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        og.simplify()
        recs, seq = og.unitigs()
        assert len(recs) > 0
        for r in recs:
            s = seq[int(r["start"]):int(r["start"]) + int(r["length"])].tobytes()
            assert s in genome or s in grc, (int(r["edge"]), int(r["length"]))
        print(f"config 2 x {scale}: {len(recs)} canonical unitigs, {int(recs['length'].sum())} bases = "
              f"{recs['length'].sum() / len(genome):.6f} of the {len(genome)}-base genome, longest {int(recs['length'].max())}")
    finally:
        ctx.close()


FULL = json.load(open(os.path.join(GOLDEN, "unitigs_full_size.json")))


@pytest.mark.gpu
@pytest.mark.parametrize("gold", FULL, ids=[f"config{g['config']}@{g['scale']}" for g in FULL])
def test_full_size_matches_golden(gold):
    from metagenomics_b200 import Context, synth
    cfg = synth.config(gold["config"], scale=gold["scale"])
    ctx = Context(0)
    try:
        ds, og = device_graph(ctx, cfg)
        assert ds.getNumberOfUniqueReads() == gold["n_unique"]
        og.simplify()
        recs, seq = og.unitigs()
        assert len(recs) == gold["unitigs"] and int(recs["length"].sum()) == gold["bases"]
        h = us.seq_hashes(seq, recs["start"], recs["length"])
        hr = us.seq_hashes(seq, recs["start"], recs["length"], reverse_complement=True)
        assert us.checksum(us.unitig_terms(recs["src"], recs["dst"], recs["orient"], h, hr)) == gold["checksum"]
    finally:
        ctx.close()


@pytest.mark.gpu
def test_two_ranks_split_the_unitigs():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29612", os.path.join(HERE, "unitig_dist_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:]
    assert r.stdout.count("unitig range identical") == 2, r.stdout[-2000:]

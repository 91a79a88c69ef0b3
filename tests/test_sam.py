"""SAM output of a sample (ogb_graph_map_reads_sam, csrc/ogb_sam.cuh).

CPU: the restatement (tests/sam_lib.py) against map_sample_approx -- pileup, NM / MD against the unitig bytes, every raw read, FLAG,
NH and record counts; the per-thread bodies of csrc/ogb_sam.cuh run on the CPU (tests/sam_emul.cpp) against the restatement byte for
byte for d = 0..3 on the fixtures, the adversarial sets and paired_mixed, both selections, with and without names, in both walk
orders; read names from FASTA / FASTQ files; the refusals without a GPU.
GPU: the device SAM against the restatement byte for byte (d = 0..3, both selections, unitig ranges); the same placements, records,
profile, hits and strata as ogb_graph_map_reads_approx, and the same bytes twice; config 3 at full size with errors (pileup = profile);
a sample across the chunk bound and many text slices; the driver's --sam; error paths."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from map_lib import filter_sample, join_reads, sm, split_reads, unitig_seqs
from sam_lib import FILTERED, check_md, header, parse, pileup, sam_records, sam_text
from test_sample_map_mismatches import (FIXTURES, adversarial_graphs, device_graph, emul as _emul_fixture, fixture, gpu_sets, spelled,  # noqa: F401
                                        substitute_read, substituted_sample)
from unitig_lib import store_layout

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EXE = os.path.join(ROOT, "metagenomics_b200", "host", "ogb_overlap")

emul = _emul_fixture


# ---------------------------------------------------------------- helpers


def build_sam_emul():
    """Compiles tests/sam_emul.cpp and returns run(words, recs, reads, m, d, first, names, reverse) -> the records' text"""
    out = os.path.join(HERE, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libsam_emul.so")
    src = os.path.join(HERE, "sam_emul.cpp")
    hdrs = [os.path.join(ROOT, "metagenomics_b200", "csrc", h) for h in ("ogb_sam.cuh", "ogb_map.cuh", "ogb_coverage.cuh", "ogb_spell.cuh")] + [
        os.path.join(ROOT, "include", "ogb.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in [src] + hdrs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.emul_sam.restype = C.c_uint64
    lib.emul_sam.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, C.POINTER(C.c_char_p)]

    def run(words, recs, reads, m, d, first=0, names=None, reverse=False):
        ks = [sm.kept(bytes(r), m) for r in reads]
        kept = [s for s in ks if s is not None]
        L = np.array([len(s) for s in kept], np.int64)
        starts = np.concatenate([[0], np.cumsum(L)])[:-1].astype(np.int64)
        fw = np.frombuffer(b"".join(kept), np.uint8).copy() if kept else np.zeros(0, np.uint8)
        rwords, rmeta = store_layout(fw, starts, L)
        rmeta = np.ascontiguousarray(rmeta if len(rmeta) else np.zeros(1, np.uint64), np.uint64)
        rwords = np.ascontiguousarray(rwords, np.uint64)
        raw, roffs = join_reads([bytes(r) for r in reads])
        raw = np.concatenate([raw, np.zeros(1, np.uint8)])
        good = np.array([s is not None for s in ks] + [0], np.uint32)
        nb = no = None
        if names is not None:
            nb, no = join_reads(names)
            nb = np.concatenate([nb, np.zeros(1, np.uint8)])
        words = np.ascontiguousarray(words, np.uint64)
        recs = np.ascontiguousarray(recs)
        txt = C.c_char_p()
        n = lib.emul_sam(words.ctypes.data, len(words), recs.ctypes.data, len(recs), raw.ctypes.data, roffs.ctypes.data, len(reads), good.ctypes.data,
                         rwords.ctypes.data, rmeta.ctypes.data, None if nb is None else nb.ctypes.data, None if no is None else no.ctypes.data, m, d,
                         first, 1 if reverse else 0, C.byref(txt))
        assert n != 2**64 - 1, "a line did not fill its counted bytes, or the emit found another placement count"
        return C.string_at(txt, n) if n else b""
    return run


def names_for(reads, seed):
    """QNAMEs over the whole allowed alphabet [!-?A-~], 1 to 254 characters"""
    rng = np.random.default_rng(seed)
    alpha = np.array([c for c in range(0x21, 0x7F) if c != 0x40], np.uint8)
    return [alpha[rng.integers(0, len(alpha), int(rng.choice([1, 5, 20, 254])))].tobytes() for _ in reads]


def edge_reads(seqs, m, rng):
    """reads that end at a unitig's end or start at 0 (either strand), and whole short unitigs, with 0 or 1 substitution"""
    out = []
    for s in seqs[:40]:
        for L in (m + 1, 2 * min(32, m + 1) + 3, 100):
            if len(s) >= L:
                for r in (s[:L], s[-L:], sm.rc(s[-L:])):
                    out.append(substitute_read(rng, r, int(rng.integers(0, 2))))
        if m < len(s) <= 300:
            out.append(s)
    return out


def check_restatement(seqs, reads, m, d, want_text, want):
    """the restatement's own invariants: pileup == depth, NM / MD against the unitig bytes, every raw read, FLAG / NH / counts"""
    lines = want_text.splitlines(keepends=True)
    recs = [parse(x) for x in lines]
    hits = want["hits"]
    assert len(recs) == sum(1 if h == FILTERED else max(1, int(h)) for h in hits)
    depth = np.concatenate(pileup(lines, [len(s) for s in seqs])) if seqs else np.zeros(0)
    assert np.array_equal(depth, want["depth"])
    k = 0
    for i, h in enumerate(hits.tolist()):
        n = 1 if h == FILTERED else max(1, h)
        for j, r in enumerate(recs[k:k + n]):
            assert r["qname"] == b"%d" % i
            if h == FILTERED:
                assert r["flag"] == 4 and r["YF"] == b"filtered"
            elif h == 0:
                assert r["flag"] == 4 and r["seq"] == sm.kept(bytes(reads[i]), m)
            else:
                assert r["flag"] & ~16 == (256 if j else 0) and r["NH"] == h and r["mapq"] == (60 if h == 1 else 0)
                u = int(r["rname"][7:])
                check_md(seqs[u][r["pos"] - 1:r["pos"] - 1 + len(r["seq"])], r["seq"], r["MD"], r["NM"])
                assert r["NM"] == want["mismatches"][i]
                assert r["seq"] == (sm.rc(sm.kept(bytes(reads[i]), m)) if r["flag"] & 16 else sm.kept(bytes(reads[i]), m))
        k += n


# ---------------------------------------------------------------- CPU


@pytest.fixture(scope="module")
def sam_emul():
    return build_sam_emul()


def test_restatement_invariants(emul):
    contract, spell_emul, _ = emul
    for cfg, edges, items in adversarial_graphs(contract):
        m = cfg["min_overlap"]
        _, _, seqs = spelled(cfg, edges, items, spell_emul, True)
        for d in range(4):
            reads = substituted_sample(seqs, m, d, seed=40 + d) + filter_sample(seqs, m)[:60] + edge_reads(seqs, m, np.random.default_rng(d))
            text, want = sam_records(seqs, reads, m, d)
            check_restatement(seqs, reads, m, d, text, want)


def check_bodies(cfg, edges, items, spell_emul, run, extra=()):
    m = cfg["min_overlap"]
    raw = split_reads(cfg["bases"], cfg["offsets"])
    for canon in (True, False):
        packed, srecs, seqs = spelled(cfg, edges, items, spell_emul, canon)
        for d in range(4):
            rng = np.random.default_rng(d)
            noisy = [substitute_read(rng, sm.kept(r, m), int(rng.integers(0, d + 2))) if sm.kept(r, m) else r for r in raw[:200]]
            samples = [noisy, filter_sample(seqs, m)[:120], substituted_sample(seqs, m, d, seed=10 + d), edge_reads(seqs, m, rng)]
            for k, reads in enumerate(samples + [s(seqs) for s in extra]):
                want, _ = sam_records(seqs, reads, m, d, first=3 * k)
                names = names_for(reads, k) if k % 2 else None
                if names is not None:
                    want, _ = sam_records(seqs, reads, m, d, first=3 * k, names=names)
                for rev in (False, True):
                    got = run(packed, srecs, reads, m, d, first=3 * k, names=names, reverse=rev)
                    assert got == want, (cfg.get("name"), canon, d, k, rev)


@pytest.mark.parametrize("name", FIXTURES)
def test_kernel_bodies_match_restatement_on_fixtures(name, emul, sam_emul):
    contract, spell_emul, _ = emul
    g, cfg = fixture(name)
    edges, items, _ = contract(g["edges"], g["len"])
    check_bodies(cfg, edges, items, spell_emul, sam_emul)


def test_kernel_bodies_match_restatement_on_adversarial_sets(emul, sam_emul):
    """tandem repeats: reads with hundreds of placements (the heap sort) and ties; palindromes: the strand rule; K < 32; samples of
    0 and 1 reads."""
    contract, spell_emul, _ = emul
    for cfg, edges, items in adversarial_graphs(contract):
        check_bodies(cfg, edges, items, spell_emul, sam_emul, extra=(lambda s: [], lambda s: [s[0]] if s else [b"ACGT"]))


def packed_layout(seqs):
    """(words, UNITIG_DTYPE records) of sequences laid out like a spell: each from a multiple of 32 bases, 2 bits a base"""
    from metagenomics_b200.api import UNITIG_DTYPE
    recs = np.zeros(len(seqs), UNITIG_DTYPE)
    words, pos = [], 0
    for u, s in enumerate(seqs):
        recs[u]["length"], recs[u]["start"] = len(s), pos
        code = np.frombuffer(bytes(s).translate(bytes.maketrans(b"ACGT", b"\0\1\2\3")), np.uint8).astype(np.uint64)
        code = np.concatenate([code, np.zeros((-len(code)) % 32, np.uint64)]).reshape(-1, 32)
        words.append((code << (np.uint64(62) - np.uint64(2) * np.arange(32, dtype=np.uint64))).sum(axis=1, dtype=np.uint64))
        pos += 32 * len(code)
    return np.concatenate(words), recs


def test_many_placements_are_sorted(sam_emul):
    """reads inside tandem repeats: hundreds of placements each (the heap-sort path of sm_sort), on both strands, with and without
    substitutions, sorted by (u, p) whatever the walk order"""
    rng = np.random.default_rng(8)
    unit = b"ACGTTGACCA"
    seqs = [unit * 60, rng.choice(list(b"ACGT"), 500).astype(np.uint8).tobytes() + unit * 40, sm.rc(unit * 50)]
    words, recs = packed_layout(seqs)
    reads = [(unit * 20)[3:103], sm.rc((unit * 20)[:100]), substitute_read(rng, (unit * 20)[5:105], 1), seqs[1][490:590], (unit * 20)[:64]]
    for d in range(4):
        text, want = sam_records(seqs, reads, 50, d)
        assert int(want["hits"].max()) > 100, want["hits"]
        check_restatement(seqs, reads, 50, d, text, want)
        assert sam_emul(words, recs, reads, 50, d) == text and sam_emul(words, recs, reads, 50, d, reverse=True) == text


def test_header_layout():
    assert header([10, 2000], 2, first=5) == (b"@HD\tVN:1.6\tSO:unsorted\n@SQ\tSN:unitig_5\tLN:10\n@SQ\tSN:unitig_6\tLN:2000\n"
                                             b"@PG\tID:ogb_map\tPN:ogb\tCL:max_mismatches=2\n")


def dataset_reads(path, keep):
    from metagenomics_b200._lib import check, lib
    ds = C.c_void_p()
    check(lib().ogb_dataset_create(C.byref(ds)))
    try:
        if keep:
            check(lib().ogb_dataset_keep_names(ds))
        check(lib().ogb_dataset_add_file(ds, str(path).encode()))
        b, o, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(lib().ogb_dataset_raw_reads(ds, C.byref(b), C.byref(o), C.byref(n)))
        offs = np.ctypeslib.as_array(C.cast(o, C.POINTER(C.c_uint64)), shape=(n.value + 1,)).copy()
        reads = [C.string_at(b.value + int(offs[i]), int(offs[i + 1] - offs[i])) for i in range(n.value)]
        names = None
        nb, no = C.c_void_p(), C.c_void_p()
        rc = lib().ogb_dataset_raw_names(ds, C.byref(nb), C.byref(no))
        if keep:
            assert rc == 0
            noff = np.ctypeslib.as_array(C.cast(no, C.POINTER(C.c_uint64)), shape=(n.value + 1,)).copy()
            names = [C.string_at(nb.value + int(noff[i]), int(noff[i + 1] - noff[i])) for i in range(n.value)]
        else:
            assert rc == 4                                                   # OGB_E_STATE: no names kept
        return reads, names
    finally:
        lib().ogb_dataset_destroy(ds)


@pytest.mark.parametrize("eol", [b"\n", b"\r\n"])
def test_parser_keeps_names(tmp_path, eol):
    fa = tmp_path / "a.fa"
    fa.write_bytes(eol.join([b">r1 some description", b"ACGT", b"acgg", b">r2\tx y", b"TTTT", b">r3", b"", b">x:y/1  z", b"GG"]) + eol)
    fq = tmp_path / "a.fq"
    fq.write_bytes(eol.join([b"@q/1 1:N:0", b"ACGTN", b"+", b"IIIII", b"@q/2\tt", b"CCC", b"+q/2", b"III", b"@q3", b"", b"+", b""]) + eol)
    for path, want_r, want_n in ((fa, [b"ACGTacgg", b"TTTT", b"", b"GG"], [b"r1", b"r2", b"r3", b"x:y/1"]),
                                 (fq, [b"ACGTN", b"CCC", b""], [b"q/1", b"q/2", b"q3"])):
        r0, n0 = dataset_reads(path, False)
        r1, n1 = dataset_reads(path, True)
        assert r0 == r1 == want_r and n0 is None and n1 == want_n, (r1, n1)


_PARSE = """
import ctypes as C, json, sys
sys.path.insert(0, sys.argv[1])
from metagenomics_b200._lib import lib
ds = C.c_void_p()
assert lib().ogb_dataset_create(C.byref(ds)) == 0
if sys.argv[3] == "1":
    assert lib().ogb_dataset_keep_names(ds) == 0
rc = lib().ogb_dataset_add_file(ds, sys.argv[2].encode())
b, o, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
assert lib().ogb_dataset_raw_reads(ds, C.byref(b), C.byref(o), C.byref(n)) == 0
offs = [C.cast(o, C.POINTER(C.c_uint64))[i] for i in range(n.value + 1)]
print(json.dumps([rc, [C.string_at(b.value + offs[i], offs[i + 1] - offs[i]).decode() for i in range(n.value)]]))
"""


@pytest.mark.parametrize("eol", [b"\n", b"\r\n"])
@pytest.mark.parametrize("body", [[b"@r1", b"ACGT", b"+", b"IIII", b""], [b"@r1", b"ACGT", b"+", b"IIII", b"", b""], [b"", b">r1", b"ACGT"],
                                  [b"", b"@r1", b"ACGT", b"+", b"IIII"], [b">r1", b"ACGT", b">", b"GG", b""], [b"@", b"ACGT", b"+", b"IIII"]],
                         ids=["fq_blank_end", "fq_two_blank_end", "fa_blank_start", "fq_blank_start", "fa_empty_header", "fq_empty_header"])
def test_parser_blank_lines_same_with_names(tmp_path, eol, body):
    """Empty lines where a header may be read (a trailing blank line, a leading one, a bare '>' or '@'): keeping names changes
    neither the return code nor the reads, and the process survives (each parse runs in its own interpreter)."""
    path = tmp_path / "s.txt"
    path.write_bytes(eol.join(body) + eol)
    got = []
    for keep in ("0", "1"):
        r = subprocess.run([sys.executable, "-c", _PARSE, ROOT, str(path), keep], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
        got.append(json.loads(r.stdout))
    assert got[0] == got[1], got


def test_keep_names_only_before_reads():
    from metagenomics_b200._lib import check, lib
    ds = C.c_void_p()
    check(lib().ogb_dataset_create(C.byref(ds)))
    try:
        b, o = join_reads([b"ACGT"])
        check(lib().ogb_dataset_add_reads(ds, b.ctypes.data, o.ctypes.data, 1))
        assert lib().ogb_dataset_keep_names(ds) == 4
    finally:
        lib().ogb_dataset_destroy(ds)


def test_entry_point_refuses_null_context_and_no_gpu(tmp_path):
    """a NULL context is OGB_E_ARG before anything is opened; without a GPU no context can be made for the call at all"""
    import torch
    from metagenomics_b200._lib import MapStats, SamStats, lib
    b, o = join_reads([b"ACGT" * 20])
    nb, no = join_reads([b"r1"])
    assert lib().ogb_graph_map_reads_sam(None, b.ctypes.data, o.ctypes.data, 1, nb.ctypes.data, no.ctypes.data, 2, str(tmp_path / "x.sam").encode(),
                                         None, None, C.byref(MapStats()), C.byref(SamStats())) == 1
    assert not (tmp_path / "x.sam").exists()
    if not torch.cuda.is_available():
        h = C.c_void_p()
        assert lib().ogb_context_create(C.byref(h), 0) != 0 and not h.value


def test_binding_and_layout():
    from metagenomics_b200._lib import PROTOTYPES, SamStats
    assert C.sizeof(SamStats) == 40
    for f in ("ogb_graph_map_reads_sam", "ogb_dataset_keep_names", "ogb_dataset_raw_names"):
        assert f in PROTOTYPES
    hdr = open(os.path.join(ROOT, "include", "ogb.h")).read()
    assert "} ogb_sam_stats; /* 40 bytes */" in hdr and "} ogb_map_stats; /* 88 bytes */" in hdr


@pytest.mark.parametrize("args", [["--sam", "out"], ["--depths", "d.tsv", "--sam", "out"], ["--samples", "1", "x.fa", "--sam", "out"],
                                  ["-s", "--samples", "1", "x.fa", "--depths", "d.tsv", "--sam", "out"],
                                  ["--samples", "2", "a/x.fa", "b/x.fa", "--depths", "d.tsv", "--sam", "out"],
                                  ["--samples", "1", "x.fa", "--depths", "d.tsv", "--sam"]])
def test_driver_refuses_sam_without_samples(tmp_path, args):
    r = subprocess.run([EXE, "-l", "50", "-se", "1", str(tmp_path / "in.fa"), "-f", str(tmp_path / "p")] + args, cwd=tmp_path,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--sam" in r.stderr, r.stderr
    assert not (tmp_path / "d.tsv").exists() and not (tmp_path / "out").exists()


# ---------------------------------------------------------------- GPU


def device_sam(og, reads, d, path, names=None, **kw):
    recs, st, hits, mis = og.map_reads(reads, hits=True, max_mismatches=d, strata=True, sam=path, names=names, **kw)
    return recs, st, hits, mis, open(path, "rb").read()


@pytest.mark.gpu
def test_device_matches_restatement(tmp_path):
    from metagenomics_b200 import Context
    from metagenomics_b200.dist import unitig_range
    ctx = Context(0)
    path = str(tmp_path / "s.sam")
    try:
        for cfg in gpu_sets():
            _, og = device_graph(ctx, cfg)
            edges, _, _ = og.simplify()
            m = cfg["min_overlap"]
            raw = split_reads(cfg["bases"], cfg["offsets"])
            for canon in (True, False):
                for d in range(4):
                    srecs, ascii = og.unitigs(canonical=canon)                # (the ranges below leave another spell behind)
                    seqs = unitig_seqs(srecs, ascii)
                    rng = np.random.default_rng(d)
                    noisy = [substitute_read(rng, sm.kept(r, m), int(rng.integers(0, d + 2))) if sm.kept(r, m) else r for r in raw[:300]]
                    samples = [noisy, substituted_sample(seqs, m, d, seed=20 + d) + filter_sample(seqs, m)[:80] + edge_reads(seqs, m, rng), []]
                    for k, reads in enumerate(samples):
                        names = names_for(reads, k) if k == 1 else None
                        _, st, hits, mis, got = device_sam(og, reads, d, path, names=names)
                        want, ref = sam_text(seqs, reads, m, d, names=names)
                        assert got == want, (cfg.get("name"), canon, d, k)
                        assert np.array_equal(hits, ref["hits"]) and np.array_equal(mis, ref["mismatches"])
                        assert st["sam"]["records"] == len(want.splitlines()) - len(seqs) - 2 and st["sam"]["bytes"] == len(want)
                    for world in ((2, 3) if d in (0, 2) else ()):
                        for r in range(world):
                            f, n = unitig_range(edges, r, world, canon)
                            srecs, ascii = og.unitigs(canonical=canon, first=f, count=n)
                            sub = unitig_seqs(srecs, ascii)
                            _, _, _, _, got = device_sam(og, noisy, d, path)
                            assert got == sam_text(sub, noisy, m, d, first=f)[0], (cfg.get("name"), canon, d, world, r)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_sam_call_is_a_pure_addition(tmp_path):
    """records, profile, hits and strata of the SAM call == ogb_graph_map_reads_approx; two runs write the same bytes; the samples
    list grows by one per call either way"""
    from metagenomics_b200 import Context, synth
    ctx = Context(0)
    try:
        cfg = synth.config(5, scale=0.01)
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        b = synth.substitute(4, cfg["bases"], 0.01)
        for d in (0, 2):
            r0, s0, h0, m0 = og.map_reads(bases=b, offsets=cfg["offsets"], hits=True, max_mismatches=d, strata=True)
            p0 = og.sample_depth()[1]
            r1, s1, h1, m1 = og.map_reads(bases=b, offsets=cfg["offsets"], hits=True, max_mismatches=d, strata=True, sam=str(tmp_path / "a.sam"))
            p1 = og.sample_depth()[1]
            og.map_reads(bases=b, offsets=cfg["offsets"], max_mismatches=d, sam=str(tmp_path / "b.sam"))
            assert r0.tobytes() == r1.tobytes() and p0.tobytes() == p1.tobytes() and h0.tobytes() == h1.tobytes() and m0.tobytes() == m1.tobytes()
            same = lambda st: {k: v for k, v in st.items() if not k.startswith("ms") and k not in ("sample", "launches", "sam")}   # noqa: E731
            assert same(s0) == same(s1) and s1["sample"] == s0["sample"] + 1 and "sam" in s1 and "sam" not in s0
            assert open(tmp_path / "a.sam", "rb").read() == open(tmp_path / "b.sam", "rb").read()
    finally:
        ctx.close()


def stream_check(path, srecs, profile, hits):
    """streaming parse of a SAM: pileup == profile on every base, record count == sum of max(1, hits) (1 per filtered read)"""
    lengths = srecs["length"].astype(np.int64)
    diff = [np.zeros(int(L) + 1, np.int64) for L in lengths]
    n = 0
    with open(path, "rb") as f:
        for ln in f:
            if ln[:1] == b"@":
                continue
            n += 1
            a = ln.split(b"\t", 6)
            if int(a[1]) & 4:
                continue
            u, p, L = int(a[2][7:]), int(a[3]) - 1, int(a[5][:-1])
            diff[u][p] += 1
            diff[u][p + L] -= 1
    h = hits.astype(np.int64)
    assert n == int(np.where(hits == FILTERED, 1, np.maximum(h, 1)).sum())
    for u, (a, L) in enumerate(zip(srecs["start"].tolist(), lengths.tolist())):
        assert np.array_equal(np.cumsum(diff[u][:-1]), profile[a:a + L].astype(np.int64)), u


@pytest.mark.gpu
def test_config3_full_size_with_errors(tmp_path):
    """config 3 at full size, its reads with 0.5 % substitutions at d = 2 (three chunks, dozens of text slices)"""
    from metagenomics_b200 import Context, synth
    cfg = synth.config(3)
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        srecs, _ = og.unitigs()
        b = synth.substitute(31, cfg["bases"], 0.005)
        path = str(tmp_path / "c3.sam")
        _, st, hits = og.map_reads(bases=b, offsets=cfg["offsets"], hits=True, max_mismatches=2, sam=path)
        profile = og.sample_depth()[1]
        assert st["reads_in"] > 2 * (1 << 22) and st["sam"]["bytes"] > 8 * (64 << 20) and os.path.getsize(path) == st["sam"]["bytes"]
        stream_check(path, srecs, profile, hits)
        print(f"config 3 SAM: {st['sam']}")
    finally:
        ctx.close()


@pytest.mark.gpu
def test_chunk_bound_and_slices(tmp_path):
    """2^22 + 5000 named reads in one call == the same reads in two calls split off the chunk bound, record for record"""
    from metagenomics_b200 import Context, synth
    cfg = synth.config(3)
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        n = (1 << 22) + 5000
        o = cfg["offsets"][:n + 1]
        b = synth.substitute(7, cfg["bases"][:int(o[-1])], 0.005)
        names = np.array([b"r%d" % i for i in range(n)], dtype=object)
        whole = str(tmp_path / "w.sam")
        og.map_reads(bases=b, offsets=o, max_mismatches=1, sam=whole, names=list(names))
        cut = (1 << 22) - 777
        parts = []
        for a, z in ((0, cut), (cut, n)):
            p = str(tmp_path / f"p{a}.sam")
            og.map_reads(bases=b[int(o[a]):int(o[z])], offsets=o[a:z + 1] - o[a], max_mismatches=1, sam=p, names=list(names[a:z]))
            parts.append(p)

        def body(p):
            with open(p, "rb") as f:
                t = f.read()
            return t[t.index(b"\n", t.index(b"@PG")) + 1:]
        w = body(whole)
        assert len(w) > 4 * (64 << 20) and w == body(parts[0]) + body(parts[1])
    finally:
        ctx.close()


@pytest.mark.gpu
def test_driver_sam_writes_what_the_api_writes(tmp_path):
    from metagenomics_b200 import Context, synth
    cfg = synth.config(5, scale=0.002)
    fa = str(tmp_path / "in.fa")
    synth.write_fasta(fa, cfg["bases"], cfg["offsets"])
    gs = [synth.genome(5, max(4000, int(20_000_000 * 0.002)))]
    os.makedirs(tmp_path / "s")
    s1, s2 = str(tmp_path / "s" / "a.fa"), str(tmp_path / "s" / "b.fq")
    b1, o1 = synth.sample_reads(21, gs, 3000, 100)
    synth.write_fasta(s1, synth.substitute(1, b1, 0.01), o1)
    b2, o2 = synth.sample_reads(22, gs, 6000, 75, 150)
    b2 = synth.substitute(2, b2, 0.01)
    with open(s2, "wb") as f:
        for i in range(len(o2) - 1):
            r = b2[int(o2[i]):int(o2[i + 1])].tobytes()
            f.write(b"@q%d extra\n%s\n+\n%s\n" % (i, r, b"I" * len(r)))
    r = subprocess.run([EXE, "-l", str(cfg["min_overlap"]), "-se", "1", fa, "-f", str(tmp_path / "x"), "--samples", "2", s1, s2, "--depths",
                        str(tmp_path / "x.tsv"), "--mismatches", "2", "--sam", str(tmp_path / "sam")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    ctx = Context(0)
    try:
        _, og = device_graph(ctx, cfg)
        og.simplify()
        og.spell()
        og.map_file(s1, max_mismatches=2, sam=str(tmp_path / "a.sam"))
        og.map_file(s2, max_mismatches=2, sam=str(tmp_path / "b.sam"))
        og.write_depths(str(tmp_path / "api.tsv"), names=["a.fa", "b.fq"])
    finally:
        ctx.close()
    assert open(tmp_path / "api.tsv", "rb").read() == open(tmp_path / "x.tsv", "rb").read()
    for x in ("a", "b"):
        got = open(tmp_path / "sam" / (x + (".fa" if x == "a" else ".fq") + ".sam"), "rb").read()
        assert got == open(tmp_path / (x + ".sam"), "rb").read()
    assert b"\nq17\t" in open(tmp_path / "b.sam", "rb").read()


@pytest.mark.gpu
def test_error_paths(tmp_path):
    from metagenomics_b200 import Context, synth
    from metagenomics_b200._lib import MapStats, SamStats, lib
    from metagenomics_b200.api import COVERAGE_DTYPE
    ctx = Context(0)
    try:
        cfg = synth.config(5, scale=0.002)
        _, og = device_graph(ctx, cfg)
        reads = split_reads(cfg["bases"], cfg["offsets"])[:100]
        b, o = join_reads(reads)
        good = join_reads([b"r%d" % i for i in range(100)])
        st, ss = MapStats(), SamStats()
        path = str(tmp_path / "x.sam")

        def call(nm, p=path, d=1):
            nb, no = nm if nm is not None else (None, None)
            return lib().ogb_graph_map_reads_sam(ctx._h, b.ctypes.data, o.ctypes.data, 100, None if nb is None else nb.ctypes.data,
                                                 None if no is None else no.ctypes.data, d, p.encode(), None, None, C.byref(st), C.byref(ss))
        assert call(good) == 4 and not os.path.exists(path)               # OGB_E_STATE: no spell
        og.simplify()
        og.spell()
        assert call(good) == 0 and st.sample == 0
        for bad in ([b"r@1"], [b""], [b"a b"], [b"x" * 255], [b"\x7f"]):
            assert call(join_reads([b"r%d" % i for i in range(99)] + bad)) == 1
            assert "read 99" in lib().ogb_last_error().decode()
        assert call(join_reads([b"!?A~" + b"x" * 250] * 100)) == 0 and st.sample == 1
        assert call(good, p=str(tmp_path / "no" / "such" / "dir.sam")) == 6                 # OGB_E_IO before any work
        assert call(good, d=9) == 1
        if os.path.exists("/dev/full"):
            assert call(good, p="/dev/full") == 6                                           # the write fails
        assert call(None) == 0 and st.sample == 2                                           # the list grew only by the calls that worked
        recs = np.zeros(len(og.unitigs()[0]) + 1, COVERAGE_DTYPE)
        og.spell()
        assert call(None) == 0 and st.sample == 0                                           # a spell starts a new list
        cov = lambda j: lib().ogb_graph_sample_coverage(ctx._h, j, recs.ctypes.data, len(recs), None, 0)   # noqa: E731
        assert cov(0) == 0 and cov(1) == 1
        with pytest.raises(ValueError):
            og.map_reads(reads, sam=path, names=[b"a"])
        with pytest.raises(ValueError):
            og.map_reads(reads, names=[b"r%d" % i for i in range(100)])           # names without a SAM would be dropped
    finally:
        ctx.close()

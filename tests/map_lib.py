"""Helpers of the sample-mapping tests (tests/test_sample_map.py)."""
import ctypes as C
import os
import subprocess

import numpy as np

from contract_lib import load_oracle_module

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sm = load_oracle_module("sample_map")
COUNTERS = ("filtered", "mapped", "multi", "placements", "index_entries", "index_buckets")


def split_reads(bases, offsets):
    """flat ASCII + offsets -> list of bytes"""
    b = np.ascontiguousarray(bases, np.uint8).tobytes()
    o = [int(x) for x in offsets]
    return [b[o[i]:o[i + 1]] for i in range(len(o) - 1)]


def join_reads(reads):
    """list of bytes -> (uint8 bases, uint64 offsets)"""
    offs = np.zeros(len(reads) + 1, np.uint64)
    offs[1:] = np.cumsum([len(r) for r in reads], dtype=np.uint64)
    return np.frombuffer(b"".join(reads), np.uint8).copy(), offs


def unitig_seqs(recs, ascii):
    """the sequences of a spell's records from its flat ASCII layout"""
    a = np.ascontiguousarray(ascii, np.uint8).tobytes()
    return [a[int(r["start"]):int(r["start"]) + int(r["length"])] for r in recs]


def decode_words(words, recs):
    """the sequences of a spell's records from its packed words"""
    acgt = np.frombuffer(b"ACGT", np.uint8)
    k = np.arange(32 * len(words), dtype=np.int64)
    flat = acgt[(words[k // 32] >> (np.uint64(62) - np.uint64(2) * (k % 32).astype(np.uint64))) & np.uint64(3)] if len(words) else np.zeros(0, np.uint8)
    return unitig_seqs(recs, flat)


def filter_sample(seqs, m, seed=5):
    """A sample with every kind of read: exact pieces of the unitigs on either strand, some in lower case, pieces with an N, reads
    of <= m bases, low-complexity reads, one of 70 000 bases, and random reads that occur nowhere."""
    rng = np.random.default_rng(seed)
    long_seqs = [s for s in seqs if len(s) > m + 1] or [b"ACGT" * (m + 1)]
    out = []
    for i in range(200):
        s = long_seqs[int(rng.integers(0, len(long_seqs)))]
        L = int(rng.integers(m + 1, min(len(s), 3 * m) + 1))
        a = int(rng.integers(0, len(s) - L + 1))
        r = s[a:a + L]
        if i % 2:
            r = sm.rc(r)
        kind = i % 10
        if kind == 3:
            r = r.lower()
        elif kind == 5:
            r = r[:L // 2] + b"N" + r[L // 2 + 1:]
        elif kind == 7:
            r = r[:m]
        out.append(r)
    out += [b"A" * (m + 20), b"AC" * m + b"A" * (8 * m), bytes(rng.choice(list(b"ACGT"), 70000).tolist())]
    out += [bytes(rng.choice(list(b"ACGT"), m + 30).tolist()) for _ in range(20)]
    return out


def build_map_emul():
    """Compiles tests/map_emul.cpp (the per-thread bodies of csrc/ogb_map.cuh on the CPU) and returns emul(...)."""
    out = os.path.join(HERE, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libmap_emul.so")
    src = os.path.join(HERE, "map_emul.cpp")
    hdrs = [os.path.join(ROOT, "metagenomics_b200", "csrc", h) for h in ("ogb_map.cuh", "ogb_coverage.cuh", "ogb_spell.cuh")] + [os.path.join(ROOT, "include", "ogb.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in [src] + hdrs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.emul_map.restype = None
    lib.emul_map.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]

    def emul(words, recs, bases, offsets, m):
        """words / recs: a spell's packed layout and records. Returns (records, uint32 depth of the layout, hits, counters)."""
        from metagenomics_b200.api import COVERAGE_DTYPE
        words = np.ascontiguousarray(words, np.uint64)
        recs = np.ascontiguousarray(recs)
        bases = np.ascontiguousarray(bases, np.uint8)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        n = len(offsets) - 1
        out = np.zeros(max(len(recs), 1), COVERAGE_DTYPE)
        depth = np.zeros(max(32 * len(words), 1), np.uint32)
        hits = np.zeros(max(n, 1), np.uint32)
        ctr = np.zeros(6, np.uint64)
        lib.emul_map(words.ctypes.data, len(words), recs.ctypes.data, len(recs), bases.ctypes.data, offsets.ctypes.data, n, m,
                     out.ctypes.data, depth.ctypes.data, hits.ctypes.data, ctr.ctypes.data)
        return out[:len(recs)].copy(), depth[:32 * len(words)].copy(), hits[:n].copy(), dict(zip(COUNTERS, (int(x) for x in ctr)))
    return emul


def index_figures(seqs, m):
    """index entries and buckets the definition implies: one entry per position p with p + K <= |S_u|"""
    K = min(32, m + 1)
    bases = sum(len(s) for s in seqs)
    b = 1
    while 2 * b < bases:
        b <<= 1
    return sum(max(0, len(s) - K + 1) for s in seqs), b


def check_against(want, recs, depth, hits, counters, srecs, m, seqs):
    """device / emulated mapping == the restatement: records, profile in the word-aligned layout, hits and counters"""
    from coverage_lib import check_records, padded_profile
    check_records(recs, want, srecs)
    assert np.array_equal(depth.astype(np.int64), padded_profile(want, srecs))
    assert np.array_equal(hits, want["hits"])
    entries, buckets = index_figures(seqs, m)
    got = {k: int(counters[k]) for k in COUNTERS}
    assert got == dict(filtered=want["filtered"], mapped=want["mapped"], multi=want["multi"], placements=want["placements"],
                       index_entries=entries, index_buckets=buckets), got

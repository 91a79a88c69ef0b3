"""Helpers of the unitig-coverage tests (tests/test_coverage.py) and of tests/golden/make_coverage_full_size.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from contract_lib import load_oracle_module

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
cv = load_oracle_module("unitig_coverage")


def sup_packed(sup_ids, lens):
    """superReadIDs (per read idx, 0 = not contained) -> K2's device form L_super << 32 | ~super_idx."""
    s = sup_ids.astype(np.int64)
    out = np.zeros(len(s), np.uint64)
    m = s > 0
    out[m] = (lens.astype(np.uint64)[s[m] - 1] << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - (s[m] - 1).astype(np.uint64))
    return out


def cover_graph(fw, starts, lens, freq, sup, edges, items, select=None, q=None):
    """coverage_all over the ogb_cedge / ogb_clist_item arrays (or a boolean selection of the edges)."""
    e = edges if select is None else edges[select]
    return cv.coverage_all(fw, starts, lens, freq, sup, e["src"].astype(np.int64), e["dst"].astype(np.int64), e["orient"], e["offset"],
                           e["list_start"], e["count"], items["read"].astype(np.int64), items["offset"], items["orient"], q=q)


def padded_profile(cov, recs):
    """the oracle's back-to-back profile in the word-aligned layout of the spell records `recs` (padding 0)"""
    words = int((recs["start"][-1] + recs["length"][-1] + 31) // 32) if len(recs) else 0
    out = np.zeros(32 * words, np.int64)
    L = recs["length"].astype(np.int64)
    idx = np.repeat(recs["start"].astype(np.int64), L) + (np.arange(int(L.sum())) - np.repeat(cov["start"], L))
    out[idx] = cov["depth"]
    return out


def build_coverage_emul():
    """Compiles tests/coverage_emul.cpp (the per-thread bodies of csrc/ogb_coverage.cuh on the CPU) and returns cover(...)."""
    out = os.path.join(HERE, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libcoverage_emul.so")
    src = os.path.join(HERE, "coverage_emul.cpp")
    hdrs = [os.path.join(ROOT, "metagenomics_b200", "csrc", h) for h in ("ogb_coverage.cuh", "ogb_spell.cuh")] + [os.path.join(ROOT, "include", "ogb.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in [src] + hdrs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.emul_coverage.restype = C.c_longlong
    lib.emul_coverage.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]

    def cover(words, meta, edges, items, recs, freq, sup):
        """words / meta: the device read store layout; recs: a spell's records; freq, sup (K2's packed form) per read idx.
        Returns (coverage records, uint32 depth of the layout, unplaced, contained placements)."""
        from metagenomics_b200.api import COVERAGE_DTYPE
        args = [np.ascontiguousarray(a) for a in (words, meta, edges, items, recs)]
        freq = np.ascontiguousarray(freq, np.uint32)
        sup = np.ascontiguousarray(sup, np.uint64)
        nw = int((recs["start"][-1] + recs["length"][-1] + 31) // 32) if len(recs) else 0
        out = np.zeros(max(len(recs), 1), COVERAGE_DTYPE)
        depth = np.zeros(max(32 * nw, 1), np.uint32)
        ncp = C.c_uint64()
        r = lib.emul_coverage(args[0].ctypes.data, args[1].ctypes.data, len(freq), args[2].ctypes.data, args[3].ctypes.data, len(items),
                              args[4].ctypes.data, len(recs), freq.ctypes.data, sup.ctypes.data, out.ctypes.data, depth.ctypes.data, nw, C.byref(ncp))
        assert r >= 0, r
        return out[:len(recs)].copy(), depth[:32 * nw].copy(), int(r), ncp.value
    return cover


def check_records(recs, cov, spell_recs):
    """device / emulated coverage records == the restatement's, field by field"""
    assert np.array_equal(recs["edge"], spell_recs["edge"]) and np.array_equal(recs["start"], spell_recs["start"])
    assert np.array_equal(recs["length"], spell_recs["length"]) and np.array_equal(recs["length"].astype(np.int64), cov["length"])
    for k in ("reads", "contained", "read_count", "depth_min", "depth_max"):
        assert np.array_equal(recs[k].astype(np.int64), cov[k].astype(np.int64)), k
    for k in ("depth_sum", "depth_sq_sum"):
        assert np.array_equal(recs[k], cov[k].astype(np.uint64)), k

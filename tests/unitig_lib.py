"""Helpers of the unitig-spelling tests (tests/test_unitigs.py) and of tests/golden/make_unitigs_full_size.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from contract_lib import load_oracle_module

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
us = load_oracle_module("unitig_spell")


def reads_ascii(ds, chunk=1 << 20):
    """Forward strands of a host Dataset's unique reads as one flat ASCII array: (fw uint8, starts int64, lens int64), read id
    i at fw[starts[i-1] : starts[i-1] + lens[i-1]] -- decoded from the packed words Dataset.packed() hands to the device."""
    words, woffs, lens = ds.packed()
    lens = lens.astype(np.int64)
    starts = np.concatenate([[0], np.cumsum(lens)])[:-1]
    fw = np.empty(int(lens.sum()), np.uint8)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    woffs = np.asarray(woffs, dtype=np.int64)
    for a in range(0, len(lens), chunk):
        b = min(len(lens), a + chunk)
        L = lens[a:b]
        n = int(L.sum())
        if n == 0:
            continue
        k = np.arange(n, dtype=np.int64) - np.repeat(starts[a:b] - starts[a], L)
        w = words[np.repeat(woffs[a:b], L) + k // 32]
        fw[starts[a]:starts[a] + n] = acgt[(w >> (np.uint64(62) - np.uint64(2) * (k % 32).astype(np.uint64))) & np.uint64(3)]
    return fw, starts, lens


def spell_graph(fw, starts, lens, edges, items, select=None):
    """spell_all over the ogb_cedge / ogb_clist_item arrays (or a boolean selection of the edges)."""
    e = edges if select is None else edges[select]
    return us.spell_all(fw, starts, lens, e["src"].astype(np.int64), e["dst"].astype(np.int64), e["orient"], e["offset"],
                        e["list_start"], e["count"], items["read"].astype(np.int64), items["offset"], items["orient"])


def build_spell_emul():
    """Compiles tests/spell_emul.cpp (the per-word body of csrc/ogb_spell.cuh on the CPU) and returns spell(...)."""
    out = os.path.join(HERE, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libspell_emul.so")
    src = os.path.join(HERE, "spell_emul.cpp")
    hdr = os.path.join(ROOT, "metagenomics_b200", "csrc", "ogb_spell.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", so], check=True)
    lib = C.CDLL(so)
    lib.emul_spell.restype = C.c_longlong
    lib.emul_spell.argtypes = [C.c_void_p] * 2 + [C.c_uint32] + [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int,
                                                                  C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]

    def spell(words, meta, n_reads, edges, items, canonical):
        """words / meta: the device read store layout (see ogb_kernels.cuh); returns (records, packed words)."""
        from metagenomics_b200.api import UNITIG_DTYPE
        words = np.ascontiguousarray(words, np.uint64)
        meta = np.ascontiguousarray(meta, np.uint64)
        edges = np.ascontiguousarray(edges)
        items = np.ascontiguousarray(items)
        L = meta & np.uint64(0xFFFF)
        cap_r = len(edges)
        cap_w = int(((edges["offset"].astype(np.int64) + L[edges["dst"].astype(np.int64) - 1].astype(np.int64) + 31) // 32).sum()) if len(edges) else 0
        recs = np.zeros(max(cap_r, 1), UNITIG_DTYPE)
        out = np.zeros(max(cap_w, 1), np.uint64)
        n = lib.emul_spell(words.ctypes.data, meta.ctypes.data, n_reads, edges.ctypes.data, len(edges), items.ctypes.data, len(items),
                           int(canonical), recs.ctypes.data, cap_r, out.ctypes.data, cap_w)
        assert n >= 0, n
        nw = int(((recs["length"][:n].astype(np.int64) + 31) // 32).sum())
        return recs[:n].copy(), out[:nw].copy()
    return spell


def store_layout(fw, starts, lens):
    """The device read store of a data set with one length or several (ogb_kernels.cuh): forward strand at word off, reverse
    complement at off + pw, pw = 2 ceil(L/64); meta[idx] = off << 16 | L. Built with the oracle's packer."""
    L = lens.astype(np.int64)
    pw = ((L + 63) // 64) * 2
    off = np.concatenate([[0], np.cumsum(2 * pw)])[:-1]
    words = np.zeros(int((2 * pw).sum()) + 8, np.uint64)
    fwd, fws = us.pack(fw, starts, L)
    rcs = np.concatenate([us._COMP[fw[int(s):int(s) + int(l)][::-1]] for s, l in zip(starts, L)]) if len(L) else np.zeros(0, np.uint8)
    rvd, rvs = us.pack(rcs, starts, L)
    nw = (L + 31) // 32
    for i in range(len(L)):
        words[off[i]:off[i] + nw[i]] = fwd[fws[i]:fws[i] + nw[i]]
        words[off[i] + pw[i]:off[i] + pw[i] + nw[i]] = rvd[rvs[i]:rvs[i] + nw[i]]
    meta = (off.astype(np.uint64) << np.uint64(16)) | L.astype(np.uint64)
    return words, meta


def canonical_mask(edges):
    return us.canonical(edges["src"].astype(np.int64), edges["dst"].astype(np.int64), edges["twin"].astype(np.int64))

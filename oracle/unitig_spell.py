"""TEST INFRASTRUCTURE (oracle/): the sequence of a unitig -- a directed edge of the simplified graph (OverlapGraph.cpp:211-215)
with its read list -- restated in plain Python. The reference's getStringInEdge (OverlapGraph.cpp:2009) is the interface this
pins; its sources are not in the repository, so what is pinned is the definition below and the properties every correct
spelling has (each read of the list is a substring at its position; S(twin(e)) == reverse_complement(S(e))). Nothing in the
product imports this module.

Edge e = (src, dst, orient, offset) with items (read_k, off_k, or_k), k = 1..c, stands for reads r_0 = src, r_1..r_c, r_{c+1} = dst:
    src forward iff orient in {2, 3};  dst forward iff orient in {1, 3};  item k forward iff or_k == 1    (mergeList, mergedEdgeOrientation)
    P_0 = 0,  P_k = off_1 + ... + off_k,  P_{c+1} = offset
    |S(e)| = offset + L[dst];  base p of S(e) = base p - P_k of the oriented read r_k, k the largest index with P_k <= p.

Canonical unitigs (saveGraphToFile, OverlapGraph.cpp:321-326): edge i with src < dst, or src == dst and i < twin[i].

Read strings are given as one flat ASCII array `fw` of the forward strands and `starts` (read id i at fw[starts[i-1] ..
starts[i-1] + L[i-1])); `spell` is the per-base restatement, `spell_all` its vectorised form for full-size data sets."""
import numpy as np

_COMP = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGT", b"TGCA"):
    _COMP[_a] = _b


def rc_bytes(s):
    return _COMP[np.frombuffer(bytes(s), dtype=np.uint8)[::-1]].tobytes()


def _pieces(src, dst, orient, offset, reads, offs, ors):
    """[(read id, forward, P_k)] for k = 0 .. c+1"""
    out, p = [(int(src), int(orient) in (2, 3), 0)], 0
    for r, o, f in zip(reads, offs, ors):
        p += int(o)
        out.append((int(r), int(f) == 1, p))
    out.append((int(dst), int(orient) in (1, 3), int(offset)))
    return out


def oriented(fw, starts, lens, rid, forward):
    a = int(starts[rid - 1])
    s = bytes(fw[a:a + int(lens[rid - 1])])
    return s if forward else rc_bytes(s)


def spell(fw, starts, lens, src, dst, orient, offset, reads, offs, ors):
    """S(e) as bytes, base by base, straight from the definition."""
    ps = _pieces(src, dst, orient, offset, reads, offs, ors)
    n = int(offset) + int(lens[int(dst) - 1])
    out = bytearray(n)
    k = 0
    strs = [oriented(fw, starts, lens, r, f) for r, f, _ in ps]
    for p in range(n):
        while k + 1 < len(ps) and ps[k + 1][2] <= p:
            k += 1
        out[p] = strs[k][p - ps[k][2]]
    return bytes(out)


def canonical(src, dst, twin):
    i = np.arange(len(src))
    return (src < dst) | ((src == dst) & (i < twin))


def spell_all(fw, starts, lens, e_src, e_dst, e_orient, e_offset, e_start, e_count, it_read, it_off, it_or):
    """Vectorised spell of edges given as arrays (items of edge i at it_*[e_start[i] : e_start[i] + e_count[i]]). Read r_k
    contributes bases [P_k, P_{k+1}) of S, r_{c+1} all of itself -- the same bases the definition assigns (the largest k with
    P_k <= p). Returns (flat uint8 ASCII of the sequences in edge order, their starts in it, their lengths)."""
    ne = len(e_src)
    cnt = e_count.astype(np.int64)
    npc = cnt + 2                                                      # pieces per edge
    first = np.concatenate([[0], np.cumsum(npc)])[:-1]
    tot = int(npc.sum())
    rid = np.empty(tot, np.int64)
    fwd = np.empty(tot, bool)
    pos = np.empty(tot, np.int64)
    rid[first] = e_src
    fwd[first] = (e_orient.astype(np.int64) & 2) != 0
    pos[first] = 0
    last = first + npc - 1
    rid[last] = e_dst
    fwd[last] = (e_orient.astype(np.int64) & 1) != 0
    pos[last] = e_offset.astype(np.int64)
    mid = np.ones(tot, bool)
    mid[first] = False
    mid[last] = False
    idx = (np.repeat(e_start.astype(np.int64), cnt) + (np.arange(int(cnt.sum())) - np.repeat(np.concatenate([[0], np.cumsum(cnt)])[:-1], cnt)))
    rid[mid] = it_read[idx]
    fwd[mid] = it_or[idx] == 1
    off = it_off[idx].astype(np.int64)
    csum = np.cumsum(off)
    base = np.repeat(np.concatenate([[0], csum])[np.concatenate([[0], np.cumsum(cnt)])[:-1]], cnt)
    pos[mid] = csum - base
    L = lens.astype(np.int64)[rid - 1]
    take = np.empty(tot, np.int64)
    take[:-1] = pos[1:] - pos[:-1]
    take[last] = L[last]
    assert (take >= 0).all() and (take <= L).all()
    seq_len = e_offset.astype(np.int64) + lens.astype(np.int64)[e_dst.astype(np.int64) - 1]
    seq_start = np.concatenate([[0], np.cumsum(seq_len)])[:-1]
    n = int(seq_len.sum())
    pstart = np.repeat(np.concatenate([[0], np.cumsum(take)])[:-1], take)
    t = np.arange(n, dtype=np.int64) - pstart                          # offset inside the piece
    pr = np.repeat(np.arange(tot), take)
    r0 = starts.astype(np.int64)[rid[pr] - 1]
    f = fwd[pr]
    src_idx = np.where(f, r0 + t, r0 + L[pr] - 1 - t)
    b = fw[src_idx]
    out = np.where(f, b, _COMP[b]).astype(np.uint8)
    assert ne == 0 or int(seq_start[-1] + seq_len[-1]) == n
    return out, seq_start, seq_len


# ---- the order-independent figure of tests/golden/unitigs_full_size.json ----

_K = [np.uint64(k) for k in (0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0x27D4EB2F165667C5, 0x94D049BB133111EB)]


def _mix(x):
    x = x ^ (x >> np.uint64(29))
    x = x * np.uint64(0xBF58476D1CE4E5B9)
    return x ^ (x >> np.uint64(32))


def seq_hashes(ascii, starts, lengths, reverse_complement=False):
    """64-bit hash of every sequence ascii[starts[i] : starts[i] + lengths[i]] (of its reverse complement when asked):
    mix(sum_j mix(base_j * K1 ^ (j + 1) * K2) + length * K3)."""
    L = lengths.astype(np.int64)
    n = int(L.sum())
    with np.errstate(over="ignore"):
        if n == 0:
            return _mix(L.astype(np.uint64) * _K[2])
        seg = np.repeat(np.arange(len(L)), L)
        segstart = np.repeat(np.concatenate([[0], np.cumsum(L)])[:-1], L)
        j = np.arange(n, dtype=np.int64) - segstart                       # position inside the sequence
        src = np.repeat(starts.astype(np.int64), L) + j
        b = ascii[src].astype(np.uint64)
        if reverse_complement:                                            # rc(S)[L-1-j] = comp(S[j])
            b = _COMP[ascii[src]].astype(np.uint64)
            j = L[seg] - 1 - j
        h = _mix(b * _K[0] ^ (j.astype(np.uint64) + np.uint64(1)) * _K[1])
        cs = np.concatenate([[np.uint64(0)], np.cumsum(h, dtype=np.uint64)])
        ends = np.cumsum(L)
        sums = cs[ends] - cs[ends - L]
        return _mix(sums + L.astype(np.uint64) * _K[2])


def unitig_terms(src, dst, orient, h, h_rc):
    """Per unitig: mix(src*K1 ^ dst*K2 ^ orient*K3 ^ hash(S)*K4). A palindromic self-edge pair (src == dst) spells S and rc(S),
    and which of its two records counts as canonical depends on the edge order; such an edge takes the smaller of its own term
    and its twin's, (dst, src, twin(orient), hash(rc(S))), so the figure does not depend on that order."""
    tw = np.array([3, 1, 2, 0], dtype=np.uint64)
    s, d, o = src.astype(np.uint64), dst.astype(np.uint64), orient.astype(np.uint64)
    with np.errstate(over="ignore"):
        a = _mix(s * _K[0] ^ d * _K[1] ^ o * _K[2] ^ h.astype(np.uint64) * _K[3])
        b = _mix(d * _K[0] ^ s * _K[1] ^ tw[orient.astype(np.int64)] * _K[2] ^ h_rc.astype(np.uint64) * _K[3])
        return np.where(src == dst, np.minimum(a, b), a)


def checksum(terms):
    """[xor, sum mod 2^64] of the terms of the canonical unitigs."""
    return [int(np.bitwise_xor.reduce(terms)) if len(terms) else 0, int(terms.sum(dtype=np.uint64))]


def pack(ascii, starts, lengths):
    """The word-aligned 2-bit layout the library returns: sequence i in words [wstart[i], wstart[i] + ceil(len/32)), base p in
    bits 63-2(p%32) .. 62-2(p%32) of its word p/32 (A0 C1 G2 T3, unused bits zero). Returns (words uint64, wstart)."""
    L = lengths.astype(np.int64)
    nw = (L + 31) // 32
    wstart = np.concatenate([[0], np.cumsum(nw)])[:-1]
    codes = np.zeros(256, dtype=np.uint64)
    for c, v in zip(b"ACGT", range(4)):
        codes[c] = v
    n = int(L.sum())
    words = np.zeros(int(nw.sum()), dtype=np.uint64)
    if n:
        segstart = np.repeat(np.concatenate([[0], np.cumsum(L)])[:-1], L)
        j = np.arange(n, dtype=np.int64) - segstart
        src = np.repeat(starts.astype(np.int64), L) + j
        w = np.repeat(wstart, L) + j // 32
        v = codes[ascii[src]] << (np.uint64(62) - np.uint64(2) * (j % 32).astype(np.uint64))
        np.bitwise_or.at(words, w, v) if n < 4096 else _or_reduce(words, w, v)
    return words, wstart


def _or_reduce(words, w, v):
    # w is non-decreasing: the bits of one word are disjoint, so their sum is their or
    cs = np.concatenate([[np.uint64(0)], np.cumsum(v, dtype=np.uint64)])
    bounds = np.flatnonzero(np.diff(w)) + 1
    lo = np.concatenate([[0], bounds])
    hi = np.concatenate([bounds, [len(w)]])
    with np.errstate(over="ignore"):
        words[w[lo]] = cs[hi] - cs[lo]

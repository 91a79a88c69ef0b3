"""TEST INFRASTRUCTURE (oracle/): per-base read depth of the unitigs of the simplified graph, restated in numpy on top of
oracle/unitig_spell.py (placements, read strings). This is the project's own definition; the reference's getBaseByBaseCoverage
(OverlapGraph.cpp:2722) is not in the repository, and no parity with it is claimed. Nothing in the product imports this module.

Unitig u = edge e with placements k = 0..c+1 (read r_k, forward?, P_k; unitig_spell._pieces). f(r) = the read's frequency.
    graph reads:     D[p] += f(r_k)  for P_k <= p < P_k + L(r_k)
    contained reads: for every read x with superReadID(x) = r_k: q_x = S.find(x) with S = r_k's forward strand and x its stored
                     strand, else S.find(reverse_complement(x)); a = P_k + q_x (r_k forward) or P_k + L(r_k) - q_x - L(x);
                     D[p] += f(x)  for a <= p < a + L(x)
A read with no occurrence is `unplaced` (K2 verified every containment, so there is none).

Read strings as in unitig_spell: flat ASCII `fw` of the stored (forward) strands, read id i at fw[starts[i-1] .. + lens[i-1]).
freq[i-1] = f(i); sup[i-1] = superReadID(i) (0: not contained)."""
import importlib.util
import os

import numpy as np

_spec = importlib.util.spec_from_file_location("unitig_spell", os.path.join(os.path.dirname(os.path.abspath(__file__)), "unitig_spell.py"))
us = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(us)

UNPLACED = -1


def locate(fw, starts, lens, sup):
    """q_x per read idx (int64): -2 = not contained, UNPLACED = no occurrence, else the shift. bytes.find gives the smallest."""
    q = np.full(len(lens), -2, np.int64)
    for i in np.flatnonzero(sup):
        x = us.oriented(fw, starts, lens, i + 1, True)
        s = us.oriented(fw, starts, lens, int(sup[i]), True)
        v = s.find(x)
        q[i] = v if v >= 0 else s.find(us.rc_bytes(x))
    return q


def profile(fw, starts, lens, freq, sup, q, src, dst, orient, offset, reads, offs, ors):
    """D of one unitig straight from the definition (int64), and its contained placements."""
    ps = us._pieces(src, dst, orient, offset, reads, offs, ors)
    D = np.zeros(int(offset) + int(lens[int(dst) - 1]), np.int64)
    nc = 0
    for r, fwd, P in ps:
        L = int(lens[r - 1])
        D[P:P + L] += int(freq[r - 1])
        for x in np.flatnonzero(sup == r):
            if q[x] < 0:
                continue
            Lx = int(lens[x])
            a = P + int(q[x]) if fwd else P + L - int(q[x]) - Lx
            D[a:a + Lx] += int(freq[x])
            nc += 1
    return D, nc


def coverage_all(fw, starts, lens, freq, sup, e_src, e_dst, e_orient, e_offset, e_start, e_count, it_read, it_off, it_or, q=None):
    """Vectorised coverage of edges given as arrays (as unitig_spell.spell_all). Returns a dict: per unitig `reads`, `contained`,
    `read_count`, `depth_sum`, `depth_sq_sum` (uint64, wraps like the device), `depth_min`, `depth_max`, `length`, `start` (in the
    flat profile), the flat int64 profile `depth` (unitigs back to back, no padding), and `unplaced`."""
    if q is None:
        q = locate(fw, starts, lens, sup)
    lens = lens.astype(np.int64)
    freq = freq.astype(np.int64)
    cnt = e_count.astype(np.int64)
    npc = cnt + 2
    first = np.concatenate([[0], np.cumsum(npc)])[:-1].astype(np.int64)
    tot = int(npc.sum())
    eid = np.repeat(np.arange(len(cnt)), npc)
    rid = np.empty(tot, np.int64)
    fwd = np.empty(tot, bool)
    pos = np.empty(tot, np.int64)
    last = first + npc - 1
    rid[first], fwd[first], pos[first] = e_src, (e_orient.astype(np.int64) & 2) != 0, 0
    rid[last], fwd[last], pos[last] = e_dst, (e_orient.astype(np.int64) & 1) != 0, e_offset.astype(np.int64)
    mid = np.ones(tot, bool)
    mid[first] = False
    mid[last] = False
    istart = np.concatenate([[0], np.cumsum(cnt)])[:-1]
    idx = np.repeat(e_start.astype(np.int64), cnt) + (np.arange(int(cnt.sum())) - np.repeat(istart, cnt))
    rid[mid] = it_read[idx]
    fwd[mid] = it_or[idx] == 1
    csum = np.cumsum(it_off[idx].astype(np.int64))
    pos[mid] = csum - np.repeat(np.concatenate([[0], csum])[istart], cnt)
    length = e_offset.astype(np.int64) + lens[e_dst.astype(np.int64) - 1]
    seg = np.concatenate([[0], np.cumsum(length)])[:-1].astype(np.int64)
    L = lens[rid - 1]
    # contained reads of every placement: CSR super read idx -> contained read idx
    placed = np.flatnonzero(q >= 0)
    sup_idx = sup.astype(np.int64)[placed] - 1
    order = np.argsort(sup_idx, kind="stable")
    clist, csup = placed[order], sup_idx[order]
    cstart = np.searchsorted(csup, np.arange(len(lens) + 1))
    nct = cstart[rid] - cstart[rid - 1]                         # contained reads of each placement
    pc = np.repeat(np.arange(tot), nct)
    x = clist[np.repeat(cstart[rid - 1], nct) + (np.arange(int(nct.sum())) - np.repeat(np.concatenate([[0], np.cumsum(nct)])[:-1], nct))]
    Lx, qx = lens[x], q[x]
    ax = np.where(fwd[pc], pos[pc] + qx, pos[pc] + L[pc] - qx - Lx)
    # intervals [seg + a, seg + a + len) with weight f
    a = np.concatenate([seg[eid] + pos, seg[eid[pc]] + ax])
    ln = np.concatenate([L, Lx])
    w = np.concatenate([freq[rid - 1], freq[x]])
    n = int(length.sum())
    diff = np.zeros(n + 1, np.int64)
    np.add.at(diff, a, w)
    np.add.at(diff, a + ln, -w)
    D = np.cumsum(diff[:-1])
    ne = len(cnt)
    out = dict(reads=npc, length=length, start=seg, depth=D, unplaced=int((q == UNPLACED).sum()))
    out["contained"] = np.bincount(eid[pc], minlength=ne).astype(np.int64)
    out["read_count"] = np.bincount(np.concatenate([eid, eid[pc]]), weights=w, minlength=ne).round().astype(np.int64) if len(w) else np.zeros(ne, np.int64)
    if n:
        with np.errstate(over="ignore"):
            out["depth_sum"] = np.add.reduceat(D.astype(np.uint64), seg) if ne else np.zeros(0, np.uint64)
            out["depth_sq_sum"] = np.add.reduceat(D.astype(np.uint64) * D.astype(np.uint64), seg) if ne else np.zeros(0, np.uint64)
        out["depth_min"] = np.minimum.reduceat(D, seg)
        out["depth_max"] = np.maximum.reduceat(D, seg)
    else:
        out["depth_sum"] = out["depth_sq_sum"] = np.zeros(ne, np.uint64)
        out["depth_min"] = out["depth_max"] = np.zeros(ne, np.int64)
    return out


# ---- the order-independent figures of tests/golden/coverage_full_size.json ----


def profile_hashes(D, starts, lengths, reverse=False):
    """64-bit hash of every profile D[starts[i] : starts[i] + lengths[i]] (read backwards when asked):
    mix(sum_j mix((D_j + 1) * K1 ^ (j + 1) * K2) + length * K3)."""
    L = lengths.astype(np.int64)
    n = int(L.sum())
    K = us._K
    with np.errstate(over="ignore"):
        if n == 0:
            return us._mix(L.astype(np.uint64) * K[2])
        segstart = np.repeat(np.concatenate([[0], np.cumsum(L)])[:-1], L)
        j = np.arange(n, dtype=np.int64) - segstart
        src = np.repeat(starts.astype(np.int64), L) + j
        if reverse:
            j = np.repeat(L, L) - 1 - j
        h = us._mix((D[src].astype(np.uint64) + np.uint64(1)) * K[0] ^ (j.astype(np.uint64) + np.uint64(1)) * K[1])
        cs = np.concatenate([[np.uint64(0)], np.cumsum(h, dtype=np.uint64)])
        ends = np.cumsum(L)
        return us._mix(cs[ends] - cs[ends - L] + L.astype(np.uint64) * K[2])


def record_terms(src, dst, cov):
    """Per unitig: mix over (src, dst, length, reads, contained, read_count, depth_sum, depth_sq_sum, min, max). Every field but
    src / dst is the same for the twin, so a self-edge's term does not depend on which half counts as canonical."""
    K = us._K
    f = [cov[k].astype(np.uint64) for k in ("length", "reads", "contained", "read_count", "depth_sum", "depth_sq_sum", "depth_min", "depth_max")]
    with np.errstate(over="ignore"):
        h = us._mix(src.astype(np.uint64) * K[0] ^ dst.astype(np.uint64) * K[1])
        for i, v in enumerate(f):
            h = us._mix(h + v * K[(i + 2) % 5])
    return h


def profile_terms(src, dst, h, h_rev):
    """Per unitig: the hash of its profile; a self-edge takes the smaller of its own and its reversed profile's, as its twin
    half holds the reversed profile."""
    return np.where(src == dst, np.minimum(h, h_rev), h)


def checksum(terms):
    return us.checksum(terms)

"""TEST INFRASTRUCTURE (oracle/): per-sample read depth of the unitigs of the simplified graph, restated in plain Python. This is
the project's own definition (csrc/ogb_map.cuh, ogb_graph_map_reads); nothing in the product imports this module.

Input: the unitig sequences S_u of a spell (bytes, in record order), the build's minOverlap m, and one sample: a list of ASCII reads.
    filter:     read s is kept iff m < len(s) < 65536, s is ACGT only with case folded, and no base occurs >= int(len(s) * .8)
                times (Dataset.cpp:155-158, :398-413; the rule k_ds_filter implements). Anything else is filtered.
    placements: (u, p) with 0 <= p <= |S_u| - L and S_u[p, p + L) == s or rc(s), s a kept read of length L; a read equal to its
                own reverse complement is tested on one strand only, so every (u, p) counts once.
    depth:      every placement adds 1 on [p, p + L) of S_u; raw reads count one by one.
    hits[i]:    the placements of read i (0: unmapped), FILTERED for a filtered read.
Records as in ogb_graph_coverage: reads = read_count = placements in the unitig, contained = 0, depth sums, min and max."""
import numpy as np

FILTERED = 0xFFFFFFFF
_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def rc(s):
    return s.translate(_COMP)[::-1]


def kept(s, m):
    """the Dataset filter for minOverlap m; returns the upper-case read, or None"""
    L = len(s)
    if not (m < L < 65536):
        return None
    u = s.upper()
    if u.translate(None, b"ACGT"):
        return None
    thr = int(L * .8)
    if any(u.count(b) >= thr for b in (b"A", b"C", b"G", b"T")):
        return None
    return u


def occurrences(hay, s):
    """every p with hay[p : p + len(s)] == s, overlapping ones included"""
    out, p = [], hay.find(s)
    while p >= 0:
        out.append(p)
        p = hay.find(s, p + 1)
    return out


def placements(hay, hstart, read, m):
    """[(u, p)] of one raw read, in (u, p) order, or None when it is filtered. hay = the unitigs joined by '|' (no occurrence
    spans two), unitig u at hay[hstart[u]:]."""
    s = kept(read, m)
    if s is None:
        return None
    strands = [s] if rc(s) == s else [s, rc(s)]
    pos = sorted(p for t in strands for p in occurrences(hay, t))
    u = np.searchsorted(hstart, pos, side="right") - 1
    return [(int(a), int(p - hstart[a])) for a, p in zip(u, pos)]


def map_sample(seqs, reads, m):
    """The depth of every unitig of `seqs` from the sample `reads` (list of bytes). Returns a dict shaped like
    unitig_coverage.coverage_all: per unitig `reads`, `contained`, `read_count`, `depth_sum`, `depth_sq_sum` (uint64), `depth_min`,
    `depth_max`, `length`, `start` (in the flat profile), the flat int64 profile `depth` (unitigs back to back); plus `hits` (uint32
    per read), `placed` ([(u, p, L, read index)]) and the counters `filtered`, `mapped`, `multi`, `placements`."""
    length = np.array([len(S) for S in seqs], np.int64)
    start = np.concatenate([[0], np.cumsum(length)])[:-1].astype(np.int64)
    n = int(length.sum())
    diff = np.zeros(n + 1, np.int64)
    count = np.zeros(len(seqs), np.int64)
    hits = np.zeros(len(reads), np.uint32)
    placed = []
    hay = b"|".join(bytes(S) for S in seqs)
    hstart = start + np.arange(len(seqs))
    for i, r in enumerate(reads):
        pl = placements(hay, hstart, bytes(r), m)
        if pl is None:
            hits[i] = FILTERED
            continue
        hits[i] = len(pl)
        for u, p in pl:
            diff[start[u] + p] += 1
            diff[start[u] + p + len(r)] -= 1
            count[u] += 1
            placed.append((u, p, len(r), i))
    D = np.cumsum(diff[:-1])
    kept_hits = hits[hits != FILTERED].astype(np.int64)
    out = dict(length=length, start=start, depth=D, hits=hits, placed=placed, reads=count, read_count=count.copy(),
               contained=np.zeros(len(seqs), np.int64), filtered=int((hits == FILTERED).sum()), mapped=int((kept_hits > 0).sum()),
               multi=int((kept_hits > 1).sum()), placements=int(kept_hits.sum()))
    with np.errstate(over="ignore"):
        Du = D.astype(np.uint64)
        out["depth_sum"] = np.array([Du[a:a + L].sum() for a, L in zip(start, length)], np.uint64)
        out["depth_sq_sum"] = np.array([(Du[a:a + L] * Du[a:a + L]).sum() for a, L in zip(start, length)], np.uint64)
    out["depth_min"] = np.array([D[a:a + L].min() for a, L in zip(start, length)], np.int64)
    out["depth_max"] = np.array([D[a:a + L].max() for a, L in zip(start, length)], np.int64)
    return out

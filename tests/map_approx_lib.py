"""TEST INFRASTRUCTURE: sample mapping with up to d substitutions per read (csrc/ogb_map.cuh, ogb_graph_map_reads_approx),
restated in plain Python next to the exact restatement oracle/sample_map.py, whose filter (kept), reverse complement (rc) and
occurrence search it uses. Nothing in the product imports this module."""
import numpy as np

from contract_lib import load_oracle_module

_sm = load_oracle_module("sample_map")
FILTERED, kept, rc, occurrences = _sm.FILTERED, _sm.kept, _sm.rc, _sm.occurrences


UNPLACED = 0xFF


def _hamming(hay, cand, t):
    """Hamming distance of hay[p : p + len(t)] and t for every p of cand (int64 array), hay and t as uint8 arrays"""
    L = len(t)
    out = np.empty(len(cand), np.int64)
    step = max(1, 4_000_000 // max(L, 1))
    for a in range(0, len(cand), step):
        c = cand[a:a + step]
        out[a:a + step] = (hay[c[:, None] + np.arange(L)] != t).sum(axis=1)
    return out


def map_sample_approx(seqs, reads, m, d):
    """map_sample with up to d substitutions per read (ogb_graph_map_reads_approx). K = min(32, m + 1); a kept read of length L is
    searched with d_r = min(d, L // K - 1). Candidates (u, p, strand): every p at which one of the d_r + 1 disjoint K-mers t[jK, jK + K)
    of the strand t (s, or rc(s)) occurs at p + jK with [p, p + L) inside S_u -- by pigeonhole every (u, p) within d_r substitutions is
    one. H = the Hamming distance of S_u[p, p + L) and t; b = the least H over both strands; the read is mapped iff b <= d_r, and its
    placements are the distinct (u, p) with min(H_fw, H_rc) == b. Returns map_sample's dict plus `mismatches` (uint8 per read: b, or
    UNPLACED for a read that is filtered or not mapped). At d = 0 this is map_sample."""
    K = min(32, m + 1)
    length = np.array([len(S) for S in seqs], np.int64)
    start = np.concatenate([[0], np.cumsum(length)])[:-1].astype(np.int64)
    n = int(length.sum())
    diff = np.zeros(n + 1, np.int64)
    count = np.zeros(len(seqs), np.int64)
    hits = np.zeros(len(reads), np.uint32)
    mis = np.full(len(reads), UNPLACED, np.uint8)
    placed = []
    hay = b"|".join(bytes(S) for S in seqs)
    harr = np.frombuffer(hay, np.uint8)
    hstart = start + np.arange(len(seqs))
    hend = hstart + length
    for i, r in enumerate(reads):
        s = kept(bytes(r), m)
        if s is None:
            hits[i] = FILTERED
            continue
        L = len(s)
        dr = min(d, L // K - 1)
        H = {}                                                         # p in hay -> min(H_fw, H_rc) over the strands that reach it
        for t in [s] if rc(s) == s else [s, rc(s)]:
            cand = set()
            for j in range(dr + 1):
                for q in occurrences(hay, t[j * K:(j + 1) * K]):
                    u = int(np.searchsorted(hstart, q, side="right")) - 1
                    p = q - j * K
                    if p >= hstart[u] and p + L <= hend[u]:
                        cand.add(p)
            cand = np.array(sorted(cand), np.int64)
            for p, h in zip(cand.tolist(), _hamming(harr, cand, np.frombuffer(t, np.uint8)).tolist()):
                H[p] = min(h, H.get(p, h))
        b = min(H.values(), default=dr + 1)
        if b > dr:
            continue
        pos = sorted(p for p, h in H.items() if h == b)
        hits[i], mis[i] = len(pos), b
        for p in pos:
            u = int(np.searchsorted(hstart, p, side="right")) - 1
            diff[start[u] + p - hstart[u]] += 1
            diff[start[u] + p - hstart[u] + L] -= 1
            count[u] += 1
            placed.append((u, int(p - hstart[u]), L, i))
    D = np.cumsum(diff[:-1])
    kept_hits = hits[hits != FILTERED].astype(np.int64)
    out = dict(length=length, start=start, depth=D, hits=hits, mismatches=mis, placed=placed, reads=count, read_count=count.copy(),
               contained=np.zeros(len(seqs), np.int64), filtered=int((hits == FILTERED).sum()), mapped=int((kept_hits > 0).sum()),
               multi=int((kept_hits > 1).sum()), placements=int(kept_hits.sum()))
    with np.errstate(over="ignore"):
        Du = D.astype(np.uint64)
        out["depth_sum"] = np.array([Du[a:a + L].sum() for a, L in zip(start, length)], np.uint64)
        out["depth_sq_sum"] = np.array([(Du[a:a + L] * Du[a:a + L]).sum() for a, L in zip(start, length)], np.uint64)
    out["depth_min"] = np.array([D[a:a + L].min() for a, L in zip(start, length)], np.int64)
    out["depth_max"] = np.array([D[a:a + L].max() for a, L in zip(start, length)], np.int64)
    return out

"""TEST INFRASTRUCTURE: writes tests/golden/coverage_full_size.json, the golden of the UNITIG COVERAGE (ogb_graph_coverage: per-base
read depth of the canonical unitigs, contained reads included) at full configuration sizes -- per entry

    {"config", "scale", "n_unique", "unitigs", "bases", "placements", "contained_placements", "unplaced", "depth_sum",
     "depth_sq_sum", "depth_min", "depth_max", "records": [xor, sum], "profile": [xor, sum]}

over the canonical unitigs (saveGraphToFile's rule, OverlapGraph.cpp:321-326). The simplified graph comes the way
make_unitigs_full_size.py gets it -- the memory-lean oracle's final edges (checked against full_size.json) through
oracle/contract_seq.cpp -- frequencies and superReadIDs from the lean oracle's read_info(), and the coverage from
oracle/unitig_coverage.py (vectorised form) over the host Dataset's reads. depth_sq_sum is mod 2^64, as on the device.

    python tests/golden/make_coverage_full_size.py 2:1.0 3:1.0 5:1.0
"""
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from contract_lib import seq_simplify  # noqa: E402
from coverage_lib import cv  # noqa: E402
from oracle_lib import LeanOracle, edge_checksum  # noqa: E402
from unitig_lib import reads_ascii  # noqa: E402
from metagenomics_b200 import Dataset, synth  # noqa: E402

OUT = os.path.join(HERE, "coverage_full_size.json")


def figures(src, dst, cov, both_halves=True):
    """The golden figures of the coverage `cov` (coverage_all or the device's, with `depth` / `start` / `length`) of unitigs whose
    ends are src / dst. both_halves: a self-edge (src == dst) appears with both halves, and each pair counts once; else (the
    canonical unitigs) with one of them."""
    self_loop = (src == dst) if both_halves else np.zeros(len(src), bool)
    assert self_loop.sum() % 2 == 0
    rt = cv.record_terms(src, dst, cov)
    h = cv.profile_hashes(cov["depth"], cov["start"], cov["length"])
    hr = cv.profile_hashes(cov["depth"], cov["start"], cov["length"], reverse=True)
    pt = cv.profile_terms(src, dst, h, hr)
    keep = ~self_loop
    pal = np.flatnonzero(self_loop)
    pal = pal[np.argsort(pt[pal], kind="stable")][0::2]         # the two halves of a pair carry the same terms: keep one of each
    keep[pal] = True
    L = cov["length"].astype(np.int64)[keep]
    mn = int(cov["depth_min"][keep].min()) if keep.any() else 0
    with np.errstate(over="ignore"):
        sq = int(cov["depth_sq_sum"].astype(np.uint64)[keep].sum(dtype=np.uint64))
    return dict(unitigs=int(keep.sum()), bases=int(L.sum()), placements=int(cov["reads"].astype(np.int64)[keep].sum()),
                contained_placements=int(cov["contained"].astype(np.int64)[keep].sum()),
                depth_sum=int(cov["depth_sum"].astype(np.uint64)[keep].sum(dtype=np.uint64)), depth_sq_sum=sq, depth_min=mn,
                depth_max=int(cov["depth_max"][keep].max()) if keep.any() else 0,
                records=cv.checksum(rt[keep]), profile=cv.checksum(pt[keep]))


def main():
    want = [(int(a.split(":")[0]), float(a.split(":")[1])) for a in sys.argv[1:]]
    gold = json.load(open(OUT)) if os.path.exists(OUT) else []
    full = json.load(open(os.path.join(HERE, "full_size.json")))
    for k, scale in want:
        t0 = time.time()
        ref = next(g for g in full if g["config"] == k and g["scale"] == scale)
        cfg = synth.config(k, scale=scale)
        o = LeanOracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run(keep_edges=True)
        e, info = o.edges(), o.read_info()
        assert edge_checksum(e) == ref["checksum"], "the lean oracle's final edges are not full_size.json's"
        st, edges, items = seq_simplify(e, info["len"])
        assert st["checksum"] == ref["simplified"]["checksum"]
        del o, e
        ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
        fw, starts, L = reads_ascii(ds)
        assert np.array_equal(L, info["len"].astype(np.int64)) and np.array_equal(ds.frequencies(), info["freq"])
        sel = edges[:, 0] <= edges[:, 1]                         # src < dst: canonical; src == dst: both halves of a pair, one counts
        g = edges[sel]
        cov = cv.coverage_all(fw, starts, L, info["freq"], info["sup"], g[:, 0].astype(np.int64), g[:, 1].astype(np.int64), g[:, 2], g[:, 3],
                              g[:, 5], g[:, 4], items[:, 0].astype(np.int64), items[:, 1], items[:, 2])
        assert cov["unplaced"] == 0
        entry = dict(config=k, scale=scale, n_unique=int(len(L)), unplaced=cov["unplaced"],
                     **figures(g[:, 0].astype(np.int64), g[:, 1].astype(np.int64), cov))
        gold = [x for x in gold if (x["config"], x["scale"]) != (k, scale)] + [entry]
        print(f"config {k} @ {scale}: {entry}  ({time.time() - t0:.0f} s)", flush=True)
        json.dump(sorted(gold, key=lambda x: (x["config"], x["scale"])), open(OUT, "w"), indent=1)


if __name__ == "__main__":
    main()

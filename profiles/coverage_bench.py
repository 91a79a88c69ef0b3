"""Unitig coverage (ogb_graph_coverage: per-base read depth of the canonical unitigs, contained reads included) on one GPU: configs 3,
2 and 5 at full size. Per config: build + simplify + spell once, then `--warmup` untimed and `--steps` timed coverage calls (device
time and its phases from the library's CUDA events, mean), and the copies to the host (records, and the per-base u32 profile; host
clock around ogb_graph_unitig_coverage, which ends in a stream synchronise).

Algorithmic bytes of one call, set against the stream peak the project measured (6540.8 GB/s on a B200):
    locate (only with contained reads): sup 8 B / read read twice + per contained read q 4 B written and read, its count and fill
        atomics 2 x 8 B, its CSR slot 4 B and start 8 B, and its stored strand plus the super read's first words 2 x 16 B
    placements: record 32 B + edge 40 B / unitig, item 8 B + position 8 B / item, meta 8 B + freq 4 B / placed read (graph and
        contained), two u32 atomics (read + write, 8 B each) / placed read, contained list 4 B + q 4 B / contained placement
    difference array 4 B / base zeroed, scan 4 B read twice + 8 B written / base, reduce 8 B read + 4 B written / base
The card's name and power limit are read in the same run.

    python profiles/coverage_bench.py [--configs 3,2,5] [--steps 10] [--warmup 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from unitig_bench import STREAM_PEAK_GBS, card  # noqa: E402


def run(k, steps, warmup):
    from metagenomics_b200 import Context, Dataset, HashTable, OverlapGraph, synth
    from metagenomics_b200._lib import CoverageStats, check, lib
    from metagenomics_b200.api import COVERAGE_DTYPE
    cfg = synth.config(k, scale=1.0)
    ctx = Context(0)
    try:
        ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
        ht = HashTable(ctx)
        ht.insertDataset(ds, cfg["min_overlap"])
        og = OverlapGraph(ht)
        edges, items, _ = og.simplify()
        sp = og.spell()
        freq = np.ascontiguousarray(ds.frequencies(), np.uint32)
        n_contained = int((og.superReadIDs()[1:] > 0).sum())

        def call():
            st = CoverageStats()
            check(lib().ogb_graph_coverage(ctx._h, freq.ctypes.data, len(freq), C.byref(st)))
            return st.as_dict()
        for _ in range(warmup):
            call()
        runs = [call() for _ in range(steps)]
        st = runs[-1]
        recs = np.zeros(st["unitigs"], COVERAGE_DTYPE)
        depth = np.zeros(32 * sp["words"], np.uint32)
        d2h = {}
        for name, dp, cap in (("records", None, 0), ("records_and_profile", depth.ctypes.data, len(depth))):
            ms = []
            for _ in range(3):
                t0 = time.perf_counter()
                check(lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), dp, cap))
                ms.append((time.perf_counter() - t0) * 1e3)
            d2h[name] = {"ms_mean": float(np.mean(ms)), "ms_min": float(np.min(ms)), "bytes": int(recs.nbytes + (depth.nbytes if dp else 0))}
        nu, ne, ni, n = st["unitigs"], len(edges), len(items), len(freq)
        npl, ncp, nb = st["placements"], st["contained_placements"], 32 * sp["words"]
        alg = {"locate": (16 * n + n_contained * (8 + 16 + 12 + 32)) if n_contained else 0,
               "placements": (32 + 40) * nu + 16 * ni + (12 + 16) * (npl + ncp) + 8 * ncp,
               "diff_scan_reduce": (4 + 16 + 12) * nb}
        tot = sum(alg.values())
        mean = float(np.mean([r["ms"] for r in runs]))
        return {
            "config": k, "n_unique": n, "contained_reads": n_contained, "unitigs": nu, "bases": st["bases"], "layout_bases": nb,
            "placements": npl, "contained_placements": ncp, "unplaced": st["unplaced"], "launches": st["launches"],
            "ms_mean": mean, "ms_min": float(np.min([r["ms"] for r in runs])), "ms_max": float(np.max([r["ms"] for r in runs])),
            "ms_locate": float(np.mean([r["ms_locate"] for r in runs])), "ms_depth": float(np.mean([r["ms_depth"] for r in runs])),
            "ms_reduce": float(np.mean([r["ms_reduce"] for r in runs])), "steps": steps, "warmup": warmup,
            "placements_per_s": (npl + ncp) / (mean * 1e-3), "bases_per_s": st["bases"] / (mean * 1e-3),
            "alg_bytes": alg, "alg_bytes_total": tot, "alg_GBps": tot / (mean * 1e-3) / 1e9,
            "share_of_stream_peak": tot / (mean * 1e-3) / 1e9 / STREAM_PEAK_GBS, "d2h": d2h, "spell_ms": sp["ms"],
        }
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="3,2,5")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.warmup < 3 or a.steps < 1:
        ap.error("--warmup >= 3 and --steps >= 1")
    res = {"card": card(), "stream_peak_GBps": STREAM_PEAK_GBS, "runs": [run(int(k), a.steps, a.warmup) for k in a.configs.split(",")]}
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()

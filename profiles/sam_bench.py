"""SAM output of a sample (ogb_graph_map_reads_sam) on one GPU, config 3 at full size. Build + simplify + spell once; then for each
sample -- the config's own 10 M reads, and the same reads with 0.5 % substitutions (seeded) -- and each d of --mismatches, `--warmup`
untimed and `--steps` timed rounds that alternate the plain mapping (ogb_graph_map_reads_approx) and the SAM call on the same reads.

Reported per (sample, d): records, bytes, the SAM stages' device times ms_emit / ms_format / ms_copy (CUDA event pairs around GPU
work only), ms_write (host wall time in fwrite / fclose) and ms_setup (host wall time: header, file, pinned buffers when they grow),
the wall time of both calls on the host clock (each ends in a device synchronise), the text rate bytes / (ms_emit + ms_format) and
bytes / (ms_emit + ms_format + ms_copy), and the plain call's ms_map next to the SAM call's (the mapping inside the SAM call is the
same work). The SAM call's wall time is split: the plain call's wall time (the same mapping, its pageable upload included), ms_setup,
ms_write, the SAM device time, and the rest ("other": host waits and launches, less the part of the device time that overlaps the
file writes). Means over the timed rounds, with min and max. The file is written under --out-dir and deleted after each call (outside
the timed calls); ms_write therefore measures the page cache of the machine's file system as much as anything.
The card's name and power limit are read in the same run.

    python profiles/sam_bench.py [--steps 3] [--warmup 1] [--mismatches 0 2] [--out-dir DIR] [--out FILE]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from unitig_bench import card  # noqa: E402


def stats(xs):
    return {"mean": float(np.mean(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--mismatches", type=int, nargs="+", default=[0, 2])
    ap.add_argument("--out-dir", default=None, help="where the SAM is written (and deleted); default: a temporary directory")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.warmup < 1 or a.steps < 1 or not all(0 <= d <= 8 for d in a.mismatches):
        ap.error("--warmup >= 1, --steps >= 1, 0 <= --mismatches <= 8")
    from metagenomics_b200 import Context, Dataset, HashTable, OverlapGraph, synth
    res = {"card": card(), "steps": a.steps, "warmup": a.warmup}
    cfg = synth.config(3)
    samples = {"own": cfg["bases"], "own_0.5pct": synth.substitute(301, cfg["bases"], 0.005)}
    o = cfg["offsets"]
    out_dir = a.out_dir or tempfile.mkdtemp(prefix="sam_bench_")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "sample.sam")
    ctx = Context(0)
    try:
        ds = Dataset(bases=cfg["bases"], offsets=o, minOverlap=cfg["min_overlap"])
        ht = HashTable(ctx)
        ht.insertDataset(ds, cfg["min_overlap"])
        og = OverlapGraph(ht)
        og.simplify()
        res["spell"] = og.spell()
        og.map_reads(bases=samples["own"], offsets=o)                          # builds the index
        res["runs"] = {}
        for name, b in samples.items():
            for d in a.mismatches:
                plain, sam, wall, wall_plain = [], [], [], []
                for step in range(a.warmup + a.steps):
                    tp = time.perf_counter()
                    _, sp = og.map_reads(bases=b, offsets=o, max_mismatches=d)
                    tp = (time.perf_counter() - tp) * 1e3
                    t0 = time.perf_counter()
                    _, ss = og.map_reads(bases=b, offsets=o, max_mismatches=d, sam=path)
                    t1 = time.perf_counter()
                    os.remove(path)
                    if step >= a.warmup:
                        plain.append(sp)
                        sam.append(ss)
                        wall.append((t1 - t0) * 1e3)
                        wall_plain.append(tp)
                s = sam[-1]["sam"]
                dev = [x["sam"]["ms_emit"] + x["sam"]["ms_format"] for x in sam]
                dev_copy = [x["sam"]["ms_emit"] + x["sam"]["ms_format"] + x["sam"]["ms_copy"] for x in sam]
                res["runs"][f"{name}_d{d}"] = {
                    "records": s["records"], "bytes": s["bytes"], "launches": s["launches"],
                    "reads_in": sam[-1]["reads_in"], "filtered": sam[-1]["filtered"], "mapped": sam[-1]["mapped"], "placements": sam[-1]["placements"],
                    **{k: stats([x["sam"][k] for x in sam]) for k in ("ms_emit", "ms_format", "ms_copy", "ms_write", "ms_setup")},
                    "wall_ms": stats(wall), "wall_plain_ms": stats(wall_plain),
                    "wall_other_ms": stats([w - wp - x["sam"]["ms_setup"] - x["sam"]["ms_write"] - t
                                            for w, wp, x, t in zip(wall, wall_plain, sam, dev_copy)]),
                    "GBps_emit_format": stats([s["bytes"] / (t * 1e-3) / 1e9 for t in dev]),
                    "GBps_emit_format_copy": stats([s["bytes"] / (t * 1e-3) / 1e9 for t in dev_copy]),
                    "plain_ms_map": stats([x["ms_map"] for x in plain]),
                    "sam_call_ms_map": stats([x["ms_map"] for x in sam]),
                    "plain_ms": stats([x["ms"] for x in plain]),
                }
                print(name, d, json.dumps(res["runs"][f"{name}_d{d}"]), flush=True)
    finally:
        ctx.close()
        if os.path.exists(path):
            os.remove(path)
        if a.out_dir is None:
            os.rmdir(out_dir)
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()

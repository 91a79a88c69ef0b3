"""Unitig spelling (ogb_graph_spell; getStringInEdge, OverlapGraph.cpp:2009) on one GPU: config 3 (the bench workload) and config 2
beside it at full size. Per config: build + simplify once, then the spell of the canonical unitigs over `--warmup` untimed and `--steps`
timed calls (device time from the library's CUDA events, mean), the copies to the host (packed words and ASCII, host clock around
ogb_graph_unitigs, which ends in a stream synchronise) and the FASTA write (ogb_graph_write_unitigs into a temporary directory).

Algorithmic bytes of one spell, set against the stream peak the project measured (6540.8 GB/s on a B200):
    packed output 8 B / word + strand gathers 16 B / word (two stored words per 32-base extract) + records 32 B / unitig
    + composite edges 40 B / edge + items 8 B read + 4 B offset written and read twice by the scan + 8 B position written / item
The card's name and power limit are read in the same run.

    python profiles/unitig_bench.py [--configs 3,2] [--steps 10] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STREAM_PEAK_GBS = 6540.8


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, timeout=60).stdout
        name, power = [x.strip() for x in out.strip().split("\n")[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                      # the measurement stands without it, but says so
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def run(k, steps, warmup):
    from metagenomics_b200 import Context, Dataset, HashTable, OverlapGraph, synth
    from metagenomics_b200._lib import check, lib
    from metagenomics_b200.api import UNITIG_DTYPE
    cfg = synth.config(k, scale=1.0)
    ctx = Context(0)
    try:
        ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
        ht = HashTable(ctx)
        ht.insertDataset(ds, cfg["min_overlap"])
        og = OverlapGraph(ht)
        edges, items, sst = og.simplify()
        for _ in range(warmup):
            og.spell()
        ms = [og.spell()["ms"] for _ in range(steps)]
        st = og.spell()
        recs = np.zeros(st["unitigs"], UNITIG_DTYPE)
        d2h = {}
        for ascii in (0, 1):
            out = np.zeros(st["words"] * (32 if ascii else 8), np.uint8)
            best = []
            for _ in range(3):
                t0 = time.perf_counter()
                check(lib().ogb_graph_unitigs(ctx._h, recs.ctypes.data, len(recs), out.ctypes.data, out.nbytes, ascii))
                best.append((time.perf_counter() - t0) * 1e3)
            d2h["ascii" if ascii else "packed"] = {"ms_mean": float(np.mean(best)), "ms_min": float(np.min(best)), "bytes": int(out.nbytes)}
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "unitigs.fa")
            t0 = time.perf_counter()
            check(lib().ogb_graph_write_unitigs(ctx._h, path.encode()))
            fasta_ms = (time.perf_counter() - t0) * 1e3
            fasta_bytes = os.path.getsize(path)
        words, nu, ne, ni = st["words"], st["unitigs"], len(edges), len(items)
        alg = {"packed_out": 8 * words, "strand_gathers": 16 * words, "records": 32 * nu, "edges": 40 * ne, "items": (8 + 3 * 4 + 8) * ni}
        tot = sum(alg.values())
        mean = float(np.mean(ms))
        return {
            "config": k, "n_unique": int(ds.getNumberOfUniqueReads()), "composite_edges": ne, "items": ni,
            "unitigs": nu, "bases": st["bases"], "words": words, "launches": st["launches"],
            "spell_ms_mean": mean, "spell_ms_min": float(np.min(ms)), "spell_ms_max": float(np.max(ms)), "steps": steps, "warmup": warmup,
            "bases_per_s": st["bases"] / (mean * 1e-3), "alg_bytes": alg, "alg_bytes_total": tot,
            "alg_GBps": tot / (mean * 1e-3) / 1e9, "share_of_stream_peak": tot / (mean * 1e-3) / 1e9 / STREAM_PEAK_GBS,
            "d2h": d2h, "fasta_write_ms": fasta_ms, "fasta_bytes": fasta_bytes, "simplify_ms": sst["ms"],
        }
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="3,2")
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

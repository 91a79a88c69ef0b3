"""Sample mapping (ogb_graph_map_reads: every read of a sample looked up exactly in the canonical unitigs) on one GPU, config 3 at full
size. Build + simplify + spell once; map the config's own 10 M raw reads (the first mapping builds the K-mer index: ms_index), then
`--warmup` untimed and `--steps` timed rounds of two samples each: the own reads again and one more sample of 10 M reads from the same
genomes with its own seeded log-normal weights. Times are the library's CUDA events (ogb_map_stats), means over the timed rounds.

Algorithmic bytes of one sample, set against the stream peak the project measured (6540.8 GB/s on a B200):
    upload (device side; the H2D copy of the ASCII crosses PCIe and is in ms_upload too): ASCII read twice (filter, pack), offsets
        8 B read twice, good 4 + position 8 + start 8 + length 2 + meta 8 (written and read) / read, packed strands 2 x 2 pw x 8 B written
    map: per kept read meta 8 B + both strands' words read, per strand two bucket starts 16 B + the bucket's entries 8 B each, per
        verified placement the layout words it spans + 1, the unitig's record 32 B and wpos 8 B, two u32 atomics on the difference
        array and two on the record (read + write, 8 B each), 4 B of hits
    reduce: difference array 4 B / base zeroed, scan 4 B read twice + 8 B written / base, reduce 8 B read + 4 B written / base
The map phase is random gathers (bucket, layout, records), so the stream peak is an upper bound it cannot reach; the share is
reported for what it is. Index, once per spell: per layout word 16 B, per entry 2 bucket atomics (16 B) and 8 B written, per bucket
4 B zeroed twice, scanned (4 B read twice + 8 B written).
The card's name and power limit are read in the same run.

    python profiles/map_bench.py [--steps 5] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from unitig_bench import STREAM_PEAK_GBS, card  # noqa: E402


def alg_bytes(st, n_bytes, mean_len, layout_bases, pw):
    kept = st["reads_in"] - st["filtered"]
    per_bucket = st["index_entries"] / max(st["index_buckets"], 1)
    words_per_placement = (mean_len + 31) // 32 + 1
    return {
        "upload": 2 * n_bytes + 16 * st["reads_in"] + (4 + 8 + 8 + 2 + 16) * st["reads_in"] + 2 * 2 * pw * 8 * kept,
        "map": kept * (8 + 2 * pw * 8 + 2 * (16 + 8 * per_bucket)) + st["placements"] * (8 * words_per_placement + 40 + 32) + 4 * st["reads_in"],
        "reduce": (4 + 16 + 12) * layout_bases,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.warmup < 1 or a.steps < 1:
        ap.error("--warmup >= 1 and --steps >= 1")
    from metagenomics_b200 import Context, Dataset, HashTable, OverlapGraph, synth
    res = {"card": card(), "stream_peak_GBps": STREAM_PEAK_GBS}
    cfg = synth.config(3)
    gs, _ = synth._metagenome(3, 20, 1e6, 5e6, 1.0)
    w = np.exp(np.random.default_rng(300).normal(0.0, 1.0, len(gs)))
    other = synth.sample_reads(300, gs, 10_000_000, 100, weights=w)
    samples = {"own": (cfg["bases"], cfg["offsets"]), "other": other}
    ctx = Context(0)
    try:
        ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
        ht = HashTable(ctx)
        ht.insertDataset(ds, cfg["min_overlap"])
        og = OverlapGraph(ht)
        og.simplify()
        sp = og.spell()
        _, first = og.map_reads(bases=samples["own"][0], offsets=samples["own"][1])
        res["spell"] = sp
        res["first_mapping"] = first
        runs = {k: [] for k in samples}
        for step in range(a.warmup + a.steps):
            for k, (b, o) in samples.items():
                _, st = og.map_reads(bases=b, offsets=o)
                if step >= a.warmup:
                    runs[k].append(st)
        layout = 32 * sp["words"]
        res["samples"] = {}
        for k, rs in runs.items():
            b, o = samples[k]
            st = rs[-1]
            mean = {f: float(np.mean([r[f] for r in rs])) for f in ("ms", "ms_index", "ms_upload", "ms_map", "ms_reduce")}
            alg = alg_bytes(st, int(o[-1] - o[0]), 100, layout, 4)
            dev = mean["ms_upload"] + mean["ms_map"] + mean["ms_reduce"]
            res["samples"][k] = {
                "stats": {f: v for f, v in st.items() if not f.startswith("ms")}, "steps": a.steps, "warmup": a.warmup,
                **{f + "_mean": v for f, v in mean.items()}, "ms_min": float(np.min([r["ms"] for r in rs])), "ms_max": float(np.max([r["ms"] for r in rs])),
                "reads_per_s": st["reads_in"] / (mean["ms"] * 1e-3), "alg_bytes": alg,
                "alg_GBps": {p: alg[p] / (mean["ms_" + p] * 1e-3) / 1e9 for p in alg},
                "share_of_stream_peak": {p: alg[p] / (mean["ms_" + p] * 1e-3) / 1e9 / STREAM_PEAK_GBS for p in alg},
                "share_of_stream_peak_all": sum(alg.values()) / (dev * 1e-3) / 1e9 / STREAM_PEAK_GBS,
            }
    finally:
        ctx.close()
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()

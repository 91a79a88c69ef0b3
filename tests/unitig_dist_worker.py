"""Worker of tests/test_unitigs.py::test_two_ranks_split_the_unitigs: every rank builds the graph through the multi-rank C ABI, simplifies
it (rank-local: every rank holds the whole graph), spells only its own range of the canonical unitigs (metagenomics_b200.dist.
unitig_range) and checks it against the same range of a spell over everything."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from metagenomics_b200 import Dataset, HashTable, OverlapGraph, synth  # noqa: E402
from metagenomics_b200.dist import make_context, unitig_range  # noqa: E402


def main():
    ctx, rank, world, local = make_context()
    torch.cuda.set_device(local)
    cfg = synth.config(3, scale=0.004)
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
    ht = HashTable(ctx)
    ht.insertDataset(ds, cfg["min_overlap"])
    og = OverlapGraph(ht)
    edges, _, _ = og.simplify()
    recs, words = og.unitigs(ascii=False)
    first, count = unitig_range(edges, rank, world)
    mine, mw = og.unitigs(ascii=False, first=first, count=count)
    assert np.array_equal(mine["edge"], recs["edge"][first:first + count]) and np.array_equal(mine["length"], recs["length"][first:first + count])
    lo = int(recs["start"][first]) // 32 if count else 0
    assert np.array_equal(mw, words[lo:lo + len(mw)])
    print(f"rank {rank}/{world}: unitig range identical ({count} of {len(recs)})", flush=True)
    ctx.close()
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

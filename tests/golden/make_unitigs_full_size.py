"""TEST INFRASTRUCTURE: writes tests/golden/unitigs_full_size.json, the golden of the UNITIG SEQUENCES of the simplified graph
(ogb_graph_spell; the reference's getStringInEdge, OverlapGraph.cpp:2009) at full configuration sizes -- per entry

    {"config", "scale", "n_unique", "unitigs", "bases", "checksum": [xor, sum]}

over the canonical unitigs (saveGraphToFile's rule, OverlapGraph.cpp:321-326). The simplified graph comes the way
make_simplified_full_size.py builds its field -- the memory-lean oracle's final edges (checked against full_size.json) through
oracle/contract_seq.cpp -- and the sequences from oracle/unitig_spell.py (vectorised form) over the host Dataset's reads.

    python tests/golden/make_unitigs_full_size.py 2:1.0 3:1.0 5:1.0
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
from oracle_lib import LeanOracle, edge_checksum  # noqa: E402
from unitig_lib import reads_ascii, us  # noqa: E402
from metagenomics_b200 import Dataset, synth  # noqa: E402

OUT = os.path.join(HERE, "unitigs_full_size.json")


def golden_entry(cfg, edges, items, fw, starts, lens):
    """edges (n, 6) [src, dst, orient, offset, count, list_start], items (m, 3) [read, offset, orientation] of a simplified graph
    (every edge with its twin) -> unitigs, bases, checksum over the canonical unitigs."""
    src, dst = edges[:, 0].astype(np.int64), edges[:, 1].astype(np.int64)
    sel = src <= dst                                     # src < dst: canonical; src == dst: both halves of a pair, one counts
    e = edges[sel]
    seq, st, ln = us.spell_all(fw, starts, lens, e[:, 0].astype(np.int64), e[:, 1].astype(np.int64), e[:, 2], e[:, 3], e[:, 5], e[:, 4],
                               items[:, 0].astype(np.int64), items[:, 1], items[:, 2])
    t = us.unitig_terms(e[:, 0], e[:, 1], e[:, 2], us.seq_hashes(seq, st, ln), us.seq_hashes(seq, st, ln, reverse_complement=True))
    self_loop = e[:, 0] == e[:, 1]
    assert self_loop.sum() % 2 == 0
    pal = np.sort(t[self_loop])                          # the two halves of a pair carry the same term: keep one of each
    assert (pal[0::2] == pal[1::2]).all()
    terms = np.concatenate([t[~self_loop], pal[0::2]])
    bases = int(ln[~self_loop].sum()) + int(ln[self_loop].sum()) // 2
    return dict(unitigs=int(len(terms)), bases=bases, checksum=us.checksum(terms))


def main():
    want = [(int(a.split(":")[0]), float(a.split(":")[1])) for a in sys.argv[1:]]
    gold = json.load(open(OUT)) if os.path.exists(OUT) else []
    full = json.load(open(os.path.join(HERE, "full_size.json")))
    for k, scale in want:
        t0 = time.time()
        ref = next(g for g in full if g["config"] == k and g["scale"] == scale)
        cfg = synth.config(k, scale=scale)
        o = LeanOracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run(keep_edges=True)
        e, lens = o.edges(), o.read_info()["len"]
        assert edge_checksum(e) == ref["checksum"], "the lean oracle's final edges are not full_size.json's"
        st, edges, items = seq_simplify(e, lens)
        assert st["checksum"] == ref["simplified"]["checksum"]
        del o, e
        ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
        fw, starts, L = reads_ascii(ds)
        assert np.array_equal(L, lens.astype(np.int64))
        entry = dict(config=k, scale=scale, n_unique=int(len(L)), **golden_entry(cfg, edges, items, fw, starts, L))
        gold = [g for g in gold if (g["config"], g["scale"]) != (k, scale)] + [entry]
        print(f"config {k} @ {scale}: {entry}  ({time.time() - t0:.0f} s)", flush=True)
        json.dump(sorted(gold, key=lambda g: (g["config"], g["scale"])), open(OUT, "w"), indent=1)


if __name__ == "__main__":
    main()

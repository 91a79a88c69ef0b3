"""Spell, coverage and sample mapping (csrc/ogb_spell.cuh, ogb_coverage.cuh, ogb_map.cuh) where their kernels switch paths or cut
their input, against the restatements oracle/unitig_spell.py, unitig_coverage.py and sample_map.py.

Seeded sets (reads of at most 250 bases, m 20 to 60):
  tiled_m20, tiled_m40  independent random genomes tiled with reads at step 1 (30 bases at m 20: K = 21; 50 at m 40: K = 32); each
                        contracts to one unitig of the genome's length. Lengths cover every residue mod 32 at least twice, most of
                        them 2-3 layout words (about 10 records per 32-word stripe of k_cov_reduce), plus four of 1-3 kb.
  contained             chains of super reads of 150-250 bases; "host" reads of 250 bases hold contained reads of 60-120 bases at
                        shift 0 and L_s - L_x, in a tandem piece (several shifts, the smallest counts) and as an even palindrome.
Samples over a spell: `spanning` (reads across the end of a unitig, into the next one or into the padding), `ends` (reads ending
at a unitig's end, starting at 0, whole unitigs, m + 1 bases), and on the GPU the chunk limits of ogb_graph_map_reads (2^22 reads,
2^30 bytes), a depth of 2^32 - 1 and the FASTA writer across its 2^20-word chunk."""
import ctypes as C
import functools

import numpy as np
import pytest

from contract_lib import build_emul, composite_records, load_oracle_module
from coverage_lib import build_coverage_emul, check_records, cover_graph, cv, padded_profile, sup_packed
from map_lib import build_map_emul, check_against, decode_words, join_reads, sm, unitig_seqs
from oracle_lib import Oracle, sort_tuples
from unitig_lib import build_spell_emul, canonical_mask, reads_ascii, spell_graph, store_layout, us

co = load_oracle_module("contract_oracle")
SETS = ["tiled_m20", "tiled_m40", "contained"]
CHUNK_READS, CHUNK_BYTES, SPELL_CHUNK_WORDS = 1 << 22, 1 << 30, 1 << 20     # ogb_device.cu


def _rand(rng, n):
    return bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), n))


def _strand(rng, s):
    return sm.rc(s) if rng.integers(0, 2) else s


def tiled(m, L, seed):
    """Genomes of every length in [L + 12, 96] twice (> DEAD_END_LENGTH list reads at step 1; 2-3 words), then 1000, 1500, 2048
    and 3000 bases; every read of L bases on a random strand."""
    rng = np.random.default_rng(seed)
    glens = list(range(L + 12, 97)) * 2 + [1000, 1500, 2048, 3000]
    genomes = [_rand(rng, g) for g in glens]
    reads = [_strand(rng, g[i:i + L]) for g in genomes for i in range(len(g) - L + 1)]
    b, o = join_reads(reads)
    return dict(name=f"tiled_m{m}", bases=b, offsets=o, min_overlap=m, genomes=genomes)


def contained(seed=33, m=40, chains=6):
    """Chains of super reads (150-200 bases at step 60, so starts and ends both increase) with two hosts of 250 bases each. A
    host's neighbours overlap it by 50 bases, so its middle 150 bases lie in no other read and whatever is cut from there has the
    host as its only (and longest) super read. Host 0 of a chain has a period-5 tandem piece in its middle, host 1 an even
    palindrome of 70 bases; every host gives contained reads at its two ends and one in between."""
    rng = np.random.default_rng(seed)
    reads = []
    for c in range(chains):
        lay, hosts, pos = [], [], 0
        for k in range(20):
            if k in (6, 13):
                h = lay[-1][0] + lay[-1][1] - 50
                lay.append((h, 250))
                hosts.append(h)
                pos = h + 200
            else:
                lay.append((pos, int(rng.integers(150, 201))))
                pos += 60
        g = bytearray(_rand(rng, lay[-1][0] + lay[-1][1]))
        unit = bytes(rng.permutation(np.frombuffer(b"ACGTA", np.uint8)))
        tandem = (unit * 20)[:74]
        g[hosts[0] + 70:hosts[0] + 144] = tandem
        y = _rand(rng, 35)
        g[hosts[1] + 90:hosts[1] + 160] = y + sm.rc(y)
        g = bytes(g)
        reads += [_strand(rng, g[a:a + n]) for a, n in lay]
        for j, h in enumerate(hosts):
            H = g[h:h + 250]
            for _ in range(2):
                Lx = int(rng.integers(60, 121))
                q = int(rng.integers(1, 250 - Lx))
                reads += [_strand(rng, H[:Lx]), _strand(rng, H[250 - Lx:]), _strand(rng, H[q:q + Lx])]
            reads.append(_strand(rng, tandem[:64]) if j == 0 else y + sm.rc(y))
    b, o = join_reads(reads)
    return dict(name="contained", bases=b, offsets=o, min_overlap=m, chains=chains)


@functools.lru_cache(maxsize=None)
def make(name):
    return {"tiled_m20": lambda: tiled(20, 30, 21), "tiled_m40": lambda: tiled(40, 50, 22), "contained": contained}[name]()


def host_reads(cfg):
    from metagenomics_b200 import Dataset
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=int(cfg["min_overlap"]))
    return ds, reads_ascii(ds)


@functools.lru_cache(maxsize=None)
def oracle_graph(name):
    """the oracle's build, simplified by the CPU bodies of csrc/ogb_contract.cuh (pinned to contract_oracle in the shape tests)"""
    cfg = make(name)
    o = Oracle(cfg["bases"], cfg["offsets"], cfg["min_overlap"]).run_all(Oracle.THREE_PHASE, threads=8)
    info = o.read_info()
    t = o.edges()
    edges, items, _ = build_emul()(t, info["len"])
    return t, info, edges, items


def spanning_sample(seqs, m):
    """Reads S_u[-a:] + what follows S_u in the word-aligned layout: S_{u+1} when |S_u| % 32 == 0 (no padding in between), else
    the A padding (code 0); after the last unitig the spare zero word. a >= K, so the read's first K-mer is indexed and only the
    unitig bound keeps it out. Both strands; reads the filter drops are left out. Returns (reads, [(u, layout offset in S_u)])."""
    K = min(32, m + 1)
    reads, where = [], []
    for u, S in enumerate(seqs):
        pad = -len(S) % 32
        nxt = b"A" * pad if pad else (seqs[u + 1] if u + 1 < len(seqs) else b"A" * 32)
        for L in (m + 1, m + 9, 2 * m):
            for a in (K, K + 3, L - 1):
                if a < K or a > len(S) or not 1 <= L - a <= len(nxt):
                    continue
                r = S[-a:] + nxt[:L - a]
                if sm.kept(r, m) is not None:
                    reads += [r, sm.rc(r)]
                    where += [(u, len(S) - a)] * 2
    return reads, where


def ends_sample(seqs, m):
    """Reads that start at 0 or end at |S_u| (m + 1 bases: exactly K when m <= 30), whole unitigs; both strands."""
    out = []
    for S in seqs:
        out += [x for L in (m + 1, m + 2, 2 * m + 1) if L <= len(S) for x in (S[:L], S[-L:])] + [S]
    out = [r for r in out if sm.kept(r, m) is not None]
    return out + [sm.rc(r) for r in out]


def padded_layout(seqs):
    """the spell's word-aligned layout as ASCII, padding A, plus the spare zero word"""
    return b"".join(S + b"A" * (-len(S) % 32) for S in seqs) + b"A" * 32


def stripe_records(lens):
    """records that touch each 32-word stripe of the word-aligned layout"""
    nw = (lens.astype(np.int64) + 31) // 32
    w0 = np.concatenate([[0], np.cumsum(nw)])[:-1]
    a, z = w0 // 32, (w0 + nw - 1) // 32
    cnt = np.zeros(int(z.max()) + 1, np.int64)
    for x, y in zip(a, z):
        cnt[x:y + 1] += 1
    return cnt, a, z


# ---------------------------------------------------------------- CPU


@pytest.mark.parametrize("name", ["tiled_m20", "tiled_m40"])
def test_tiled_set_has_its_shape(name):
    cfg = make(name)
    t, info, edges, items = oracle_graph(name)
    assert composite_records(edges, items) == co.Graph(t.tolist(), info["len"].tolist()).simplify().edge_records()
    _, (fw, st, L) = host_reads(cfg)
    sel = canonical_mask(edges)
    flat, starts, lens = spell_graph(fw, st, L, edges, items, sel)
    genomes = cfg["genomes"]
    assert sorted(lens.tolist()) == sorted(len(g) for g in genomes)                # one unitig per genome
    for a, n in zip(starts, lens):
        s = flat[a:a + n].tobytes()
        assert s in genomes or sm.rc(s) in genomes
    assert np.bincount(lens % 32, minlength=32).min() >= 2
    cnt, a, z = stripe_records(lens)
    assert cnt.max() >= 8 and (z > a).sum() >= 4                                  # dense stripes, and records across stripes
    assert (lens <= 96).mean() > 0.9


def test_contained_set_has_its_shape():
    cfg = make("contained")
    t, info, edges, items = oracle_graph("contained")
    assert composite_records(edges, items) == co.Graph(t.tolist(), info["len"].tolist()).simplify().edge_records()
    _, (fw, st, L) = host_reads(cfg)
    sup = info["sup"].astype(np.int64)
    q = cv.locate(fw, st, L, sup)
    idx = np.flatnonzero(sup)
    assert len(idx) >= 10 * cfg["chains"] and (q[idx] >= 0).all()
    Ls, Lx = L[sup[idx] - 1], L[idx]
    assert (q[idx] == 0).any() and (q[idx] == Ls - Lx).any()
    strs = [(us.oriented(fw, st, L, int(sup[i]), True), us.oriented(fw, st, L, i + 1, True)) for i in idx]
    assert any(x not in s for s, x in strs)                                        # found only as the reverse complement
    occ = [len(sm.occurrences(s, x if x in s else sm.rc(x))) for s, x in strs]
    assert sum(o >= 3 for o in occ) >= cfg["chains"]                                # the tandem pieces
    assert sum(x == sm.rc(x) and len(x) % 2 == 0 for _, x in strs) >= cfg["chains"]   # even palindromes
    sel = canonical_mask(edges)
    assert sel.sum() == cfg["chains"]
    hosts = set(sup[idx].tolist())
    strands = set()
    for e in edges[sel]:
        it = items[int(e["list_start"]):int(e["list_start"]) + int(e["count"])]
        strands |= {f for r, f, _ in us._pieces(e["src"], e["dst"], e["orient"], e["offset"], it["read"], it["offset"], it["orient"]) if r in hosts}
    assert strands == {True, False}                                                 # hosts placed forward and reversed


@pytest.mark.parametrize("name", ["tiled_m20", "tiled_m40"])
def test_spanning_reads_bite(name):
    """Every spanning read lies in the padded layout where it was cut (so a search without the unitig bound finds it), and the
    restatement does not place it there."""
    cfg = make(name)
    _, info, edges, items = oracle_graph(name)
    _, (fw, st, L) = host_reads(cfg)
    m = cfg["min_overlap"]
    for canon in (True, False):
        flat, starts, lens = spell_graph(fw, st, L, edges, items, canonical_mask(edges) if canon else np.ones(len(edges), bool))
        seqs = [flat[a:a + n].tobytes() for a, n in zip(starts, lens)]
        reads, where = spanning_sample(seqs, m)
        assert sum(len(seqs[u]) % 32 == 0 for u, _ in where) >= 8 and len(reads) >= 100
        lay = padded_layout(seqs)
        w0 = np.concatenate([[0], np.cumsum((lens + 31) // 32)])
        for r, (u, p) in zip(reads, where):
            at = 32 * int(w0[u]) + p
            assert lay[at:at + len(r)] in (r, sm.rc(r))
        got = sm.map_sample(seqs, reads, m)
        bad = {(u, p, i) for u, p, _, i in got["placed"]}
        assert not any((u, p, i) in bad for i, (u, p) in enumerate(where))


@pytest.fixture(scope="module")
def emul():
    return build_spell_emul(), build_coverage_emul(), build_map_emul()


@pytest.mark.parametrize("name", SETS)
def test_kernel_bodies_match_restatement(name, emul):
    spell_emul, cover_emul, map_emul = emul
    cfg = make(name)
    _, info, edges, items = oracle_graph(name)
    _, (fw, st, L) = host_reads(cfg)
    m = cfg["min_overlap"]
    words, meta = store_layout(fw, st, L)
    sup_ids = info["sup"].astype(np.int64)
    q = cv.locate(fw, st, L, sup_ids)
    for canon in (True, False):
        sel = canonical_mask(edges) if canon else np.ones(len(edges), bool)
        srecs, packed = spell_emul(words, meta, len(L), edges, items, canon)
        flat, starts, lens = spell_graph(fw, st, L, edges, items, sel)
        want_w, wstart = us.pack(flat, starts, lens)
        assert np.array_equal(srecs["length"], lens) and np.array_equal(srecs["start"], 32 * wstart) and np.array_equal(packed, want_w)
        recs, depth, unplaced, ncp = cover_emul(words, meta, edges, items, srecs, info["freq"], sup_packed(sup_ids, L))
        want = cover_graph(fw, st, L, info["freq"], sup_ids, edges, items, sel, q=q)
        assert unplaced == want["unplaced"] == 0 and ncp == int(want["contained"].sum())
        check_records(recs, want, srecs)
        assert np.array_equal(depth.astype(np.int64), padded_profile(want, srecs))
        seqs = decode_words(packed, srecs)
        for reads in (spanning_sample(seqs, m)[0], ends_sample(seqs, m)):
            b, o = join_reads(reads)
            check_against(sm.map_sample(seqs, reads, m), *map_emul(packed, srecs, b, o, m), srecs, m, seqs)


# ---------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def ctx():
    from metagenomics_b200 import Context
    c = Context(0)
    yield c
    c.close()


def device_graph(ctx, cfg):
    from metagenomics_b200 import Dataset, HashTable, OverlapGraph
    ds = Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"])
    ht = HashTable(ctx)
    ht.insertDataset(ds, cfg["min_overlap"])
    return ds, OverlapGraph(ht)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SETS)
def test_build_matches_oracle(ctx, name):
    from metagenomics_b200 import edges_as_tuples
    cfg = make(name)
    t, info, _, _ = oracle_graph(name)
    _, og = device_graph(ctx, cfg)
    assert np.array_equal(sort_tuples(edges_as_tuples(og.edges())), sort_tuples(t))
    assert np.array_equal(og.superReadIDs()[1:], info["sup"])


def in_range(sel, first, count):
    rank = np.cumsum(sel) - 1
    return sel & (rank >= first) & (rank < first + (len(sel) if count is None else count))


def check_device(og, cfg, graph, canon, first=0, count=None):
    """spell (records, ASCII and packed), coverage (records, profile) and the mapping of the spanning and ends samples of the range
    against the restatements"""
    edges, items, fw, st, L, freq, sup, q = graph
    m = cfg["min_overlap"]
    sel = in_range(canonical_mask(edges) if canon else np.ones(len(edges), bool), first, count)
    flat, starts, lens = spell_graph(fw, st, L, edges, items, sel)
    recs, seq = og.unitigs(canonical=canon, ascii=True, first=first, count=count)
    assert np.array_equal(recs["edge"], np.flatnonzero(sel)) and np.array_equal(recs["length"], lens)
    assert np.array_equal(recs["src"], edges["src"][sel]) and np.array_equal(recs["orient"], edges["orient"][sel])
    idx = np.repeat(recs["start"].astype(np.int64), lens) + (np.arange(int(lens.sum())) - np.repeat(starts, lens))
    assert np.array_equal(seq[idx], flat)
    recs2, words = og.unitigs(canonical=canon, ascii=False, first=first, count=count)
    want_w, wstart = us.pack(flat, starts, lens)
    assert np.array_equal(recs2, recs) and np.array_equal(recs["start"], 32 * wstart) and np.array_equal(words, want_w)
    crecs, depth = og.depth(canonical=canon, first=first, count=count)
    want = cover_graph(fw, st, L, freq, sup, edges, items, sel, q=q)
    check_records(crecs, want, recs)
    assert np.array_equal(depth.astype(np.int64), padded_profile(want, recs))
    seqs = unitig_seqs(recs, seq)
    for reads in (spanning_sample(seqs, m)[0], ends_sample(seqs, m)):
        b, o = join_reads(reads)
        mrecs, mst, hits = og.map_reads(bases=b, offsets=o, hits=True)
        check_against(sm.map_sample(seqs, reads, m), mrecs, og.sample_depth()[1], hits, mst, recs, m, seqs)
    return recs


@pytest.mark.gpu
@pytest.mark.parametrize("name", SETS)
def test_device_matches_restatement(ctx, name):
    cfg = make(name)
    ds, og = device_graph(ctx, cfg)
    edges, items, _ = og.simplify()
    fw, st, L = reads_ascii(ds)
    sup = og.superReadIDs()[1:].astype(np.int64)
    graph = (edges, items, fw, st, L, ds.frequencies(), sup, cv.locate(fw, st, L, sup))
    for canon in (True, False):
        recs = check_device(og, cfg, graph, canon)
    # a range whose first record starts mid-stripe in the whole layout: the ranged layout starts at word 0 all the same
    w0 = np.concatenate([[0], np.cumsum((recs["length"].astype(np.int64) + 31) // 32)])
    first = int(np.flatnonzero(w0[1:-1] % 32)[0]) + 1
    got = check_device(og, cfg, graph, False, first=first, count=len(recs) // 2)
    assert got["start"][0] == 0 and len(got) == len(recs) // 2


def weighted(seqs, distinct, m, pat):
    """sm.map_sample of the raw reads distinct[pat[i]], from the distinct reads once and their multiplicities"""
    one = sm.map_sample(seqs, distinct, m)
    w = np.bincount(pat, minlength=len(distinct)).astype(np.int64)
    start, length = one["start"], one["length"]
    diff = np.zeros(int(length.sum()) + 1, np.int64)
    count = np.zeros(len(seqs), np.int64)
    for u, p, n, i in one["placed"]:
        diff[start[u] + p] += w[i]
        diff[start[u] + p + n] -= w[i]
        count[u] += w[i]
    D = np.cumsum(diff[:-1])
    h = one["hits"]
    kept = h != sm.FILTERED
    out = dict(length=length, start=start, depth=D, hits=h[pat], reads=count, read_count=count.copy(), contained=np.zeros(len(seqs), np.int64),
               filtered=int(w[~kept].sum()), mapped=int(w[kept & (h > 0)].sum()), multi=int(w[kept & (h > 1)].sum()),
               placements=int((w[kept] * h[kept].astype(np.int64)).sum()))
    Du = D.astype(np.uint64)
    with np.errstate(over="ignore"):
        out["depth_sum"] = np.array([Du[a:a + n].sum() for a, n in zip(start, length)], np.uint64)
        out["depth_sq_sum"] = np.array([(Du[a:a + n] * Du[a:a + n]).sum() for a, n in zip(start, length)], np.uint64)
    out["depth_min"] = np.array([D[a:a + n].min() for a, n in zip(start, length)], np.int64)
    out["depth_max"] = np.array([D[a:a + n].max() for a, n in zip(start, length)], np.int64)
    return out


def tile_sample(distinct, n):
    """n raw reads distinct[i % len(distinct)], as flat bases + offsets built with numpy"""
    lens = np.array([len(r) for r in distinct], np.uint64)
    period = np.frombuffer(b"".join(distinct), np.uint8)
    reps = n // len(distinct) + 1
    offs = (np.arange(reps, dtype=np.uint64)[:, None] * np.uint64(len(period)) + np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)[None, :]).ravel()
    offs = offs[:n + 1].copy()
    return np.tile(period, reps)[:int(offs[n])], offs, np.arange(n) % len(distinct)


def check_split(og, b, o, cut, recs, depth, hits):
    """the sample mapped as two samples [0, cut) and [cut, n) adds up to the whole"""
    r1, _, h1 = og.map_reads(bases=b, offsets=o[:cut + 1], hits=True)
    d1 = og.sample_depth()[1].astype(np.int64)
    r2, _, h2 = og.map_reads(bases=b, offsets=o[cut:], hits=True)
    d2 = og.sample_depth()[1].astype(np.int64)
    assert np.array_equal(d1 + d2, depth.astype(np.int64)) and np.array_equal(np.concatenate([h1, h2]), hits)
    for k in ("reads", "read_count", "depth_sum"):
        assert np.array_equal(r1[k].astype(np.int64) + r2[k].astype(np.int64), recs[k].astype(np.int64)), k


@pytest.mark.gpu
def test_chunk_reads(ctx):
    """2^22 - 1, 2^22 and 2^22 + 1 raw reads: one chunk, one full chunk, a second chunk of one read. The reads at the last index of
    each chunk are mapped, so a hit count that is not copied back shows."""
    cfg = make("tiled_m20")
    m = cfg["min_overlap"]
    _, og = device_graph(ctx, cfg)
    og.simplify()
    srecs, ascii = og.unitigs()
    seqs = unitig_seqs(srecs, ascii)
    rng = np.random.default_rng(41)
    pieces = []
    for _ in range(250):
        S = seqs[int(rng.integers(0, len(seqs)))]
        L = int(rng.integers(m + 1, min(len(S), 60) + 1))
        a = int(rng.integers(0, len(S) - L + 1))
        pieces.append(_strand(rng, S[a:a + L]))
    pieces[::7] = [p.lower() for p in pieces[::7]]
    dropped = [p[:10] + b"N" + p[11:] for p in pieces[:20]] + [p[:m] for p in pieces[20:40]] + [_rand(rng, 45) for _ in range(20)]
    distinct = pieces[:]
    for i, x in zip(range(3, len(distinct), 5), dropped):
        distinct.insert(i, x)
    D = len(distinct)
    must = {(CHUNK_READS - 2) % D, (CHUNK_READS - 1) % D, CHUNK_READS % D}
    ok = [j for j in range(D) if distinct[j] in pieces and j not in must]
    for r in must:
        if distinct[r] not in pieces:
            j = ok.pop()
            distinct[r], distinct[j] = distinct[j], distinct[r]
    for n in (CHUNK_READS - 1, CHUNK_READS, CHUNK_READS + 1):
        b, o, pat = tile_sample(distinct, n)
        want = weighted(seqs, distinct, m, pat)
        recs, st, hits = og.map_reads(bases=b, offsets=o, hits=True)
        depth = og.sample_depth()[1]
        check_against(want, recs, depth, hits, st, srecs, m, seqs)
        assert hits[-1] not in (0, sm.FILTERED) and hits[min(n, CHUNK_READS) - 1] not in (0, sm.FILTERED)
        assert 0 < want["filtered"] and 0 < want["mapped"] < n
        check_split(og, b, o, n // 2, recs, depth, hits)


@pytest.mark.gpu
def test_chunk_bytes(ctx):
    """Reads of 65 535 .. 128 bases cut from the longest unitig of config 2 x 0.1 (and one of 65 536, filtered) repeated past
    2^30 bytes, so the byte bound cuts the sample; against the same reads as two samples below 2^30 bytes each."""
    from metagenomics_b200 import synth
    cfg = synth.config(2, scale=0.1)
    m = cfg["min_overlap"]
    _, og = device_graph(ctx, cfg)
    og.simplify()
    srecs, ascii = og.unitigs()
    seqs = unitig_seqs(srecs, ascii)
    S = max(seqs, key=len)
    assert len(S) >= 65535
    group = []
    for i, L in enumerate((65535, 40000, 1025, 1024, 1023, 129, 128)):
        a = (len(S) - L) * i // 7
        group += [S[a:a + L], sm.rc(S[a:a + L])]
    group.append(S[:65535] + b"C")
    n = len(group) * (CHUNK_BYTES // sum(len(r) for r in group) + 1)
    b, o, pat = tile_sample(group, n)
    assert int(o[-1]) > CHUNK_BYTES
    want = weighted(seqs, group, m, pat)
    assert want["filtered"] == n // len(group) and want["mapped"] == n - want["filtered"]
    recs, st, hits = og.map_reads(bases=b, offsets=o, hits=True)
    depth = og.sample_depth()[1]
    check_against(want, recs, depth, hits, st, srecs, m, seqs)
    cut = n // 2
    assert int(o[cut]) <= CHUNK_BYTES and int(o[-1] - o[cut]) <= CHUNK_BYTES
    check_split(og, b, o, cut, recs, depth, hits)


@pytest.mark.gpu
def test_depth_of_2_32_minus_1_and_refusal(ctx):
    """Frequencies summing to 2^32 - 1, all of it on 30 reads that cover one base: depth_max 0xFFFFFFFF, depth_sq_sum wraps mod 2^64
    on the device and in the restatement alike. One more is refused with OGB_E_ARG and leaves the result as it was."""
    from metagenomics_b200._lib import CoverageStats, lib
    from metagenomics_b200.api import COVERAGE_DTYPE
    cfg = make("tiled_m20")
    ds, og = device_graph(ctx, cfg)
    edges, items, _ = og.simplify()
    fw, st, L = reads_ascii(ds)
    sup = og.superReadIDs()[1:].astype(np.int64)
    e = int(np.argmax(edges["count"]))
    a = int(edges["list_start"][e]) + 100
    heavy = items["read"][a:a + 30].astype(np.int64) - 1
    freq = np.zeros(len(L), np.uint32)
    freq[heavy] = (2**32 - 1) // 30
    freq[heavy[0]] += (2**32 - 1) % 30
    assert int(freq.sum(dtype=np.uint64)) == 2**32 - 1
    q = cv.locate(fw, st, L, sup)
    cst = CoverageStats()
    for canon in (True, False):
        srecs, words = og.unitigs(canonical=canon, ascii=False)                    # the spell the coverage runs on
        assert lib().ogb_graph_coverage(ctx._h, freq.ctypes.data, len(freq), C.byref(cst)) == 0
        recs = np.zeros(len(srecs), COVERAGE_DTYPE)
        depth = np.zeros(32 * len(words), np.uint32)
        assert lib().ogb_graph_unitig_coverage(ctx._h, recs.ctypes.data, len(recs), depth.ctypes.data, len(depth)) == 0
        want = cover_graph(fw, st, L, freq, sup, edges, items, canonical_mask(edges) if canon else np.ones(len(edges), bool), q=q)
        assert int(want["depth"].max()) == 0xFFFFFFFF and (want["depth"] > 2**31).sum() >= 20 and int(want["read_count"].max()) < 2**53
        check_records(recs, want, srecs)
        assert np.array_equal(depth.astype(np.int64), padded_profile(want, srecs))
        over = freq.copy()
        over[heavy[1]] += 1
        assert lib().ogb_graph_coverage(ctx._h, over.ctypes.data, len(over), C.byref(cst)) == 1
        assert str(2**32) in lib().ogb_last_error().decode()
        recs2 = np.zeros_like(recs)
        depth2 = np.zeros_like(depth)
        assert lib().ogb_graph_unitig_coverage(ctx._h, recs2.ctypes.data, len(recs2), depth2.ctypes.data, len(depth2)) == 0
        assert recs2.tobytes() == recs.tobytes() and np.array_equal(depth2, depth)


@pytest.mark.gpu
def test_fasta_across_the_writer_chunk(ctx, tmp_path):
    """Config 3 at full size: a ranged spell whose layout holds more than 2^20 words and a unitig across word 2^20 (the writer's
    chunk). The FASTA equals one composed from ogb_graph_unitigs byte for byte."""
    from metagenomics_b200 import synth
    from metagenomics_b200._lib import check, lib
    cfg = synth.config(3)
    _, og = device_graph(ctx, cfg)
    edges, _, _ = og.simplify()
    whole, _ = og.unitigs(ascii=False)
    W = np.concatenate([[0], np.cumsum((whole["length"].astype(np.int64) + 31) // 32)])
    b1 = 32 * SPELL_CHUNK_WORDS
    first = next(f for f in range(1, len(whole)) if
                 ((32 * (W[f:-1] - W[f]) < b1) & (32 * (W[f:-1] - W[f]) + whole["length"][f:].astype(np.int64) > b1)).any())
    recs, seq = og.unitigs(first=first)
    assert int(recs["start"][-1] + recs["length"][-1]) > b1
    assert ((recs["start"].astype(np.int64) < b1) & (recs["start"].astype(np.int64) + recs["length"].astype(np.int64) > b1)).any()
    path = tmp_path / "u.fa"
    check(lib().ogb_graph_write_unitigs(og.ctx._h, str(path).encode()))
    parts = []
    for i, r in enumerate(recs):
        a, n = int(r["start"]), int(r["length"])
        parts.append(b">unitig_%d src=%d dst=%d orient=%d reads=%d length=%d\n" % (first + i, r["src"], r["dst"], r["orient"],
                                                                                   edges["count"][r["edge"]] + 2, n))
        parts += [seq[a:a + n].tobytes(), b"\n"]
    assert path.read_bytes() == b"".join(parts)

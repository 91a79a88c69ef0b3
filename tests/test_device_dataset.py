"""The Dataset stage on the GPU (ogb_dataset_finalize_device: k_ds_filter / k_ds_compact, k_ds_canon, the LSD radix sort
k_ds_key / k_rs_orand / k_rs_hist / k_rs_scatter, k_ds_heads / k_ds_unique / k_ds_emit, and k_pack_words for the resident
read store) against the host Dataset (ogb_dataset_finalize), on sets built to reach the points where the device stage
changes behaviour: row widths W = ceil(longest / 32) from 1 to 2048 words, key bytes the sort skips, reads that tie on every
word and differ in length only, duplicate runs longer than a 2048-pair scatter tile, canonical strands decided at an inner
word, the filter's length and base-count edges, and every length residue mod 32 of the resident store.

`restate` is the stage in a few lines of plain Python (Dataset.cpp:155-167, 197-202, 316-345, 398-413). The CPU tests pin
the host Dataset to it on every set; the GPU tests then require the device stage to give the host's answers, and build the
overlap graph from the reads the device stage leaves in HBM."""
import ctypes as C
import functools
import re
from collections import Counter

import numpy as np
import pytest

import datasets
from oracle_lib import Oracle, sort_tuples

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = str.maketrans("ACGTacgt", "TGCAtgca")
_NOT_ACGT = str.maketrans("", "", "ACGT")
NONE_KEPT = (2 ** 64 - 1, 0)            # shortest / longest of a data set without a kept read (Dataset.cpp initial values)


def rc(s):
    return s.translate(_COMP)[::-1]


def keeps(read, m):
    """The filter: m < length < 65536, ACGT only after upper-casing, no base count reaching (UINT64)(length * .8)."""
    L = len(read)
    if not m < L < 65536:
        return False
    s = read.upper()
    return not s.translate(_NOT_ACGT) and max(s.count(b) for b in "ACGT") < int(L * 0.8)


def restate(reads, m):
    """reads: ASCII strings. Returns (sorted unique canonical strings -- read ID i is entry i - 1 --, their frequencies,
    n_good, (shortest, longest) of the kept reads)."""
    kept = []
    for r in reads:
        if keeps(r, m):
            s = r.upper()
            kept.append(min(s, rc(s)))
    freq = Counter(kept)
    uniq = sorted(freq)
    span = (min(map(len, kept)), max(map(len, kept))) if kept else NONE_KEPT
    return uniq, [freq[s] for s in uniq], len(kept), span


def reads_of(cfg):
    raw, o = cfg["bases"].tobytes().decode("ascii"), cfg["offsets"].tolist()
    return [raw[o[i]:o[i + 1]] for i in range(len(o) - 1)]


def _seq(rng, n):
    return _ACGT[rng.integers(0, 4, n)].tobytes().decode()


def _sample(rng, genome, n, lmin, lmax):
    """n reads of lengths lmin..lmax from random positions of genome, each on a random strand."""
    out = []
    for L in rng.integers(lmin, lmax + 1, n):
        st = int(rng.integers(0, len(genome) - L + 1))
        s = genome[st:st + int(L)]
        out.append(s if rng.integers(0, 2) else rc(s))
    return out


def _shuffled(rng, reads):
    return [reads[i] for i in rng.permutation(len(reads))]


# ---- seeded sets (datasets.from_strings layout) ----

WIDTHS = (32, 33, 64, 65, 257, 1000, 4097, 65535)


def widths(longest, seed=31):
    """Short reads (lengths 21..min(120, longest), 40..120 once the longest read exceeds 65 bases) of a 20 kb genome plus a
    few long random reads, the longest exactly `longest` bases -- which sets the row width of every read. That read is also
    there on the other strand and with its last base changed. At most about 2 000 reads once W = 2048 (n * W * 8 < 64 MB)."""
    rng = np.random.default_rng(seed + longest)
    W = (longest + 31) // 32
    n = min(20000, 2000 * 2048 // W)
    lo = 21 if longest <= 65 else 40
    reads = _sample(rng, _seq(rng, 20000), n, lo, min(120, longest))
    top = _seq(rng, longest)
    last = "ACGT"[("ACGT".index(top[-1]) + 1) % 4]
    reads += [top, rc(top), top[:-1] + last] + [_seq(rng, int(L)) for L in rng.integers(min(121, longest), longest + 1, 4)]
    return datasets.from_strings(_shuffled(rng, reads), 20, f"widths_{longest}")


def prefix_family(seed=32):
    """A 300-base s that starts with 'A', its prefixes s[:k] for k = 41..300 and s[:k] + 'A' * j for j = 1..3, shuffled. Padding
    is 'A', so s[:k] and s[:k] + 'A' * j have equal rows and only the length key separates them; lengths 41..303 cross
    255/256, so the length key varies in two bytes."""
    rng = np.random.default_rng(seed)
    s = "A" + _seq(rng, 299)
    reads = [s[:k] for k in range(41, 301)] + [s[:k] + "A" * j for k in range(41, 301) for j in (1, 2, 3)]
    return datasets.from_strings(_shuffled(rng, reads), 40, "prefix_family")


def late_difference(seed=33):
    """Reads p + b (b = A, C, G, T) that share their first L - 1 bases (and hence every word but the last) at lengths around
    word boundaries, some given on the other strand; and reads x + y + rc(x) with |x| a multiple of 32, whose forward and
    reverse-complement rows agree on every word except the one holding y. y and rc(y) give the same canonical read
    (frequency 2). Every such read r also comes as r[d:] + d random bases (d = 1..20), which overlaps it by L - d >= 45
    bases, so the graph built from these reads has edges through the late words. All reads are at most 300 bases."""
    rng = np.random.default_rng(seed)
    reads = []
    for L in (64, 65, 96, 97, 128, 250, 300):
        p = "AC" + _seq(rng, L - 4) + "A"                      # forward is the smaller strand for every b
        reads += [p + b for b in "ACGT"]
    for nx in (32, 64, 96, 128):
        x = _seq(rng, nx)
        for ny in (1, 2, 31, 32, 33):
            ys = [_seq(rng, ny) for _ in range(3)]
            ys.append(rc(ys[0]))
            reads += [x + y + rc(x) for y in ys]
    shifted = [r[d:] + _seq(rng, d) for r, d in zip(reads, rng.integers(1, 21, len(reads)))]
    reads = [r if rng.integers(0, 3) else rc(r) for r in reads + shifted]
    return datasets.from_strings(_shuffled(rng, reads), 40, "late_difference")


DUPLICATES = ("one_read_5000", "tile_runs", "n1", "n2", "n257", "n2049", "identical", "rc_pairs")


def duplicates(kind, seed=34):
    """one_read_5000: one read 5 000 times on both strands among 3 000 others. tile_runs: ten reads 2047, 2048 or 2049 times
    each, shuffled among 3 000 others. nK: K reads of a 3 kb genome, drawn with repeats. identical: 3 000 copies of one read
    (no key byte varies). rc_pairs: 40 reads, each also given as its reverse complement (every frequency is 2)."""
    rng = np.random.default_rng(seed + DUPLICATES.index(kind))
    g = _seq(rng, 3000)
    if kind == "one_read_5000":
        r = _seq(rng, 150)
        reads = [r if i % 2 else rc(r) for i in range(5000)] + _sample(rng, g, 3000, 80, 200)
    elif kind == "tile_runs":
        reads = _sample(rng, g, 3000, 80, 200)
        for i, r in enumerate(_sample(rng, g, 10, 100, 100)):
            reads += [r] * (2047 + i % 3)
    elif kind.startswith("n"):
        n = int(kind[1:])
        pool = _sample(rng, g, max(1, 2 * n // 3), 60, 140)
        reads = [pool[i] if rng.integers(0, 2) else rc(pool[i]) for i in rng.integers(0, len(pool), n)]
    elif kind == "identical":
        reads = [_seq(rng, 120)] * 3000
    else:
        pool = _sample(rng, g, 40, 60, 140)
        reads = pool + [rc(r) for r in pool]
    return datasets.from_strings(_shuffled(rng, reads), 30, f"dup_{kind}")


def palindromes(seed=35):
    """h + rc(h) (even length, equal to its own reverse complement, given on both strands) and h + b + rc(h) (odd length:
    the strands differ in the middle base only), half lengths 21..100, plus reads of a genome holding them."""
    rng = np.random.default_rng(seed)
    reads, genome = [], ""
    for k in (21, 31, 32, 33, 48, 63, 64, 100):
        h = _seq(rng, k)
        pal = h + rc(h)
        odd = h + _seq(rng, 1) + rc(h)
        reads += [pal, pal, odd, rc(odd), odd]
        genome += _seq(rng, 150) + pal + _seq(rng, 150) + odd
    reads += _sample(rng, genome + _seq(rng, 150), 600, 60, 200)
    return datasets.from_strings(_shuffled(rng, reads), 30, "palindromes")


FILTER_M = 50


def filter_edge_reads(seed=36):
    """(read, kept?) pairs at the filter's edges for minOverlap FILTER_M: lengths m / m + 1 / 65535 / 65536; lower and mixed
    case (one read four times, once as its lower-case reverse complement: one entry of frequency 4); 'N', 'n' and '*' at
    the first or the last position; one base exactly int(0.8 L) times (dropped) and once less (kept), for every base and
    several L."""
    rng = np.random.default_rng(seed)
    m = FILTER_M
    out = [(_seq(rng, m), False), (_seq(rng, m + 1), True), (_seq(rng, 65535), True), (_seq(rng, 65536), False)]
    r = _seq(rng, 90)
    mixed = "".join(c.lower() if i % 3 else c for i, c in enumerate(r))
    out += [(r, True), (r.lower(), True), (mixed, True), (rc(r).lower(), True)]
    for bad in "Nn*":
        s = _seq(rng, 80)
        out += [(bad + s[1:], False), (s[:-1] + bad, False), (s, True)]
    for L in (m + 1, 100, 256, 1001):
        thr = int(L * 0.8)
        for b in "ACGT":
            others = [c for c in "ACGT" if c != b]
            for c, keep in ((thr, False), (thr - 1, True)):
                s = list(b * c + "".join(rng.choice(others, L - c)))
                rng.shuffle(s)
                out.append(("".join(s) if rng.integers(0, 2) else "".join(s).lower(), keep))
    return [out[i] for i in rng.permutation(len(out))]


def filter_edges(kind):
    if kind == "edges":
        return datasets.from_strings([r for r, _ in filter_edge_reads()], FILTER_M, "filter_edges")
    if kind == "none_kept":
        reads = ["N" * 60, "A" * 60, "ACGT" * 12, "acgtn" * 20, "G" * 49 + "C" * 11, "ACGTAC" * 8 + "x" * 3, "T" * 56 + "acg" * 4 + "ac"]
        return datasets.from_strings(reads, FILTER_M, "filter_none_kept")
    return datasets.from_strings([], FILTER_M, "filter_empty")


def pack_residues(seed=37):
    """20 reads of every length 33..96 from a 4 kb genome, both strands, minOverlap 30: L mod 32 takes all 32 values on both
    sides of a word boundary, and the reads overlap densely, so a wrong reverse-complement word of the store changes edges."""
    rng = np.random.default_rng(seed)
    g = _seq(rng, 4000)
    reads = [r for L in range(33, 97) for r in _sample(rng, g, 20, L, L)]
    return datasets.from_strings(_shuffled(rng, reads), 30, "pack_residues")


def config3_duplicated(seed=38):
    """Config-3 shape at 0.17 (1.7 M reads of 100 bases) plus 10 % exact duplicates and 5 % reverse-complement duplicates,
    shuffled: about 2 M reads in a thousand scatter tiles, several byte passes for every word."""
    from metagenomics_b200 import synth
    cfg = synth.config(3, scale=0.17)
    rows = cfg["bases"].reshape(-1, 100)
    rng = np.random.default_rng(seed)
    comp = np.zeros(256, np.uint8)
    comp[np.frombuffer(b"ACGT", np.uint8)] = np.frombuffer(b"TGCA", np.uint8)
    n = len(rows)
    rows = np.concatenate([rows, rows[rng.integers(0, n, n // 10)], comp[rows[rng.integers(0, n, n // 20)][:, ::-1]]])
    rows = rows[rng.permutation(len(rows))]
    offs = np.arange(len(rows) + 1, dtype=np.uint64) * np.uint64(100)
    return dict(name="config3_duplicated", bases=np.ascontiguousarray(rows).ravel(), offsets=offs, min_overlap=cfg["min_overlap"], paired=False)


def config5_scaled():
    from metagenomics_b200 import synth
    return synth.config(5, scale=0.2)


SETS = {f"widths_{L}": functools.partial(widths, L) for L in WIDTHS}
SETS.update(prefix_family=prefix_family, late_difference=late_difference)
SETS.update({f"dup_{k}": functools.partial(duplicates, k) for k in DUPLICATES})
SETS.update(palindromes=palindromes, pack_residues=pack_residues)
SETS.update({f"filter_{k}": functools.partial(filter_edges, k) for k in ("edges", "none_kept", "empty")})
SETS.update(scale_config5=config5_scaled, scale_config3_duplicated=config3_duplicated)


@functools.lru_cache(maxsize=None)
def get(name):
    return SETS[name]()


def sample_ids(n, seed=39):
    """Every ID of a set under 10 000 unique reads, else 2 000 seeded ones plus the first and the last."""
    if n < 10000:
        return list(range(1, n + 1))
    rng = np.random.default_rng(seed)
    return sorted(set((rng.choice(n, 2000, replace=False) + 1).tolist()) | {1, n})


def dataset(cfg, device=None):
    from metagenomics_b200 import Dataset
    return Dataset(bases=cfg["bases"], offsets=cfg["offsets"], minOverlap=cfg["min_overlap"], device=device)


def words_of(s, W):
    """The 2-bit row of s (A C G T = 0 1 2 3, first base in the top bits), zero-padded to W words."""
    codes = np.zeros(32 * W, np.uint64)
    codes[:len(s)] = np.frombuffer(s.translate(str.maketrans("ACGT", "\0\1\2\3")).encode(), np.uint8)
    return (codes.reshape(W, 32) << (np.uint64(62) - np.uint64(2) * np.arange(32, dtype=np.uint64))).sum(axis=1, dtype=np.uint64)


def restated_passes(uniq):
    """Byte passes of the device sort: for every key word (the length, then words W-1 .. 0 of the canonical rows), one pass per
    byte in which two keys differ. Duplicates change no OR / AND, so the unique reads give the count."""
    if not uniq:
        return 0
    W = (max(map(len, uniq)) + 31) // 32
    rows = np.stack([words_of(s, W) for s in uniq])
    keys = np.concatenate([rows, np.array([[len(s)] for s in uniq], np.uint64)], axis=1)
    varying = np.bitwise_or.reduce(keys, axis=0) ^ np.bitwise_and.reduce(keys, axis=0)
    return sum(int((int(v) >> s) & 255 != 0) for v in varying for s in range(0, 64, 8))


# ---- CPU: the host Dataset equals the restatement ----

@pytest.mark.parametrize("name", list(SETS))
def test_host_dataset_equals_restatement(name):
    cfg = get(name)
    uniq, freq, n_good, span = restate(reads_of(cfg), cfg["min_overlap"])
    ds = dataset(cfg)
    assert ds.getNumberOfReads() == n_good and ds.getNumberOfUniqueReads() == len(uniq)
    assert (ds.shortestReadLength, ds.longestReadLength) == span
    assert ds.lengths().tolist() == [len(s) for s in uniq]
    assert ds.frequencies().tolist() == freq
    for i in sample_ids(len(uniq)):
        assert ds.getReadFromID(i) == uniq[i - 1], i


def test_sets_reach_their_branches():
    """Each set has the shape it is meant to have (checked on the restatement, so it holds for whatever it tests)."""
    for L in WIDTHS:
        uniq, freq, n_good, span = restate(reads_of(get(f"widths_{L}")), 20)
        assert span[1] == L and n_good * ((L + 31) // 32) * 8 < 64 << 20
    assert (restate(reads_of(get("widths_65535")), 20)[3][1] + 31) // 32 == 2048
    uniq = restate(reads_of(get("prefix_family")), 40)[0]
    assert min(map(len, uniq)) <= 255 < 256 <= max(map(len, uniq))
    have = set(uniq)
    assert sum(s + "A" in have for s in uniq) > 100                       # rows that tie, the length decides
    uniq = restate(reads_of(get("late_difference")), 40)[0]
    assert sum(a[:-1] == b[:-1] and len(a) == len(b) for a, b in zip(uniq, uniq[1:])) >= 7 * 3
    inner = 0
    for s in uniq:
        W = (len(s) + 31) // 32
        d = np.nonzero(words_of(s, W) != words_of(rc(s), W))[0]
        inner += len(d) == 1 and 0 < d[0] < W - 1
    assert inner >= 12
    assert max(restate(reads_of(get("dup_one_read_5000")), 30)[1]) == 5000
    freq = restate(reads_of(get("dup_tile_runs")), 30)[1]
    assert max(freq) > 2048 and {2047, 2048, 2049} <= set(freq)
    assert [restate(reads_of(get(f"dup_n{n}")), 30)[2] for n in (1, 2, 257, 2049)] == [1, 2, 257, 2049]
    assert len(restate(reads_of(get("dup_identical")), 30)[0]) == 1
    assert set(restate(reads_of(get("dup_rc_pairs")), 30)[1]) == {2}
    uniq = restate(reads_of(get("palindromes")), 30)[0]
    assert any(s == rc(s) and len(s) % 2 == 0 for s in uniq) and any(len(s) % 2 for s in uniq)
    pairs = filter_edge_reads()
    assert [keeps(r, FILTER_M) for r, _ in pairs] == [k for _, k in pairs]
    assert restate(reads_of(get("filter_none_kept")), FILTER_M)[2] == 0
    assert sorted(set(map(len, restate(reads_of(get("pack_residues")), 30)[0]))) == list(range(33, 97))


# ---- GPU: the device stage equals the host Dataset ----

@pytest.fixture(scope="module")
def ctx():
    from metagenomics_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SETS))
def test_device_dataset_equals_host(ctx, name):
    cfg = get(name)
    host, dev = dataset(cfg), dataset(cfg, ctx)
    n = host.getNumberOfUniqueReads()
    assert dev.getNumberOfReads() == host.getNumberOfReads() and dev.getNumberOfUniqueReads() == n
    assert (dev.shortestReadLength, dev.longestReadLength) == (host.shortestReadLength, host.longestReadLength)
    assert np.array_equal(dev.lengths(), host.lengths()) and np.array_equal(dev.frequencies(), host.frequencies())
    hw, ho, _ = host.packed(); dw, do, _ = dev.packed()
    assert np.array_equal(do, ho) and np.array_equal(dw, hw)
    ids = sample_ids(n)
    for i in ids:
        assert dev.getReadFromID(i) == host.getReadFromID(i) and dev.getReadFromID(i, reverse=True) == host.getReadFromID(i, reverse=True), i
    for i in ids[::max(1, len(ids) // 200)]:
        f = host.getReadFromID(i)
        assert dev.getReadFromString(f) == i and dev.getReadFromString(rc(f).lower()) == i, i


@pytest.mark.gpu
def test_radix_pass_counts(ctx, monkeypatch, capfd):
    """The sort takes one pass per varying key byte: none for identical reads or a single read, two length passes plus the
    word passes for the prefix family -- the counts the restatement predicts."""
    monkeypatch.setenv("OGB_DBG_TIMING", "1")
    got = {}
    for name in ("dup_identical", "dup_n1", "prefix_family", "widths_33", "late_difference"):
        cfg = get(name)
        capfd.readouterr()
        dataset(cfg, ctx)
        found = re.findall(r"\[finalize_device\] (\d+) radix passes", capfd.readouterr().err)
        assert len(found) == 1, name
        got[name] = int(found[0])
        assert got[name] == restated_passes(restate(reads_of(cfg), cfg["min_overlap"])[0]), name
    assert got["dup_identical"] == 0 and got["dup_n1"] == 0 and got["prefix_family"] >= 2


GRAPH_SETS = ("pack_residues", "late_difference", "palindromes", "dup_n1", "dup_n2", "dup_n257", "dup_n2049", "dup_identical", "dup_rc_pairs")


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAPH_SETS)
def test_graph_from_resident_reads_matches_oracle(ctx, name):
    """K0 from the device stage's own words (k_pack_words, no second upload): k_verify compares bases against the stored
    strands, so a wrong reverse-complement word shows up as a wrong edge or superReadID."""
    from metagenomics_b200 import HashTable, OverlapGraph, edges_as_tuples
    cfg = get(name)
    m = cfg["min_overlap"]
    assert max(np.diff(cfg["offsets"].astype(np.int64))) <= 300
    dev = dataset(cfg, ctx)
    ht = HashTable(ctx)
    ht.insertDataset(dev, m)
    og = OverlapGraph(ht, keep_pre=True)
    orc = Oracle(cfg["bases"], cfg["offsets"], m).run_all(Oracle.BFS)
    assert dev.getNumberOfUniqueReads() == orc.n
    assert np.array_equal(og.superReadIDs()[1:], orc.read_info()["sup"])
    for pre in (True, False):
        got, want = sort_tuples(edges_as_tuples(og.edges(pre=pre))), orc.edges(pre=pre)
        assert got.shape == want.shape and np.array_equal(got, want), (name, "pre" if pre else "post", len(got), len(want))


@pytest.mark.gpu
def test_refused_calls_leave_the_dataset_usable(ctx):
    """A second finalize of a finalized data set is OGB_E_STATE and changes nothing; minOverlap < 2 is OGB_E_ARG, after which
    the raw reads are still there and the host finalize still succeeds."""
    from metagenomics_b200._lib import OGB_E_ARG, OGB_E_STATE, OGB_OK, lib
    cfg = get("pack_residues")
    m = cfg["min_overlap"]
    dev = dataset(cfg, ctx)
    freq, n = dev.frequencies(), dev.getNumberOfUniqueReads()
    assert lib().ogb_dataset_finalize_device(dev._h, ctx._h, m) == OGB_E_STATE
    assert lib().ogb_dataset_finalize(dev._h, m) == OGB_E_STATE
    assert dev.getNumberOfUniqueReads() == n and np.array_equal(dev.frequencies(), freq)
    uniq = restate(reads_of(cfg), m)[0]
    assert dev.getReadFromID(n) == uniq[-1]
    h = C.c_void_p()
    assert lib().ogb_dataset_create(C.byref(h)) == OGB_OK
    try:
        bases, offs = cfg["bases"], cfg["offsets"]
        assert lib().ogb_dataset_add_reads(h, bases.ctypes.data, offs.ctypes.data, len(offs) - 1) == OGB_OK
        for bad in (0, 1):
            assert lib().ogb_dataset_finalize_device(h, ctx._h, bad) == OGB_E_ARG
        bp, op, nr = C.c_void_p(), C.c_void_p(), C.c_uint64()
        assert lib().ogb_dataset_raw_reads(h, C.byref(bp), C.byref(op), C.byref(nr)) == OGB_OK
        assert nr.value == len(offs) - 1 and C.string_at(bp.value, len(bases)) == bases.tobytes()
        assert lib().ogb_dataset_finalize(h, m) == OGB_OK
        assert lib().ogb_dataset_n_unique(h) == len(uniq) and lib().ogb_dataset_n_reads(h) == restate(reads_of(cfg), m)[2]
    finally:
        lib().ogb_dataset_destroy(h)

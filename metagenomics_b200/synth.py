"""Seeded synthetic read sets: the five BASELINE.json configurations (SURVEY.md 8(d)) plus
adversarial genomes for the parity tests. Generation runs in libogb's host code (ogb_synth_*)."""
import ctypes as C

import numpy as np

from ._lib import check, lib


def genome(seed, length):
    out = np.empty(length, dtype=np.uint8)
    check(lib().ogb_synth_genome(seed, length, out.ctypes.data))
    return out


def sample_reads(seed, genomes, n_reads, len_min, len_max=None, weights=None, paired=False, insert_mean=300.0,
                 insert_sd=30.0):
    """genomes: list of uint8 arrays. Returns (bases uint8, offsets uint64[n_reads+1])."""
    len_max = len_max or len_min
    g_offs = np.zeros(len(genomes) + 1, dtype=np.uint64)
    g_offs[1:] = np.cumsum([len(g) for g in genomes], dtype=np.uint64)
    flat = np.ascontiguousarray(np.concatenate(genomes)) if len(genomes) > 1 else np.ascontiguousarray(genomes[0])
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
    cap = int(n_reads) * int(len_max)
    bases = np.empty(cap, dtype=np.uint8)
    offs = np.zeros(n_reads + 1, dtype=np.uint64)
    check(lib().ogb_synth_reads(seed, flat.ctypes.data, g_offs.ctypes.data, None if w is None else w.ctypes.data,
                                len(genomes), n_reads, len_min, len_max, 1 if paired else 0, insert_mean, insert_sd,
                                bases.ctypes.data, cap, offs.ctypes.data))
    return bases[:int(offs[-1])], offs


def substitute(seed, bases, rate):
    """Sequencing substitutions: every base of the flat ASCII `bases` (upper-case ACGT) is replaced, independently with probability
    `rate`, by one of the other three bases, uniformly. Returns a new array (bases itself when rate is 0)."""
    if rate <= 0 or len(bases) == 0:
        return bases
    rng = np.random.default_rng(seed)
    n = len(bases)
    gaps = []
    total = 0
    while total < n:                                              # a Bernoulli process as geometric gaps between substituted bases
        g = rng.geometric(rate, int(n * rate * 1.05) + 64)
        gaps.append(g)
        total += int(g.sum())
    pos = np.cumsum(np.concatenate(gaps)) - 1
    pos = pos[pos < n]
    code = np.full(256, 0, np.uint8)
    code[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)
    out = np.array(bases, dtype=np.uint8, copy=True)
    out[pos] = np.frombuffer(b"ACGT", np.uint8)[(code[out[pos]] + rng.integers(1, 4, len(pos), dtype=np.uint8)) % 4]
    return out


def _metagenome(seed, n_genomes, len_lo, len_hi, scale):
    rng = np.random.default_rng(seed)
    lens = (rng.uniform(len_lo, len_hi, n_genomes) * scale).astype(np.int64)
    lens = np.maximum(lens, 2000)
    weights = np.exp(rng.normal(0.0, 1.0, n_genomes))
    gs = [genome(seed * 1000 + i, int(l)) for i, l in enumerate(lens)]
    return gs, weights


def config(k, scale=1.0):
    """BASELINE.json configs[k-1], optionally scaled down (genome length and read count together,
    so coverage -- hence degree, hit rate and bytes per read -- stays that of the named config).
    Returns dict(name, bases, offsets, min_overlap, paired)."""
    s = float(scale)
    if k == 1:
        g = [genome(1, max(2000, int(100_000 * s)))]
        b, o = sample_reads(1, g, max(100, int(10_000 * s)), 100)
        return dict(name="config1: 100 kb genome, 10k x 100 bp, minOverlap 40", bases=b, offsets=o, min_overlap=40, paired=False)
    if k == 2:
        g = [genome(2, max(4000, int(5_000_000 * s)))]
        n = max(100, int(750_000 * s)) * 2
        b, o = sample_reads(2, g, n, 100, paired=True, insert_mean=300.0, insert_sd=30.0)
        return dict(name="config2: 5 Mb genome, 30x, 1.5M x 100 bp paired-end, minOverlap 50", bases=b, offsets=o, min_overlap=50, paired=True)
    if k == 3:
        gs, w = _metagenome(3, 20, 1e6, 5e6, s)
        b, o = sample_reads(3, gs, max(1000, int(10_000_000 * s)), 100, weights=w)
        return dict(name="config3: 20 genomes log-normal abundance, 10M x 100 bp, minOverlap 50", bases=b, offsets=o, min_overlap=50, paired=False)
    if k == 4:
        gs, w = _metagenome(4, 200, 1e6, 8e6, s)
        b, o = sample_reads(4, gs, max(1000, int(50_000_000 * s)), 150, weights=w)
        return dict(name="config4: 200 genomes, 50M x 150 bp, minOverlap 60", bases=b, offsets=o, min_overlap=60, paired=False)
    if k == 5:
        return containment_stress(5, genome_len=max(4000, int(20_000_000 * s)), n_primary=max(200, int(1_600_000 * s)))
    raise ValueError("config 1..5")


def containment_stress(seed, genome_len, n_primary, len_min=75, len_max=250, derived_frac=0.25, min_overlap=50):
    """Config 5: mixed 75-250 bp reads + 20 % derived reads (half exact duplicates on a random
    strand, half proper substrings) -- exercises contained-read marking and the reduction."""
    g = [genome(seed, genome_len)]
    b, o = sample_reads(seed, g, n_primary, len_min, len_max)
    rng = np.random.default_rng(seed)
    n_der = int(n_primary * derived_frac)       # 0.25 of primary = 20 % of the total
    src = rng.integers(0, n_primary, n_der)
    comp = np.zeros(256, dtype=np.uint8)
    for a, c in zip(b"ACGT", b"TGCA"):
        comp[a] = c
    pieces = []
    for i, r in enumerate(src):
        s = b[int(o[r]):int(o[r + 1])]
        if i % 2 == 1 and len(s) > len_min:
            ln = int(rng.integers(len_min, len(s)))       # proper substring, length len_min..len-1
            st = int(rng.integers(0, len(s) - ln + 1))
            s = s[st:st + ln]
        if rng.integers(0, 2):
            s = comp[s[::-1]]
        pieces.append(s)
    bases = np.concatenate([b] + pieces) if pieces else b
    offs = np.zeros(n_primary + n_der + 1, dtype=np.uint64)
    offs[:n_primary + 1] = o
    if pieces:
        offs[n_primary + 1:] = o[-1] + np.cumsum([len(p) for p in pieces], dtype=np.uint64)
    return dict(name="config5: containment/duplication stress, mixed 75-250 bp, 20% duplicate+contained, minOverlap 50",
                bases=bases, offsets=offs, min_overlap=min_overlap, paired=False)


def write_fasta(path, bases, offsets):
    """One sequence per record, single line -- the input format of the reference binary."""
    with open(path, "wb") as f:
        mv = memoryview(np.ascontiguousarray(bases))
        for i in range(len(offsets) - 1):
            f.write(b">r%d\n" % i)
            f.write(mv[int(offsets[i]):int(offsets[i + 1])])
            f.write(b"\n")

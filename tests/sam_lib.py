"""TEST INFRASTRUCTURE: the SAM of a sample (ogb_graph_map_reads_sam, csrc/ogb_sam.cuh) restated in plain Python on top of
map_approx_lib.map_sample_approx, which gives the placements; this module adds each placement's strand and MD string and writes the
header and records as include/ogb.h defines them. Also a line parser and the pileup of a SAM. Nothing in the product imports this."""
import numpy as np

from map_approx_lib import FILTERED, UNPLACED, kept, map_sample_approx, rc

HEADER_PG = b"@PG\tID:ogb_map\tPN:ogb\tCL:max_mismatches=%d\n"


def header(lengths, d, first=0):
    out = [b"@HD\tVN:1.6\tSO:unsorted\n"]
    out += [b"@SQ\tSN:unitig_%d\tLN:%d\n" % (first + u, int(L)) for u, L in enumerate(lengths)]
    out.append(HEADER_PG % d)
    return b"".join(out)


def hamming(a, b):
    return int((np.frombuffer(a, np.uint8) != np.frombuffer(b, np.uint8)).sum())


def md_string(ref, t):
    """SAM MD of t against ref (same length, substitutions only): counts and reference bases, a count first and last"""
    out, run = [], 0
    for x, y in zip(ref, t):
        if x == y:
            run += 1
        else:
            out.append(b"%d%c" % (run, x))
            run = 0
    out.append(b"%d" % run)
    return b"".join(out)


def filtered_seq(r):
    s = bytes(c - 32 if 97 <= c <= 122 else c if 65 <= c <= 90 else 78 for c in r)
    return s or b"*"


def sam_records(seqs, reads, m, d, first=0, names=None, want=None):
    """(records text, map_sample_approx's dict) of one sample; names: None (QNAME = index) or one bytes name per read"""
    want = want if want is not None else map_sample_approx(seqs, reads, m, d)
    per = {}
    for u, p, L, i in want["placed"]:
        per.setdefault(i, []).append((u, p))
    out = []
    for i, r in enumerate(reads):
        q = names[i] if names is not None else b"%d" % i
        s = kept(bytes(r), m)
        if s is None:
            assert want["hits"][i] == FILTERED
            out.append(q + b"\t4\t*\t0\t0\t*\t*\t0\t0\t" + filtered_seq(bytes(r)) + b"\t*\tYF:Z:filtered\n")
            continue
        pl = per.get(i, [])
        if not pl:
            out.append(q + b"\t4\t*\t0\t0\t*\t*\t0\t0\t" + s + b"\t*\n")
            continue
        b, h, L = int(want["mismatches"][i]), len(pl), len(s)
        assert h == int(want["hits"][i]) and pl == sorted(pl)
        for k, (u, p) in enumerate(pl):
            ref = seqs[u][p:p + L]
            strand = 0 if hamming(ref, s) == b else 1
            t = s if strand == 0 else rc(s)
            assert hamming(ref, t) == b
            out.append(b"%s\t%d\tunitig_%d\t%d\t%d\t%dM\t*\t0\t0\t%s\t*\tNM:i:%d\tMD:Z:%s\tNH:i:%d\n"
                       % (q, 16 * strand + 256 * (k > 0), first + u, p + 1, 60 if h == 1 else 0, L, t, b, md_string(ref, t), h))
    return b"".join(out), want


def sam_text(seqs, reads, m, d, first=0, names=None):
    """the whole file: header, then the records"""
    rec, want = sam_records(seqs, reads, m, d, first, names)
    return header([len(s) for s in seqs], d, first) + rec, want


def parse(line):
    """one record line -> dict of its fields and tags"""
    f = line.rstrip(b"\n").split(b"\t")
    out = dict(qname=f[0], flag=int(f[1]), rname=f[2], pos=int(f[3]), mapq=int(f[4]), cigar=f[5], seq=f[9])
    assert f[6:9] == [b"*", b"0", b"0"] and f[10] == b"*", f
    for t in f[11:]:
        k, typ, v = t.split(b":", 2)
        out[k.decode()] = int(v) if typ == b"i" else v
    return out


def check_md(ref, seq, md, nm):
    """MD and NM of a record agree with SEQ against the reference bytes"""
    assert md_string(ref, seq) == md and hamming(ref, seq) == nm


def pileup(lines, lengths, first=0):
    """per-unitig int64 depth of every mapped record: +1 on [POS - 1, POS - 1 + L)"""
    diff = [np.zeros(int(L) + 1, np.int64) for L in lengths]
    for ln in lines:
        f = ln.split(b"\t", 6)
        if int(f[1]) & 4:
            continue
        u = int(f[2][7:]) - first
        p = int(f[3]) - 1
        L = int(f[5][:-1])
        diff[u][p] += 1
        diff[u][p + L] -= 1
    return [np.cumsum(x[:-1]) for x in diff]


__all__ = ["FILTERED", "UNPLACED", "header", "md_string", "sam_records", "sam_text", "parse", "check_md", "pileup", "filtered_seq"]

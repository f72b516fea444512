"""CPU restatement of the strand switches and inversion calls (test infrastructure; no reference counterpart, DESIGN.md
section 5.5f; include/gavisunk_b200.h gvs_strand_switches, cli.inversion_texts).

Brute force from the definition: per read, rows sorted by (pos, row), every row tested against every other row, runs
built with itertools.groupby and merged by looking at the previous block.  The kind, the clusters and the calls are
restated here as well.  No logic is shared with the device code or with gavisunk_b200.cli.

Inputs: kept rows (read, pos, contig, start, ID) in row order; a read is every row with the same read key (reads in order
of first appearance), its rows on the contig of its first row count; bad = set of (contig, ID); rlen: read -> length."""
import itertools
from collections import defaultdict

import numpy as np

CHAIN, MIN_READS, MIN_IDS = 10000, 3, 3


def strands(rows):
    """rows of ONE read: (ID, start, pos), already ordered -> per row 0 ('+'), 1 ('-') or None.  Every pair is tested in
    an m x m table (the GPU tests' reads carry thousands of rows) with the ratio test 9*ds < 10*dp < 11*ds in exact
    integers (process-by-contig_lowmem_AR.py:145-147, Q12)."""
    if not rows:
        return []
    g, s, p = (np.asarray([r[k] for r in rows], np.int64) for k in range(3))
    ds, dp = np.abs(s[None, :] - s[:, None]), np.abs(p[None, :] - p[:, None])
    ok = (9 * ds < 10 * dp) & (10 * dp < 11 * ds) & (g[None, :] != g[:, None])
    rising = (p[None, :] > p[:, None]) == (s[None, :] > s[:, None])
    up, down = (ok & rising).sum(1), (ok & ~rising).sum(1)
    return [0 if u > d else (1 if d > u else None) for u, d in zip(up.tolist(), down.tolist())]


def read_blocks(rows):
    """rows of ONE read: (ID, start, pos) ordered -> blocks [(strand, [rows])]"""
    st = strands(rows)
    oriented = [(d, r) for d, r in zip(st, rows) if d is not None]
    runs = [(d, [r for _, r in g]) for d, g in itertools.groupby(oriented, key=lambda x: x[0])]
    runs = [(d, g) for d, g in runs if len({r[0] for r in g}) >= MIN_IDS]
    blocks = []
    for d, g in runs:
        if blocks and blocks[-1][0] == d:
            blocks[-1] = (d, blocks[-1][1] + g)
        else:
            blocks.append((d, g))
    return blocks


def switches(rows, rlen, bad=frozenset(), minlen=10000):
    """-> records in (read, block) order: (read, contig, side1, side2), a side = (strand, ids, lo, hi, (ID, start, pos))
    with side1 at B_i's last row and side2 at B_i+1's first row"""
    by_read = defaultdict(list)
    for k, r in enumerate(rows):
        by_read[r[0]].append((k, r))
    out = []
    for rd, rr in by_read.items():
        if rlen.get(rd, 0) < minlen:
            continue
        c0 = rr[0][1][2]
        use = sorted(((r[1], k, (int(r[4]), int(r[3]), int(r[1]))) for k, r in rr if r[2] == c0 and (r[2], r[4]) not in bad))
        blocks = read_blocks([u[2] for u in use])
        side = lambda d, b, row: (d, len({r[0] for r in b}), min(r[1] for r in b), max(r[1] for r in b), row)
        for (d1, b1), (d2, b2) in zip(blocks, blocks[1:]):
            out.append((rd, c0, side(d1, b1, b1[-1]), side(d2, b2, b2[0])))
    return out


def kind(rec):
    _, _, a, b = rec
    return "foldback" if max(a[2], b[2]) <= min(a[3], b[3]) else "inversion"


def _chain(items, key):
    out = []
    for t in sorted(items, key=key):
        if out and key(t) - key(out[-1][-1]) <= CHAIN:
            out[-1].append(t)
        else:
            out.append([t])
    return out


def calls(records, min_reads=MIN_READS):
    """(contig, start, end, reads, switches, spanning), sorted"""
    groups = defaultdict(list)
    for rec in records:
        if kind(rec) == "inversion":
            s1, s2 = rec[2][4][1], rec[3][4][1]
            groups[rec[1]].append((min(s1, s2), max(s1, s2), rec[0]))
    med = lambda v: sorted(v)[(len(v) - 1) // 2]
    out = []
    for c, items in groups.items():
        for ch in _chain(items, lambda t: t[0]):
            for cl in _chain(ch, lambda t: t[1]):
                n = defaultdict(int)
                for t in cl:
                    n[t[2]] += 1
                if len(n) >= min_reads:
                    out.append((c, med([t[0] for t in cl]), med([t[1] for t in cl]), len(n), len(cl), sum(1 for v in n.values() if v >= 2)))
    return sorted(out)


def texts(records, contigs, hap_contigs, read_name, read_len):
    """the two files of one haplotype as str: inversions.reads.tsv, inversions.bed; contigs: [(name, length)];
    read_name(read) / read_len(read): what is written for a read key"""
    names = [n for n, _ in contigs]
    hc = set(hap_contigs)
    sel = [i for i, r in enumerate(records) if r[1] in hc]
    sel.sort(key=lambda i: (read_name(records[i][0]).encode(), i))
    sd = "+-"
    lines = []
    for i in sel:
        rd, c, a, b = records[i]
        cols = [names[c], read_name(rd), read_len(rd)]
        for d, n, lo, hi, (g, s, p) in (a, b):
            cols += [sd[d], n, lo, hi, g, s, p]
        cols += [b[4][2] - a[4][2], kind(records[i])]
        lines.append("\t".join(str(x) for x in cols) + "\n")
    reads = ("contig\tread\tread_len\tstrand1\tids1\tlo1\thi1\tid1\tstart1\tpos1\tstrand2\tids2\tlo2\thi2\tid2\tstart2\tpos2\t"
             "read_gap\tkind\n") + "".join(lines)
    bed = "".join(f"{names[c]}\t{a}\t{b}\tinversion\t{n}\t{k}\t{sp}\n" for c, a, b, n, k, sp in calls([records[i] for i in sel]))
    return reads, bed

"""CPU restatement of the junctions (test infrastructure; no reference counterpart, DESIGN.md section 5.5c).

Brute force from the definition in include/gavisunk_b200.h, from every match row (no screen, no stash): per read, every
row is tested against every other row, runs are built with itertools.groupby and merged by looking at the previous
block, strands count every pair.  The host columns and the clusters are restated here as well.  No logic is shared with
the device code or with gavisunk_b200.cli."""
import itertools

CHAIN = 10000


def _ratio_ok(ds, dp):
    """0.9 < dp/ds < 1.1 in exact integers (process-by-contig_lowmem_AR.py:145-147, Q12)"""
    return 9 * ds < 10 * dp < 11 * ds


def _strand(block):
    up = down = 0
    for x, y in itertools.combinations(block, 2):
        if x[1] == y[1] or not _ratio_ok(abs(x[2] - y[2]), abs(x[3] - y[3])):
            continue
        if (y[3] - x[3]) * (y[2] - x[2]) > 0:
            up += 1
        else:
            down += 1
    return "+" if up >= down else "-"


def read_blocks(rows, bad=frozenset()):
    """rows of ONE read: (contig, ID, start, pos) in row order -> its blocks, lists of rows"""
    rs = [r for r in rows if (r[0], r[1]) not in bad]
    anch = [r for r in rs if any(o[0] == r[0] and o[1] != r[1] and _ratio_ok(abs(o[2] - r[2]), abs(o[3] - r[3])) for o in rs)]
    ids = {}
    for r in anch:
        ids.setdefault(r[0], set()).add(r[1])
    qual = {c for c, s in ids.items() if len(s) >= 3}
    kept = [r for r in anch if r[0] in qual]
    runs = [list(g) for _, g in itertools.groupby(kept, key=lambda r: r[0])]
    runs = [g for g in runs if len({r[1] for r in g}) >= 3]
    blocks = []
    for g in runs:
        if blocks and blocks[-1][0][0] == g[0][0]:
            blocks[-1] = blocks[-1] + g
        else:
            blocks.append(g)
    return blocks


def junctions(rows, rlen, bad=frozenset(), minlen=10000):
    """rows: (read, pos, contig, start, ID) in row order, a read = a run of consecutive rows with one read key; rlen:
    read -> length; bad: set of (contig, ID).  -> records (read, side1, side2) in (read, block) order, a side =
    (contig, strand '+'/'-', distinct IDs, (ID, start, pos))"""
    out = []
    for read, g in itertools.groupby(rows, key=lambda r: r[0]):
        if rlen.get(read, 0) < minlen:
            continue
        blocks = read_blocks([(r[2], int(r[4]), int(r[3]), int(r[1])) for r in g], bad)
        for b1, b2 in zip(blocks, blocks[1:]):
            l, f = b1[-1], b2[0]
            out.append((read, (l[0], _strand(b1), len({r[1] for r in b1}), (l[1], l[2], l[3])),
                        (f[0], _strand(b2), len({r[1] for r in b2}), (f[1], f[2], f[3]))))
    return out


def host_columns(rec, contig_len):
    """(read_gap, leave1, enter2, implied_gap, class) of one record; contig_len: contig -> length"""
    _, (c1, d1, _, (_, s1, p1)), (c2, d2, _, (_, s2, p2)) = rec
    read_gap = p2 - p1
    leave1 = contig_len[c1] - s1 if d1 == "+" else s1
    enter2 = s2 if d2 == "+" else contig_len[c2] - s2
    cls = "link" if leave1 + enter2 <= read_gap + read_gap // 10 + 1000 else "breakpoint"
    return read_gap, leave1, enter2, read_gap - leave1 - enter2, cls


def _chain(items, key):
    """maximal chains of items sorted by key, consecutive keys at most CHAIN apart"""
    out = []
    for t in sorted(items, key=key):
        if out and key(t) - key(out[-1][-1]) <= CHAIN:
            out[-1].append(t)
        else:
            out.append([t])
    return out


def clusters(records, contig_len, contig_hap, order):
    """records of junctions(); contig_hap: contig -> 0 / 1 (missing: neither); order: contig -> rank (fai1-then-fai2).
    -> clusters (contig1, strand1, hap1, start1, contig2, strand2, hap2, start2, records, links, median implied gap,
    class), sorted by (contig1, start1, contig2, start2), then strands"""
    flip = {"+": "-", "-": "+"}
    groups = {}
    for rec in records:
        _, a, b = rec
        gap, cls = host_columns(rec, contig_len)[3:]
        sa, sb = (a[0], a[1], a[3][1]), (b[0], b[1], b[3][1])
        if (order[sb[0]], sb[2]) < (order[sa[0]], sa[2]):
            sa, sb = (sb[0], flip[sb[1]], sb[2]), (sa[0], flip[sa[1]], sa[2])
        groups.setdefault((sa[0], sa[1], sb[0], sb[1]), []).append((sa[2], sb[2], gap, cls))
    med = lambda v: sorted(v)[(len(v) - 1) // 2]
    hap = lambda c: {0: "1", 1: "2"}.get(contig_hap.get(c), ".")
    out = []
    for (c1, d1, c2, d2), items in groups.items():
        for ch in _chain(items, lambda t: t[0]):
            for cl in _chain(ch, lambda t: t[1]):
                links = sum(1 for t in cl if t[3] == "link")
                out.append((c1, d1, hap(c1), med([t[0] for t in cl]), c2, d2, hap(c2), med([t[1] for t in cl]), len(cl), links,
                            med([t[2] for t in cl]), "link" if links * 2 > len(cl) else "breakpoint"))
    out.sort(key=lambda t: (order[t[0]], t[3], order[t[4]], t[7], t[1], t[5]))
    return out


def reads_tsv_lines(records, rlen, contig_len):
    """rows of hap{N}.junctions.reads.tsv (no header): by read name bytewise, then record order"""
    idx = sorted(range(len(records)), key=lambda i: (records[i][0].encode(), i))
    out = []
    for i in idx:
        rec = records[i]
        read, a, b = rec
        cols = [read, rlen[read]]
        for c, d, n, (i_, s, p) in (a, b):
            cols += [c, d, n, i_, s, p]
        out.append("\t".join(str(x) for x in cols + list(host_columns(rec, contig_len))))
    return out


def clusters_tsv_lines(cl):
    return ["\t".join(str(x) for x in t) for t in cl]

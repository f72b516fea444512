"""CPU restatement of the gap evidence (test infrastructure; no reference counterpart, DESIGN.md section 5.5b).

Brute force from the definition: for every gap and every read, the read's rows on the gap's contig are split into
sides by ID, every row is tested against every other row of its side, and the flanks are picked with max() / min()
over explicit keys.  No logic is shared with the device algorithm (no candidate ranges, no packed keys)."""
from collections import OrderedDict


def _ratio_ok(ds, dp):
    """0.9 < dp/ds < 1.1 in exact integers (process-by-contig_lowmem_AR.py:145-147, Q12)"""
    return 9 * ds < 10 * dp < 11 * ds


def _anchored(row, side):
    """row = (ID, start, pos): another row of the side with a different ID passes the ratio test with it"""
    return any(o[0] != row[0] and _ratio_ok(abs(o[1] - row[1]), abs(o[2] - row[2])) for o in side)


def gap_evidence(rows, rlen, bad, gaps, minlen=10000, anchored=True):
    """rows: (read, pos, contig, start, ID); rlen: read -> length; bad: set of (contig, ID); gaps: [(contig, gs, ge)] in
    gaps.bed order.  anchored=False: the bare rule (every row of a side counts, flanks by start alone, then pos).
    -> records (gap index, read, (left ID, start, pos), (right ID, start, pos), delta, consistent), sorted by gap index,
    then read name bytewise"""
    by_read = OrderedDict()
    for r in rows:
        by_read.setdefault(r[0], []).append((r[2], int(r[4]), int(r[3]), int(r[1])))  # (contig, ID, start, pos)
    out = []
    for gi, (c, gs, ge) in enumerate(gaps):
        gs, ge = int(gs), int(ge)
        for read, rs in by_read.items():
            if rlen.get(read, 0) < minlen:
                continue
            mine = [(i, s, p) for cc, i, s, p in rs if cc == c and (cc, i) not in bad]
            left = [x for x in mine if x[0] <= gs]
            right = [x for x in mine if x[0] >= ge + 1]
            if not left or not right:
                continue
            if anchored:
                left = [x for x in left if _anchored(x, left)]
                right = [x for x in right if _anchored(x, right)]
            if not left or not right:
                continue
            lf = max(left, key=lambda x: (x[1], -x[2], -x[0]))
            rf = min(right, key=lambda x: (x[1], x[2], x[0]))
            ds, dp = rf[1] - lf[1], abs(rf[2] - lf[2])
            out.append((gi, read, lf, rf, dp - ds, _ratio_ok(ds, dp)))
    out.sort(key=lambda t: (t[0], t[1].encode() if isinstance(t[1], str) else t[1]))
    return out


def summary(records, gaps):
    """per gap: (contig, gs, ge, bridging reads, consistent reads, min delta, lower median delta, max delta), the three
    deltas None without a bridging read"""
    out = []
    for gi, (c, gs, ge) in enumerate(gaps):
        d = sorted(r[4] for r in records if r[0] == gi)
        n_cons = sum(1 for r in records if r[0] == gi and r[5])
        out.append((c, gs, ge, len(d), n_cons) + ((d[0], d[(len(d) - 1) // 2], d[-1]) if d else (None, None, None)))
    return out


def reads_tsv_lines(records, gaps, rlen):
    """the rows of hap{N}.gaps.reads.tsv (without the header) for records of gap_evidence()"""
    return [f"{gaps[gi][0]}\t{gaps[gi][1]}\t{gaps[gi][2]}\t{read}\t{rlen[read]}\t{lf[0]}\t{lf[1]}\t{lf[2]}\t{rf[0]}\t{rf[1]}\t{rf[2]}\t"
            f"{delta}\t{int(cons)}" for gi, read, lf, rf, delta, cons in records]

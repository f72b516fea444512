"""CPU oracle of the distance discordance (include/gavisunk_b200.h gvs_spans / gvs_discordance; cli.discordance_texts):
the definition restated by brute force, for the GPU tests to compare against.

Inputs: kept rows (read, pos, contig, start, ID) with contig an index into `contigs` = [(name, length)]; bad = set of
(contig, ID); validated = set of (read, ID) (the rows of inter_outs); groups = set of (contig, ID), the group table
behind the ranks.  A read is every row with the same read key, in row order; its rows on the contig of its first row
count."""
from collections import defaultdict

MIN_DELTA, REL_PERMILLE, MIN_READS = 300, 30, 3


def spans(rows, bad, validated, min_delta=MIN_DELTA, rel_permille=REL_PERMILLE):
    """every span of every read, in (read first appearance, span) order: (read, contig, (id, start, pos) of a, of b,
    delta, kind) with kind 'longer', 'shorter' or None"""
    by_read = defaultdict(list)
    for r in rows:
        by_read[r[0]].append(r)
    out = []
    for rd, rr in by_read.items():
        c0 = rr[0][2]
        cand = [r for r in rr if r[2] == c0 and (r[2], r[4]) not in bad and (rd, r[4]) in validated]
        n_id = defaultdict(int)
        for r in cand:
            n_id[r[4]] += 1
        use = sorted((r for r in cand if n_id[r[4]] == 1), key=lambda r: (r[3], r[4]))
        for a, b in zip(use, use[1:]):
            ds = b[3] - a[3]
            delta = abs(b[1] - a[1]) - ds
            bound = 1000 * min_delta + rel_permille * ds
            kind = "longer" if 1000 * delta >= bound else ("shorter" if -1000 * delta >= bound else None)
            out.append((rd, c0, (a[4], a[3], a[1]), (b[4], b[3], b[1]), delta, kind))
    return out


def records(sp):
    return [s for s in sp if s[5] is not None]


def segments(sp, groups, contigs):
    """per contig, its groups in start order as segments [ID_r, ID_r+1 or the contig's end) with the counts of the spans
    that cover them (rank(a) <= r < rank(b)): {contig: [(start, end, spans, longer, shorter)]}"""
    out = {}
    for c, (_, ln) in enumerate(contigs):
        ids = sorted(i for cc, i in groups if cc == c)
        cnt = [[0, 0, 0] for _ in ids]
        at = {i: k for k, i in enumerate(ids)}
        for s in sp:
            if s[1] != c:
                continue
            for r in range(at[s[2][0]], at[s[3][0]]):
                cnt[r][0] += 1
                if s[5] == "longer":
                    cnt[r][1] += 1
                elif s[5] == "shorter":
                    cnt[r][2] += 1
        out[c] = [(i, ids[k + 1] if k + 1 < len(ids) else ln, *cnt[k]) for k, i in enumerate(ids)]
    return out


def runs(sp, groups, contigs):
    """(contig, start, end, spans, longer, shorter) tiling every contig, maximal, contigs in index order"""
    segs = segments(sp, groups, contigs)
    out = []
    for c, (_, ln) in enumerate(contigs):
        cur = []
        pieces = segs[c]
        if not pieces or pieces[0][0] != 0:
            cur.append([c, 0, pieces[0][0] if pieces else ln, 0, 0, 0])
        for a, b, n, lo, sh in pieces:
            if cur and cur[-1][3:] == [n, lo, sh]:
                cur[-1][2] = b
            else:
                cur.append([c, a, b, n, lo, sh])
        out += [tuple(x) for x in cur]
    return out


def calls(recs, rn, min_reads=MIN_READS):
    """(contig, start, end, kind, peak_start, peak_end, spans, supporting, size or None) from the records and the runs"""
    out, cur = [], None

    def close():
        c, kind, a, b, members = cur
        sup = lambda m: m[4] if kind == "collapse" else m[5]
        best = members[0]
        for m in members[1:]:
            if sup(m) > sup(best) or (sup(m) == sup(best) and sup(m) * best[3] > sup(best) * m[3]):
                best = m
        want = "longer" if kind == "collapse" else "shorter"
        d = sorted(r[4] for r in recs if r[1] == c and r[5] == want and r[2][0] <= best[1] < r[3][0])
        out.append((c, a, b, kind, best[1], best[2], best[3], sup(best), d[(len(d) - 1) // 2] if d else None))
    for run in rn:
        c, a, b, n, lo, sh = run
        kind = "collapse" if lo >= min_reads and 2 * lo > n else ("expansion" if sh >= min_reads and 2 * sh > n else None)
        if cur is not None and (kind is None or cur[0] != c or cur[1] != kind or cur[3] != a):
            close()
            cur = None
        if kind is not None:
            if cur is None:
                cur = [c, kind, a, b, [run]]
            else:
                cur[3] = b
                cur[4].append(run)
    if cur is not None:
        close()
    return out


def texts(recs, rn, contigs, hap_contigs, read_name, read_len):
    """the three files of one haplotype (hap_contigs: its contig indices) as str: reads.tsv, tsv, bed.  read_name(read) is
    the name written for a read key, read_len(read) its length."""
    names = [n for n, _ in contigs]
    hc = set(hap_contigs)
    rs = sorted((r for r in recs if r[1] in hc), key=lambda r: (r[1], r[2][1], r[3][1], read_name(r[0]).encode()))
    reads = "contig\tread\tread_len\tid1\tstart1\tpos1\tid2\tstart2\tpos2\tdelta\tkind\n" + "".join(
        f"{names[r[1]]}\t{read_name(r[0])}\t{read_len(r[0])}\t{r[2][0]}\t{r[2][1]}\t{r[2][2]}\t{r[3][0]}\t{r[3][1]}\t{r[3][2]}\t"
        f"{r[4]}\t{r[5]}\n" for r in rs)
    hr = [r for r in rn if r[0] in hc]
    tsv = "contig\tstart\tend\tspans\tlonger\tshorter\n" + "".join(f"{names[c]}\t{a}\t{b}\t{n}\t{lo}\t{sh}\n" for c, a, b, n, lo, sh in hr)
    bed = "".join(f"{names[c]}\t{a}\t{b}\t{k}\t{ps}\t{pe}\t{n}\t{s}\t{'.' if z is None else z}\n"
                  for c, a, b, k, ps, pe, n, s, z in calls(recs, hr))
    return reads, tsv, bed

"""CPU oracle of the SUNK hit depth (include/gavisunk_b200.h gvs_sunk_depth / gvs_depth_runs, cli.depth_calls, DESIGN.md
section 5.5g), restated by brute force from row tuples: per-group counts, runs, size classes and baselines with their
fallback, states, clusters, calls and the three file texts.

Groups are (contig, start) pairs; contigs are ids into a list of (name, length); reads are any hashable record keys."""
from collections import defaultdict

HIGH, LOW, MAX_GAP, MIN_GROUPS, MIN_CLASS = 1750, 250, 2, 5, 100


def counts(match_rows, groups):
    """match_rows: (read, contig, start) of every match row.  -> {group: (hits, reads)} over `groups`"""
    hits = {g: 0 for g in groups}
    seen = {g: set() for g in groups}
    for r, c, s in match_rows:
        hits[(c, s)] += 1
        seen[(c, s)].add(r)
    return {g: (hits[g], len(seen[g])) for g in groups}


def runs(values, contigs):
    """values: {group: tuple of ints}; contigs: [(name, length)] by id.  -> [(contig, start, end, *values)] tiling every
    contig: a zero head run unless its first group starts at 0, then a run wherever the values change"""
    nv = len(next(iter(values.values()))) if values else 3
    out = []
    for c, (_, ln) in enumerate(contigs):
        mine = []
        starts = sorted(s for (cc, s) in values if cc == c)
        if not starts or starts[0] != 0:
            mine.append([0, (0,) * nv])
        for s in starts:
            v = tuple(values[(c, s)])
            if not mine or mine[-1][1] != v:
                mine.append([s, v])
        for i, (s, v) in enumerate(mine):
            out.append((c, s, mine[i + 1][0] if i + 1 < len(mine) else ln) + v)
    return out


def size_class(sunks):
    q = 0
    while q < 5 and sunks >= 2 ** (q + 1):
        q += 1
    return q


def lower_median(v):
    v = sorted(v)
    return v[(len(v) - 1) // 2]


def baselines(hap_groups, hits, sunks, min_class=MIN_CLASS):
    """[(groups, hit groups, baseline or None, fallback)] of classes 0..5 over the haplotype's groups"""
    every = [hits[g] for g in hap_groups if hits[g] >= 1]
    out = []
    for q in range(6):
        mine = [g for g in hap_groups if size_class(sunks[g]) == q]
        hq = [hits[g] for g in mine if hits[g] >= 1]
        fb = len(hq) < min_class
        b = None if not every else (lower_median(every) if fb else lower_median(hq))
        out.append((len(mine), len(hq), b, fb))
    return out


def calls(hap_contigs, contigs, hits, reads, sunks, bad, high=HIGH, low=LOW, max_gap=MAX_GAP, min_groups=MIN_GROUPS,
          min_class=MIN_CLASS):
    """hits / reads / sunks: {group: int} over every group; bad: set of groups; hap_contigs: the haplotype's contig ids in
    .fai order.  -> (calls [(contig, start, end, kind, groups, marked, ratio, copies, tandem or None, bad)], baselines)"""
    hap_groups = [g for g in hits if g[0] in set(hap_contigs)]
    base = baselines(hap_groups, hits, sunks, min_class)
    if base[0][2] is None:
        return [], base
    B = {g: base[size_class(sunks[g])][2] for g in hap_groups}
    state = {}
    for g in hap_groups:
        state[g] = "high" if 1000 * hits[g] >= high * B[g] else ("low" if 1000 * hits[g] <= low * B[g] else None)
    out = []
    for c in hap_contigs:
        gs = sorted(g for g in hap_groups if g[0] == c)
        for st, kind in (("high", "collapse"), ("low", "depleted")):
            clusters, last = [], None
            for i, g in enumerate(gs):
                if state[g] != st:
                    continue
                if last is not None and i - last - 1 <= max_gap:
                    clusters[-1].append(i)
                else:
                    clusters.append([i])
                last = i
            for cl in clusters:
                if len(cl) < min_groups:
                    continue
                m = [gs[i] for i in cl]
                end = gs[cl[-1] + 1][1] if cl[-1] + 1 < len(gs) else contigs[c][1]
                ratio = lower_median([1000 * hits[g] // B[g] for g in m])
                tandem = (1 if 2 * sum(hits[g] for g in m) >= 3 * sum(reads[g] for g in m) else 0) if kind == "collapse" else None
                out.append((c, m[0][1], end, kind, cl[-1] - cl[0] + 1, len(m), ratio, (ratio + 500) // 1000, tandem,
                            sum(1 for g in m if g in bad)))
    pos = {c: i for i, c in enumerate(hap_contigs)}
    out.sort(key=lambda t: (pos[t[0]], t[1], t[2], t[3]))
    return out, base


def texts(hap_contigs, contigs, hits, reads, kept, sunks, bad, **kw):
    """(depth.bedgraph, depth.bed, depth.tsv) strings of one haplotype; kept: {group: int}"""
    rn = runs({g: (hits[g], reads[g], kept[g]) for g in hits}, contigs)
    hc = set(hap_contigs)
    bedgraph = "".join("\t".join([contigs[r[0]][0]] + [str(x) for x in r[1:]]) + "\n" for r in rn if r[0] in hc)
    cl, base = calls(hap_contigs, contigs, hits, reads, sunks, bad, **kw)
    bed = "".join("\t".join([contigs[t[0]][0]] + [str(x) for x in t[1:8]] + ["." if t[8] is None else str(t[8]), str(t[9])]) + "\n"
                  for t in cl)
    tsv = ["class\tmin_sunks\tmax_sunks\tgroups\thit_groups\tbaseline\tfallback\n"]
    for q, (n, nh, b, fb) in enumerate(base):
        tsv.append(f"{q}\t{2 ** q}\t{2 ** (q + 1) - 1 if q < 5 else '.'}\t{n}\t{nh}\t{'.' if b is None else b}\t"
                   f"{'.' if b is None else (1 if fb else 0)}\n")
    return bedgraph, bed, "".join(tsv)


def from_files(loc_rows, detailed_rows, kept_rows, bad_lines, contigs):
    """The oracle's inputs from the per-rule files: loc_rows (contig name, start, kmer, group) of kmer.loc (identical rows
    once), detailed_rows / kept_rows: (name, pos, contig name, start, group) of both haplotypes' files in order (a read =
    a run of consecutive rows with one name, per file: lists of lists), bad_lines: lines of bad_sunks.txt.
    -> (hits, reads, kept, sunks, bad) dicts / set"""
    cidx = {}
    for i, (n, _) in enumerate(contigs):
        cidx.setdefault(n, i)
    sunks = defaultdict(int)
    for c, s, k, g in dict.fromkeys(loc_rows):
        sunks[(cidx[c], g)] += 1
    groups = list(sunks)
    rows = []
    for f, part in enumerate(detailed_rows):
        rid, prev = -1, None
        for name, _, c, _, g in part:
            if name != prev:
                rid += 1
                prev = name
            rows.append(((f, rid), cidx[c], g))
    cnt = counts(rows, groups)
    kept = {g: 0 for g in groups}
    for part in kept_rows:
        for _, _, c, _, g in part:
            kept[(cidx[c], g)] += 1
    bad = set()
    for b in bad_lines:
        c, _, g = b.partition(":")
        if c in cidx and (cidx[c], int(g)) in sunks:
            bad.add((cidx[c], int(g)))
    return {g: cnt[g][0] for g in groups}, {g: cnt[g][1] for g in groups}, kept, dict(sunks), bad

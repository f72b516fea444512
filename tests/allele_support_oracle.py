"""CPU oracle of the allele support (include/gavisunk_b200.h gvs_allele_support / gvs_allele_runs, cli.allele_calls,
DESIGN.md section 5.5h), restated by brute force: per-group (own, other) from distinct (read, group) pairs, runs, calls
straight from the definition and the four file texts.

Groups are (contig, start) pairs; contigs are ids into a list of (name, length); reads are any hashable record keys."""
from sunk_depth_oracle import baselines, lower_median, runs, size_class  # noqa: F401 -- the shared pieces

MIN_READS, FLIP, MIN_BASELINE, MAX_GAP, MIN_SWITCH, MIN_CLASS = 3, 200, 10, 2, 3, 100


def counts(match_rows, read_hap, contig_hap, groups):
    """match_rows: (read, contig, start) of every match row; read_hap: {read: 0 / 1}; contig_hap: haplotype by contig id.
    -> {group: (own, other)} over `groups`"""
    pairs = {(r, (c, s)) for r, c, s in match_rows}
    out = {g: [0, 0] for g in groups}
    for r, g in pairs:
        h = contig_hap[g[0]]
        if h in (0, 1):
            out[g][0 if read_hap[r] == h else 1] += 1
    return {g: tuple(v) for g, v in out.items()}


def calls(hap_contigs, own, other, sunks, end, min_reads=MIN_READS, flip=FLIP, min_baseline=MIN_BASELINE, max_gap=MAX_GAP,
          min_switch=MIN_SWITCH, min_class=MIN_CLASS):
    """own / other / sunks / end: {group: int} over every group; hap_contigs: the haplotype's contig ids in .fai order.
    -> (calls [(contig, start, end, kind, groups, marked, own, other)], per contig (groups, assessed, flipped, flips,
    switches, errors, error_eligible, shared), baselines of own)"""
    hc = set(hap_contigs)
    hap_groups = [g for g in own if g[0] in hc]
    base = baselines(hap_groups, own, sunks, min_class)
    out, per = [], []
    for c in hap_contigs:
        gs = sorted(g for g in hap_groups if g[0] == c)
        t = {g: own[g] + other[g] for g in gs}
        assessed = {g: t[g] >= min_reads for g in gs}
        flipped = {g: other[g] >= min_reads and 1000 * own[g] <= flip * t[g] for g in gs}
        shared = {g: own[g] >= min_reads and other[g] >= min_reads and not flipped[g] for g in gs}
        eligible = {}
        for g in gs:
            b = base[size_class(sunks[g])][2]
            eligible[g] = b is not None and b >= min_baseline
        mine = []
        chain = []
        for i, g in enumerate(gs):
            if not flipped[g]:
                continue
            if chain:
                gap = sum(1 for j in range(chain[-1] + 1, i) if assessed[gs[j]] and not flipped[gs[j]])
                if gap > max_gap:
                    mine.append(chain)
                    chain = []
            chain.append(i)
        if chain:
            mine.append(chain)
        cl = []
        for ch in mine:
            if len(ch) >= min_switch:
                cl.append(("switch", ch))
            else:
                cl += [("flip", [i]) for i in ch]
        for i, g in enumerate(gs):
            if t[g] == 0 and eligible[g] and 0 < i < len(gs) - 1 and assessed[gs[i - 1]] and assessed[gs[i + 1]]:
                cl.append(("error", [i]))
        for kind, ix in cl:
            m = [gs[i] for i in ix]
            out.append((c, m[0][1], end[m[-1]], kind, ix[-1] - ix[0] + 1, len(m), sum(own[g] for g in m), sum(other[g] for g in m)))
        per.append((len(gs), sum(assessed.values()), sum(flipped.values()), sum(1 for k, _ in cl if k == "flip"),
                    sum(1 for k, _ in cl if k == "switch"), sum(1 for k, _ in cl if k == "error"), sum(eligible.values()),
                    sum(shared.values())))
    pos = {c: i for i, c in enumerate(hap_contigs)}
    out.sort(key=lambda x: (pos[x[0]], x[1], x[2], x[3]))
    return out, per, base


def texts(hap_contigs, contigs, own, other, sunks, end, **kw):
    """(alleles.bedgraph, alleles.bed, alleles.tsv, alleles.classes.tsv) strings of one haplotype"""
    rn = runs({g: (own[g], other[g]) for g in own}, contigs)
    hc = set(hap_contigs)
    bedgraph = "".join("\t".join([contigs[r[0]][0]] + [str(x) for x in r[1:]]) + "\n" for r in rn if r[0] in hc)
    cl, per, base = calls(hap_contigs, own, other, sunks, end, **kw)
    bed = "".join("\t".join([contigs[x[0]][0]] + [str(v) for v in x[1:]]) + "\n" for x in cl)
    tsv = ["contig\tgroups\tassessed\tflipped\tflips\tswitches\terrors\terror_eligible\tshared\thamming_ppm\tswitch_ppm\n"]
    total = tuple(sum(v[i] for v in per) for i in range(8))
    for name, v in [(contigs[c][0], v) for c, v in zip(hap_contigs, per)] + [("*", total)]:
        ppm = lambda x: str(1000000 * x // v[1]) if v[1] else "."
        tsv.append("\t".join([name] + [str(x) for x in v] + [ppm(v[2]), ppm(2 * v[4])]) + "\n")
    cls = ["class\tmin_sunks\tmax_sunks\tgroups\town_groups\tbaseline\tfallback\n"]
    for q, (n, nh, b, fb) in enumerate(base):
        cls.append(f"{q}\t{2 ** q}\t{2 ** (q + 1) - 1 if q < 5 else '.'}\t{n}\t{nh}\t{'.' if b is None else b}\t"
                   f"{'.' if b is None else (1 if fb else 0)}\n")
    return bedgraph, bed, "".join(tsv), "".join(cls)


def from_files(loc_rows, detailed_rows, contigs, k):
    """The oracle's inputs from the per-rule files: loc_rows (contig name, start, kmer, group) of kmer.loc (identical rows
    once), detailed_rows: (name, pos, contig name, start, group) of both haplotypes' _detailed.sunkpos in order (a read = a
    run of consecutive rows with one name; the file gives its haplotype).  -> (match rows (read, contig, start), read
    haplotypes, groups, sunks, end) for counts / calls"""
    cidx = {}
    for i, (n, _) in enumerate(contigs):
        cidx.setdefault(n, i)
    sunks, end = {}, {}
    for c, s, _, g in dict.fromkeys(loc_rows):
        key = (cidx[c], g)
        sunks[key] = sunks.get(key, 0) + 1
        end[key] = max(end.get(key, 0), s + k)
    groups = list(sunks)
    rows, read_hap = [], {}
    for f, part in enumerate(detailed_rows):
        rid, prev = -1, None
        for name, _, c, _, g in part:
            if name != prev:
                rid += 1
                prev = name
            read_hap[(f, rid)] = f
            rows.append(((f, rid), cidx[c], g))
    return rows, read_hap, groups, sunks, end

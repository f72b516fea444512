"""SUNK hit depth on the host (cli.depth_calls / cli.depth_texts, DESIGN.md section 5.5g) against the brute-force oracle
(tests/sunk_depth_oracle.py) on hand-made groups and counts.  CPU only: the per-group counts and runs come from the
oracle here; tests/test_gpu_sunk_depth.py checks the device's against it."""
import numpy as np
import pytest

import sunk_depth_oracle as O

from gavisunk_b200 import cli


def _host(groups, hits, reads, sunks, kept=None):
    """engine-like tables of hand-made per-group dicts, in the order of `groups` (the group index)"""
    g = dict(contig=np.asarray([c for c, _ in groups], np.uint32), group=np.asarray([s for _, s in groups], np.uint32))
    kept = kept or {x: 0 for x in groups}
    dp = dict(hits=np.asarray([hits[x] for x in groups], np.int32), reads=np.asarray([reads[x] for x in groups], np.int32),
              sunks=np.asarray([sunks[x] for x in groups], np.uint32), kept=np.asarray([kept[x] for x in groups], np.int32))
    return g, dp


def _calls(groups, hits, reads, sunks, bad, hap_contigs, contigs, **kw):
    g, dp = _host(groups, hits, reads, sunks)
    bidx = [i for i, x in enumerate(groups) if x in bad]
    got, base = cli.depth_calls(g["contig"], g["group"], dp["hits"], dp["reads"], dp["sunks"], bidx, hap_contigs,
                                [l for _, l in contigs], **kw)
    want, wbase = O.calls(hap_contigs, contigs, hits, reads, sunks, bad, **kw)
    assert got == want and base == wbase
    return got, base


def _line(n=120, step=500, hit=10, sunks=20, contig=0):
    """n class-4 groups of one contig, `step` apart from 1000 on, `hit` hits and reads each"""
    groups = [(contig, 1000 + step * i) for i in range(n)]
    return groups, {x: hit for x in groups}, {x: hit for x in groups}, {x: sunks for x in groups}


def test_counts_reentry_two_contigs_and_zero_hit_groups():
    groups = [(0, 100), (0, 200), (0, 300), (1, 50)]
    rows = [("a", 0, 100), ("a", 0, 200), ("a", 0, 100), ("b", 0, 200), ("b", 1, 50), ("c", 1, 50), ("c", 1, 50)]
    cnt = O.counts(rows, groups)
    assert cnt == {(0, 100): (2, 1), (0, 200): (2, 2), (0, 300): (0, 0), (1, 50): (3, 2)}
    rn = O.runs({g: cnt[g] + (0,) for g in groups}, [("c0", 1000), ("c1", 60)])
    assert rn == [(0, 0, 100, 0, 0, 0), (0, 100, 200, 2, 1, 0), (0, 200, 300, 2, 2, 0), (0, 300, 1000, 0, 0, 0),
                  (1, 0, 50, 0, 0, 0), (1, 50, 60, 3, 2, 0)]


def test_class_fallback_below_100_groups():
    groups, hits, reads, sunks = _line(150, hit=10)
    small = [(0, 200000 + 500 * i) for i in range(99)]
    for i, x in enumerate(small):  # class 1 (2-3 SUNKs): 99 groups with a hit, one short of a baseline of its own
        groups.append(x)
        hits[x] = reads[x] = 4 + i % 2
        sunks[x] = 2 + i % 2
    _, base = _calls(groups, hits, reads, sunks, set(), [0], [("c0", 300000)])
    assert base[4] == (150, 150, 10, False)
    assert base[1] == (99, 99, 10, True)  # lower median of all 249 hit groups
    x = (0, 260000)
    groups.append(x)
    hits[x], reads[x], sunks[x] = 6, 6, 3
    _, base = _calls(groups, hits, reads, sunks, set(), [0], [("c0", 300000)])
    assert base[1] == (100, 100, 4, False)  # 100 groups: the class's own lower median (50 x 4, 49 x 5, 1 x 6 hits)


def test_gap_of_two_chains_gap_of_three_splits_and_five_marked_make_a_call():
    groups, hits, reads, sunks = _line()
    for i in (10, 11, 12, 15, 16):  # two groups between 12 and 15: one cluster of 5
        hits[groups[i]] = 20
    for i in (40, 41, 42, 46, 47):  # three between 42 and 46: clusters of 3 and 2
        hits[groups[i]] = 20
    for i in (70, 71, 72, 73):  # 4 marked
        hits[groups[i]] = 18
    for i in (90, 91, 92, 93, 94):  # 5 marked, the last group of the call followed by group 95
        hits[groups[i]] = 35
    got, _ = _calls(groups, hits, reads, sunks, {groups[11], groups[93]}, [0], [("c0", 100000)])
    assert [(t[1], t[2], t[4], t[5]) for t in got] == [(groups[10][1], groups[17][1], 7, 5), (groups[90][1], groups[95][1], 5, 5)]
    assert [(t[3], t[6], t[7], t[8], t[9]) for t in got] == [("collapse", 2000, 2, 1, 1), ("collapse", 3500, 4, 1, 1)]


def test_interleaved_high_and_low_clusters_and_contig_end():
    groups, hits, reads, sunks = _line()
    for i in range(60, 70):
        hits[groups[i]] = 20 if i % 2 == 0 else 2
    for i in range(113, 120):  # depleted up to the contig's end
        hits[groups[i]] = 0
    got, _ = _calls(groups, hits, reads, sunks, set(), [0], [("c0", 61000)])
    assert [(t[1], t[2], t[3], t[4], t[5], t[6], t[7], t[8]) for t in got] == [
        (groups[60][1], groups[69][1], "collapse", 9, 5, 2000, 2, 1),
        (groups[61][1], groups[70][1], "depleted", 9, 5, 200, 0, None),
        (groups[113][1], 61000, "depleted", 7, 7, 0, 0, None)]


def test_haplotype_without_hits_has_no_states():
    groups, hits, reads, sunks = _line(20, hit=0)
    g2, h2, r2, s2 = _line(130, hit=12, contig=1)
    groups += g2
    hits.update(h2), reads.update(r2), sunks.update(s2)
    contigs = [("a", 20000), ("b", 80000)]
    got, base = _calls(groups, hits, reads, sunks, set(), [0], contigs)
    assert got == [] and all(b[2] is None for b in base) and base[4][0] == 20
    g, dp = _host(groups, hits, reads, sunks)
    rn = O.runs({x: (hits[x], reads[x], 0) for x in groups}, contigs)
    runs = {c: np.asarray([r[i] for r in rn], np.uint32) for i, c in enumerate(("contig", "start", "end", "hits", "reads", "kept"))}
    bg, bed, tsv = cli.depth_texts([0], [n for n, _ in contigs], [l for _, l in contigs], g, dp, runs, [])
    assert bed == b"" and tsv.decode().splitlines()[5] == "4\t16\t31\t20\t0\t.\t."
    assert bg.decode().splitlines() == ["a\t0\t20000\t0\t0\t0"]


@pytest.mark.parametrize("extra", [0, 1])
def test_tandem_at_its_boundary(extra):
    groups, hits, reads, sunks = _line()
    for i in range(30, 35):  # 2 * 5 * 30 = 300 >= 3 * (100 - extra)
        hits[groups[i]] = 30
        reads[groups[i]] = 20
    reads[groups[30]] += extra
    got, _ = _calls(groups, hits, reads, sunks, set(), [0], [("c0", 100000)])
    assert [(t[3], t[7], t[8]) for t in got] == [("collapse", 3, 1 - extra)]


@pytest.mark.parametrize("seed", range(6))
def test_files_equal_oracle_on_random_tables(seed):
    """two haplotypes of random groups: zero-hit groups, every size class, runs of raised and lowered hits, bad groups,
    and the thresholds as keyword arguments"""
    rng = np.random.default_rng(seed)
    contigs = [("h1a", 400000), ("h1b", 90000), ("h2a", 300000), ("h2b", 5000)]
    groups = []
    for c, (_, ln) in enumerate(contigs):
        st = np.unique(rng.integers(0, ln, int(ln // 900)))
        if seed % 2 and c == 0:
            st[0] = 0
        groups += [(c, int(s)) for s in st]
    rng.shuffle(groups)
    groups = [tuple(int(v) for v in x) for x in groups]
    sunks = {x: int(rng.choice([1, 2, 3, 5, 9, 20, 20, 20, 40, 70])) for x in groups}
    lam = {x: 12 * (0.54 if sunks[x] == 1 else 0.95) for x in groups}
    for c in range(len(contigs)):
        mine = sorted(x for x in groups if x[0] == c)
        for _ in range(3):
            a = int(rng.integers(0, max(1, len(mine) - 12)))
            f = float(rng.choice([0.0, 0.1, 2.0, 3.0]))
            for x in mine[a:a + int(rng.integers(3, 12))]:
                lam[x] *= f
    hits = {x: int(rng.poisson(lam[x])) for x in groups}
    reads = {x: int(rng.binomial(hits[x], 0.7)) if hits[x] else 0 for x in groups}
    kept = {x: int(rng.binomial(hits[x], 0.8)) for x in groups}
    bad = {x for x in groups if rng.random() < 0.2}
    kw = dict(high=1700, low=300, max_gap=1, min_groups=4, min_class=40) if seed >= 4 else {}
    ckw = dict(high_permille=kw["high"], low_permille=kw["low"], max_gap_groups=kw["max_gap"], min_groups=kw["min_groups"],
               min_class_groups=kw["min_class"]) if kw else {}
    g, dp = _host(groups, hits, reads, sunks, kept)
    rn = O.runs({x: (hits[x], reads[x], kept[x]) for x in groups}, contigs)
    runs = {c: np.asarray([r[i] for r in rn], np.uint32) for i, c in enumerate(("contig", "start", "end", "hits", "reads", "kept"))}
    bidx = [i for i, x in enumerate(groups) if x in bad]
    n_calls = 0
    for hap_contigs in ([0, 1], [2, 3]):
        if kw:
            got_calls, _ = cli.depth_calls(g["contig"], g["group"], dp["hits"], dp["reads"], dp["sunks"], bidx, hap_contigs,
                                           [l for _, l in contigs], **ckw)
            assert got_calls == O.calls(hap_contigs, contigs, hits, reads, sunks, bad, **kw)[0]
            n_calls += len(got_calls)
            continue
        got = cli.depth_texts(hap_contigs, [n for n, _ in contigs], [l for _, l in contigs], g, dp, runs, bidx)
        want = O.texts(hap_contigs, contigs, hits, reads, kept, sunks, bad)
        assert [t.decode() for t in got] == list(want)
        n_calls += len(want[1].splitlines())
    assert n_calls > 0

"""The gap-evidence oracle (tests/gap_evidence_oracle.py) on hand-made cases pinned to explicit records, and on the
reference-made rows of the bundled hg02723 sample, where the README's gap has no bridging read.  CPU only."""
from conftest import load_golden
from gavisunk_b200 import io as gio

import gap_evidence_oracle as O

GAP = [("a", 1000, 1999)]  # left: ID <= 1000, right: ID >= 2000
LONG = 20000


def _rows(read, triples, contig="a"):
    """(ID, start, pos) triples -> sunkpos rows (read, pos, contig, start, ID)"""
    return [(read, p, contig, s, i) for i, s, p in triples]


# a forward read that agrees with the assembly: two anchored rows on each side
BASE = [(500, 500, 100), (1000, 1000, 600), (2000, 2000, 1600), (2500, 2500, 2100)]


def _one(rows, gaps=GAP, bad=(), rlen=None, minlen=10000):
    rl = rlen or {r[0]: LONG for r in rows}
    return O.gap_evidence(rows, rl, set(bad), gaps, minlen)


def test_plain_read():
    assert _one(_rows("r", BASE)) == [(0, "r", (1000, 1000, 600), (2000, 2000, 1600), 0, True)]


def test_bad_flank_is_skipped():
    rows = _rows("r", [(400, 400, 0), (700, 700, 300), (1000, 1000, 600)] + BASE[2:])
    assert _one(rows)[0][2] == (1000, 1000, 600)
    assert _one(rows, bad=[("a", 1000)]) == [(0, "r", (700, 700, 300), (2000, 2000, 1600), 0, True)]


def test_short_read_is_ignored():
    rows = _rows("r", BASE)
    assert _one(rows, rlen={"r": 9999}) == []
    assert len(_one(rows, rlen={"r": 10000})) == 1


def test_two_hits_of_the_flank_sunk_take_the_smallest_pos():
    rows = _rows("r", [(500, 500, 100), (1000, 1000, 640), (1000, 1000, 600)] + BASE[2:])
    assert _one(rows) == [(0, "r", (1000, 1000, 600), (2000, 2000, 1600), 0, True)]
    right = _rows("r", BASE[:2] + [(2000, 2000, 1640), (2000, 2000, 1600), (2500, 2500, 2100)])
    assert _one(right)[0][3] == (2000, 2000, 1600)


def test_anchored_on_one_side_only_does_not_bridge():
    # two left rows that fail the ratio test with each other: neither is anchored
    rows = _rows("r", [(500, 500, 100), (1000, 1000, 9000)] + BASE[2:])
    assert _one(rows) == []


def test_single_stray_row_does_not_bridge():
    rows = _rows("r", [(30, 30, 40000)] + BASE[2:])
    assert _one(rows) == []
    assert O.gap_evidence(rows, {"r": LONG}, set(), GAP, anchored=False) == [(0, "r", (30, 30, 40000), (2000, 2000, 1600), 36430, False)]


def test_stray_row_nearer_the_gap_is_passed_over():
    rows = _rows("r", [(500, 500, 100), (800, 800, 400), (1000, 1000, 50000)] + BASE[2:])
    assert _one(rows) == [(0, "r", (800, 800, 400), (2000, 2000, 1600), 0, True)]


def test_read_spanning_two_gaps_gives_two_records():
    gaps = [("a", 1000, 1999), ("a", 3000, 3999)]
    rows = _rows("r", BASE + [(4000, 4000, 3600), (4500, 4500, 4100)])
    assert _one(rows, gaps=gaps) == [(0, "r", (1000, 1000, 600), (2000, 2000, 1600), 0, True),
                                     (1, "r", (2500, 2500, 2100), (4000, 4000, 3600), 0, True)]


def test_side_is_decided_by_id_not_start():
    rows = _rows("r", [(500, 500, 100), (1000, 1010, 610)] + BASE[2:])
    assert _one(rows) == [(0, "r", (1000, 1010, 610), (2000, 2000, 1600), 0, True)]


def test_reverse_strand_twin_has_the_same_delta():
    ins = [(500, 500, 100), (1000, 1000, 600), (2000, 2000, 2100), (2500, 2500, 2600)]  # 500 bases the assembly lacks
    fwd = _one(_rows("f", ins))
    rev = _one(_rows("v", [(i, s, 30000 - p) for i, s, p in ins]))
    assert fwd == [(0, "f", (1000, 1000, 600), (2000, 2000, 2100), 500, False)]
    assert rev == [(0, "v", (1000, 1000, 29400), (2000, 2000, 27900), 500, False)]


def test_lower_median_of_an_even_count():
    rows = []
    for name, shift in (("r1", 0), ("r2", 100), ("r3", 200), ("r4", 300)):
        rows += _rows(name, BASE[:2] + [(i, s, p + shift) for i, s, p in BASE[2:]])
    recs = _one(rows)
    assert [r[1] for r in recs] == ["r1", "r2", "r3", "r4"]
    assert O.summary(recs, GAP) == [("a", 1000, 1999, 4, 1, 0, 100, 300)]


def test_consistent_flips_at_the_ratio_boundaries():
    """flanks 1000 apart on the assembly: consistent iff 900 < dp < 1100"""
    got = {}
    for dp in (900, 901, 1099, 1100):
        rows = _rows("r", BASE[:2] + [(2000, 2000, 600 + dp), (2500, 2500, 1100 + dp)])
        (rec,) = _one(rows)
        got[dp] = (rec[4], rec[5])
    assert got == {900: (-100, False), 901: (-99, True), 1099: (99, True), 1100: (100, False)}


def test_readme_gap_of_the_bundled_sample_has_no_bridging_read():
    """the reference-made rows of AMY_h1 (hg02723 sample): no read validly reaches both sides of the README's gap.  The
    bare rule would report four reads, each through a single stray hit hundreds of kb away: anchoring is what keeps
    them out."""
    case = load_golden("j1_amy_hg02723")
    rows = gio.parse_sunkpos(case["breaks"]["AMY_h1_hap1.sunkpos"])
    rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in case["hap"]["1"]["rlen"].splitlines()}
    bad = {(b.split(":")[0], int(b.split(":")[1])) for b in case["bad_sunks"]}
    gaps = [(p[0], int(p[1]), int(p[2])) for p in (l.split("\t") for l in case["final_out"]["hap1.gaps.bed"].splitlines())]
    assert ("AMY_h1", 284861, 324275) in gaps
    gi = gaps.index(("AMY_h1", 284861, 324275))
    for minlen in (10000, 0):
        assert [r for r in O.gap_evidence(rows, rlen, bad, gaps, minlen) if r[0] == gi] == []
    bare = [r for r in O.gap_evidence(rows, rlen, bad, gaps, anchored=False) if r[0] == gi]
    assert [r[1] for r in bare] == ["h1r000020", "h1r000114", "h1r000357", "h1r000486"]
    for r in bare:
        left = [x for x in rows if x[0] == r[1] and x[2] == "AMY_h1" and ("AMY_h1", x[4]) not in bad and x[4] <= 284861]
        assert len(left) == 1
        assert -347386 <= r[4] <= -39468 and not r[5]

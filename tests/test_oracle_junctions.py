"""The junctions oracle (tests/junctions_oracle.py) pinned to explicit answers on hand-made reads: every rule of the
definition in include/gavisunk_b200.h, the host columns and the clustering.  CPU only."""
import junctions_oracle as O

ORDER = {"A": 0, "B": 1, "C": 2}
HAP = {"A": 0, "B": 0, "C": 1}
LEN = {"A": 100000, "B": 100000, "C": 100000}


def run(contig, ids, pos0, strand="+", step=1000):
    """rows (contig, ID, start, pos) of one colinear run: start = ID, pos rising by `step` per row; strand '-': the IDs
    are taken in falling order"""
    ids = list(ids) if strand == "+" else sorted(ids, reverse=True)
    return [(contig, i, i, pos0 + k * step) for k, i in enumerate(ids)]


def read(name, *runs):
    """(read, pos, contig, start, ID) rows of one read from runs of (contig, ID, start, pos)"""
    return [(name, p, c, s, i) for r in runs for c, i, s, p in r]


def test_a_b_a_gives_two_records():
    rows = read("r1", run("A", [1000, 2000, 3000], 0), run("B", [10000, 11000, 12000], 5000), run("A", [20000, 21000, 22000], 10000))
    got = O.junctions(rows, {"r1": 20000})
    assert got == [("r1", ("A", "+", 3, (3000, 3000, 2000)), ("B", "+", 3, (10000, 10000, 5000))),
                   ("r1", ("B", "+", 3, (12000, 12000, 7000)), ("A", "+", 3, (20000, 20000, 10000)))]


def test_one_contig_gives_nothing():
    rows = read("r1", run("A", [1000, 2000, 3000], 0), run("A", [50000, 51000, 52000], 10000))
    assert O.junctions(rows, {"r1": 20000}) == []


def test_short_run_dropped_and_neighbours_merged():
    """A1, B1 (2 IDs: dropped), A2, B2: the A runs merge into one block of 6 IDs, one record A -> B2"""
    rows = read("r1", run("A", [1000, 2000, 3000], 0), run("B", [10000, 11000], 3000), run("A", [4000, 5000, 6000], 5000),
                run("B", [20000, 21000, 22000], 9000))
    assert O.junctions(rows, {"r1": 20000}) == [("r1", ("A", "+", 6, (6000, 6000, 7000)), ("B", "+", 3, (20000, 20000, 9000)))]
    blocks = O.read_blocks([(r[2], r[4], r[3], r[1]) for r in rows])
    assert [len(b) for b in blocks] == [6, 3]


def test_bad_group_removes_the_third_id():
    rows = read("r1", run("A", [1000, 2000, 3000], 0), run("B", [10000, 11000, 12000], 5000))
    assert len(O.junctions(rows, {"r1": 20000})) == 1
    assert O.junctions(rows, {"r1": 20000}, bad={("B", 12000)}) == []
    # a bad group elsewhere changes nothing
    assert len(O.junctions(rows, {"r1": 20000}, bad={("C", 12000)})) == 1


def test_anchoring_needs_a_ratio_partner():
    """B's third ID sits far off the diagonal of the other two: it is not anchored, B does not qualify"""
    rows = read("r1", run("A", [1000, 2000, 3000], 0), run("B", [10000, 11000], 5000), [("B", 30000, 30000, 7000)])
    assert O.junctions(rows, {"r1": 20000}) == []


def test_min_read_len_is_inclusive():
    rows = read("r1", run("A", [1000, 2000, 3000], 0), run("B", [10000, 11000, 12000], 5000))
    assert len(O.junctions(rows, {"r1": 10000}, minlen=10000)) == 1
    assert O.junctions(rows, {"r1": 9999}, minlen=10000) == []


def test_strand_tie_is_plus_and_minus_strand():
    """block A: one rising pair (1000, 2000) and one falling pair (3000, 4000), no other pair passes -> '+'; block B
    runs with falling starts -> '-'"""
    a = [("A", 1000, 1000, 5000), ("A", 2000, 2000, 6000), ("A", 3000, 3000, 10000), ("A", 4000, 4000, 9000)]
    rows = read("r1", a, run("B", [10000, 11000, 12000], 20000, strand="-"))
    got = O.junctions(rows, {"r1": 30000})
    assert got == [("r1", ("A", "+", 4, (4000, 4000, 9000)), ("B", "-", 3, (12000, 12000, 20000)))]


def test_host_columns_and_link_rule_both_sides():
    """A '+' leaves through its end (len - start1), B '+' is entered through its start (start2); read_gap 10000 allows
    leave1 + enter2 <= 10000 + 1000 + 1000"""
    def rec(start1, start2, d1="+", d2="+"):
        return ("r", ("A", d1, 3, (start1, start1, 1000)), ("B", d2, 3, (start2, start2, 11000)))
    assert O.host_columns(rec(95000, 7000), LEN) == (10000, 5000, 7000, -2000, "link")
    assert O.host_columns(rec(95000, 7001), LEN) == (10000, 5000, 7001, -2001, "breakpoint")
    # '-' sides: leave1 = start1, enter2 = len2 - start2
    assert O.host_columns(rec(4000, 92000, "-", "-"), LEN) == (10000, 4000, 8000, -2000, "link")
    assert O.host_columns(rec(4000, 91999, "-", "-"), LEN)[4] == "breakpoint"


def _rec(read, c1, s1, c2, s2, d1="+", d2="+", p1=1000, p2=2000):
    return (read, (c1, d1, 3, (s1, s1, p1)), (c2, d2, 3, (s2, s2, p2)))


def test_canonical_swap_and_flip():
    """B+ -> A+ is A- -> B- read the other way; it joins A- -> B- records, not A+ -> B+ ones"""
    recs = [_rec("r1", "B", 5000, "A", 90000), _rec("r2", "A", 90500, "B", 5200, "-", "-"), _rec("r3", "A", 90000, "B", 5000)]
    cl = O.clusters(recs, LEN, HAP, ORDER)
    assert [(t[0], t[1], t[4], t[5], t[8]) for t in cl] == [("A", "+", "B", "+", 1), ("A", "-", "B", "-", 2)]
    assert cl[1][3] == 90000 and cl[1][7] == 5000  # lower medians of (90000, 90500) and (5000, 5200)


def test_chaining_at_10000_and_10001():
    recs = [_rec("r1", "A", 10000, "B", 5000), _rec("r2", "A", 20000, "B", 5000), _rec("r3", "A", 30001, "B", 5000)]
    cl = O.clusters(recs, LEN, HAP, ORDER)
    assert [(t[3], t[8]) for t in cl] == [(10000, 2), (30001, 1)]
    # the second chaining pass on start2
    recs = [_rec("r1", "A", 10000, "B", 5000), _rec("r2", "A", 10000, "B", 15000), _rec("r3", "A", 10000, "B", 25001)]
    cl = O.clusters(recs, LEN, HAP, ORDER)
    assert [(t[7], t[8]) for t in cl] == [(5000, 2), (25001, 1)]


def test_cluster_class_haplotypes_and_median_gap():
    """link records: A+ near its end -> C+ near its start (C is hap 2); the cluster is a link only with a strict
    majority of link records"""
    link = lambda r, s2: _rec(r, "A", 99000, "C", s2, p1=0, p2=5000)
    brk = lambda r: _rec(r, "A", 99000, "C", 9000, p1=0, p2=5000)
    cl = O.clusters([link("r1", 1000), link("r2", 2000), brk("r3")], LEN, HAP, ORDER)
    assert len(cl) == 1
    c = cl[0]
    assert (c[2], c[6], c[8], c[9], c[11]) == ("1", "2", 3, 2, "link")
    assert c[10] == 5000 - 1000 - 2000  # lower median of the implied gaps 3000, 2000, -5000
    cl = O.clusters([link("r1", 1000), brk("r3")], LEN, HAP, ORDER)
    assert cl[0][11] == "breakpoint" and cl[0][9] == 1
    assert O.clusters([_rec("r", "A", 1000, "X", 2000)], {**LEN, "X": 5000}, HAP, {**ORDER, "X": 3})[0][6] == "."


def test_reads_tsv_order_and_columns():
    recs = [_rec("r2", "A", 95000, "B", 7000, p1=1000, p2=11000), _rec("r10", "A", 95000, "B", 7001, p1=1000, p2=11000)]
    lines = O.reads_tsv_lines(recs, {"r2": 20000, "r10": 30000}, LEN)
    assert lines == ["r10\t30000\tA\t+\t3\t95000\t95000\t1000\tB\t+\t3\t7001\t7001\t11000\t10000\t5000\t7001\t-2001\tbreakpoint",
                     "r2\t20000\tA\t+\t3\t95000\t95000\t1000\tB\t+\t3\t7000\t7000\t11000\t10000\t5000\t7000\t-2000\tlink"]

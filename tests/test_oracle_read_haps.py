"""The read-haplotype oracle (tests/read_haps_oracle.py) pinned to explicit answers on hand-made chunks, and the host
formatting of the two files of `fused --read-haplotypes` (gavisunk_b200.cli.read_hap_texts).  CPU only."""
import numpy as np

import read_haps_oracle as O

HAP = [{"A", "B", "h1tg000000l", "h1tg000001l"}, {"C", "D"}]


def run(read, contig, ids, pos0=0, step=3000, strand="+"):
    """(read, pos, contig, start, group) rows of one colinear run: group = start = the ID, pos rising by `step` (as the
    IDs of ids(): only the diagonal of the read's strand holds more than one row in band); strand '-': IDs taken in
    falling order"""
    ids = list(ids) if strand == "+" else sorted(ids, reverse=True)
    return [(read, pos0 + k * step, contig, i, i) for k, i in enumerate(ids)]


def ids(n, first=100000, step=3000):
    return [first + k * step for k in range(n)]


def test_votes_on_both_haplotypes():
    rows = run("r1", "A", ids(5)) + run("r1", "C", ids(3, 500000), 5000, strand="-")
    got = O.read_haps([(O.ANY, rows)], HAP)
    assert got["records"] == [("r1", ("A", 5, "+"), ("C", 3, "-"), 0)]
    assert got["kept"] == [r for r in rows if r[2] == "A"]
    # binned to hap 2 (mis-binned): the rows stay on C, the hap-1 vote is only reported
    got = O.read_haps([(1, rows)], HAP)
    assert got["records"] == [("r1", ("A", 5, "+"), ("C", 3, "-"), 0)]
    assert got["kept"] == [r for r in rows if r[2] == "C"]


def test_equal_votes_are_a_tie():
    rows = run("r1", "B", ids(4)) + run("r1", "D", ids(4, 700000), 4000)
    got = O.read_haps([(O.ANY, rows)], HAP)
    assert got["records"] == [("r1", ("B", 4, "+"), ("D", 4, "+"), "tie")]
    assert got["kept"] == []  # an unbinned tie keeps nothing
    assert O.read_haps([(0, rows)], HAP)["kept"] == [r for r in rows if r[2] == "B"]
    assert O.file_haps(["r0", "r1", "r2"], [O.ANY] * 3, got["assigned"]) == [0, 1, 0]  # placed by parity


def test_one_group_is_no_vote():
    """two rows of one group on C: good = 1, no hap-2 vote (maxgood > 1 is needed); a read with only that has no record"""
    one = [("r1", 0, "C", 500000, 500000), ("r1", 10, "C", 500000, 500000)]
    got = O.read_haps([(O.ANY, run("r1", "A", ids(3)) + [(r, p + 9000, c, s, g) for r, p, c, s, g in one])], HAP)
    assert got["records"] == [("r1", ("A", 3, "+"), None, 0)]
    got = O.read_haps([(O.ANY, one)], HAP)
    assert got["records"] == [] and got["assigned"] == {"r1": None}
    assert O.file_haps(["r0", "r1"], [O.ANY, O.ANY], got["assigned"]) == [0, 1]


X, Y = "h1tg000000l", "h1tg000001l"  # Nim hash slots 29 < 36 at capacity 64, 93 > 36 at capacity 128


def _tie_read(name):
    """a read whose hap-1 optimum is shared by X and Y (3 groups, 3 rows each), plus a hap-2 vote of 2 groups on C"""
    return run(name, "C", ids(2, 900000)) + run(name, X, ids(3)) + run(name, Y, ids(3, 300000), 3000)


def test_tie_replays_the_table_with_both_haplotypes_contigs():
    """The tie between X and Y on hap 1 is decided by Table slot order, which the hap-2 contigs share: 43 distinct
    contigs in the first read keep capacity 64 (X first), a 44th -- a hap-2 contig -- grows it to 128 for the rest of
    the chunk (Y first)"""
    def filler(n_hap1, n_hap2):
        rows = run("r0", "A", ids(3))
        rows += [("r0", 50000 + k, f"f1_{k}", 0, 0) for k in range(n_hap1)]
        rows += [("r0", 90000 + k, f"f2_{k}", 0, 0) for k in range(n_hap2)]
        return rows
    hap = [HAP[0] | {f"f1_{k}" for k in range(10)}, HAP[1] | {f"f2_{k}" for k in range(34)}]
    small = O.read_haps([(O.ANY, filler(10, 32) + _tie_read("r1"))], hap)["records"]  # 43 distinct contigs in r0
    big = O.read_haps([(O.ANY, filler(10, 33) + _tie_read("r1"))], hap)["records"]    # 44: the table grows
    assert small[-1] == ("r1", (X, 3, "+"), ("C", 2, "+"), 0)
    assert big[-1] == ("r1", (Y, 3, "+"), ("C", 2, "+"), 0)
    # each chunk starts over at capacity 64
    again = O.read_haps([(O.ANY, filler(10, 33)), (O.ANY, _tie_read("r1"))], hap)["records"]
    assert again[-1] == ("r1", (X, 3, "+"), ("C", 2, "+"), 0)


def test_host_files():
    from gavisunk_b200 import cli, io as gio
    names = ["A", "B", "C", "D"]
    contig_hap = np.array([0, 0, 1, 1], np.uint8)
    N = 0xFFFFFFFF
    rh = {"read": np.array([0, 1, 3], np.uint32), "contig1": np.array([0, 1, N], np.uint32), "n1": np.array([5, 4, 0], np.uint32),
          "strand1": np.array([0, 0, 0], np.uint32), "contig2": np.array([2, 3, 2], np.uint32), "n2": np.array([3, 4, 2], np.uint32),
          "strand2": np.array([1, 0, 0], np.uint32), "hap": np.array([0, 2, 1], np.uint32)}
    read_bin = np.array([2, 2, 2, 0], np.uint8)
    read_hap = cli.file_haps(read_bin, rh)
    assert read_hap.tolist() == [0, 1, 0, 0]  # assigned, tie -> odd index, no vote -> even index, binned
    rtab = gio.NameTable(["rb", "rc", "rd", "ra"])
    lens = np.array([20000, 30000, 15000, 12000], np.uint32)
    rank = cli.bytewise_rank(rtab)
    reads1, contigs1 = cli.read_hap_texts(0, names, contig_hap, rh, read_bin, read_hap, rtab, lens, rank)
    assert reads1.decode() == (cli.READ_HAP_READS_HEADER + "ra\t12000\thap1\t.\t0\t.\tC\t2\t+\thap2\n"
                               "rb\t20000\tunbinned\tA\t5\t+\tC\t3\t-\thap1\n")
    assert contigs1.decode() == ("contig\treads\tassigned_hap1\tassigned_hap2\ttie\tno_vote_reads\tno_vote_bases\n"
                                 "A\t1\t1\t0\t0\t.\t.\nB\t1\t0\t0\t1\t.\t.\ntotal\t2\t1\t0\t1\t1\t15000\n")
    reads2, contigs2 = cli.read_hap_texts(1, names, contig_hap, rh, read_bin, read_hap, rtab, lens, rank)
    assert reads2.decode() == cli.READ_HAP_READS_HEADER + "rc\t30000\tunbinned\tB\t4\t+\tD\t4\t+\ttie\n"
    assert contigs2.decode() == ("contig\treads\tassigned_hap2\tassigned_hap1\ttie\tno_vote_reads\tno_vote_bases\n"
                                 "C\t2\t1\t1\t0\t.\t.\nD\t1\t0\t0\t1\t.\t.\ntotal\t3\t1\t1\t1\t0\t0\n")

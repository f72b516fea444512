"""Strand switches and inversion calls (include/gavisunk_b200.h gvs_strand_switches, cli.inversion_texts): the CPU
oracle (tests/inversions_oracle.py) on hand-made reads, the host files against it, and why the feature is needed: the
validation joins the flanks of an inversion.  No GPU needed."""
import numpy as np

import gavisunk_oracle as G
import inversions_oracle as O

STEP = 500


def read_across(segs, read="r", contig=0, step=STEP, pos0=0):
    """kept rows (read, pos, contig, start, ID) of one read made of assembly pieces [(lo, hi, strand)] in read order, one
    SUNK group every `step` bases (ID = start)"""
    rows, p = [], pos0
    for lo, hi, d in segs:
        ss = list(range(lo, hi, step)) if d == 0 else list(range(hi - step, lo - step, -step))
        rows += [(read, p + k * step, contig, s, s) for k, s in enumerate(ss)]
        p += hi - lo
    return rows


def sides(recs):
    """(strand1, start1, strand2, start2) of every record"""
    return [(a[0], a[4][1], b[0], b[4][1]) for _, _, a, b in recs]


RLEN = {"r": 50000}


def test_read_spanning_an_inversion_names_both_ends():
    recs = O.switches(read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)]), RLEN)
    assert sides(recs) == [(0, 19500, 1, 29500), (1, 20000, 0, 30000)]
    assert [O.kind(r) for r in recs] == ["inversion", "inversion"]
    assert [(r[2][1:4], r[3][1:4]) for r in recs] == [((20, 10000, 19500), (18, 20000, 29500)), ((18, 20000, 29500), (30, 30000, 44500))]


def test_read_across_one_breakpoint_of_a_long_inversion():
    recs = O.switches(read_across([(10000, 20000, 0), (200000, 230000, 1)]), RLEN)
    assert sides(recs) == [(0, 19500, 1, 229500)] and O.kind(recs[0]) == "inversion"


def test_foldback_read():
    recs = O.switches(read_across([(10000, 30000, 0), (15000, 30000, 1)]), RLEN)
    assert len(recs) == 1 and O.kind(recs[0]) == "foldback"
    assert recs[0][2][2:4] == (10000, 29500) and recs[0][3][2:4] == (15000, 29000)


def test_plain_read_has_no_record():
    assert O.switches(read_across([(10000, 45000, 0)]), RLEN) == []
    assert O.switches(read_across([(10000, 45000, 1)]), RLEN) == []


def test_short_run_is_dropped_and_its_neighbours_merge():
    """two rows of a far-away inverted pair between two '+' pieces: the pair is a '-' run of 2 IDs, dropped, and the '+'
    runs around it merge into one block; with a third ID the run is a block and the read has two records"""
    def rows(n_mid):
        left = read_across([(10000, 15000, 0)])
        mid = [("r", 5000 + k * STEP, 0, 100000 + (n_mid - 1 - k) * STEP, 100000 + (n_mid - 1 - k) * STEP) for k in range(n_mid)]
        right = read_across([(15000, 25000, 0)], pos0=5000 + n_mid * STEP)
        return left + mid + right
    st = O.strands([(r[4], r[3], r[1]) for r in rows(2)])
    assert st[10:12] == [1, 1] and all(d == 0 for d in st[:10] + st[12:])
    assert O.switches(rows(2), RLEN) == []
    assert [(a[0], b[0]) for _, _, a, b in O.switches(rows(3), RLEN)] == [(0, 1), (1, 0)]


def test_up_equal_down_stays_unoriented():
    """X pairs once rising (with U) and once falling (with D); a row without a partner is unoriented too"""
    x, u, d, lone = (1, 5000, 5000), (2, 6000, 6000), (3, 4000, 6000), (4, 900000, 7000)
    assert O.strands([x, u, d, lone]) == [None, 0, 1, None]


def test_repeated_ids_count_once_and_never_pair():
    rows = read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)])
    twin = [r for r in rows if r[4] == 12000][0]
    rows.insert(rows.index(twin) + 1, ("r", twin[1] + 2, 0, twin[3] + 2, twin[4]))  # the same ID again
    recs = O.switches(rows, RLEN)
    assert sides(recs) == [(0, 19500, 1, 29500), (1, 20000, 0, 30000)] and recs[0][2][1] == 20
    # a '-' run of three rows with two distinct IDs is dropped like a run of two rows
    mid = [("r", 5000, 0, 100500, 100500), ("r", 5500, 0, 100000, 100000), ("r", 5502, 0, 100002, 100000)]
    rows = read_across([(10000, 15000, 0)]) + mid + read_across([(15000, 25000, 0)], pos0=6500)
    assert O.strands([(r[4], r[3], r[1]) for r in rows])[10:13] == [1, 1, 1]
    assert O.switches(rows, RLEN) == []


def test_bad_rows_are_ignored():
    rows = read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)])
    bad = {(0, s) for s in range(20000, 30000, STEP)}
    assert O.switches(rows, RLEN, bad) == []
    bad = {(0, s) for s in range(20000, 29000, STEP)}  # two inverted IDs left: a dropped run
    assert O.switches(rows, RLEN, bad) == []


def test_rows_on_another_contig_and_row_order():
    """rows off the first row's contig do not count; rows are taken in pos order whatever their row order"""
    rows = read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)])
    want = O.switches(rows, RLEN)
    other = [("r", 100 + k, 1, 5000 - k * 600, 7000 + k) for k in range(20)]
    assert O.switches(rows[:1] + other + rows[1:], RLEN) == want
    rng = np.random.default_rng(3)
    shuffled = [rows[0]] + [rows[i] for i in 1 + rng.permutation(len(rows) - 1)]
    assert O.switches(shuffled, RLEN) == want


def test_read_length_at_the_minimum():
    rows = read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)])
    assert len(O.switches(rows, {"r": 10000}, minlen=10000)) == 2
    assert O.switches(rows, {"r": 9999}, minlen=10000) == []


# ------------------------------------------------------------------------------------------------
# host files (cli.inversion_texts) against the oracle's
# ------------------------------------------------------------------------------------------------
def _columns(recs, read_index):
    from gavisunk_b200.engine import Engine
    cols = {c: [] for c in Engine.SWITCH_COLUMNS}
    for rd, c, a, b in recs:
        cols["read"].append(read_index[rd])
        cols["contig"].append(c)
        for side, (d, n, lo, hi, (g, s, p)) in (("1", a), ("2", b)):
            for k, v in zip(("strand", "ids", "lo", "hi", "id", "start", "pos"), (d, n, lo, hi, g, s, p)):
                cols[k + side].append(v)
    return {k: np.asarray(v, np.uint32) for k, v in cols.items()}


def test_host_files_equal_oracle():
    """three reads across the breakpoints of [20 kb, 30 kb) (one spanning it), two reads across another inversion (no
    call), a fold-back read, records chained apart by more than the chain distance, and a record on another
    haplotype's contig"""
    from gavisunk_b200 import cli, io as gio
    rows = []
    rows += read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)], read="zspan")
    rows += read_across([(5000, 20000, 0), (20000, 26000, 1)], read="b_left")
    rows += read_across([(24000, 30000, 1), (30000, 42000, 0)], read="a_right")
    rows += read_across([(12000, 20000, 0), (20000, 27000, 1)], read="c_left")
    rows += read_across([(100000, 120000, 0), (200000, 215000, 1)], read="far1")
    rows += read_across([(105000, 120000, 0), (200000, 212000, 1)], read="far2")
    rows += read_across([(60000, 80000, 0), (65000, 80000, 1)], read="fold")
    rows += read_across([(10000, 20000, 0), (20000, 30000, 1)], read="otherhap", contig=1)
    reads = list(dict.fromkeys(r[0] for r in rows))
    rlen = {r: 40000 + 1000 * i for i, r in enumerate(reads)}
    recs = O.switches(rows, rlen)
    contigs = [("ctg0", 300000), ("ctg1", 50000)]
    want = O.texts(recs, contigs, [0], lambda r: r, lambda r: rlen[r])
    assert want[1] == "ctg0\t19500\t29500\tinversion\t4\t5\t1\n"
    idx = {r: i for i, r in enumerate(reads)}
    sw = _columns(recs, idx)
    rtab = gio.NameTable(reads)
    lens = np.asarray([rlen[r] for r in reads], np.uint32)
    got = cli.inversion_texts([0], [n for n, _ in contigs], sw, rtab, lens, cli.bytewise_rank(rtab))
    assert got == (want[0].encode(), want[1].encode())
    assert b"\tfoldback\n" in got[0] and b"otherhap" not in got[0]
    got1 = cli.inversion_texts([1], [n for n, _ in contigs], sw, rtab, lens, cli.bytewise_rank(rtab))
    assert got1 == tuple(t.encode() for t in O.texts(recs, contigs, [1], lambda r: r, lambda r: rlen[r])) and got1[1] == b""


def test_host_files_without_records():
    from gavisunk_b200 import cli, io as gio
    from gavisunk_b200.engine import Engine
    sw = {c: np.zeros(0, np.uint32) for c in Engine.SWITCH_COLUMNS}
    rtab = gio.NameTable(["a"])
    got = cli.inversion_texts([0], ["ctg0"], sw, rtab, np.asarray([5], np.uint32), cli.bytewise_rank(rtab))
    assert got == (O.texts([], [("ctg0", 1)], [0], str, len)[0].encode(), b"")


# ------------------------------------------------------------------------------------------------
# why: the validation joins the flanks of an inversion
# ------------------------------------------------------------------------------------------------
def test_validation_joins_across_an_inversion():
    rows = read_across([(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)])
    ids = G.validate_read(sorted(((r[1], r[3], r[4]) for r in rows), key=lambda t: t[1]))
    assert len(rows) == 70 and len(ids) == 54
    assert min(ids) == 10000 and max(ids) == 44500
    assert sum(1 for i in ids if 20000 <= i < 30000) == 4

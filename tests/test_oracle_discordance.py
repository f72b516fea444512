"""The distance-discordance oracle (tests/discordance_oracle.py) on hand-made reads with explicit expected records, and the
host side of `fused --discordance` (cli.discordance_texts: reads.tsv, runs, calls) against the oracle's files."""
import numpy as np
import pytest

import discordance_oracle as O

CONTIGS = [("c0", 20000), ("c1", 8000), ("c2", 5000)]
IDS = (1000, 3000, 5000, 7000, 9000)  # groups of c0; c1 has a group at 0, c2 none
GROUPS = {(0, i) for i in IDS} | {(1, 0), (1, 4000)}


def _read(name, shift_after, sign=1, ids=IDS, event=6000, c=0, base=1000):
    """rows of a read over the groups `ids` (starts = ID + 5): pos = base + start on the + strand (sign 1) or
    base + 30000 - start on the - strand; the read carries `shift_after` extra bases past the event"""
    out = []
    for i in ids:
        s = i + 5
        p = (base + s if sign > 0 else base + 30000 - s) + (shift_after if s > event else 0) * sign
        out.append((name, p, c, s, i))
    return out


def _all_validated(rows):
    return {(r[0], r[4]) for r in rows}


def test_plus_and_minus_read_across_an_insertion_and_a_deletion():
    rows = _read("p", 1000) + _read("m", 1000, sign=-1) + _read("e", -500)
    sp = O.spans(rows, set(), _all_validated(rows))
    assert O.records(sp) == [
        ("p", 0, (5000, 5005, 6005), (7000, 7005, 9005), 1000, "longer"),
        ("m", 0, (5000, 5005, 25995), (7000, 7005, 22995), 1000, "longer"),
        ("e", 0, (5000, 5005, 6005), (7000, 7005, 7505), -500, "shorter"),
    ]
    assert len(sp) == 12 and all(s[4] == 0 for s in sp if s[5] is None)
    rn = O.runs(sp, GROUPS, CONTIGS)
    assert rn == [(0, 0, 1000, 0, 0, 0), (0, 1000, 5000, 3, 0, 0), (0, 5000, 7000, 3, 2, 1), (0, 7000, 9000, 3, 0, 0),
                  (0, 9000, 20000, 0, 0, 0), (1, 0, 8000, 0, 0, 0), (2, 0, 5000, 0, 0, 0)]
    assert O.calls(O.records(sp), rn, min_reads=2) == [(0, 5000, 7000, "collapse", 5000, 7000, 3, 2, 1000)]
    assert O.calls(O.records(sp), rn) == []


def test_repeated_validated_id_is_skipped_and_its_neighbours_span_across():
    rows = _read("d", 1000)
    rows.insert(3, ("d", 6010, 0, 5010, 5000))  # a second row of group 5000
    sp = O.spans(rows, set(), _all_validated(rows))
    assert [(s[2][0], s[3][0]) for s in sp] == [(1000, 3000), (3000, 7000), (7000, 9000)]
    assert O.records(sp) == [("d", 0, (3000, 3005, 4005), (7000, 7005, 9005), 1000, "longer")]
    seg = O.segments(sp, GROUPS, CONTIGS)[0]
    assert [x[2:] for x in seg] == [(1, 0, 0), (1, 1, 0), (1, 1, 0), (1, 0, 0), (0, 0, 0)]


def test_bad_row_and_non_validated_row_are_not_usable():
    rows = _read("b", 1000)
    sp = O.spans(rows, {(0, 5000)}, _all_validated(rows) - {("b", 9000)})
    assert [(s[2][0], s[3][0], s[5]) for s in sp] == [(1000, 3000, None), (3000, 7000, "longer")]


def test_span_that_skips_groups_covers_every_segment_between():
    rows = _read("s", 1000, ids=(1000, 9000))
    sp = O.spans(rows, set(), _all_validated(rows))
    assert O.records(sp) == [("s", 0, (1000, 1005, 2005), (9000, 9005, 11005), 1000, "longer")]
    rn = O.runs(sp, GROUPS, CONTIGS)
    assert rn[:3] == [(0, 0, 1000, 0, 0, 0), (0, 1000, 9000, 1, 1, 0), (0, 9000, 20000, 0, 0, 0)]


def test_rows_on_another_contig_than_the_first_do_not_count():
    rows = _read("x", 1000) + [("x", 50000, 1, 4005, 4000)]
    assert len(O.spans(rows, set(), _all_validated(rows))) == 4


@pytest.mark.parametrize("min_delta,rel,delta,kind", [
    (300, 30, 360, "longer"), (300, 30, 359, None), (300, 30, -360, "shorter"), (300, 30, -359, None),
    (300, 0, 300, "longer"), (300, 0, 299, None), (300, 0, -300, "shorter"), (300, 0, -299, None),
    (0, 30, 60, "longer"), (0, 30, 59, None), (0, 30, -60, "shorter"), (0, 30, -59, None)])
def test_threshold_equality(min_delta, rel, delta, kind):
    rows = [("t", 1005, 0, 1005, 1000), ("t", 3005 + delta, 0, 3005, 3000)]  # dstart = 2000
    sp = O.spans(rows, set(), _all_validated(rows), min_delta, rel)
    assert [(s[4], s[5]) for s in sp] == [(delta, kind)]


def test_head_runs_and_contig_ends():
    rows = [("h", 5, 1, 5, 0), ("h", 5005, 1, 4005, 4000)]  # c1: a group at 0, a span of +1000 from it
    sp = O.spans(rows, set(), _all_validated(rows))
    rn = O.runs(sp, GROUPS, CONTIGS)
    assert [r for r in rn if r[0] == 1] == [(1, 0, 4000, 1, 1, 0), (1, 4000, 8000, 0, 0, 0)]
    assert [r for r in rn if r[0] == 2] == [(2, 0, 5000, 0, 0, 0)]
    assert [r for r in rn if r[0] == 0] == [(0, 0, 20000, 0, 0, 0)]


def _merge_case():
    # three reads longer over [3000, 7000) (segments 3000 and 5000), one concordant read over segment 3000 only
    rows = []
    for k in range(3):
        rows += [(f"r{k}", 4005, 0, 3005, 3000), (f"r{k}", 9005 + k, 0, 7005, 7000)]
    rows += [("q", 4005, 0, 3005, 3000), ("q", 6005, 0, 5005, 5000)]
    return rows


def test_adjacent_called_segments_merge_and_the_peak_takes_the_larger_fraction():
    rows = _merge_case()
    sp = O.spans(rows, set(), _all_validated(rows))
    rn = O.runs(sp, GROUPS, CONTIGS)
    assert [r for r in rn if r[0] == 0][1:4] == [(0, 3000, 5000, 4, 3, 0), (0, 5000, 7000, 3, 3, 0), (0, 7000, 20000, 0, 0, 0)]
    assert O.calls(O.records(sp), rn) == [(0, 3000, 7000, "collapse", 5000, 7000, 3, 3, 1001)]


def _tie_case():
    # segments 1000 and 3000 both with 3 longer of 4 spans; a concordant read over the first, a shorter one over the second
    rows = []
    for k in range(3):
        rows += [(f"a{k}", 2005, 0, 1005, 1000), (f"a{k}", 5005, 0, 3005, 3000)]  # +1000 over segment 1000
        rows += [(f"b{k}", 4005, 0, 3005, 3000), (f"b{k}", 7005 + 2 * k, 0, 5005, 5000)]  # +1000.. over segment 3000
    rows += [("c", 2005, 0, 1005, 1000), ("c", 4005, 0, 3005, 3000), ("s", 4005, 0, 3005, 3000), ("s", 5505, 0, 5005, 5000)]
    return rows


def test_peak_ties_go_to_the_first_run():
    rows = _tie_case()
    sp = O.spans(rows, set(), _all_validated(rows))
    rn = O.runs(sp, GROUPS, CONTIGS)
    assert rn[1:3] == [(0, 1000, 3000, 4, 3, 0), (0, 3000, 5000, 4, 3, 1)]
    assert O.calls(O.records(sp), rn) == [(0, 1000, 5000, "collapse", 1000, 3000, 4, 3, 1000)]


def _cli_texts(rows, validated, hap_contigs):
    from gavisunk_b200 import cli
    from gavisunk_b200 import io as gio
    sp = O.spans(rows, set(), validated)
    recs = O.records(sp)
    rn = O.runs(sp, GROUPS, CONTIGS)
    names = sorted({r[0] for r in rows})
    idx = {n: i for i, n in enumerate(names)}
    u = lambda v: np.asarray(v, np.uint32)
    rec = dict(read=u([idx[r[0]] for r in recs]), contig=u([r[1] for r in recs]), id1=u([r[2][0] for r in recs]),
               start1=u([r[2][1] for r in recs]), pos1=u([r[2][2] for r in recs]), id2=u([r[3][0] for r in recs]),
               start2=u([r[3][1] for r in recs]), pos2=u([r[3][2] for r in recs]))
    runs = {c: u([r[k] for r in rn]) for k, c in enumerate(("contig", "start", "end", "spans", "longer", "shorter"))}
    lens = u([10000 + i for i in range(len(names))])
    rtab = gio.NameTable(names)
    got = cli.discordance_texts(hap_contigs, [n for n, _ in CONTIGS], rec, runs, rtab, lens, np.arange(len(names)))
    want = O.texts(recs, rn, CONTIGS, hap_contigs, lambda r: r, lambda r: 10000 + idx[r])
    return got, want


@pytest.mark.parametrize("case", ["mixed", "merge", "ties"])
def test_host_texts_equal_oracle(case):
    if case == "mixed":
        rows = _read("p", 1000) + _read("m", 1000, sign=-1) + _read("e", -1500) + _read("f", -1500, sign=-1) + _read("g", -1500)
        rows += [("h", 5, 1, 5, 0), ("h", 5005, 1, 4005, 4000)]
    elif case == "merge":
        rows = _merge_case()
    else:
        rows = _tie_case()
    got, want = _cli_texts(rows, _all_validated(rows), [0, 1, 2])
    assert [g.decode() for g in got] == list(want)
    assert want[2]  # every case makes a call
    got1, want1 = _cli_texts(rows, _all_validated(rows), [1])
    assert [g.decode() for g in got1] == list(want1)

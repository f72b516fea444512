"""cli.allele_calls / cli.allele_texts (the host side of the allele support, DESIGN.md section 5.5h) against the brute-force
oracle (tests/allele_support_oracle.py) on hand-made group tables: the chaining slack, the neighbour rule, the baseline
and its fallback, the summary arithmetic and the file formats.  No GPU."""
import numpy as np
import pytest

import allele_support_oracle as O

K = 20


def _table(rows):
    """rows: (contig, start, own, other, sunks) -> the column dicts of Engine.groups() / Engine.alleles()"""
    a = np.asarray(rows, np.int64).reshape(-1, 5)
    groups = dict(contig=a[:, 0].astype(np.uint32), group=a[:, 1].astype(np.uint32))
    al = dict(own=a[:, 2].astype(np.int32), other=a[:, 3].astype(np.int32), sunks=a[:, 4].astype(np.uint32),
              end=(a[:, 1] + K + 10 * (a[:, 4] - 1)).astype(np.uint32))
    return groups, al


def _dicts(groups, al):
    keys = list(zip(groups["contig"].tolist(), groups["group"].tolist()))
    return [dict(zip(keys, al[c].tolist())) for c in ("own", "other", "sunks", "end")]


def _calls(groups, al, hap_contigs, **kw):
    from gavisunk_b200 import cli
    got = cli.allele_calls(groups["contig"], groups["group"], al["end"], al["own"], al["other"], al["sunks"], hap_contigs, **kw)
    okw = {dict(min_class_groups="min_class", max_gap_groups="max_gap", min_switch_groups="min_switch",
                flip_permille="flip").get(k, k): v for k, v in kw.items()}
    want = O.calls(hap_contigs, *_dicts(groups, al), **okw)
    assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2]
    return got


def _row(c, i, own, other, sunks=4):
    return (c, 1000 + 100 * i, own, other, sunks)


def test_chaining_slack():
    """flipped groups chain across at most max_gap_groups assessed, non-flipped groups; unassessed groups are free"""
    st = [(0, 20), (1, 20), (20, 0), (0, 1), (20, 0), (2, 20), (20, 0), (20, 0), (20, 0), (0, 20)]
    groups, al = _table([_row(0, i, o, t) for i, (o, t) in enumerate(st)])
    calls, per, _ = _calls(groups, al, [0], min_class_groups=1)
    assert [c[3] for c in calls] == ["switch", "flip"]
    sw = calls[0]
    assert (sw[1], sw[2], sw[4], sw[5], sw[6], sw[7]) == (1000, 1500 + K + 30, 6, 3, 3, 60)
    assert per[0][:6] == (10, 9, 4, 1, 1, 0)
    calls, _, _ = _calls(groups, al, [0], min_class_groups=1, max_gap_groups=1)
    assert [c[3] for c in calls] == ["flip"] * 4
    calls, _, _ = _calls(groups, al, [0], min_class_groups=1, min_switch_groups=4)
    assert [c[3] for c in calls] == ["flip"] * 4


def test_flip_threshold_is_exact():
    """1000*own <= flip_permille*(own+other), other >= min_reads: 1 of 5 is flipped at 200 permille, 3 of 13 is not (and
    shared), 0 of 2 is not assessed"""
    groups, al = _table([_row(0, 0, 1, 4), _row(0, 1, 3, 10), _row(0, 2, 0, 2), _row(0, 3, 0, 3)])
    calls, per, _ = _calls(groups, al, [0], min_class_groups=1)
    assert [(c[1], c[3]) for c in calls] == [(1000, "flip"), (1300, "flip")]
    assert per[0][1:3] == (3, 2) and per[0][7] == 1  # (3, 10): shared


def test_neighbour_rule():
    """an unsupported group is an error only with an assessed group on both sides: not at a contig end, nor next to a
    coverage hole"""
    st = [(0, 0), (20, 0), (0, 0), (20, 0), (1, 1), (0, 0), (20, 0), (20, 0), (0, 0)]
    groups, al = _table([_row(0, i, o, t) for i, (o, t) in enumerate(st)] + [_row(1, 0, 20, 0), _row(1, 1, 0, 0)])
    calls, per, _ = _calls(groups, al, [0, 1], min_class_groups=1)
    assert [(c[0], c[1], c[3]) for c in calls] == [(0, 1200, "error")]
    assert calls[0][2] == 1200 + K + 30 and calls[0][4:] == (1, 1, 0, 0)
    assert per[0][5:7] == (1, 9) and per[1][5:7] == (0, 2)


def test_baseline_and_fallback():
    """B = lower median of own over the class's groups with an own read; a class with fewer than min_class_groups such
    groups falls back to the haplotype's; a group whose B is below min_baseline is not eligible for an error"""
    rows = [_row(0, i, 20, 0, sunks=4) for i in range(6)] + [_row(0, 6, 0, 0, sunks=4), _row(0, 7, 20, 0, sunks=4)]
    rows += [_row(0, 8 + i, 4, 0, sunks=40) for i in range(3)] + [_row(0, 11, 0, 0, sunks=40), _row(0, 12, 4, 0, sunks=40)]
    groups, al = _table(rows)
    calls, per, base = _calls(groups, al, [0], min_class_groups=4)
    assert base[2][1:] == (7, 20, False) and base[5][1:] == (4, 4, False)
    assert [(c[1], c[3]) for c in calls] == [(1600, "error")] and per[0][6] == 8
    calls, per, base = _calls(groups, al, [0], min_class_groups=5)  # class 5 falls back to the lower median of all 11
    assert base[5][1:] == (4, 20, True)
    assert [(c[1], c[3]) for c in calls] == [(1600, "error"), (2100, "error")] and per[0][6] == 13
    calls, per, _ = _calls(groups, al, [0], min_class_groups=4, min_baseline=21)
    assert calls == [] and per[0][6] == 0


def test_no_read_at_all():
    groups, al = _table([_row(0, i, 0, 0) for i in range(5)])
    calls, per, base = _calls(groups, al, [0])
    assert calls == [] and per == [(5, 0, 0, 0, 0, 0, 0, 0)] and all(b[2] is None for b in base)


def _random_table(seed, n=600):
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(n):
        c = int(rng.integers(0, 4))
        kind = rng.random()
        own, other = (int(rng.integers(8, 20)), int(rng.integers(0, 3)))
        if kind < 0.08:
            own, other = other, own
        elif kind < 0.12:
            own, other = 0, 0
        elif kind < 0.16:
            own, other = int(rng.integers(0, 3)), int(rng.integers(0, 3))
        rows.append((c, 10 * i + int(rng.integers(0, 5)), own, other, int(rng.integers(1, 80))))
    return rows


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_tables_and_texts(seed):
    from gavisunk_b200 import cli
    groups, al = _table(_random_table(seed))
    contigs = [(f"c{i}", 7000 + 10 * i) for i in range(4)]
    own, other, sunks, end = _dicts(groups, al)
    rn = O.runs({g: (own[g], other[g]) for g in own}, contigs)
    runs = {c: np.asarray([r[i] for r in rn], np.uint32) for i, c in enumerate(("contig", "start", "end", "own", "other"))}
    for hap_contigs in ([0, 2], [3, 1]):
        kw = dict(min_class_groups=30)
        calls, per, _ = _calls(groups, al, hap_contigs, **kw)
        assert {c[3] for c in calls} >= {"flip", "error"}
        got = cli.allele_texts(hap_contigs, [n for n, _ in contigs], [l for _, l in contigs], groups, al, runs, **kw)
        want = O.texts(hap_contigs, contigs, own, other, sunks, end, min_class=30)
        assert [g.decode() if isinstance(g, bytes) else bytes(g).decode() for g in got] == list(want)
        total = want[2].splitlines()[-1].split("\t")
        assert total[0] == "*" and int(total[9]) == 10 ** 6 * int(total[3]) // int(total[2])
        assert int(total[10]) == 10 ** 6 * 2 * int(total[5]) // int(total[2])

"""The oracle's diag vote (oracle/gavisunk_oracle.py: _trunc_median, diag_filter_v3) on large candidates.

The reference-recorded goldens pin the oracle only up to 23 rows per (read, contig) candidate.  Here it is checked at
every size tier of the GPU vote (2-48, 49-256, > 256 rows) and on the diagonal shapes those kernels treat specially,
against an independent statement: the median as an exact Fraction truncated toward zero, the band vote as a
brute-force count of distinct groups.  The candidate generator below also feeds tests/test_gpu_diag_vote.py, which
compares the CUDA kernels with this oracle.

A candidate is a list of rows (pos, start, group).  Its reverse diagonal is pos + start, its forward one start - pos.
"""
import random
from fractions import Fraction

import pytest

import gavisunk_oracle as O

BAND = 2500
U32 = (1 << 32) - 1
SIZES = (2, 3, 47, 48, 49, 50, 255, 256, 257, 1023, 1024, 1025, 4999, 5000)
WARP_MAX, RANK_MAX = 256, 48  # largest candidate of the warp kernel, and of its all-pairs rank path


def diag(rows, orient):
    """0: reverse diagonal (pos + start), 1: forward diagonal (start - pos)"""
    return [s + p if orient == 0 else s - p for p, s, _ in rows]


def is_sorted(v):
    return all(a <= b for a, b in zip(v, v[1:])) or all(a >= b for a, b in zip(v, v[1:]))


def exact_median(vals):
    """percentile 50 with linear interpolation, as an exact fraction, truncated toward zero"""
    a = sorted(vals)
    lo = (len(a) - 1) // 2
    m = Fraction(a[lo]) if len(a) % 2 else Fraction(a[lo] + a[lo + 1], 2)
    q = abs(m.numerator) // m.denominator
    return q if m >= 0 else -q


def brute_vote(rows, orient):
    """distinct groups among the rows whose diagonal lies strictly within BAND of the median"""
    v = diag(rows, orient)
    med = exact_median(v)
    inband = sorted(g for x, (_, _, g) in zip(v, rows) if -BAND < x - med < BAND)
    return sum(1 for i, g in enumerate(inband) if i == 0 or g != inband[i - 1])


def expected_best(rows):
    """(good, dir) of a read whose only contig is this candidate: reverse is tried first, forward wins only on more"""
    g0, g1 = brute_vote(rows, 0), brute_vote(rows, 1)
    return (g1, "+") if g1 > g0 else (g0, "-")


# ---- group ids --------------------------------------------------------------------------------
def set_groups(rows, mode, rng):
    """up / down: strictly monotone; flat: monotone with equal neighbours; perm: distinct, not monotone;
    dup: repeated ids in random order (in and out of the band)"""
    n = len(rows)
    g0 = rng.randrange(1, 1 << 20)
    if mode == "up":
        gs = [g0 + 3 * i for i in range(n)]
    elif mode == "down":
        gs = [g0 + 3 * (n - i) for i in range(n)]
    elif mode == "flat":
        gs, g = [], g0
        for i in range(n):
            g += 0 if i % 3 == 1 else 1
            gs.append(g)
    elif mode == "perm":
        gs = [g0 + i for i in range(n)]
        rng.shuffle(gs)
        if n > 1 and gs == sorted(gs):
            gs[0], gs[1] = gs[1], gs[0]
    elif mode == "dup":
        pool = [g0 + i for i in range(max(1, n // 3))]
        gs = [rng.choice(pool) for _ in range(n)]
    else:
        raise ValueError(mode)
    return [(p, s, g) for (p, s, _), g in zip(rows, gs)]


# ---- diagonal shapes ----------------------------------------------------------------------------
def one_strand(rng, n, fwd, jitter=3500):
    """a read along one strand: the true diagonal is jittery, the other one is sorted along the rows (pos steps
    exceed the jitter).  Group ids follow the contig coordinate, so they are strictly monotone."""
    s0 = 200_000_000
    rows, p = [], rng.randrange(0, 5000)
    for i in range(n):
        p += rng.randrange(4000, 6000)
        j = rng.randrange(-jitter, jitter + 1)
        rows.append((p, s0 + p + j if fwd else s0 - p + j, 0))
    return set_groups(rows, "up" if fwd else "down", rng)


def plateau(rng, n, fwd):
    """one_strand with equal neighbours on the sorted diagonal: pairs (p, s) and (p + t, s - t) (forward read) or
    (p + t, s + t) (reverse read)"""
    rows = one_strand(rng, n, fwd)
    for i in range(1, n, 2):
        p, s, g = rows[i - 1]
        t = rng.randrange(0, 400)
        rows[i] = (p + t, s - t if fwd else s + t, rows[i][2])
    return rows


def strand_flip(rng, n):
    """the read changes strand half way at the same locus: neither diagonal is sorted"""
    s0 = 200_000_000
    rows, p = [], 0
    for i in range(n):
        p += rng.randrange(800, 1200)
        j = rng.randrange(-3000, 3001)
        rows.append((p, s0 + p + j if i < n // 2 else s0 + 2 * (n // 2) * 1000 - p + j, 0))
    return set_groups(rows, "perm", rng)


def chimera(rng, n):
    """a forward read whose last 40 % maps to a second locus 3 Mb upstream on the same contig"""
    rows = one_strand(rng, n, True)
    cut = (n * 3) // 5
    return [(p, s - 3_000_000 if i >= cut else s, g) for i, (p, s, g) in enumerate(rows)]


def designed(rng, n, orient, V, D, ties, upper_ties=0):
    """an unsorted candidate whose `orient` diagonal has the value V at rank lo = (n - 1) // 2, V + D at rank lo + 1
    (even n), `ties` extra copies of V just below rank lo and `upper_ties` copies of V + D just above rank lo + 1,
    and rows at 2498 / 2499 below and 2499 / 2500 / 2501 above the median (when the ranks leave room).  The edges
    are asymmetric so that moving the median by one changes the vote.  The other diagonal is spread far wider
    than the band, so this one decides the read."""
    lo = (n - 1) // 2
    med = exact_median([V, V + D] if n % 2 == 0 else [V])
    below = [V] * min(ties, lo)
    for e in (2499, 2498):
        if len(below) < lo and med - e <= V:
            below.append(med - e)
    while len(below) < lo:
        below.append(V - rng.randrange(3000, 4_000_000))
    n_up = n - lo - 1 - (n % 2 == 0)
    above = [V + D] * min(upper_ties, n_up)
    for e in (2499, 2500, 2501):
        if len(above) < n_up and med + e >= V + D:
            above.append(med + e)
    while len(above) < n_up:
        above.append(V + D + rng.randrange(3000, 4_000_000))
    vals = below + [V] + ([V + D] if n % 2 == 0 else []) + above
    assert len(vals) == n and sorted(vals)[lo] == V
    rng.shuffle(vals)
    if n > 2 and is_sorted(vals):
        vals[0], vals[-1] = vals[-1], vals[0]
    return rows_on_diag(rng, vals, orient)


def rows_on_diag(rng, vals, orient, step=(6000, 9000)):
    """rows whose `orient` diagonal takes the given values in order; pos grows by `step` along the rows"""
    lo_v = min(vals)
    p = max(0, -lo_v) if orient == 1 else 0  # forward: start = v + pos >= 0
    rows = []
    for v in vals:
        p += rng.randrange(*step)
        s = v + p if orient == 1 else v - p
        rows.append((p, s, 0))
    if orient == 0 and min(s for _, s, _ in rows) < 0:  # reverse: start = v - pos: shift the diagonal up
        sh = -min(s for _, s, _ in rows)
        rows = [(p, s + sh, 0) for p, s, _ in rows]
    assert all(0 <= p <= U32 and 0 <= s <= U32 for p, s, _ in rows)
    return set_groups(rows, "perm", rng)


def spread(rng, n):
    """pos and start near 0 and near 2^32 - 1 on one candidate: both diagonals span about 2^33.  A cluster of rows
    around the middle carries the vote."""
    rows = []
    corners = [(0, 0), (0, U32), (U32, 0), (U32, U32), (1, 2), (U32 - 3, U32 - 1)]
    for i in range(n):
        if i % 4 == 0:
            p, s = corners[(i // 4) % len(corners)]
            p += rng.randrange(0, 50) if p < (1 << 31) else -rng.randrange(0, 50)
            s += rng.randrange(0, 50) if s < (1 << 31) else -rng.randrange(0, 50)
        else:
            p = (1 << 31) + rng.randrange(0, 1 << 24)
            s = (1 << 31) + rng.randrange(-4000, 4000) + (p - (1 << 31)) * (i % 2)
        rows.append((p, s, 0))
    rng.shuffle(rows)
    return set_groups(rows, "perm", rng)


def tie_both(rng, n):
    """every row within the band in both orientations: good0 == good1, so the reverse strand must win"""
    rows = [(rng.randrange(10_000, 10_600), rng.randrange(50_000, 50_600), 0) for _ in range(n)]
    return set_groups(rows, "perm", rng)


def candidate_zoo(seed):
    """(label, rows) for every shape at every size of SIZES (a few shapes only where the size allows)"""
    rng = random.Random(seed)
    out = []
    for n in SIZES:
        out.append((f"fwd_{n}", one_strand(rng, n, True)))
        out.append((f"rev_{n}", one_strand(rng, n, False)))
        out.append((f"tie_both_{n}", tie_both(rng, n)))
        if n >= 4:
            out.append((f"plateau_fwd_{n}", plateau(rng, n, True)))
            out.append((f"plateau_rev_{n}", plateau(rng, n, False)))
            out.append((f"flip_{n}", strand_flip(rng, n)))
            out.append((f"chimera_{n}", chimera(rng, n)))
            out.append((f"spread_{n}", spread(rng, n)))
            out.append((f"fwd_dupgroups_{n}", set_groups(one_strand(rng, n, True), "dup", rng)))
            out.append((f"rev_flatgroups_{n}", set_groups(one_strand(rng, n, False), "flat", rng)))
        if n >= 8:
            lo = (n - 1) // 2
            for orient in (0, 1):
                # V negative: a forward diagonal with pos > start; D odd: the median is an x.5 before truncation
                for V in ((-50_001, 50_001) if orient == 1 else (7_000_001,)):
                    out.append((f"odd_gap_o{orient}_V{V}_{n}", designed(rng, n, orient, V, 2001, 0)))
                    out.append((f"ties_below_o{orient}_V{V}_{n}", designed(rng, n, orient, V, 1999, lo // 2)))
                    out.append((f"ties_across_o{orient}_V{V}_{n}", designed(rng, n, orient, V, 0, lo // 2, 3)))
                # the value of rank lo is the diagonal's minimum (lo + 1 copies) / lo + 2 copies: count_le(vlo) = lo + 1
                # < lo + 2 and >= lo + 2
                out.append((f"min_at_lo_o{orient}_{n}", designed(rng, n, orient, 90_000_001, 1001, lo)))
                out.append((f"min_across_o{orient}_{n}", designed(rng, n, orient, 90_000_001, 0, lo, 1)))
                # the value of rank lo is the diagonal's maximum
                out.append((f"max_at_lo_o{orient}_{n}", designed(rng, n, orient, 90_000_001, 0, 0, n)))
    return out


ZOO = candidate_zoo(7)


def _vote_by_oracle(rows):
    got = O.diag_filter_v3([("r", p, "c", s, g) for p, s, g in rows], {"c"})
    return (got[0][2], got[0][3]) if got else None


@pytest.mark.parametrize("vals", [
    [-3, -2], [2, 3], [-3, 4], [-4, 3], [-1, 0], [0, 1], [-(1 << 33), 1 << 33], [-(1 << 33), (1 << 33) - 1],
    [-(1 << 33) + 1, 1 << 33], [U32, U32 + 2], [-U32, -U32 + 1], [5], [-5], [-7, -7, -7], [1, 1, 2, 2],
])
def test_trunc_median_edges(vals):
    assert O._trunc_median(vals) == exact_median(vals)


def test_trunc_median_zoo():
    for label, rows in ZOO:
        for orient in (0, 1):
            v = diag(rows, orient)
            assert O._trunc_median(v) == exact_median(v), (label, orient)


def test_vote_zoo():
    for label, rows in ZOO:
        good, d = expected_best(rows)
        assert _vote_by_oracle(rows) == ((good, d) if good > 1 else None), label


def test_zoo_reaches_every_tier():
    """the shapes the GPU vote treats differently all occur above each tier boundary, within the u32 range of the
    .sunkpos columns"""
    assert all(0 <= p <= U32 and 0 <= s <= U32 for _, rows in ZOO for p, s, _ in rows)  # .sunkpos columns are u32
    big = [(label, rows) for label, rows in ZOO if len(rows) > WARP_MAX]
    mid = [(label, rows) for label, rows in ZOO if RANK_MAX < len(rows) <= WARP_MAX]
    for group in (big, mid):
        assert any(not is_sorted(diag(r, 0)) and not is_sorted(diag(r, 1)) for _, r in group)
        assert any(is_sorted(diag(r, 0)) != is_sorted(diag(r, 1)) for _, r in group)
        assert any(not (len({g for _, _, g in r}) == len(r)) for _, r in group)
    for label, rows in ZOO:
        if label.startswith("spread_"):
            v = diag(rows, 0)
            assert max(v) - min(v) > (1 << 33) - 1000, label
    # the band edge decides: some candidates have rows at exactly 2499 and 2500 from the median
    n_edge = 0
    for label, rows in ZOO:
        for orient in (0, 1):
            v = diag(rows, orient)
            m = exact_median(v)
            n_edge += any(abs(x - m) == BAND - 1 for x in v) and any(abs(x - m) == BAND for x in v)
    assert n_edge > 50


def test_vote_shapes_change_the_count():
    """the designed candidates are sensitive to the median: moving it by one, or taking the lower middle element
    for the median of an even count, changes the vote"""
    for label, rows in ZOO:
        if not label.startswith(("odd_gap", "ties_below")):
            continue
        orient = int(label.split("_o")[1][0])
        v = diag(rows, orient)
        m = exact_median(v)
        a = sorted(v)
        lo = (len(a) - 1) // 2

        def count(med):
            return len({g for x, (_, _, g) in zip(v, rows) if abs(x - med) < BAND})
        assert count(m) != count(m - 1), label
        if len(v) % 2 == 0:
            assert count(m) != count(a[lo]), label

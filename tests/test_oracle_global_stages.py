"""The oracle's run-wide stages against independent statements of the same rules, on seeded adversarial inputs: the
bad groups of badsunks_AR.py (O.bad_sunks_one_hap), the contig-wide components and intervals of
process-by-contig_lowmem_AR.py (O.process_by_contig) and the gaps of get_gaps.py (O.get_gaps).  The GPU suite compares
the kernels with these functions, so they are pinned here first."""
from collections import Counter

import numpy as np
import pytest

import gavisunk_oracle as O


# ------------------------------------------------------------------------------------------------
# bad groups
# ------------------------------------------------------------------------------------------------
def _rows_of_counts(counts, rng):
    """one row per count unit of every (contig, group), in random order"""
    rows = [("r", 0, c, g, g) for (c, g), v in counts.items() for _ in range(v)]
    return [rows[i] for i in rng.permutation(len(rows))]


def _bad_plain(counts, own):
    """the rule in Counter terms: the mode is the smallest of the most frequent counts of the haplotype's own contigs;
    v > m + 4*sqrt(m) in exact integers is v > m and (v - m)^2 > 16m; own contigs also drop counts below 2, other
    contigs only answer to the upper limit"""
    freq = Counter(v for (c, _), v in counts.items() if c in own)
    top = max(freq.values())
    m = min(v for v, f in freq.items() if f == top)
    over = lambda v: v > m and (v - m) ** 2 > 16 * m
    bad = {k for k, v in counts.items() if (over(v) or v < 2) if k[0] in own}
    bad |= {k for k, v in counts.items() if k[0] not in own and over(v)}
    return bad, m


def _counts(spec):
    """spec: {contig: [count of group 0, count of group 1, ...]} -> {(contig, start): count}"""
    return {(c, 10 + 25 * i): v for c, vs in spec.items() for i, v in enumerate(vs)}


@pytest.mark.parametrize("m", [1, 4, 9, 16, 25, 2025, 2500, 4096, 10 ** 6])
def test_bad_limit_at_perfect_square_modes(m):
    """m + 4*sqrt(m) is an integer: a count there stays, one above is bad"""
    rng = np.random.default_rng(m)
    lim = m + 4 * int(round(m ** 0.5))
    counts = _counts({"a": [m] * 4 + [lim, lim + 1, 1, 2], "b": [lim, lim + 1, 1]})
    bad, mode = O.bad_sunks_one_hap(_rows_of_counts(counts, rng) if m < 10 ** 5 else
                                    [("r", 0, c, g, g) for (c, g), v in counts.items() for _ in range(v)], {"a"})
    assert (bad, mode) == _bad_plain(counts, {"a"})
    assert mode == m
    assert {counts[k] for k in bad if k[0] == "a"} == {lim + 1, 1}
    assert {counts[k] for k in bad if k[0] == "b"} == {lim + 1}


def test_bad_mode_ties_take_the_smallest_count():
    rng = np.random.default_rng(1)
    for spec, want in [({"a": [2047] * 3 + [2048] * 3 + [5, 1]}, 2047), ({"a": [2048] * 3 + [2047] * 2 + [9] * 3}, 9),
                       ({"a": [7, 3, 7, 3, 100]}, 3), ({"a": [12] * 5 + [1, 2, 3]}, 12)]:
        counts = _counts(spec)
        bad, mode = O.bad_sunks_one_hap(_rows_of_counts(counts, rng), {"a"})
        assert mode == want
        assert (bad, mode) == _bad_plain(counts, {"a"})


def test_bad_groups_random():
    """random counts on own and other contigs, many seeds: the oracle equals the plain statement"""
    for seed in range(40):
        rng = np.random.default_rng(100 + seed)
        spec = {f"c{c}": rng.integers(1, rng.integers(3, 60), rng.integers(1, 40)).tolist() for c in range(4)}
        counts = _counts(spec)
        own = {"c0", "c2"} if seed % 2 else {"c1"}
        got = O.bad_sunks_one_hap(_rows_of_counts(counts, rng), own)
        assert got == _bad_plain(counts, own)


def test_bad_groups_without_own_contigs_raise():
    with pytest.raises(IndexError):
        O.bad_sunks_one_hap([("r", 0, "b", 10, 10)], {"a"})


# ------------------------------------------------------------------------------------------------
# components and intervals
# ------------------------------------------------------------------------------------------------
def _read_rows(name, contig, starts, p0=500):
    """a read that validates by construction: pos = start - s0 + p0 passes every pair test"""
    s0 = min(starts)
    return [(name, s - s0 + p0, contig, s, s) for s in sorted(starts)]


def _components(reads, bad, contig):
    """scipy's connected components of the union of the reads' validated ID sets, components of >= 3 groups as
    [min, max] sorted by start"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    sets = [sorted({s for s in st if (contig, s) not in bad}) for st in reads]
    sets = [s for s in sets if len(s) >= 2]
    ids = sorted({i for s in sets for i in s})
    if not ids:
        return []
    ix = {v: i for i, v in enumerate(ids)}
    a = [ix[s[j]] for s in sets for j in range(len(s) - 1)]
    b = [ix[s[j + 1]] for s in sets for j in range(len(s) - 1)]
    n, lab = connected_components(coo_matrix((np.ones(len(a)), (a, b)), shape=(len(ids), len(ids))), directed=False)
    out = []
    for c in range(n):
        mem = [ids[i] for i in np.nonzero(lab == c)[0]]
        if len(mem) >= 3:
            out.append((contig, min(mem), max(mem)))
    return sorted(out, key=lambda t: t[1])


@pytest.mark.parametrize("seed", range(12))
def test_components_and_intervals_against_scipy(seed):
    """random reads over a contig's groups: chains, pairs (components of 2 groups), triples, interleaved and nested
    components, reads on bad groups; the oracle's intervals are the connected components of >= 3 groups"""
    rng = np.random.default_rng(seed)
    ng = int(rng.integers(50, 400))
    groups = np.sort(rng.choice(np.arange(0, 100 * ng), ng, replace=False))
    reads = []
    for _ in range(int(rng.integers(20, 150))):
        kind = rng.integers(0, 4)
        if kind == 0:     # an edge
            i, j = rng.choice(ng, 2, replace=False)
            reads.append([groups[i], groups[j]])
        elif kind == 1:   # a local run
            i = int(rng.integers(0, ng - 6))
            reads.append(list(groups[i:i + int(rng.integers(2, 6))]))
        elif kind == 2:   # interleaved: every p-th group
            p = int(rng.integers(2, 5))
            i = int(rng.integers(0, ng - 3 * p))
            reads.append(list(groups[i:i + 3 * p:p]))
        else:             # scattered
            reads.append(list(rng.choice(groups, int(rng.integers(2, 7)), replace=False)))
    bad = {("c", int(g)) for g in rng.choice(groups, ng // 20, replace=False)}
    rows, rlen = [], {}
    for i, st in enumerate(reads):
        name = f"r{i:05d}"
        rows += _read_rows(name, "c", [int(s) for s in set(st)])
        rlen[name] = 10 ** 7
    inter, bed = O.process_by_contig(rows, rlen, bad, "c", minlen=10000)
    want = _components([[int(s) for s in st] for st in reads], bad, "c")
    assert (bed or []) == want
    # every read with >= 2 non-bad IDs validates to all of them, in start order
    exp_inter = []
    for i, st in enumerate(reads):
        ids = sorted({int(s) for s in st if ("c", int(s)) not in bad})
        if len(ids) >= 2:
            exp_inter += [(s, f"r{i:05d}") for s in ids]
    assert (inter or []) == exp_inter


def test_read_of_one_id_at_two_starts_adds_no_vertex():
    """rows repeating one ID at two starts validate to that ID alone: no vertex, no edge"""
    rows = [("r0", 1000, "c", 5000, 5000), ("r0", 2000, "c", 6000, 5000), ("r0", 900_000, "c", 7000, 7000)]
    rows += _read_rows("r1", "c", [7000, 8000, 9000])
    rows += _read_rows("r2", "c", [4000, 4500])
    inter, bed = O.process_by_contig(rows, {"r0": 10 ** 6, "r1": 10 ** 6, "r2": 10 ** 6}, set(), "c", minlen=10000)
    assert [i for i, r in inter if r == "r0"] == [5000]
    assert bed == [("c", 7000, 9000)]   # 5000 would join 4000-4500 into a component of 3 if it were a vertex
    rows += _read_rows("r3", "c", [4500, 5000])
    _, bed = O.process_by_contig(rows, {f"r{i}": 10 ** 6 for i in range(4)}, set(), "c", minlen=10000)
    assert bed == [("c", 4000, 5000), ("c", 7000, 9000)]


# ------------------------------------------------------------------------------------------------
# gaps
# ------------------------------------------------------------------------------------------------
def _gaps_by_coverage(fai, beds):
    """per-base coverage: an interval (s, e) covers [s, e); a gap is a maximal uncovered run [a, b) between covered
    bases of a contig, written (a, b - 1); a contig without intervals is nodata (0, len)"""
    gaps, nodata = [], []
    for ctg, ln in fai:
        iv = beds.get(ctg)
        if not iv:
            nodata.append((ctg, 0, ln))
            continue
        top = max(e for _, e in iv) + 2
        cov = np.zeros(top + 1, np.int64)
        for s, e in iv:
            cov[s] += 1
            cov[e] -= 1
        on = np.cumsum(cov)[:top] > 0
        lo, hi = int(np.argmax(on)), top - int(np.argmax(on[::-1]))
        d = np.diff(np.concatenate([[0], (~on[lo:hi]).astype(np.int8), [0]]))
        gaps += [(ctg, int(a) + lo, int(b) + lo - 1) for a, b in zip(np.nonzero(d == 1)[0], np.nonzero(d == -1)[0])]
    return gaps, nodata


def test_gaps_of_identical_nested_touching_adjacent_intervals():
    beds = {"a": [(100, 400), (100, 400), (150, 300), (400, 700), (701, 900), (950, 1000), (1000, 1001), (1003, 1500)]}
    fai = [("a", 2000), ("b", 300), ("c", 10)]
    got = O.get_gaps(fai, beds)
    assert got == _gaps_by_coverage(fai, beds)
    assert got[0] == [("a", 700, 700), ("a", 900, 949), ("a", 1001, 1002)]
    assert got[1] == [("b", 0, 300), ("c", 0, 10)]


@pytest.mark.parametrize("seed", range(20))
def test_gaps_random_against_coverage(seed):
    rng = np.random.default_rng(seed)
    fai = [(f"c{i}", int(rng.integers(500, 5000))) for i in range(int(rng.integers(1, 8)))]
    beds = {}
    for ctg, ln in fai:
        if rng.random() < 0.3:
            continue
        iv = []
        for _ in range(int(rng.integers(1, 30))):
            s = int(rng.integers(0, ln - 50))
            iv.append((s, s + int(rng.integers(1, 120))))
        if rng.random() < 0.5 and iv:   # touching and adjacent neighbours
            s, e = iv[-1]
            iv += [(e, e + 5), (e + 6, e + 9)]
        beds[ctg] = [iv[i] for i in rng.permutation(len(iv))]
    assert O.get_gaps(fai, beds) == _gaps_by_coverage(fai, beds)

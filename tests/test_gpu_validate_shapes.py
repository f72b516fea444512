"""Per-read validation (k_validate, csrc/validate_reads.cu) against the oracle's restatement of
process-by-contig_lowmem_AR.py at the shapes where that kernel can go wrong: bad rows removed in every row-count
tier (with the cross-warp prefix of the compaction) and reads landing on the tier edges after removal, orientation
and component ties, reads whose clean-up leaves no edge, working storage reused by later reads of a thread group,
the narrow/wide switch of the ratio test, the length filter, repeated IDs and two rows at one read position.

The oracle's validate_read tests every pair in Python; for reads of hundreds of rows in the thousands that is too
slow, so the reads go through `_validate_np`, the same rule with the pair mask, the multipos counts and the
components in numpy, itself pinned to O.validate_read on small reads (test_numpy_oracle_matches_validate_read).

No test reaches the 4096-round cap of the label propagation: a component needs a path of > 4096 edges whose ends
are not linked more directly, and rows along one diagonal pass the ratio test pairwise (the mediant of two ratios
in (0.9, 1.1) is in it too), so such graphs collapse to diameter 1 or 2."""
from collections import defaultdict

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

import gavisunk_oracle as O

pytestmark = pytest.mark.gpu

U32 = 0xFFFFFFFF


# ------------------------------------------------------------------------------------------------
# the oracle's per-read rule in numpy
# ------------------------------------------------------------------------------------------------
def _validate_np(rows):
    """O.validate_read on rows [(pos, start, ID)] sorted by start (stable) -> (IDs in vertex order or None, orientation,
    status): status 'nopair' (no pair passes), 'empty' (the clean-up dropped every oriented edge) or 'ok'"""
    a = np.asarray(rows, np.int64).reshape(-1, 3)
    P, S, ID = a[:, 0], a[:, 1], a[:, 2]
    n = len(a)
    i, j = np.triu_indices(n, 1)
    ds = np.abs(S[i] - S[j])
    dp = np.abs(P[i] - P[j])
    ok = (9 * ds < 10 * dp) & (10 * dp < 11 * ds)
    i, j = i[ok], j[ok]                       # (i, j) in the reference's loop order
    sg = (P[i] > P[j]).astype(np.int64)
    n1 = int(sg.sum())
    n0 = len(sg) - n1
    if n0 + n1 < 1:
        return None, None, "nopair"
    orient = 1 if n1 > n0 else 0
    i, j = i[sg == orient], j[sg == orient]
    # rows coded by ID and by (ID, pos); first appearances by writing indices in reverse (the earliest write wins)
    uid, idc = np.unique(ID, return_inverse=True)
    _, pc = np.unique(np.stack([ID, P], 1), axis=0, return_inverse=True)
    pc = pc.reshape(-1)

    def first_seen(codes, k):
        f = np.full(k, len(codes))
        f[codes[::-1]] = np.arange(len(codes))[::-1]
        return f

    # multipos over M = left ends in edge order, then right ends, as (ID, pos) pairs
    M = np.concatenate([pc[i], pc[j]])
    k = int(pc.max()) + 1
    cnt, first = np.bincount(M, minlength=k), first_seen(M, k)
    code_id, code_pos = np.empty(k, np.int64), np.empty(k, np.int64)
    code_id[pc], code_pos[pc] = idc, P
    seen = np.flatnonzero(cnt)
    # good position per ID: most entries, ties -> first appearance in M
    o = seen[np.lexsort((first[seen], -cnt[seen], code_id[seen]))]
    head = np.r_[True, code_id[o][1:] != code_id[o][:-1]]
    n_pos = np.diff(np.r_[np.flatnonzero(head), len(o)])
    gp_of = np.full(len(uid), -1, np.int64)
    gp_of[code_id[o][head][n_pos > 1]] = code_pos[o][head][n_pos > 1]   # multi-positioned IDs only
    gp = gp_of[idc[i]]
    drop = (gp >= 0) & (P[i] != gp) & (P[j] != gp)
    i, j = i[~drop], j[~drop]
    if len(i) == 0:
        return None, orient, "empty"
    # vertices by first appearance (source before target), components, largest (ties: earliest vertex)
    seq = np.stack([idc[i], idc[j]], 1).ravel()
    fv = first_seen(seq, len(uid))
    order = np.flatnonzero(fv < len(seq))
    order = order[np.argsort(fv[order], kind="stable")]   # vertex v's ID code
    vnum = np.empty(len(uid), np.int64)
    vnum[order] = np.arange(len(order))
    ev = vnum[seq].reshape(-1, 2)
    nv = len(order)
    g = coo_matrix((np.ones(len(ev)), (ev[:, 0], ev[:, 1])), shape=(nv, nv))
    _, lab = connected_components(g, directed=False)
    size = np.bincount(lab)
    best = None
    for v in range(nv):  # labels in vertex order: the first component of the largest size
        if best is None or size[lab[v]] > size[best]:
            best = lab[v]
    return [int(x) for x in uid[order][lab == best]], orient, "ok"


class _Memo(dict):
    """_validate_np by the read's rows: the oracle's loop and the per-read checks share one evaluation"""

    def __missing__(self, key):
        v = self[key] = _validate_np(list(key))
        return v

    def validate_read(self, rows):
        return self[tuple(rows)][0]


def _per_read(rows, rlen, bad, minlen, memo):
    """read name -> (rows as the reference's loop sees them, (IDs, orientation, status)) on one contig's rows"""
    rows = [r for r in rows if (r[2], int(r[4])) not in bad]
    ids = defaultdict(set)
    for r in rows:
        ids[r[0]].add(r[4])
    sub = sorted((r for r in rows if len(ids[r[0]]) > 1), key=lambda r: (r[0], r[3]))
    by_read = defaultdict(list)
    for r in dict.fromkeys(sub):
        if rlen.get(r[0], -1) >= minlen:
            by_read[r[0]].append((r[1], r[3], r[4]))
    return {n: (rr, memo[tuple(rr)]) for n, rr in by_read.items()}


# ------------------------------------------------------------------------------------------------
# shapes and the engine run
# ------------------------------------------------------------------------------------------------
def _diag(rng, m, strand="+", gap=(15, 3000), wobble=3, jitter=0, s0=10_000, p0=500):
    """m rows (pos, start) along one strand: starts ascending, positions following them (or falling against them)"""
    start = s0 + np.cumsum(rng.integers(gap[0], gap[1], m))
    d = (start - start[0]) + rng.integers(-wobble, wobble + 1, m).cumsum()
    pos = p0 + d if strand == "+" else p0 + 5_000_000 - d
    if jitter:
        pos = pos + rng.integers(-jitter, jitter + 1, m)
    return np.maximum(pos, 0), start


def _shape(rng, m, kind):
    """rows (pos, start, ID) of one read in input order (rising read position); kinds: fwd, rev, fwd_jitter,
    rev_jitter, fwd_dupid, rev_dupid, sparse"""
    strand = "-" if kind.startswith("rev") else "+"
    pos, start = _diag(rng, m, strand, jitter=40 if kind.endswith("jitter") else 0)
    if kind == "sparse":
        pos = 500 + ((start - start[0]) * 1.3).astype(np.int64)    # ratio 1.3: no pair passes ...
        k = rng.choice(m, min(m, max(3, m // 3)), replace=False)
        pos[k] = 500 + (start[k] - start[0])                         # ... except among these rows
    ids = start.copy()
    if kind.endswith("dupid") and m > 3:
        j = rng.choice(m - 2, max(1, m // 12), replace=False)
        ids[j + 2] = ids[j]                                          # the same group again two rows later
    order = np.argsort(pos, kind="stable")
    return [(int(pos[t]), int(start[t]), int(ids[t])) for t in order]


class Case:
    """reads laid out on contigs, each read on its own stretch (IDs never shared across reads), for one engine run"""

    def __init__(self):
        self.reads = []   # (name, contig, [(pos, start, ID)], rlen)
        self.bad = set()  # (contig name, ID)
        self._ctg, self._at = 0, 0

    def add(self, rows, rlen=None, bad_ids=(), shift=True, name=None):
        """rows relative to their own first start; shifted onto a free stretch of the current contig"""
        rows = list(dict.fromkeys((int(p), int(s), int(g)) for p, s, g in rows))  # drop_duplicates (:104)
        if not shift and self._at:
            self._ctg, self._at = self._ctg + 1, 0
        if shift:
            lo = min(min(s for _, s, _ in rows), min(g for _, _, g in rows))
            hi = max(max(s for _, s, _ in rows), max(g for _, _, g in rows))
            if self._at + (hi - lo) + 1_000_000 > U32:
                self._ctg, self._at = self._ctg + 1, 0
            d = self._at - lo + 1_000_000
            rows = [(p, s + d, g + d) for p, s, g in rows]
            bad_ids = [g + d for g in bad_ids]
            self._at += hi - lo + 2_000_000
        ctg = f"c{self._ctg}"
        name = name or f"r{len(self.reads):06d}"
        if rlen is None:
            rlen = max(p for p, _, _ in rows) + 10_000
        self.reads.append((name, ctg, rows, min(int(rlen), U32)))
        self.bad |= {(ctg, int(g)) for g in bad_ids}
        if not shift:
            self._ctg, self._at = self._ctg + 1, 0  # the read keeps its own coordinates: a contig to itself
        return name

    def sunkpos_rows(self):
        return [(n, p, c, s, g) for n, c, rows, _ in self.reads for p, s, g in rows]


def _run(case, minlen=10000, min_pairs=1):
    """the engine's validation + intervals of `case` against the oracle, contig by contig: validated (ID, read) pairs in
    order, per-read orientation (strand of the placements), the count of reads the clean-up emptied, the intervals.
    Returns (oracle per read name, engine pairs as [(ID, name)])."""
    from gavisunk_b200.engine import Engine
    names = sorted(n for n, _, _, _ in case.reads)
    assert len(set(names)) == len(names)
    ridx = {n: i for i, n in enumerate(names)}
    rlen = {n: l for n, _, _, l in case.reads}
    ctgs = sorted({c for _, c, _, _ in case.reads}, key=lambda c: int(c[1:]))
    cidx = {c: i for i, c in enumerate(ctgs)}
    rows = sorted(case.sunkpos_rows(), key=lambda r: ridx[r[0]])  # stable: a read's rows in input order
    eng = Engine(20)
    eng.contig_names = ctgs
    eng.set_reads_meta(np.array([rlen[n] for n in names], np.uint32))
    eng.set_rows(1, [ridx[r[0]] for r in rows], [r[1] for r in rows], [cidx[r[2]] for r in rows], [r[3] for r in rows],
                 [r[4] for r in rows], n_contigs=len(ctgs))
    eng.set_contigs([0] * len(ctgs))
    if case.bad:
        bad = sorted(case.bad)
        eng.bad_set([cidx[c] for c, _ in bad], [g for _, g in bad])
    eng.validate(minlen)
    p = eng.pairs()
    got = [(int(g), names[int(r)]) for g, r in zip(p["group"], p["read"])]
    got_by_ctg = defaultdict(list)
    for (g, n), c in zip(got, p["contig"]):
        got_by_ctg[ctgs[c]].append((g, n))
    pl = eng.placements()
    got_strand = {names[int(r)]: int(s) for r, s in zip(pl["read"], pl["strand"])}
    n_empty = eng.validate_empty_reads()
    eng.components_local()
    iv = eng.intervals()
    got_bed = defaultdict(list)
    for c, s, e in zip(iv["contig"], iv["start"], iv["end"]):
        got_bed[ctgs[c]].append((ctgs[c], int(s), int(e)))
    by_ctg = defaultdict(list)
    for r in case.sunkpos_rows():
        by_ctg[r[2]].append(r)
    per_read, exp_empty, n_pairs = {}, 0, 0
    memo = _Memo()
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(O, "validate_read", memo.validate_read)
        for c in ctgs:
            inter, bed = O.process_by_contig(by_ctg[c], rlen, case.bad, c, minlen=minlen)
            assert got_by_ctg.get(c, []) == (inter or []), c
            assert got_bed.get(c, []) == (bed or []), c
            n_pairs += len(inter or [])
            pr = _per_read(by_ctg[c], rlen, case.bad, minlen, memo)
            per_read.update(pr)
            exp_empty += sum(v[1][2] == "empty" for v in pr.values())
    exp_strand = {n: v[1][1] for n, v in per_read.items() if v[1][2] == "ok" and len(v[1][0]) >= 2}
    assert got_strand == exp_strand
    assert n_empty == exp_empty
    assert n_pairs >= min_pairs
    return per_read, got


def _n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------
# the numpy rule against the oracle's own
# ------------------------------------------------------------------------------------------------
def _fuzz_read(rng, m, n_ids=None, pos_repeat=0.0):
    """a short read with repeated IDs and repeated read positions: rows near a diagonal of either strand, some IDs
    drawn from a few values, some positions copied from a neighbour"""
    pos, start = _diag(rng, m, "+" if rng.random() < 0.5 else "-", gap=(50, 400), wobble=10, jitter=int(rng.integers(0, 30)))
    ids = start.copy() if n_ids is None else rng.choice(start[: max(2, n_ids)], m)
    if pos_repeat:
        k = np.flatnonzero(rng.random(m - 1) < pos_repeat)
        pos[k + 1] = pos[k]
    off = rng.random(m) < 0.1
    start[off] += rng.integers(-5000, 5000, off.sum())
    order = np.argsort(pos, kind="stable")
    return [(int(pos[t]), int(start[t]), int(ids[t])) for t in order]


def test_numpy_oracle_matches_validate_read():
    rng = np.random.default_rng(7)
    seen = defaultdict(int)
    reads = [_fuzz_read(rng, int(m), n_ids=int(rng.integers(2, m + 2)) if t % 2 else None, pos_repeat=0.3 if t % 3 == 0 else 0.0)
             for t, m in enumerate(rng.integers(2, 40, 1500))] + _empty_reads(rng, 20)
    for rows in reads:
        rows.sort(key=lambda r: r[1])
        ids, orient, status = _validate_np(rows)
        assert ids == O.validate_read(rows)
        seen[status] += 1
        seen[f"o{orient}"] += 1
    assert min(seen["ok"], seen["empty"], seen["nopair"], seen["o0"], seen["o1"]) > 10, dict(seen)


# ------------------------------------------------------------------------------------------------
# 1. bad rows in every tier
# ------------------------------------------------------------------------------------------------
def _bad_rows(rng, rows, pattern):
    """IDs to mark bad in a read: a random 10-60 %, every other, runs across 32-row warp boundaries, all but one ID,
    all but one row"""
    ids = [g for _, _, g in rows]
    uniq = list(dict.fromkeys(ids))
    m = len(rows)
    if pattern == "random":
        return [g for g in uniq if rng.random() < rng.uniform(0.1, 0.6)]
    if pattern == "every_other":
        return uniq[::2]
    if pattern == "straddle":
        out = set()
        for b in range(32, m + 31, 32):  # rows b-3 .. b+2 around every warp boundary, and a longer run at random
            out |= {ids[i] for i in range(max(0, b - 3), min(m, b + 3))}
        if m > 40:
            a = int(rng.integers(0, m - 40))
            out |= set(ids[a:a + 37])
        return sorted(out)
    if pattern == "all_but_one_id":
        keep = uniq[int(rng.integers(0, len(uniq)))]
        return [g for g in uniq if g != keep]
    if pattern == "all_but_one_row":
        keep = int(rng.integers(0, m))
        return [g for g in uniq if g != ids[keep]]
    raise ValueError(pattern)


@pytest.mark.parametrize("pattern", ["random", "every_other", "straddle", "all_but_one_id", "all_but_one_row"])
def test_bad_rows_in_every_tier(pattern):
    rng = np.random.default_rng(sum(map(ord, pattern)))
    case = Case()
    for m in [2, 33, 64, 65, 100, 512, 513, 700, 3000]:
        for kind in ("fwd", "rev_jitter", "fwd_dupid"):
            rows = _shape(rng, m, kind)
            case.add(rows, bad_ids=_bad_rows(rng, rows, pattern))
    _run(case, min_pairs=0 if pattern.startswith("all_but") else 100)


def test_bad_rows_land_on_tier_edges():
    """reads placed in a tier by their row count before removal whose kept rows are exactly 1, 2, 64, 65, 512 or 513
    (every count from every larger tier), and reads left with a single ID"""
    rng = np.random.default_rng(3)
    case = Case()
    for m0 in (40, 64, 70, 300, 512, 600, 1100):
        for target in (1, 2, 64, 65, 512, 513):
            if target >= m0:
                continue
            for kind in ("fwd", "rev", "fwd_jitter"):
                rows = _shape(rng, m0, kind)
                keep = set(rng.choice(m0, target, replace=False).tolist())
                case.add(rows, bad_ids=[rows[i][2] for i in range(m0) if i not in keep])
        rows = _shape(rng, m0, "fwd")
        rows = [(p, s, rows[0][2] if i % 3 else rows[1][2]) for i, (p, s, _) in enumerate(rows)]  # two IDs ...
        case.add(rows, bad_ids=[rows[1][2]])                                                     # ... one bad
    per_read, got = _run(case, min_pairs=1000)
    assert {len(v[0]) for v in per_read.values()} >= {2, 64, 65, 512, 513}


# ------------------------------------------------------------------------------------------------
# 2. orientation tie   3. component ties and order
# ------------------------------------------------------------------------------------------------
def _cluster(k, strand, s0, p0, step=1000):
    """k rows on one exact diagonal: every pair passes, k(k-1)/2 pairs of one sign"""
    return [(p0 + (i if strand == "+" else k - 1 - i) * step, s0 + i * step, s0 + i * step) for i in range(k)]


def _join(*clusters):
    rows = [r for c in clusters for r in c]
    return sorted(rows, key=lambda r: r[0])


@pytest.mark.parametrize("m_scale", [1, 10, 30, 90])
def test_orientation_tie_and_off_by_one(m_scale):
    """a forward and a reverse cluster far apart in one read: equal passing pairs keep orientation 0; an extra lone
    pair of either sign tips it.  Sizes scale the read through the three tiers."""
    case = Case()
    k = 3 * m_scale
    for first in ("+", "-"):
        for extra in (None, "+", "-"):
            f = _cluster(k, "+", 100_000, 10_000)
            r = _cluster(k, "-", 50_000_000, 90_000_000)
            if first == "-":  # the reverse cluster at the lower starts
                f, r = _cluster(k, "+", 50_000_000, 10_000), _cluster(k, "-", 100_000, 90_000_000)
            parts = [f, r]
            if extra:
                parts.append(_cluster(2, extra, 200_000_000, 500_000_000))
            case.add(_join(*parts))
    per_read, _ = _run(case, min_pairs=10)
    assert sorted(v[1][1] for v in per_read.values()) == [0] * 4 + [1] * 2


@pytest.mark.parametrize("strand", ["+", "-"])
@pytest.mark.parametrize("k", [3, 20, 200])
def test_component_ties_and_order(strand, k):
    """disjoint diagonals of one orientation in one read: two or three of equal size (the one holding the earliest
    vertex wins), the larger one later in start order, and a component whose lowest row index is not its earliest
    vertex (a row of its ID that has no edge sits before everything else, and the multipos drop takes the edges of a
    repeated ID)"""
    case = Case()
    c = lambda i, kk: _cluster(kk, strand, 1_000_000 + i * 40_000_000, 500_000 + i * 45_000_000)
    case.add(_join(c(0, k), c(1, k)))
    case.add(_join(c(0, k), c(1, k), c(2, k)))
    case.add(_join(c(0, k), c(1, k + 1)))
    case.add(_join(c(0, k), c(1, k), c(2, k + 1)))
    # an edgeless first row carrying an ID of the second cluster: that cluster's label is the lowest, yet the first
    # cluster's vertex was inserted first
    b = c(1, k)
    lone = (5_000_000_000 % U32, 10, b[k // 2][2])
    case.add(_join(c(0, k), b, [lone]))
    case.add(_join(c(0, k), c(1, k + 1), [(4_000_000_000, 10, b[0][2])]))
    # the same ID again inside the first cluster at another read position with fewer edges: its edges go
    a = c(0, k + 1)
    dup = (a[-1][0] + 77, a[-1][1] + 500_000, c(1, k)[0][2])
    case.add(_join(a, c(1, k), [dup]))
    _run(case, min_pairs=10)


# ------------------------------------------------------------------------------------------------
# 4. empty after clean-up
# ------------------------------------------------------------------------------------------------
def _empty_reads(rng, n):
    """short reads whose multipos clean-up drops every oriented edge: IDs X and Y, each on two rows that are only left
    ends (one edge each) and on one row that is the right end of both edges of the other ID.  That row's position is
    the ID's good position (2 edge ends against 1 and 1), so every left end is off its ID's good position and every
    right end is off it too (it holds the other ID).  Scaled, shifted and mirrored at random."""
    out = []
    for _ in range(n):
        k = int(rng.integers(1, 20))
        # (start, pos) of two left ends in the backward ratio cone of a right end at (0, 0), not in each other's
        left = [(-100_000 * k, -108_999 * k), (-10_000 * k, -9_100 * k)]
        rows = []
        for g, (ds, dp) in enumerate([(0, 0), (10_000_000, 30_000_000)]):
            right_id, left_id = (2_000_000, 1_000_000) if g == 0 else (1_000_000, 2_000_000)
            base_s, base_p = 5_000_000 + ds, 5_000_000 + dp
            rows.append((base_p, base_s, right_id))
            rows += [(base_p + p, base_s + s, left_id) for s, p in left]
        if rng.random() < 0.5:
            rows = [(60_000_000 - p, s, g) for p, s, g in rows]
        out.append(sorted(rows))
    return out


def test_reads_emptied_by_the_clean_up_report_nothing():
    rng = np.random.default_rng(11)
    case = Case()
    for rows in _empty_reads(rng, 60):
        case.add(rows)
    per_read, got = _run(case, min_pairs=0)
    assert got == []
    assert sum(v[1][2] == "empty" for v in per_read.values()) == 60
    # and next to reads that do validate, in every tier
    case = Case()
    for i, rows in enumerate(_empty_reads(rng, 40)):
        case.add(rows)
        case.add(_shape(rng, [5, 64, 65, 300, 513][i % 5], "fwd_dupid"))
    _run(case, min_pairs=100)


# ------------------------------------------------------------------------------------------------
# 5. working storage reused across reads
# ------------------------------------------------------------------------------------------------
def test_working_storage_reused_by_every_group():
    """more reads than thread groups in every tier (warp tier: 8 groups per block, 5 blocks per SM; block tier: 5
    blocks per SM; global-scratch tier: one block per SM), large and small sizes interleaved, so that every group takes
    reads of both orders of size and stale state of a larger earlier read would show"""
    n_sm = _n_sm()
    rng = np.random.default_rng(5)
    n_small, n_mid, n_big = 2 * 40 * n_sm + 13, 2 * 5 * n_sm + 7, 2 * n_sm + 5
    sizes = np.concatenate([rng.integers(2, 65, n_small), rng.integers(65, 513, n_mid), rng.integers(513, 901, n_big)])
    rng.shuffle(sizes)
    kinds = ["fwd", "rev", "fwd_jitter", "rev_jitter", "fwd_dupid", "rev_dupid", "sparse"]
    case = Case()
    for i, m in enumerate(sizes.tolist()):
        kind = kinds[i % len(kinds)]
        pos, start = _diag(rng, m, "-" if kind.startswith("rev") else "+", gap=(15, 1500),
                           jitter=40 if kind.endswith("jitter") else 0)
        rows = _shape(rng, m, kind) if kind == "sparse" else None
        if rows is None:
            ids = start.copy()
            if kind.endswith("dupid") and m > 3:
                j = rng.choice(m - 2, max(1, m // 12), replace=False)
                ids[j + 2] = ids[j]
            order = np.argsort(pos, kind="stable")
            rows = [(int(pos[t]), int(start[t]), int(ids[t])) for t in order]
        bad = [g for _, _, g in rows if rng.random() < 0.05] if i % 4 == 0 else []
        case.add(rows, bad_ids=bad)
    for rows in _empty_reads(rng, 50):
        case.add(rows)
    per_read, got = _run(case, min_pairs=100_000)
    assert len({n for _, n in got}) > n_small + n_mid


# ------------------------------------------------------------------------------------------------
# 6. width and length edges
# ------------------------------------------------------------------------------------------------
def _span_read(m, start_span, pos_span, s0, p0, strand="+"):
    """m rows from one corner of a (start_span x pos_span) box to the other, evenly spaced"""
    t = np.linspace(0.0, 1.0, m)
    start = s0 + np.round(t * start_span).astype(np.int64)
    d = np.round(t * pos_span).astype(np.int64)
    pos = p0 + (d if strand == "+" else pos_span - d)
    start[-1], pos[-1 if strand == "+" else 0] = s0 + start_span, p0 + pos_span
    order = np.argsort(pos, kind="stable")
    return [(int(pos[i]), int(start[i]), int(start[i])) for i in order]


@pytest.mark.parametrize("m", [6, 64, 65, 300, 513])
def test_span_switch_and_top_of_range(m):
    """start span and position span of exactly 2^28 - 1 and 2^28, each on its own; spans where the 32-bit form of the
    ratio test would overflow (11 * 2^32/11, 10 * 2^32/10); coordinates up to 2^32 - 1; pairs exactly on 0.9 and 1.1"""
    case = Case()
    B = 1 << 28
    for ss, ps in [(B - 1, B - 1), (B, B - 1), (B - 1, B), (B, B), (B, B + B // 12), (B + B // 12, B),
                   (U32 // 11 + 1, U32 // 11 + 1), (U32 // 10 + 2, U32 // 11 + 9), (U32 // 10 + 5, U32 // 10 + 5)]:
        for strand in ("+", "-"):
            case.add(_span_read(m, ss, ps, 1000, 7, strand), shift=False)
            case.add(_span_read(m, ss, ps, U32 - ss, U32 - ps, strand), shift=False)
    # two clusters 420M apart (over 2^32 / 11, under 2^29), rows of a cluster off each other's ratio (1.3): every passing
    # pair spans the whole read, so a 32-bit ratio test below the 2^28 switch would lose all of them
    for strand in ("+", "-"):
        d = 420_000_000
        rows = [(5000 + 1300 * i + d * c, 1000 + 1000 * i + d * c, 1000 + 1000 * i + d * c) for c in (0, 1) for i in range(max(2, m // 2))]
        if strand == "-":
            rows = [(U32 - 10 - p, s, g) for p, s, g in rows]
        case.add(sorted(rows), shift=False)
    # exact ratio boundaries: 10*dp == 11*ds and 9*ds == 10*dp fail, one step inside passes
    for s0, p0 in [(1000, 5), (U32 - 50_000_000, U32 - 60_000_000)]:
        rows = []
        for i in range(max(3, m // 3)):
            s = s0 + i * 100_000
            p = p0 + i * 100_000
            rows += [(p, s, s), (p + 11_000, s + 10_000, s + 10_000), (p + 9_000, s + 10_001, s + 10_001),
                     (p + 10_999, s + 10_002, s + 10_002)]
        case.add(sorted(rows), shift=False)
    _run(case, min_pairs=50)


@pytest.mark.parametrize("m", [5, 64, 65, 512, 513, 900])
def test_min_read_len_edge(m):
    rng = np.random.default_rng(m)
    case = Case()
    names = {}
    for kind in ("fwd", "rev_dupid"):
        for d in (0, -1, 1):
            names[(kind, d)] = case.add(_shape(rng, m, kind), rlen=123_457 + d)
    per_read, got = _run(case, minlen=123_457, min_pairs=m)
    valid = {n for _, n in got}
    assert all((names[(k, d)] in valid) == (d >= 0) for k, d in names)


# ------------------------------------------------------------------------------------------------
# 7. repeated IDs and repeated read positions
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["fwd_dupid", "rev_dupid"])
def test_repeated_ids_both_strands_every_tier(kind):
    rng = np.random.default_rng(sum(map(ord, kind)))
    case = Case()
    for m in [4, 17, 64, 65, 257, 512, 513, 800, 1500]:
        for _ in range(3):
            case.add(_shape(rng, m, kind))
    _run(case, min_pairs=1000)


def _same_position_reads():
    """the read of the multipos example: a 7-row forward diagonal, a row repeating the diagonal's ID 106000 at its read
    position 7000 but at a far start, then a 4-row diagonal from that row on; and variants"""
    diag = [(1000 * (k + 1), 100_000 + 1000 * k, 100_000 + 1000 * k) for k in range(7)]
    far = (7000, 900_000, 106_000)
    diag2 = [(7000 + 1000 * j, 900_000 + 1000 * j, 900_000 + 1000 * j) for j in range(1, 5)]
    out = [diag + [far] + diag2]
    # the same, reverse strand
    out.append([(20_000 - p, s, g) for p, s, g in out[0]][::-1])
    # different IDs at one position: ID X at its good position 7000 and at an off position; the off row's partner
    # is another ID's row sitting at X's good position
    x_off = (2500, 40_000, 106_000)
    y_at_good = (7000, 44_500, 777_000)
    out.append(diag + [x_off, y_at_good] + diag2[:2])
    # the same ID at one position with different starts, both with many edges (counts add up per position)
    out.append(diag + [(3000, 950_000, 102_000)] + [(3000 + 1000 * j, 950_000 + 1000 * j, 950_000 + 1000 * j) for j in range(1, 8)])
    return [sorted(r, key=lambda t: t[0]) for r in out]


def test_two_rows_at_one_read_position():
    rng = np.random.default_rng(17)
    case = Case()
    first = None
    for rows in _same_position_reads():
        n = case.add(rows)
        first = first or n
    for m in (6, 30, 64, 65, 200, 512, 513, 700):
        for t in range(12):
            case.add(_fuzz_read(rng, m, n_ids=int(rng.integers(2, m)) if t % 2 else None, pos_repeat=0.25))
    per_read, got = _run(case, min_pairs=1000)
    assert sum(n == first for _, n in got) == 11  # the far row keeps its 4 edges


def test_cli_process_by_contig_read_name_in_two_chunks(tmp_path):
    """a .sunkpos in which one read name occurs twice (two chunk files concatenated): the read's rows merge, and two of
    them share a read position.  inter_outs TSV and BED against the oracle."""
    from gavisunk_b200 import cli
    rows = []
    reads = _same_position_reads()
    for i, rr in enumerate(reads):
        rows += [(f"rd{i}", p, "chrA", s + 10_000_000 * i, g + 10_000_000 * i) for p, s, g in rr]
    # rd0 once more as a second chunk: its far row and second diagonal again (the first chunk keeps the first diagonal)
    dup = [r for r in rows if r[0] == "rd0" and r[3] >= 900_000]
    first = [r for r in rows if not (r[0] == "rd0" and r[3] >= 900_000)]
    rows = first + dup + [r for r in rows if r[0] == "rd0" and r[3] >= 900_000][:1]  # (an identical row: dropped)
    sp = tmp_path / "chrA_hap1.sunkpos"
    sp.write_text("".join(f"{r[0]}\t{r[1]}\t{r[2]}\t{r[3]}\t{r[4]}\n" for r in rows))
    rl = tmp_path / "hap1.rlen"
    rl.write_text("".join(f"rd{i}\t50000\n" for i in range(len(reads))))
    bs = tmp_path / "bad_sunks.txt"
    bs.write_text(f"chrA:{10_000_000 * 3 + 950_000 + 7000}\n")
    loc = tmp_path / "chrA_hap1.loc"
    loc.write_text("")
    tsv, bed = tmp_path / "out.tsv", tmp_path / "out.bed"
    assert cli.main(["process_by_contig", str(loc), str(sp), str(rl), str(bs), str(tsv), str(bed)]) == 0
    bad = {("chrA", 10_000_000 * 3 + 950_000 + 7000)}
    inter, exp_bed = O.process_by_contig(list(dict.fromkeys(rows)), {f"rd{i}": 50000 for i in range(len(reads))}, bad, "chrA")
    assert tsv.read_text() == "".join(f"{g}\t{n}\n" for g, n in inter)
    assert bed.read_text() == "".join(f"{c}\t{s}\t{e}\n" for c, s, e in sorted(exp_bed, key=lambda t: t[1]))
    assert sum(n == "rd0" for _, n in inter) == 11

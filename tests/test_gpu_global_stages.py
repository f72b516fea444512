"""The run-wide stages against plain references, at the shapes where they go wrong: the per-haplotype mode and the bad
groups (k_hist, k_hist_max, k_cnt_hist, k_mode, k_bad_flag), the contig-wide union-find and its multi-rank merge
(k_comp_pairs, k_comp_flatten, k_comp_merge_all), the per-root statistics (k_comp_stats), the intervals (k_iv_write) and
the gap scan of gvs_gaps.

The group table is a kmer.loc of distinct random 20-mers with group = start, loaded sorted or shuffled, so several
engines can share one dense index.  Reads are fed as kept rows (set_rows(1, ...)), every read on one contig with
pos = start - s0 + p0: such a read passes every pair test, so its validated IDs are all of its non-bad groups and it
joins them into one component.  Small and medium cases are compared with the oracle; at scale with scipy's connected
components and with the pairs the construction implies (the Python oracle is too slow there)."""
import math
from collections import Counter

import numpy as np
import pytest

import gavisunk_oracle as O

pytestmark = pytest.mark.gpu

K = 20
P0 = 1000       # read position of a read's first row
MINLEN = 1000   # every read is at least P0 + 1000 long


# ------------------------------------------------------------------------------------------------
# group tables
# ------------------------------------------------------------------------------------------------
def _random_kmers(rng, n):
    """n distinct random 20-mers as bytes"""
    codes = np.unique(rng.integers(0, 1 << (2 * K), int(n * 1.1) + 64, dtype=np.uint64))
    codes = rng.permutation(codes)[:n]
    assert len(codes) == n
    digits = (codes[:, None] >> (2 * np.arange(K - 1, -1, -1, dtype=np.uint64))) & np.uint64(3)
    buf = np.frombuffer(b"ACGT", np.uint8)[digits.astype(np.int64)].tobytes()
    return [buf[i * K:(i + 1) * K] for i in range(n)]


class Table:
    """groups (contig, start) of a kmer.loc with group = start; order: 'sorted', 'shuffled' or a permutation"""

    def __init__(self, rng, starts_per_contig):
        self.nc = len(starts_per_contig)
        self.names = [f"ctg{c}" for c in range(self.nc)]
        self.contig = np.concatenate([np.full(len(s), c, np.uint32) for c, s in enumerate(starts_per_contig)]).astype(np.uint32)
        self.start = np.concatenate([np.asarray(s, np.int64) for s in starts_per_contig]).astype(np.uint32)
        key = (self.contig.astype(np.uint64) << np.uint64(32)) | self.start.astype(np.uint64)
        assert len(np.unique(key)) == len(key)
        o = np.argsort(key, kind="stable")
        self.contig, self.start = self.contig[o], self.start[o]
        self.kmers = _random_kmers(rng, len(self.start))
        self.contig_len = np.array([min(int(self.start[self.contig == c].max()) + 1000, (1 << 32) - 1) if (self.contig == c).any()
                                    else 5000 for c in range(self.nc)], np.int64)

    def engine(self, rng, order="sorted"):
        from gavisunk_b200.engine import Engine
        n = len(self.start)
        perm = np.arange(n) if order == "sorted" else rng.permutation(n)
        loc = [(self.names[self.contig[i]], int(self.start[i]), self.kmers[i], int(self.start[i])) for i in perm]
        eng = Engine(K)
        eng.load_loc_text(list(self.kmers), loc, self.names)
        g = eng.groups()
        assert np.array_equal(g["contig"], self.contig[perm]) and np.array_equal(g["group"], self.start[perm])
        if order != "sorted" and n > 64:
            assert not _sorted_table(g), "the shuffled kmer.loc gave a sorted group table"
        return eng


def _sorted_table(g):
    key = (g["contig"].astype(np.uint64) << np.uint64(32)) | g["group"].astype(np.uint64)
    return bool(np.all(key[1:] > key[:-1]))


# ------------------------------------------------------------------------------------------------
# reads: flat rows (read, contig, start), rows of a read contiguous, on one contig, distinct increasing starts
# ------------------------------------------------------------------------------------------------
class Reads:
    def __init__(self, read, contig, start):
        self.read = np.asarray(read, np.int64)
        self.contig = np.asarray(contig, np.uint32)
        self.start = np.asarray(start, np.int64)
        n = len(self.read)
        assert n == 0 or (np.all(np.diff(self.read) >= 0) and self.read[0] >= 0)
        self.n_reads = int(self.read.max()) + 1 if n else 0
        first = np.ones(n, bool)
        first[1:] = self.read[1:] != self.read[:-1]
        head = np.maximum.accumulate(np.where(first, np.arange(n), 0))
        same = ~first
        assert np.all(self.contig[same] == self.contig[head[same]])       # one contig per read
        assert np.all(self.start[1:][same[1:]] > self.start[:-1][same[1:]])  # increasing starts
        self.pos = self.start - self.start[head] + P0
        assert n == 0 or self.pos.max() < (1 << 32) - 2000
        self.rlen = np.full(self.n_reads, P0 + 1000, np.int64)
        if n:
            np.maximum.at(self.rlen, self.read, self.pos + 1000)

    @staticmethod
    def of_pairs(contig, a, b):
        """2-row reads: one edge between groups a and b (starts) of contig each"""
        contig, a, b = (np.asarray(x, np.int64) for x in (contig, a, b))
        lo, hi = np.minimum(a, b), np.maximum(a, b)
        keep = lo != hi
        contig, lo, hi = contig[keep], lo[keep], hi[keep]
        m = len(lo)
        return Reads(np.repeat(np.arange(m), 2), np.repeat(contig, 2), np.stack([lo, hi], 1).ravel())

    @staticmethod
    def of_lists(reads):
        """reads = [(contig, [starts ...]), ...]"""
        r, c, s = [], [], []
        for i, (ctg, st) in enumerate(reads):
            st = sorted(set(int(x) for x in st))
            r += [i] * len(st)
            c += [ctg] * len(st)
            s += st
        return Reads(r, c, s)

    def subset(self, read_mask):
        """the reads where read_mask is set, renumbered densely"""
        keep = read_mask[self.read]
        new = np.cumsum(read_mask) - 1
        return Reads(new[self.read[keep]], self.contig[keep], self.start[keep])

    def feed(self, eng, nc, contig_hap=None):
        eng.set_reads_meta(np.maximum(self.rlen, 1).astype(np.uint32) if self.n_reads else np.zeros(1, np.uint32))
        eng.set_rows(1, self.read, self.pos, self.contig, self.start, self.start, n_contigs=nc)
        eng.set_contigs(np.zeros(nc, np.uint8) if contig_hap is None else contig_hap)


def _expected(reads, bad=frozenset()):
    """the pairs and intervals the construction implies, via scipy: (pairs as (read, contig, start) rows, intervals as
    (contig, start, end) rows in (contig, start) order, component labels of the present groups)"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    n = len(reads.read)
    if n == 0:
        return (np.zeros(0, np.int64),) * 3, [], None
    isbad = np.array([(int(c), int(s)) in bad for c, s in zip(reads.contig, reads.start)], bool) if bad else np.zeros(n, bool)
    ok = ~isbad
    per_read = np.bincount(reads.read[ok], minlength=reads.n_reads)
    val = ok & (per_read[reads.read] >= 2)
    pr, pc, ps = reads.read[val], reads.contig[val], reads.start[val]
    pairs = (pr, pc, ps)
    key = (pc.astype(np.uint64) << np.uint64(32)) | ps.astype(np.uint64)
    if len(key) == 0:
        return pairs, [], None
    uk, inv = np.unique(key, return_inverse=True)
    nxt = np.nonzero(pr[1:] == pr[:-1])[0]
    g = coo_matrix((np.ones(len(nxt)), (inv[nxt], inv[nxt + 1])), shape=(len(uk), len(uk)))
    ncomp, lab = connected_components(g, directed=False)
    uc = (uk >> np.uint64(32)).astype(np.int64)
    us = (uk & np.uint64(0xFFFFFFFF)).astype(np.int64)
    cnt = np.bincount(lab, minlength=ncomp)
    mn = np.full(ncomp, 1 << 40, np.int64)
    mx = np.full(ncomp, -1, np.int64)
    np.minimum.at(mn, lab, us)
    np.maximum.at(mx, lab, us)
    ctg = np.zeros(ncomp, np.int64)
    ctg[lab] = uc
    iv = sorted((int(ctg[i]), int(mn[i]), int(mx[i])) for i in range(ncomp) if cnt[i] >= 3)
    return pairs, iv, (uk, lab)


def _oracle(reads, table, bad=frozenset()):
    """pairs and intervals of the oracle's restatement of process-by-contig_lowmem_AR.py, contig by contig"""
    rname = lambda r: f"r{int(r):09d}"
    rlen = {rname(r): int(reads.rlen[r]) for r in range(reads.n_reads)}
    by_ctg = {}
    for r, p, c, s in zip(reads.read, reads.pos, reads.contig, reads.start):
        by_ctg.setdefault(int(c), []).append((rname(r), int(p), table.names[c], int(s), int(s)))
    badn = {(table.names[c], s) for c, s in bad}
    pairs, iv = [], []
    for c in range(table.nc):
        inter, bed = O.process_by_contig(by_ctg[c], rlen, badn, table.names[c], minlen=MINLEN) if c in by_ctg else (None, None)
        pairs += [(int(nm[1:]), c, g) for g, nm in inter or []]
        iv += [(c, s, e) for _, s, e in bed or []]
    pairs.sort(key=lambda t: t[0])  # stable: per read in vertex order
    return pairs, iv


def _gaps_oracle(table, iv):
    fai = [(table.names[c], int(table.contig_len[c])) for c in range(table.nc)]
    beds = {}
    for c, s, e in iv:
        beds.setdefault(table.names[c], []).append((s, e))
    return O.get_gaps(fai, beds)


def _run(eng, reads, table, bad=frozenset()):
    """validation -> local forest -> intervals -> gaps of one engine"""
    reads.feed(eng, table.nc)
    if bad:
        cs = sorted(bad)
        eng.bad_set([c for c, _ in cs], [s for _, s in cs])
    eng.validate(MINLEN)
    eng.components_local()
    return _results(eng, table)


def _results(eng, table):
    iv = eng.intervals()
    gaps, nodata = eng.gaps(table.contig_len.astype(np.uint32))
    got_iv = list(zip(iv["contig"].tolist(), iv["start"].tolist(), iv["end"].tolist()))
    got_gaps = [(table.names[c], s, e) for c, s, e in zip(gaps["contig"].tolist(), gaps["start"].tolist(), gaps["end"].tolist())]
    got_nd = [(table.names[c], 0, int(table.contig_len[c])) for c in nodata.tolist()]
    return got_iv, got_gaps, got_nd


def _check_pairs(eng, want):
    p = eng.pairs()
    if isinstance(want, tuple):
        r, c, s = want
        assert np.array_equal(p["read"], r) and np.array_equal(p["contig"], c) and np.array_equal(p["group"], s)
    else:
        assert list(zip(p["read"].tolist(), p["contig"].tolist(), p["group"].tolist())) == want
    g = eng.groups()
    assert np.array_equal(g["contig"][p["gidx"]], p["contig"]) and np.array_equal(g["group"][p["gidx"]], p["group"])
    return len(p["read"])


def _max_roots_per_warp(eng, comp):
    """largest number of distinct component roots (smallest group index of the component) among the 32 groups of one warp
    of k_comp_stats, from the expected components"""
    uk, lab = comp
    g = eng.groups()
    key = (g["contig"].astype(np.uint64) << np.uint64(32)) | g["group"].astype(np.uint64)
    o = np.argsort(key)
    gi = o[np.searchsorted(key[o], uk)]   # group index of every present group
    root = np.full(lab.max() + 1, 1 << 40, np.int64)
    np.minimum.at(root, lab, gi)
    warp = gi // 32
    pairs = np.unique(np.stack([warp, root[lab]], 1), axis=0)
    return int(np.bincount(pairs[:, 0]).max())


ORDERS = ["sorted", "shuffled"]


def _check_case(table, reads, rng, bad=frozenset(), oracle=False, orders=ORDERS, rows_table=True):
    """one case on a sorted and a shuffled kmer.loc and on a rows-derived table: pairs, intervals in (contig, start)
    order and gaps straight after them, against scipy (and the oracle); returns the expected components"""
    pairs, iv, comp = _expected(reads, bad)
    if oracle:
        opairs, oiv = _oracle(reads, table, bad)
        assert oiv == iv
        assert opairs == list(zip(*(x.tolist() for x in pairs)))
    want_gaps = _gaps_oracle(table, iv)
    engines = [table.engine(rng, o) for o in orders]
    if rows_table:
        from gavisunk_b200.engine import Engine
        e = Engine(K)
        e.contig_names = list(table.names)
        engines.append(e)
    for eng in engines:
        got = _run(eng, reads, table, bad)
        if len(pairs[0]):
            _check_pairs(eng, pairs)
        assert got[0] == iv
        assert (got[1], got[2]) == want_gaps
        eng.close()
    return pairs, iv, comp


# ------------------------------------------------------------------------------------------------
# components, intervals, gaps
# ------------------------------------------------------------------------------------------------
def test_chain_unioned_in_shuffled_order():
    """one chain of 2*10^5 groups, one 2-row read per link, reads in random order: the longest paths the union-find has
    to walk, with the hooks coming from everywhere at once"""
    rng = np.random.default_rng(1)
    n = 200_000
    starts = np.sort(rng.choice(np.arange(100, 60 * n), n, replace=False))
    table = Table(rng, [starts])
    o = rng.permutation(n - 1)
    reads = Reads.of_pairs(np.zeros(n - 1), starts[o], starts[o + 1])
    _, iv, _ = _check_case(table, reads, rng)
    assert iv == [(0, int(starts[0]), int(starts[-1]))]


def test_stars_on_hubs():
    """a star of 10^5 edges on one hub (every union contends for the hub's root), a star whose leaves lie on both sides
    of its hub, and small stars next to it"""
    rng = np.random.default_rng(2)
    c0 = np.sort(rng.choice(np.arange(0, 2_000_000), 20_000, replace=False))
    c1 = np.sort(rng.choice(np.arange(0, 8_000_000), 100_500, replace=False))
    table = Table(rng, [c0, c1])
    hub1 = c1[77_777]
    leaves1 = np.setdiff1d(c1, [hub1])[:100_000]
    hub0 = c0[10_000]
    leaves0 = c0[5000:15_000][c0[5000:15_000] != hub0]
    small = [(c0[i], c0[i + 1: i + 4]) for i in range(16_000, 19_000, 10)]
    a = np.concatenate([np.full(len(leaves1), hub1), np.full(len(leaves0), hub0)] + [np.full(3, h) for h, _ in small])
    b = np.concatenate([leaves1, leaves0] + [lv for _, lv in small])
    c = np.concatenate([np.ones(len(leaves1)), np.zeros(len(leaves0) + 3 * len(small))])
    o = rng.permutation(len(a))
    reads = Reads.of_pairs(c[o], a[o], b[o])
    assert int(np.sum((reads.contig == 1) & (reads.start == hub1))) == 100_000
    _, iv, _ = _check_case(table, reads, rng)
    assert (1, int(leaves1.min()), int(leaves1.max())) in iv and len(iv) == 2 + len(small)


@pytest.mark.parametrize("p", [2, 3, 7, 33])
def test_interleaved_components(p):
    """group g of a contig in component g mod p: nested, overlapping intervals, and every warp of k_comp_stats sees
    min(p, 32) roots.  A second contig holds the same starts: neighbours in the index, never joined."""
    rng = np.random.default_rng(10 + p)
    n = 20_000   # a multiple of 32: no warp straddles the two contigs
    starts = np.arange(n, dtype=np.int64) * 50 + 7
    table = Table(rng, [starts, starts])
    j = np.arange(n - p)
    c = np.concatenate([np.zeros(len(j)), np.ones(len(j))])
    a = np.concatenate([starts[j], starts[j]])
    b = np.concatenate([starts[j + p], starts[j + p]])
    o = rng.permutation(len(a))
    reads = Reads.of_pairs(c[o], a[o], b[o])
    _, iv, comp = _check_case(table, reads, rng, rows_table=(p == 7))
    assert len(iv) == 2 * p
    eng = table.engine(rng, "sorted")
    roots = _max_roots_per_warp(eng, comp)
    eng.close()
    assert roots == min(p, 32)


def test_sizes_two_and_three_nested_adjacent_and_edges_of_the_start_range():
    """components of exactly 2 groups (no interval) next to ones of exactly 3; components nested inside a long one;
    adjacent intervals (a gap (e, e)); groups at start 0 and 2^32-1; a contig whose groups never occur in a read; bad
    groups inside reads -- against scipy and the oracle"""
    rng = np.random.default_rng(3)
    top = (1 << 32) - 1
    c0 = np.arange(0, 200_000, 100, dtype=np.int64)
    c1 = np.concatenate([[0], np.arange(5000, 6000, 10), np.arange(7000, 7010), [top - 4000, top - 2000, top]])
    c2 = np.arange(1000, 50_000, 500, dtype=np.int64)
    c3 = np.arange(10, 3000, 30, dtype=np.int64)
    table = Table(rng, [c0, c1, c2, c3])
    reads = []
    for i in range(0, len(c0) - 10, 10):   # contig 0: a component of 2 groups, then one of 3
        reads += [(0, c0[i:i + 2]), (0, c0[i + 3:i + 5]), (0, c0[i + 4:i + 6])]
    reads += [(3, [c3[0], c3[50]]), (3, [c3[50], c3[99]])]                  # contig 3: a long component ...
    reads += [(3, c3[10:14]), (3, [c3[20], c3[21]]), (3, [c3[21], c3[22]])]  # ... around short ones
    reads += [(1, [0, 5000, 5010]), (1, [5010, 5020]), (1, [5030, 5040, 5050]), (1, [5100, 5110, 5120, 5130])]
    reads += [(1, [7000, 7001, 7002]), (1, [7003, 7004]), (1, [7004, 7005])]  # adjacent: [7000, 7002], [7003, 7005]
    reads += [(1, [top - 4000, top - 2000]), (1, [top - 2000, top])]
    rd = Reads.of_lists(reads)
    bad = {(0, int(c0[5])), (0, int(c0[15])), (3, int(c3[11]))}
    _, iv, _ = _check_case(table, rd, rng, bad=bad, oracle=True)
    assert (1, 0, 5020) in iv and (1, top - 4000, top) in iv and not any(c == 2 for c, _, _ in iv)
    assert (1, 7000, 7002) in iv and (1, 7003, 7005) in iv
    assert (3, int(c3[0]), int(c3[99])) in iv and (3, int(c3[10]), int(c3[13])) in iv and (3, int(c3[20]), int(c3[22])) in iv
    assert (0, int(c0[3]), int(c0[5])) not in iv and (0, int(c0[13]), int(c0[15])) not in iv and (0, int(c0[23]), int(c0[25])) in iv


def test_rows_repeating_one_id_add_no_vertex():
    """rows-derived table (no database): a read whose only validated ID is one group seen at two starts joins nothing"""
    from gavisunk_b200.engine import Engine
    rows = []  # (read, pos, contig, start, ID)
    rows += [("r000000000", 1000, "c0", 5000, 5000), ("r000000000", 2000, "c0", 6000, 5000), ("r000000000", 900_000, "c0", 7000, 7000)]
    rows += [("r000000001", 1000, "c0", 8000, 8000), ("r000000001", 2000, "c0", 9000, 9000), ("r000000001", 3000, "c0", 10000, 10000)]
    rows += [("r000000002", 1000, "c0", 7000, 7000), ("r000000002", 4000, "c0", 10000, 10000)]
    rlen = {f"r{i:09d}": 1_000_000 for i in range(3)}
    inter, bed = O.process_by_contig(rows, rlen, set(), "c0", minlen=MINLEN)
    assert (5000, "r000000000") in inter and bed == [("c0", 7000, 10000)]
    eng = Engine(K)
    eng.contig_names = ["c0"]
    eng.set_reads_meta(np.full(3, 1_000_000, np.uint32))
    eng.set_rows(1, [int(r[0][1:]) for r in rows], [r[1] for r in rows], np.zeros(len(rows)), [r[3] for r in rows],
                 [r[4] for r in rows], n_contigs=1)
    eng.set_contigs([0])
    eng.validate(MINLEN)
    p = eng.pairs()
    assert [(int(g), f"r{int(r):09d}") for g, r in zip(p["group"], p["read"])] == inter
    eng.components_local()
    iv = eng.intervals()
    assert [("c0", int(s), int(e)) for s, e in zip(iv["start"], iv["end"])] == bed
    eng.close()


def test_groups_in_first_appearance_order_give_sorted_intervals():
    """groups of contig 1 appear first, and a component's first-seen group is not its leftmost: intervals() still comes
    in (contig, start) order and gaps() sees every gap, on every kind of group table"""
    rng = np.random.default_rng(4)
    c = np.arange(0, 10_000, 100)
    table = Table(rng, [c, c])
    reads = [(1, c[60:64]), (1, c[20:22]), (0, c[70:74]), (1, [c[15], c[20]]), (0, c[40:42]), (0, c[5:9]), (0, [c[35], c[40]])]
    rd = Reads.of_lists(reads)
    _, iv, _ = _check_case(table, rd, rng, oracle=True)
    assert iv == [(0, 500, 800), (0, 3500, 4100), (0, 7000, 7300), (1, 1500, 2100), (1, 6000, 6300)]
    from gavisunk_b200.engine import Engine
    eng = Engine(K)
    eng.contig_names = list(table.names)
    rd.feed(eng, table.nc)
    assert not _sorted_table(eng.groups())   # the rows-derived table above was unsorted
    eng.close()


def test_several_million_pairs():
    """random short-range edges plus hubs over 4.2*10^5 groups on 6 contigs, reads in random order: more than 10^6
    validated pairs in one run"""
    rng = np.random.default_rng(5)
    per = 70_000
    st = np.stack([np.sort(rng.choice(np.arange(0, 30 * per), per, replace=False)) for _ in range(6)])
    table = Table(rng, list(st))
    m = 1_300_000
    c = rng.integers(0, 6, m)
    i = rng.integers(0, per - 40, m)
    a, b = st[c, i], st[c, i + rng.integers(1, 40, m)]
    hubs = rng.integers(0, per, 6)
    hc = rng.integers(0, 6, 200_000)
    ha, hb = st[hc, hubs[hc]], st[hc, rng.integers(0, per, len(hc))]
    o = rng.permutation(m + len(hc))
    reads = Reads.of_pairs(np.concatenate([c, hc])[o], np.concatenate([a, ha])[o], np.concatenate([b, hb])[o])
    pairs, _, _ = _check_case(table, reads, rng, orders=["shuffled"], rows_table=False)
    assert len(pairs[0]) > 2_000_000


# ------------------------------------------------------------------------------------------------
# forest merge across ranks
# ------------------------------------------------------------------------------------------------
def _merge(table, reads, parts, rng, order):
    """engines holding the read subsets `parts` (boolean masks over reads), one shared dense index; the forests gathered
    with torch.stack of aliased arrays and merged on every rank"""
    import torch
    from gavisunk_b200.parallel import alias_device_array
    dev = torch.device("cuda", 0)
    engines = [table.engine(np.random.default_rng(99), order) for _ in parts]
    ng = engines[0].db_groups()
    forests = []
    for e, mask in zip(engines, parts):
        sub = reads.subset(mask)
        sub.feed(e, table.nc)
        e.validate(MINLEN)
        forests.append(e.components_local())
        e.sync()
    gathered = torch.stack([alias_device_array(f, ng, "<i4", dev) for f in forests])
    torch.cuda.synchronize()
    res = []
    for r, e in enumerate(engines):
        e.components_merge_all(int(gathered.data_ptr()), len(engines), r)
        res.append(_results(e, table))
    for e in engines:
        e.close()
    return res


@pytest.mark.parametrize("R", [2, 3, 8])
@pytest.mark.parametrize("split", ["round_robin", "one_idle", "random"])
def test_merge_of_rank_forests(R, split):
    """every rank's intervals and gaps after components_merge_all equal one engine holding every read, and the oracle"""
    rng = np.random.default_rng(100 + R)
    n = 3000
    starts = [np.arange(0, 50 * n, 50), np.sort(rng.choice(np.arange(10, 50 * n), n, replace=False))]
    table = Table(rng, starts)
    # contig 0: one chain; contig 1: random short edges (many components, some of 2 groups)
    j = np.arange(n - 1)
    e1 = rng.integers(0, n - 8, 1500)
    reads = Reads.of_pairs(np.concatenate([np.zeros(n - 1), np.ones(len(e1))]),
                           np.concatenate([starts[0][j], starts[1][e1]]),
                           np.concatenate([starts[0][j + 1], starts[1][e1 + rng.integers(1, 8, len(e1))]]))
    nr = reads.n_reads
    if split == "round_robin":
        owner = np.arange(nr) % R            # no rank holds two neighbouring links of the chain
    elif split == "one_idle":
        owner = rng.integers(1, R, nr) if R > 1 else np.zeros(nr, np.int64)
    else:
        owner = rng.integers(0, R, nr)
    parts = [owner == r for r in range(R)]
    if split == "one_idle":
        assert not parts[0].any()
    _, iv, _ = _expected(reads)
    oiv = _oracle(reads, table)[1]
    assert oiv == iv
    want = (iv, *_gaps_oracle(table, iv))
    for order in ORDERS:
        one = table.engine(rng, order)
        assert _run(one, reads, table) == want
        one.close()
        for got in _merge(table, reads, parts, rng, order):
            assert got == want


# ------------------------------------------------------------------------------------------------
# gaps through set_intervals
# ------------------------------------------------------------------------------------------------
def test_gaps_of_given_intervals():
    """identical, nested, touching (start == previous end) and adjacent (start == previous end + 1) intervals, in random
    input order, and many contigs without any interval, against the oracle and a per-base coverage count"""
    from gavisunk_b200.engine import Engine
    rng = np.random.default_rng(6)
    nc = 400
    lens = rng.integers(2000, 6000, nc)
    ivs = []
    for c in range(0, nc, 5):   # 4 of 5 contigs have no interval
        base = [(100, 400), (100, 400), (150, 300), (400, 700), (701, 900), (950, 1000), (1000, 1001), (1003, 1500)]
        ivs += [(c, s, e) for s, e in base]
        for _ in range(rng.integers(0, 12)):
            s = int(rng.integers(0, lens[c] - 200))
            ivs.append((c, s, s + int(rng.integers(1, 200))))
    o = rng.permutation(len(ivs))
    ivs = [ivs[i] for i in o]
    eng = Engine(K)
    eng.set_intervals([t[0] for t in ivs], [t[1] for t in ivs], [t[2] for t in ivs], nc)
    gaps, nodata = eng.gaps(lens.astype(np.uint32))
    names = [f"ctg{c}" for c in range(nc)]
    beds = {}
    for c, s, e in ivs:
        beds.setdefault(names[c], []).append((s, e))
    eg, en = O.get_gaps([(names[c], int(lens[c])) for c in range(nc)], beds)
    assert [(names[c], s, e) for c, s, e in zip(gaps["contig"].tolist(), gaps["start"].tolist(), gaps["end"].tolist())] == eg
    assert [(names[c], 0, int(lens[c])) for c in nodata.tolist()] == en
    assert ("ctg0", 900, 949) in eg and ("ctg0", 700, 700) in eg and ("ctg0", 1001, 1002) in eg
    # per-base coverage: a gap is a maximal run of uncovered bases [e, s) between covered ones, written (e, s - 1)
    for c in range(0, nc, 5):
        cov = np.zeros(int(lens[c]) + 2, np.int64)
        for cc, s, e in ivs:
            if cc == c:
                cov[s] += 1
                cov[e] -= 1
        cov = np.cumsum(cov) > 0
        first, last = int(np.argmax(cov)), len(cov) - int(np.argmax(cov[::-1]))
        unc = ~cov[first:last]
        edges = np.diff(np.concatenate([[0], unc.astype(np.int8), [0]]))
        runs = list(zip((np.nonzero(edges == 1)[0] + first).tolist(), (np.nonzero(edges == -1)[0] + first).tolist()))
        assert [(names[c], a, b - 1) for a, b in runs] == [g for g in eg if g[0] == names[c]]


# ------------------------------------------------------------------------------------------------
# mode and bad groups
# ------------------------------------------------------------------------------------------------
def _bad_reference(counts, code):
    """counts: {(contig, start): rows}; code[contig]: 0 / 1 own haplotype, 2 / 3 other-haplotype contig under the limit
    of haplotype 0 / 1, 255 neither.  The mode in plain Counter terms, the limit in exact integer form."""
    modes = []
    for h in (0, 1):
        freq = Counter(v for (c, _), v in counts.items() if code[c] == h and v > 0)
        top = max(freq.values()) if freq else 0
        modes.append(min(v for v, f in freq.items() if f == top) if freq else 0)
    over = lambda v, m: m > 0 and v > m and (v - m) ** 2 > 16 * m
    bad = set()
    for (c, s), v in counts.items():
        h = code[c]
        if v > 0 and h in (0, 1) and (over(v, modes[h]) or v < 2):
            bad.add((c, s))
        elif v > 0 and h in (2, 3) and over(v, modes[h - 2]):
            bad.add((c, s))
    return modes, bad


def _bad_case(counts_per_contig, code, rng, order="shuffled", parts=1):
    """rows with the designed per-group counts; returns (modes, bad set, hist) of the engine after checking them"""
    starts = [np.arange(len(cnts), dtype=np.int64) * 40 + 3 for cnts in counts_per_contig]
    table = Table(rng, starts)
    counts = {}
    for c, cnts in enumerate(counts_per_contig):
        for s, v in zip(starts[c], cnts):
            counts[(c, int(s))] = int(v)
    keys = list(counts)
    rc = np.repeat([k[0] for k in keys], [counts[k] for k in keys]).astype(np.uint32)
    rs = np.repeat([k[1] for k in keys], [counts[k] for k in keys]).astype(np.uint32)
    o = rng.permutation(len(rc))
    rc, rs = rc[o], rs[o]
    eng = table.engine(rng, order)
    eng.set_reads_meta(np.full(1, 20000, np.uint32))
    eng.set_contigs(np.asarray(code, np.uint8))
    for i, sl in enumerate(np.array_split(np.arange(len(rc)), parts)):
        eng.set_rows(1, np.zeros(len(sl), np.uint32), np.arange(len(sl)), rc[sl], rs[sl], rs[sl], n_contigs=table.nc)
        eng.group_hist(accumulate=i > 0)
    eng.bad_groups()
    g = eng.groups(with_hist=True)
    got_counts = {(int(c), int(s)): int(v) for c, s, v in zip(g["contig"], g["group"], g["count"])}
    assert got_counts == counts
    want_modes, want_bad = _bad_reference(counts, code)
    bl = eng.bad_list()
    got_bad = {(int(g["contig"][i]), int(g["group"][i])) for i in bl}
    assert len(got_bad) == len(bl)
    assert eng.modes == want_modes
    assert got_bad == want_bad
    # the oracle's statement of badsunks_AR.py, per haplotype whose contigs have groups
    names = table.names
    for h in (0, 1):
        own = {names[c] for c in range(table.nc) if code[c] == h}
        rows = [("r", 0, names[c], s, s) for (c, s), v in counts.items() if code[c] in (h, 2 + h) for _ in range(v)]
        if any(code[c] == h and v > 0 for (c, _), v in counts.items()):
            ob, om = O.bad_sunks_one_hap(rows, own)
            assert om == want_modes[h]
            assert ob == {(names[c], s) for c, s in want_bad if code[c] in (h, 2 + h)}
    eng.close()
    return want_modes, want_bad, counts


def test_mode_ties_across_the_shared_bins():
    """equal top frequency at 2047 (privatised shared bins) and 2048 (global atomics): the smaller count wins either way
    round; then 2048 alone on top"""
    rng = np.random.default_rng(7)
    a = [2047] * 3 + [2048] * 3 + [5, 5, 9, 9, 1, 3000, 2100]
    modes, _, counts = _bad_case([a, [7] * 4 + [2] * 4 + [1, 40]], [0, 1], rng)
    assert modes == [2047, 2]
    b = [2047] * 3 + [2048] * 4 + [10, 10, 10, 11]
    modes, bad, counts = _bad_case([b, [3, 3]], [0, 1], rng)
    assert modes == [2048, 3] and max(counts.values()) >= 2048
    # the mode is the largest count of the run (the top bin of the count table)
    modes, bad, counts = _bad_case([[12] * 5 + [3, 4, 1], [6, 6, 2]], [0, 1], rng)
    assert modes == [12, 6] and max(counts.values()) == 12


@pytest.mark.parametrize("m", [9, 16, 2500, 4096])
def test_limit_at_perfect_square_modes(m):
    """mode m a perfect square: m + 4*sqrt(m) is an integer; a count exactly there stays, one above is bad; count 1 is
    bad, count 2 is not"""
    rng = np.random.default_rng(m)
    lim = m + 4 * math.isqrt(m)
    own = [m] * 6 + [lim, lim, lim + 1, 1, 2, m - 1, m + 1]
    other = [lim, lim + 1, 1]
    modes, bad, counts = _bad_case([own, [4] * 3, other, other, other], [0, 1, 2, 3, 255], rng, parts=3)
    assert modes == [m, 4]
    assert {counts[k] for k in bad if k[0] == 0} == {lim + 1, 1}
    assert {counts[k] for k in bad if k[0] == 2} == {lim + 1}   # other-haplotype contig: the upper limit only
    assert {counts[k] for k in bad if k[0] == 3} == {lim, lim + 1}   # haplotype 1's limit: 4 + 4*2 = 12 < lim
    assert not any(k[0] == 4 for k in bad)                        # neither haplotype


def test_haplotype_without_groups_and_a_huge_group():
    """no group on haplotype 1's contigs (mode 0: nothing is over its limit), and one group of ~10^6 rows (a large count
    table for the mode)"""
    rng = np.random.default_rng(8)
    modes, bad, counts = _bad_case([[30] * 50 + [1_000_003, 31, 1], [5, 90, 1]], [0, 3], rng, order="sorted")
    assert modes == [30, 0]
    assert max(counts.values()) > 10 ** 6
    assert {counts[k] for k in bad} == {1_000_003, 1}   # contig 1 answers to haplotype 1's limit, which is none


def test_accumulated_histogram_equals_one_call():
    """group_hist(accumulate=True) over three set_rows calls gives the histogram and bad groups of one call"""
    rng = np.random.default_rng(9)
    cnts = rng.integers(1, 60, 3000).tolist() + [2500, 2049, 2048]
    r1 = _bad_case([cnts, cnts[::-1]], [0, 1], rng, parts=1)
    r3 = _bad_case([cnts, cnts[::-1]], [0, 1], rng, parts=3)
    assert r1 == r3

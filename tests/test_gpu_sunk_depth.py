"""SUNK hit depth (Engine.sunk_depth / depth / depth_runs, csrc/depth.cu; `fused --sunk-depth`, `cli sunk_depth`): per-group
counts and runs against the CPU oracle (tests/sunk_depth_oracle.py) over one vs several batches and contexts, hand-set
rows, known answers on an assembly with a planted interspersed collapse, tandem collapse and deletion, and the
reference's bundled samples.  No reference counterpart."""
import os
import sys
import threading

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

import sunk_depth_oracle as O

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

SPLITS = [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]]
CONTIGS = (300000, 200000)
# Per haplotype.  The 1.75x bound is 12.5 % below the 2x of an interspersed collapse, and the hits of a group follow the
# reads covering it (about Poisson, correlated over a read length): at 30x a 2-copy stretch has ~60 reads and dips below
# the bound in stretches; at 200x (~400 reads, sd 5 %) it stays 2.5 sd above, and single-copy groups stay far from 1.75x
# and 0.25x.
COV = 200.0
MEDIAN_LEN, MAX_LEN = 30000, 120000
COPY = (40000, 80000)      # hap 1: this segment of contig 0 is also inserted into contig 1 at COPY_AT
COPY_AT = 150000
TANDEM = (180000, 188000)  # hap 1: this unit of contig 0 is repeated 3 times in place
DELETED = (50000, 80000)   # hap 1: deleted from contig 1
SLACK = 2000


def _planted(seed=71, edit=True):
    """a synthetic diploid assembly (database built from it unedited) and 12 chunks of reads (6 per haplotype) simulated
    from its contigs, with the three edits made to hap 1 when `edit`.  Reads are drawn from every contig flanked by MAX_LEN
    random bases on both sides that the assembly lacks, as a genome goes on past an assembly's contig ends: drawn from
    the bare contigs, reads up to MAX_LEN long would thin out towards the ends (rightly called depleted) and cover a short
    contig's interior more deeply than a long one's."""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    eng = Engine(20)
    wl = W.make_assembly(eng, list(CONTIGS), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    W.build_db(eng, wl)
    asm = wl.asm.cpu().numpy()
    off = wl.contig_off.cpu().numpy()
    seqs = [asm[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(wl.contig_names))]
    if edit:
        c0, c1 = seqs[0], seqs[1]
        unit = c0[TANDEM[0]:TANDEM[1]]
        seqs[0] = c0[:TANDEM[1]] + unit + unit + c0[TANDEM[1]:]
        seqs[1] = c1[:DELETED[0]] + c1[DELETED[1]:COPY_AT] + c0[COPY[0]:COPY[1]] + c1[COPY_AT:]
    nc = len(CONTIGS)
    chunks, chunk_hap = [], []
    rng = np.random.default_rng(seed + 1)
    flank = lambda: np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, MAX_LEN)].tobytes()
    seqs = [flank() + q + flank() for q in seqs]
    for hap in range(2):
        contigs = [(wl.contig_names[hap * nc + i], seqs[hap * nc + i]) for i in range(nc)]
        want = COV * sum(len(s) for _, s in contigs)
        lengths = []
        while sum(lengths) < want:
            lengths.append(int(min(MAX_LEN, max(1000, rng.lognormal(np.log(MEDIAN_LEN), 0.6)))))
        reads = S.simulate(contigs, lengths, seed + 10 + hap, f"h{hap + 1}_")
        chunks += S.split_round_robin(reads, 6)
        chunk_hap += [hap] * 6
    return eng, wl, chunks, np.asarray(chunk_hap, np.uint8)


def _host_batches(chunks, chunk_hap, groups):
    out = []
    for g in groups:
        reads = [r for c in g for r in chunks[c]]
        off = np.zeros(len(reads) + 1, np.uint64)
        off[1:] = np.cumsum([len(s) for _, s in reads])
        cf = np.cumsum([0] + [len(chunks[c]) for c in g]).astype(np.uint64)
        out.append((np.frombuffer(b"".join(s for _, s in reads), np.uint8), off, cf, chunk_hap[g]))
    return out


def _binds(hb):
    return [(lambda e, b=b: e.set_reads(b[0], b[1], b[2], b[3])) for b in hb]


def _run(eng, wl, hb, **kw):
    """run_batches with the depth stage; -> the match rows of every batch as oracle tuples (run-wide read, contig, start)"""
    rows = []

    def on_batch(e, b, base):
        r0 = e.rows(0)
        rows.extend(zip((r0["read"].astype(np.int64) + base).tolist(), r0["contig"].tolist(), r0["group"].tolist()))
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=3000, on_batch=on_batch, sunk_depth=True, **kw)
    return rows


def _tables(eng, contig_len, allreduce=None):
    gt = eng.groups()
    groups = list(zip(gt["contig"].tolist(), gt["group"].tolist()))
    dp = eng.depth(allreduce=allreduce)
    rn = eng.depth_runs(contig_len)
    runs = [tuple(int(rn[c][i]) for c in eng.DEPTH_COLUMNS) for i in range(len(rn["contig"]))]
    return gt, groups, dp, rn, runs


def _oracle(groups, match_rows, kept_rows, contig_len):
    cnt = O.counts(match_rows, groups)
    kept = {g: 0 for g in groups}
    for c, s in kept_rows:
        kept[(c, s)] += 1
    runs = O.runs({g: cnt[g] + (kept[g],) for g in groups}, [(str(i), int(l)) for i, l in enumerate(contig_len)])
    return cnt, kept, runs


def _check(eng, wl, match_rows):
    gt, groups, dp, rn, runs = _tables(eng, wl.contig_len)
    k1 = eng.rows(1)
    cnt, kept, want_runs = _oracle(groups, match_rows, zip(k1["contig"].tolist(), k1["group"].tolist()), wl.contig_len)
    assert [(int(h), int(r)) for h, r in zip(dp["hits"], dp["reads"])] == [cnt[g] for g in groups]
    assert dp["kept"].tolist() == [kept[g] for g in groups]
    assert runs == want_runs
    return gt, dp, rn


def _calls(eng, wl, gt, dp, hap):
    from gavisunk_b200 import cli
    hc = [i for i, h in enumerate(wl.contig_hap) if h == hap]
    calls, _ = cli.depth_calls(gt["contig"], gt["group"], dp["hits"], dp["reads"], dp["sunks"], eng.bad_list(), hc, wl.contig_len)
    groups = list(zip(gt["contig"].tolist(), gt["group"].tolist()))
    d = lambda col: dict(zip(groups, dp[col].tolist()))
    bad = {groups[i] for i in eng.bad_list().tolist()}
    assert calls == O.calls(hc, [(str(i), int(l)) for i, l in enumerate(wl.contig_len)], d("hits"), d("reads"), d("sunks"), bad)[0]
    return calls


@pytest.fixture(scope="module")
def planted():
    eng, wl, chunks, chunk_hap = _planted()
    return dict(eng=eng, wl=wl, chunks=chunks, chunk_hap=chunk_hap, calls={})


@pytest.mark.parametrize("split", SPLITS)
def test_counts_and_runs_equal_oracle(planted, split):
    eng, wl = planted["eng"], planted["wl"]
    rows = _run(eng, wl, _host_batches(planted["chunks"], planted["chunk_hap"], split))
    gt, dp, _ = _check(eng, wl, rows)
    assert int(dp["hits"].sum()) == len(rows) and (dp["reads"] < dp["hits"]).any() and (dp["sunks"] > 0).all()
    planted["calls"][len(split)] = [_calls(eng, wl, gt, dp, h) for h in range(2)]
    assert planted["calls"][len(split)] == next(iter(planted["calls"].values()))


def test_planted_events_are_called(planted):
    """one call per edit, of its kind, copies and tandem flag, both ends within SLACK; no other call"""
    eng, wl = planted["eng"], planted["wl"]
    if not planted["calls"]:
        _run(eng, wl, _host_batches(planted["chunks"], planted["chunk_hap"], SPLITS[0]))
        gt, _, _, _, _ = _tables(eng, wl.contig_len)
        planted["calls"][1] = [_calls(eng, wl, gt, eng.depth(), h) for h in range(2)]
    hap1, hap2 = next(iter(planted["calls"].values()))
    print("hap1 calls:", hap1)
    assert hap2 == []
    want = [(0, COPY, "collapse", 2, 0), (0, (TANDEM[0], TANDEM[1]), "collapse", 3, 1), (1, DELETED, "depleted", 0, None)]
    assert len(hap1) == len(want), hap1
    for c, (a, b), kind, copies, tandem in want:
        hit = [t for t in hap1 if t[0] == c and abs(t[1] - a) <= SLACK and abs(t[2] - b) <= SLACK]
        assert len(hit) == 1 and hit[0][3] == kind and hit[0][8] == tandem, (c, a, b, hap1)
        if kind == "collapse":
            assert hit[0][7] == copies, hit


def test_two_contexts_equal_one(planted):
    """two contexts on one GPU, half of the batches each, exchanging through parallel.ThreadExchange: the summed counts and
    the runs are the single context's on both"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    from gavisunk_b200 import workload as W
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], [[0, 1, 2], [3], [4, 5, 6], [7, 8, 9, 10, 11]])
    _run(eng, wl, hb)
    _, _, want_dp, _, want_runs = _tables(eng, wl.contig_len)
    eng2 = Engine(20)
    W.build_db(eng2, wl)
    engines = [eng, eng2]
    xch = ThreadExchange(engines)
    out, errs = [None, None], []

    def work(i):
        try:
            cx = xch.for_rank(i)
            engines[i].run_batches(_binds(hb[:2] if i == 0 else hb[2:]), wl.contig_hap, min_read_len=3000,
                                   allreduce_hist=cx.allreduce_hist, gather_forests=cx.gather_forests, sunk_depth=True)
            out[i] = _tables(engines[i], wl.contig_len, allreduce=cx.allreduce_hist)
            again = engines[i].depth(allreduce=cx.allreduce_hist)  # summed once per sunk_depth(), not again
            assert np.array_equal(again["hits"], out[i][2]["hits"]) and np.array_equal(again["reads"], out[i][2]["reads"])
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    for o in out:
        assert o[4] == want_runs
        for c in ("hits", "reads", "sunks", "kept"):
            assert np.array_equal(o[2][c], want_dp[c]), c
    eng2.close()


def test_rank_without_a_batch_takes_part(planted):
    """a rank with no batch of its own still sums its (zero) counts with the other's"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    from gavisunk_b200 import workload as W
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], [[0, 1, 2, 3, 4, 5], [6, 7, 8, 9, 10, 11]])
    _run(eng, wl, hb)
    _, _, want_dp, _, want_runs = _tables(eng, wl.contig_len)
    eng2 = Engine(20)
    W.build_db(eng2, wl)
    engines = [eng, eng2]
    xch = ThreadExchange(engines)
    out, errs = [None, None], []

    def work(i):
        try:
            cx = xch.for_rank(i)
            engines[i].run_batches(_binds(hb if i == 0 else []), wl.contig_hap, min_read_len=3000, allreduce_hist=cx.allreduce_hist,
                                   gather_forests=cx.gather_forests, sunk_depth=True)
            out[i] = _tables(engines[i], wl.contig_len, allreduce=cx.allreduce_hist)
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    for o in out:
        assert o[4] == want_runs and np.array_equal(o[2]["hits"], want_dp["hits"])
    eng2.close()


def test_unedited_reads_make_no_call():
    eng, wl, chunks, chunk_hap = _planted(edit=False)
    _run(eng, wl, _host_batches(chunks, chunk_hap, SPLITS[0]))
    gt, _, dp, _, _ = _tables(eng, wl.contig_len)
    assert int(dp["hits"].sum()) > 0
    assert [_calls(eng, wl, gt, dp, h) for h in range(2)] == [[], []]
    eng.close()


# ------------------------------------------------------------------------------------------------
# hand-set rows (gvs_rows_set(0), no database: groups in first-appearance order)
# ------------------------------------------------------------------------------------------------
def _hand_rows(seed=5):
    """read 0: 1500 rows over 300 groups in a random order (non-monotone, re-entering groups); read 1: 50 rows of one
    group; read 2: two groups alternating 20 times; reads 3-12: one row each; read 13: 40 monotone rows with repeats;
    read 14: 1100 rows descending; reads 15 and 16 (first, so that their groups take the group indices 0-39 in order):
    monotone but for one row 32 that re-enters the group of row 30 (15, ascending) or row 30 (16, descending), so that
    only the carry from the first 32-row chunk shows that they are not monotone"""
    rng = np.random.default_rng(seed)
    cg = lambda i: CARRY_BASE + 100 * i
    rows = [(15, k, 0, cg(i), cg(i)) for k, i in enumerate(list(range(32)) + [30] + list(range(32, 40)))]
    rows += [(16, k, 0, cg(i), cg(i)) for k, i in enumerate(list(range(39, 7, -1)) + [9] + list(range(7, -1, -1)))]
    for k in range(1500):
        g = int(rng.integers(0, 300))
        rows.append((0, k, 0, 1000 + 100 * g, 1000 + 100 * g))
    rows += [(1, k, 0, 5000, 5000) for k in range(50)]
    rows += [(2, k, 1, 700 + 300 * (k % 2), 700 + 300 * (k % 2)) for k in range(40)]
    rows += [(r, 0, r % 2, 100 * r + 50, 100 * r + 50) for r in range(3, 13)]
    rows += [(13, k, 0, 1000 + 100 * (k // 3), 1000 + 100 * (k // 3)) for k in range(40)]
    rows += [(14, k, 0, 1000 + 100 * (1099 - k), 1000 + 100 * (1099 - k)) for k in range(1100)]
    return rows


CARRY_BASE = 3000000


def _hand_engine(rows, n_reads=17, match=True, hist=True):
    """an engine without a database; hist: the rows' histogram first (set_rows(1), group_hist), so that depth() has
    `kept`; match: then the rows as match rows (set_rows(0): the same rows give the same group table)"""
    from gavisunk_b200.engine import Engine
    eng = Engine(20)
    eng.set_reads_meta(np.full(n_reads, 50000, np.uint32))
    cols = [np.asarray([r[k] for r in rows], np.uint32) for k in range(5)]
    if hist:
        eng.set_rows(1, *cols, n_contigs=2)
        eng.group_hist()
    if match:
        eng.set_rows(0, *cols, n_contigs=2)
    return eng


def test_hand_set_rows():
    rows = _hand_rows()
    eng = _hand_engine(rows)
    eng.sunk_depth()
    dp = eng.depth()
    gt = eng.groups()
    groups = list(zip(gt["contig"].tolist(), gt["group"].tolist()))
    cnt = O.counts([(r[0], r[2], r[4]) for r in rows], groups)
    assert [(int(h), int(r)) for h, r in zip(dp["hits"], dp["reads"])] == [cnt[g] for g in groups]
    assert cnt[(0, 5000)][0] >= 50 and cnt[(1, 700)] == (20, 1) and cnt[(1, 1000)] == (20, 1)
    assert cnt[(0, CARRY_BASE + 3000)] == (3, 2) and cnt[(0, CARRY_BASE + 900)] == (3, 2)
    assert gt["group"][:40].tolist() == [CARRY_BASE + 100 * i for i in range(40)]  # group index = i: monotone up to row 32
    assert not dp["sunks"].any()  # no database: no .loc rows
    assert np.array_equal(dp["kept"], dp["hits"])
    eng.sunk_depth(accumulate=True)
    dp2 = eng.depth()
    assert np.array_equal(dp2["hits"], 2 * dp["hits"]) and np.array_equal(dp2["reads"], 2 * dp["reads"])
    eng.sunk_depth()  # accumulate = 0 replaces
    assert np.array_equal(eng.depth()["hits"], dp["hits"])
    eng.close()


def test_stage_order_errors():
    from gavisunk_b200._lib import GavisunkError
    rows = _hand_rows()
    eng = _hand_engine(rows, hist=False)
    with pytest.raises(GavisunkError):
        eng.depth()  # before gvs_sunk_depth
    eng.sunk_depth()
    with pytest.raises(GavisunkError):
        eng.depth_runs([200000, 200000])  # before gvs_group_hist
    eng.close()
    eng = _hand_engine(rows, match=False)
    with pytest.raises(GavisunkError):
        eng.depth_runs([200000, 200000])  # before gvs_sunk_depth
    eng.close()


def test_empty_batch_adds_nothing(planted):
    eng, wl = planted["eng"], planted["wl"]
    _run(eng, wl, _host_batches(planted["chunks"], planted["chunk_hap"], SPLITS[1]))
    want = eng.depth()
    eng.set_reads_meta(np.zeros(1, np.uint32))
    eng.set_rows(0, *[np.zeros(0, np.uint32)] * 5)
    eng.sunk_depth(accumulate=True)
    got = eng.depth()
    assert np.array_equal(got["hits"], want["hits"]) and np.array_equal(got["reads"], want["reads"])
    eng.sunk_depth()
    assert not eng.depth()["hits"].any()


def test_no_new_launches_without_the_flag(planted):
    """run_batches without sunk_depth launches the same on every run, and the stage only adds launches of its own"""
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], SPLITS[1])
    counts = []
    for _ in range(2):
        l0 = eng.launches
        eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=3000)
        counts.append(eng.launches - l0)
    l0 = eng.launches
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=3000, sunk_depth=True)
    assert counts[0] == counts[1] and eng.launches - l0 > counts[0]


# ------------------------------------------------------------------------------------------------
# the reference's bundled samples (BASELINE configs 1-2)
# ------------------------------------------------------------------------------------------------
FILES = ("depth.bedgraph", "depth.bed", "depth.tsv")
AMY_GAP = ("AMY_h1", 284861, 324275)


def _fused_argv(case, asm, chunks):
    return ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1], "--detailed"]


@pytest.fixture(scope="module", params=["j1_amy_pseudodip", "j1_amy_hg02723"])
def runs(request, tmp_path_factory):
    from gavisunk_b200 import cli
    from gavisunk_b200.engine import Engine
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_sunk_depth")
    asm, fai, chunks = _materialise(case, tmp)
    out = {}
    real = (Engine.sunk_depth, Engine.depth, Engine.depth_runs)

    def refuse(*a, **kw):
        raise AssertionError("fused without --sunk-depth ran a depth stage")
    for name, extra in (("plain", []), ("sd", ["--sunk-depth"]), ("two", ["--sunk-depth", "--devices", "0,0", "--batch-files", "3"])):
        out[name] = tmp / name
        Engine.sunk_depth, Engine.depth, Engine.depth_runs = (refuse,) * 3 if not extra else real
        try:
            assert cli.main(_fused_argv(case, asm, chunks) + ["--outdir", str(out[name])] + extra) == 0, name
        finally:
            Engine.sunk_depth, Engine.depth, Engine.depth_runs = real
    return dict(name=request.param, case=case, tmp=tmp, asm=asm, fai=fai, out=out)


def _files(root):
    got = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            got[os.path.relpath(p, root)] = open(p, "rb").read()
    return got


def test_flag_adds_only_its_six_files(runs):
    plain, sd = _files(runs["out"]["plain"]), _files(runs["out"]["sd"])
    new = {os.path.join("final_out", f"hap{h}.{t}") for h in (1, 2) for t in FILES}
    assert set(sd) == set(plain) | new and not (set(plain) & new)
    for k, v in plain.items():
        assert sd[k] == v, k
    two = _files(runs["out"]["two"])
    for k in new:
        assert two[k] == sd[k], k


def _oracle_texts(d, fai_paths):
    from gavisunk_b200 import io as gio
    contigs = [(n, l) for p in fai_paths for n, l in gio.read_fai(p)]
    sp = lambda *p: os.path.join(d, "sunkpos", *p)
    loc = list(zip(*gio.read_loc(os.path.join(d, "mrsfast", "kmer.loc"))))
    det = [gio.read_sunkpos(sp(f"hap{h}_detailed.sunkpos")) for h in (1, 2)]
    kept = [gio.read_sunkpos(sp(f"hap{h}.sunkpos")) for h in (1, 2)]
    hits, reads, kp, sunks, bad = O.from_files(loc, det, kept, open(sp("bad_sunks.txt")).read().split(), contigs)
    n1 = len(gio.read_fai(fai_paths[0]))
    return [O.texts(list(range(n1)) if h == 0 else list(range(n1, len(contigs))), contigs, hits, reads, kp, sunks, bad)
            for h in range(2)], contigs


def test_files_equal_oracle(runs):
    d = runs["out"]["sd"]
    want, contigs = _oracle_texts(str(d), runs["fai"])
    for h in (1, 2):
        for t, w in zip(FILES, want[h - 1]):
            assert open(d / "final_out" / f"hap{h}.{t}").read() == w, (h, t)
    if runs["name"] == "j1_amy_hg02723":  # what the track shows at the README gap (reads simulated from the assembly)
        c, a, b = AMY_GAP
        for l in want[0][0].splitlines():
            p = l.split("\t")
            if p[0] == c and int(p[2]) > a and int(p[1]) < b:
                print("AMY gap run:", l)
        print("AMY hap1 calls:", want[0][1].splitlines())


def test_shim_reproduces_fused(runs):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["sd"], runs["tmp"]
    sp = lambda *p: str(d / "sunkpos" / os.path.join(*p))
    for h in (1, 2):
        outs = [str(tmp / f"shim_hap{h}.{t}") for t in FILES]
        assert cli.main(["sunk_depth", str(d / "mrsfast" / "kmer.loc"), *runs["fai"], sp("bad_sunks.txt"), sp("hap1_detailed.sunkpos"),
                         sp("hap2_detailed.sunkpos"), sp("hap1.sunkpos"), sp("hap2.sunkpos"), f"hap{h}", *outs]) == 0
        for t, o in zip(FILES, outs):
            assert open(o, "rb").read() == open(d / "final_out" / f"hap{h}.{t}", "rb").read(), (h, t)


def test_shim_missing_input_writes_nothing(runs, capsys):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["sd"], runs["tmp"]
    sp = lambda *p: str(d / "sunkpos" / os.path.join(*p))
    outs = [str(tmp / f"missing.{t}") for t in FILES]
    rc = cli.main(["sunk_depth", str(d / "mrsfast" / "kmer.loc"), *runs["fai"], sp("bad_sunks.txt"), sp("hap1_detailed.sunkpos"),
                   str(tmp / "no_detailed.sunkpos"), sp("hap1.sunkpos"), sp("hap2.sunkpos"), "hap1", *outs])
    assert rc == 1 and "no_detailed.sunkpos" in capsys.readouterr().err
    assert not any(os.path.exists(o) for o in outs)

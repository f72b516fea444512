"""Junctions (Engine.junction_screen / Engine.junctions, csrc/junctions.cu; `fused --junctions`, `cli junctions`): records
against the CPU oracle (tests/junctions_oracle.py) on an assembly with a planted split, misjoin and phase switch, one vs
several batches and contexts, on hand-set rows, and on the reference's bundled samples.  No reference counterpart."""
import os
import sys
import threading

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

import junctions_oracle as O

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

SPLITS = [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]]
MINLEN = 3000
CONTIGS = (250000, 200000, 200000, 200000)  # per haplotype: T0 .. T3
CUT, MISSING = 120000, 6000  # T0 of hap 1 is split at CUT into two contigs, MISSING bases lost between them
AT = 100000  # T1 / T2 of hap 1 are misjoined here, and T3's haplotypes switch here


def _tol(size):
    return 250 + 0.03 * size


def _rname(i):
    return f"r{int(i):08d}"  # bytewise order == read index order


def _planted(seed=61, cov_per_hap=15.0):
    """truth: a synthetic diploid assembly (hap 2 heterozygous where hap 1 loses bases); the database: its hap 1 with T0 split (MISSING bases lost), T1 and T2
    misjoined reciprocally at AT, and T3's haplotypes switched at AT.  12 chunks of reads (6 per haplotype) are
    simulated from the truth."""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    tmp = Engine(20)
    wl = W.make_assembly(tmp, list(CONTIGS), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    asm = wl.asm.cpu().numpy()
    off = wl.contig_off.cpu().numpy()
    names = list(wl.contig_names)
    seqs = [asm[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(names))]
    tmp.close()
    nc = len(CONTIGS)
    # the lost bases must occur nowhere else in the database: through a copy on hap 2 the reads would hit one long SUNK
    # run, and kmerpos_annot3 prints only its first hit while later positions drift by the suppressed hits (Q3), which
    # shrinks read_gap.  So hap 2 carries other sequence there (a heterozygous stretch).
    rng = np.random.default_rng(seed)
    seqs[nc] = seqs[nc][:CUT] + np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, MISSING)].tobytes() + seqs[nc][CUT + MISSING:]
    h1, h2 = seqs[:nc], seqs[nc:]
    db = [(names[0] + "_a", h1[0][:CUT]), (names[0] + "_b", h1[0][CUT + MISSING:]), (names[1], h1[1][:AT] + h1[2][AT:]),
          (names[2], h1[2][:AT] + h1[1][AT:]), (names[3], h1[3][:AT] + h2[3][AT:])]
    db += [(names[nc + i], h2[i]) for i in range(nc - 1)] + [(names[2 * nc - 1], h2[3][:AT] + h1[3][AT:])]
    eng = Engine(20)
    eng.build_db(db)
    contig_hap = np.asarray([0] * (nc + 1) + [1] * nc, np.uint8)
    contig_len = np.asarray([len(s) for _, s in db], np.uint32)
    chunks, chunk_hap = [], []
    for hap in range(2):
        contigs = [(names[hap * nc + i], seqs[hap * nc + i]) for i in range(nc)]
        want = cov_per_hap * sum(len(s) for _, s in contigs)
        lengths = []
        while sum(lengths) < want:
            lengths.append(int(min(50000, max(1000, rng.lognormal(np.log(14000), 0.6)))))
        reads = S.simulate(contigs, lengths, seed + 10 + hap, f"h{hap + 1}_")
        chunks += S.split_round_robin(reads, 6)
        chunk_hap += [hap] * 6
    return eng, db, contig_hap, contig_len, chunks, np.asarray(chunk_hap, np.uint8)


def _host_batches(chunks, chunk_hap, groups):
    out, r0 = [], 0
    for g in groups:
        reads = [r for c in g for r in chunks[c]]
        lens = np.asarray([len(s) for _, s in reads], np.uint64)
        off = np.zeros(len(reads) + 1, np.uint64)
        off[1:] = np.cumsum(lens)
        cf = np.cumsum([0] + [len(chunks[c]) for c in g]).astype(np.uint64)
        seq = np.frombuffer(b"".join(s for _, s in reads), np.uint8)
        out.append((seq, off, cf, chunk_hap[g], r0, lens))
        r0 += len(reads)
    return out


def _binds(hb):
    return [(lambda e, b=b: e.set_reads(b[0], b[1], b[2], b[3])) for b in hb]


def _records(jn, name=_rname):
    """device records as oracle tuples, in device order"""
    sd = "+-"
    out = []
    for i in range(len(jn["read"])):
        side = lambda k: (int(jn["contig" + k][i]), sd[int(jn["strand" + k][i])], int(jn["ids" + k][i]),
                          (int(jn["id" + k][i]), int(jn["start" + k][i]), int(jn["pos" + k][i])))
        out.append((name(jn["read"][i]), side("1"), side("2")))
    return out


def _bad(eng):
    gt = eng.groups()
    return {(int(gt["contig"][i]), int(gt["group"][i])) for i in eng.bad_list().tolist()}


def _run(eng, contig_hap, hb, **kw):
    """run_batches with the junction screen; -> (records, every batch's match rows as oracle rows)"""
    rows0 = []

    def on_batch(e, b, base):
        r = e.rows(0)
        rows0.extend(zip((_rname(x + base) for x in r["read"].tolist()), r["pos"].tolist(), r["contig"].tolist(), r["start"].tolist(),
                         r["group"].tolist()))
    eng.run_batches(_binds(hb), contig_hap, min_read_len=MINLEN, on_batch=on_batch, junctions=True, **kw)
    return eng.junctions(), rows0


@pytest.fixture(scope="module")
def planted():
    eng, db, contig_hap, contig_len, chunks, chunk_hap = _planted()
    hb = _host_batches(chunks, chunk_hap, SPLITS[0])
    rlen = {_rname(i): int(l) for i, l in enumerate(hb[0][5])}
    return dict(eng=eng, db=db, contig_hap=contig_hap, contig_len=contig_len, chunks=chunks, chunk_hap=chunk_hap, rlen=rlen, oracle={})


def _clusters(recs, contig_len, contig_hap):
    n = len(contig_len)
    return O.clusters(recs, {c: int(contig_len[c]) for c in range(n)}, {c: int(contig_hap[c]) for c in range(n)}, {c: c for c in range(n)})


def _check_known_answers(recs, contig_len, contig_hap):
    cl = _clusters(recs, contig_len, contig_hap)
    joins = lambda t, a, b: {t[0], t[4]} == {a, b}
    near = lambda t: abs(t[3] - AT) <= 3000 and abs(t[7] - AT) <= 3000
    split = [t for t in cl if joins(t, 0, 1) and t[11] == "link" and t[8] >= 3]
    assert split, cl
    assert any(abs(t[10] - MISSING) <= _tol(MISSING) for t in split), split
    mis = [t for t in cl if joins(t, 2, 3) and t[11] == "breakpoint"]
    assert len(mis) == 2 and all(near(t) for t in mis), mis
    switch = [t for t in cl if joins(t, 4, 8) and t[11] == "breakpoint" and t[2] != t[6] and near(t)]
    assert switch, cl
    known = set(map(id, split + mis + switch))
    assert not [t for t in cl if t[8] >= 3 and id(t) not in known], cl


@pytest.mark.parametrize("split", SPLITS)
def test_records_equal_oracle(planted, split):
    eng = planted["eng"]
    jn, rows0 = _run(eng, planted["contig_hap"], _host_batches(planted["chunks"], planted["chunk_hap"], split))
    got = _records(jn)
    if "want" not in planted["oracle"]:
        planted["oracle"]["want"] = O.junctions(rows0, planted["rlen"], _bad(eng), MINLEN)
    assert got == planted["oracle"]["want"]
    _check_known_answers(got, planted["contig_len"], planted["contig_hap"])


def test_two_contexts_equal_one(planted):
    """two contexts on one GPU, half of the batches each, exchanging through parallel.ThreadExchange: each resolves
    its own reads with the shared bad groups, and the records of the two concatenate to the single context's"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    eng, contig_hap = planted["eng"], planted["contig_hap"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], [[0, 1, 2], [3], [4, 5, 6], [7, 8, 9, 10, 11]])
    want = _records(_run(eng, contig_hap, hb)[0])
    eng2 = Engine(20)
    eng2.build_db(planted["db"])
    engines = [eng, eng2]
    xch = ThreadExchange(engines)
    out, errs = [None, None], []

    def work(i):
        try:
            cx = xch.for_rank(i)
            part = hb[:2] if i == 0 else hb[2:]
            out[i] = _run(engines[i], contig_hap, part, allreduce_hist=cx.allreduce_hist, gather_forests=cx.gather_forests)[0]
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    jn = {c: np.concatenate([out[0][c], out[1][c] + (np.uint32(hb[2][4]) if c == "read" else np.uint32(0))]) for c in out[0]}
    assert _records(jn) == want and len(want) > 0
    eng2.close()


def test_default_run_batches_launches_nothing_new(planted):
    """run_batches without junctions=True launches exactly the kernels of a screened run minus the screens' own"""
    eng = planted["eng"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], SPLITS[1])
    l0 = eng.launches
    eng.run_batches(_binds(hb), planted["contig_hap"], min_read_len=MINLEN)
    plain = eng.launches - l0
    screen = []
    real = eng.junction_screen

    def counted(*a, **kw):
        n0 = eng.launches
        out = real(*a, **kw)
        screen.append(eng.launches - n0)
        return out
    eng.junction_screen = counted
    try:
        l0 = eng.launches
        eng.run_batches(_binds(hb), planted["contig_hap"], min_read_len=MINLEN, junctions=True)
        screened = eng.launches - l0
    finally:
        del eng.junction_screen
    assert len(screen) == len(hb) and min(screen) > 0
    assert plain == screened - sum(screen)


# ------------------------------------------------------------------------------------------------
# rows set by hand (gvs_rows_set(0)): long reads, reads at the length limit, equal starts, bad groups
# ------------------------------------------------------------------------------------------------
N_CONTIGS = 40


def _colinear(rng, contig, n, pos0, start0, strand, ids):
    """n rows of one contig whose positions follow the starts (rising or falling) within +-10 bp"""
    st = start0 + np.cumsum(rng.integers(200, 1500, n))
    if strand < 0:
        st = st[::-1]
    pos = pos0 + 200 + np.abs(st - st[0]) + rng.integers(-10, 11, n)
    return [(int(p), contig, int(s), ids(int(s))) for p, s in zip(pos, st)], int(pos.max()) + 10


def _hand_rows(seed):
    rng = np.random.default_rng(seed)
    reads, lens = [], []
    # one read of > 1024 rows over 40 contigs: colinear runs of 2..12 rows, stray rows and repeated IDs
    rows, pos = [], 0
    while len(rows) < 1300:
        c = int(rng.integers(0, N_CONTIGS))
        run, pos = _colinear(rng, c, int(rng.integers(2, 13)), pos, int(rng.integers(0, 5)) * 100000, 1 if rng.random() < 0.6 else -1,
                             lambda s: s - s % 100)
        rows += run
        if rng.random() < 0.3:
            rows.append((pos + 10, int(rng.integers(0, N_CONTIGS)), int(rng.integers(0, 10 ** 6)), int(rng.integers(0, 10 ** 6))))
        if rng.random() < 0.2 and rows:
            p, c2, s2, i2 = rows[int(rng.integers(0, len(rows)))]
            rows.append((pos + 20, c2, s2 + 5, i2))  # an ID seen before, elsewhere in the read
    reads.append(rows)
    lens.append(pos + 1000)
    # reads exactly at the limit, one below, and reads with equal starts across different IDs
    for L in (MINLEN, MINLEN - 1, MINLEN, MINLEN + 1):
        rows, pos = [], 0
        for c in rng.choice(N_CONTIGS, 3, replace=False).tolist():
            run, pos = _colinear(rng, c, 5, pos, int(rng.integers(0, 3)) * 50000, 1, lambda s: s)
            rows += run
        s = rows[2][2]
        rows.insert(3, (rows[2][0] + 1, rows[2][1], s, s + 7))  # equal start, another ID
        reads.append(rows)
        lens.append(L)
    # random reads of 2..6 runs on 2..4 contigs (A -> B -> A and friends)
    for _ in range(300):
        cs = rng.choice(N_CONTIGS, int(rng.integers(2, 5)), replace=False).tolist()
        rows, pos = [], 0
        for _r in range(int(rng.integers(2, 7))):
            run, pos = _colinear(rng, cs[int(rng.integers(0, len(cs)))], int(rng.integers(1, 8)), pos, int(rng.integers(0, 4)) * 40000,
                                 1 if rng.random() < 0.5 else -1, lambda s: s)
            rows += run
        reads.append(rows)
        lens.append(int(rng.integers(MINLEN - 500, 4 * MINLEN)))
    return reads, lens


@pytest.mark.parametrize("seed", [1, 2])
def test_hand_set_rows_equal_oracle(seed):
    from gavisunk_b200.engine import Engine
    reads, lens = _hand_rows(seed)
    cols = [[], [], [], [], []]
    for r, rows in enumerate(reads):
        for p, c, s, i in rows:
            for k, v in enumerate((r, p, c, s, i)):
                cols[k].append(v)
    rng = np.random.default_rng(seed + 100)
    pairs = sorted({(c, i) for c, i in zip(cols[2], cols[4])})
    bad = [pairs[j] for j in rng.choice(len(pairs), len(pairs) // 20, replace=False).tolist()]
    eng = Engine(20)
    eng.contig_names = [f"c{i}" for i in range(N_CONTIGS)]
    eng.set_reads_meta(np.asarray(lens, np.uint32))
    eng.set_rows(0, *cols)
    orows = list(zip(cols[0], cols[1], cols[2], cols[3], cols[4]))
    rlen = {r: l for r, l in enumerate(lens)}
    # no bad groups, then the bad groups (the screen does not depend on them)
    assert eng.junction_screen(MINLEN)[1] > 0
    want0 = O.junctions(orows, rlen, set(), MINLEN)
    assert _records(eng.junctions(), int) == want0
    eng.bad_set([c for c, _ in bad], [i for _, i in bad])
    want = O.junctions(orows, rlen, set(bad), MINLEN)
    assert _records(eng.junctions(), int) == want and want != want0
    # a second screen outside a batches run replaces the stash
    n = eng.junction_screen(MINLEN)
    assert eng.junction_screen(MINLEN) == n
    assert _records(eng.junctions(), int) == want
    assert any(len(r) > 1024 for r in reads) and 0 in {x[0] for x in want0}
    assert {x[0] for x in want0} & {1, 3} and 2 not in {x[0] for x in want0}
    eng.close()


# ------------------------------------------------------------------------------------------------
# the reference's bundled samples (BASELINE configs 1-2)
# ------------------------------------------------------------------------------------------------
FILES = ("junctions.reads.tsv", "junctions.tsv")


def _fused_argv(case, asm, chunks):
    return ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1], "--detailed"]


@pytest.fixture(scope="module", params=["j1_amy_pseudodip", "j1_amy_hg02723"])
def runs(request, tmp_path_factory):
    from gavisunk_b200 import cli
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_junctions")
    asm, fai, chunks = _materialise(case, tmp)
    out = {}
    for name, extra in (("plain", []), ("jn", ["--junctions"]), ("two", ["--junctions", "--devices", "0,0", "--batch-files", "3"])):
        out[name] = tmp / name
        assert cli.main(_fused_argv(case, asm, chunks) + ["--outdir", str(out[name])] + extra) == 0, name
    return dict(name=request.param, case=case, tmp=tmp, asm=asm, fai=fai, out=out)


def _files(root):
    got = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            got[os.path.relpath(p, root)] = open(p, "rb").read()
    return got


def test_flag_adds_only_the_four_files(runs):
    plain, jn = _files(runs["out"]["plain"]), _files(runs["out"]["jn"])
    new = {os.path.join("final_out", f"hap{h}.{t}") for h in (1, 2) for t in FILES}
    assert set(jn) == set(plain) | new and not (set(plain) & new)
    for k, v in plain.items():
        assert jn[k] == v, k
    two = _files(runs["out"]["two"])
    assert set(two) == set(jn)
    for k in new:
        assert two[k] == jn[k], k


def test_files_equal_oracle(runs):
    from gavisunk_b200 import io as gio
    d = runs["out"]["jn"]
    fai = [gio.read_fai(p) for p in runs["fai"]]
    names = [n for f in fai for n, _ in f]
    clen = {n: l for f in fai for n, l in f}
    chap = {n: h for h in range(2) for n, _ in fai[h]}
    order = {n: i for i, n in enumerate(names)}
    bad = {(b.split(":")[0], int(b.split(":")[1])) for b in open(d / "sunkpos" / "bad_sunks.txt").read().split()}
    n_rec = 0
    for h in (1, 2):
        rows = gio.read_sunkpos(d / "sunkpos" / f"hap{h}_detailed.sunkpos")
        rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in open(d / "sunkpos" / f"hap{h}.rlen").read().splitlines()}
        recs = O.junctions(rows, rlen, bad)
        n_rec += len(recs)
        lines = open(d / "final_out" / f"hap{h}.junctions.reads.tsv").read().splitlines()
        assert lines[0].split("\t") == ["read", "read_len", "contig1", "strand1", "ids1", "id1", "start1", "pos1", "contig2", "strand2",
                                        "ids2", "id2", "start2", "pos2", "read_gap", "leave1", "enter2", "implied_gap", "class"]
        assert lines[1:] == O.reads_tsv_lines(recs, rlen, clen)
        lines = open(d / "final_out" / f"hap{h}.junctions.tsv").read().splitlines()
        assert lines[0].split("\t") == ["contig1", "strand1", "hap1", "start1", "contig2", "strand2", "hap2", "start2", "records", "links",
                                        "median_implied_gap", "class"]
        assert lines[1:] == O.clusters_tsv_lines(O.clusters(recs, clen, chap, order))
    print(runs["name"], "junction records:", n_rec)


def test_shim_reproduces_fused(runs):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["jn"], runs["tmp"]
    for h in (1, 2):
        outs = [str(tmp / f"shim_hap{h}.{t}") for t in FILES]
        assert cli.main(["junctions", str(d / "sunkpos" / f"hap{h}_detailed.sunkpos"), str(d / "sunkpos" / f"hap{h}.rlen"),
                         str(d / "sunkpos" / "bad_sunks.txt"), runs["fai"][0], runs["fai"][1], *outs]) == 0
        for t, o in zip(FILES, outs):
            assert open(o, "rb").read() == open(d / "final_out" / f"hap{h}.{t}", "rb").read(), (h, t)


def test_shim_missing_input_writes_nothing(runs, capsys):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["jn"], runs["tmp"]
    outs = [str(tmp / f"missing.{t}") for t in FILES]
    rc = cli.main(["junctions", str(d / "sunkpos" / "hap1_detailed.sunkpos"), str(tmp / "no.rlen"), str(d / "sunkpos" / "bad_sunks.txt"),
                   runs["fai"][0], runs["fai"][1], *outs])
    assert rc == 1 and "no.rlen" in capsys.readouterr().err
    assert not any(os.path.exists(o) for o in outs)

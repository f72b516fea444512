"""Distance discordance (Engine.spans / Engine.discordance, csrc/discordance.cu; `fused --discordance`, `cli discordance`):
records and runs against the CPU oracle (tests/discordance_oracle.py) on an assembly with a planted 1 kb insertion and
1 kb deletion that the validation lets through, one vs several batches and contexts, hand-set rows, and the reference's
bundled samples.  No reference counterpart."""
import os
import sys
import threading

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

import discordance_oracle as O

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

SPLITS = [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]]
MINLEN = 3000
CONTIGS = (300000, 200000)
P, Q, EVENT = 150000, 100000, 1000  # EVENT random bases inserted into contig 0 at P, deleted from contig 1 at Q
MEDIAN_LEN, MAX_LEN = 30000, 120000  # reads reach far past 10 x EVENT: they validate across both events


def _rname(i):
    return f"r{int(i):08d}"  # bytewise order == read index order


def _planted(seed=61, cov_per_hap=15.0, edit=True):
    """a synthetic diploid assembly (database built from it unedited) and 12 chunks of reads (6 per haplotype) simulated
    from its contigs, with the two events planted into hap 1 when `edit`"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    eng = Engine(20)
    wl = W.make_assembly(eng, list(CONTIGS), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    W.build_db(eng, wl)
    asm = wl.asm.cpu().numpy()
    off = wl.contig_off.cpu().numpy()
    seqs = [asm[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(wl.contig_names))]
    rng = np.random.default_rng(seed)
    if edit:
        seqs[0] = seqs[0][:P] + np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, EVENT)].tobytes() + seqs[0][P:]
        seqs[1] = seqs[1][:Q] + seqs[1][Q + EVENT:]
    nc = len(CONTIGS)
    chunks, chunk_hap = [], []
    rng = np.random.default_rng(seed + 1)
    for hap in range(2):
        contigs = [(wl.contig_names[hap * nc + i], seqs[hap * nc + i]) for i in range(nc)]
        want = cov_per_hap * sum(len(s) for _, s in contigs)
        lengths = []
        while sum(lengths) < want:
            lengths.append(int(min(MAX_LEN, max(1000, rng.lognormal(np.log(MEDIAN_LEN), 0.6)))))
        reads = S.simulate(contigs, lengths, seed + 10 + hap, f"h{hap + 1}_")
        chunks += S.split_round_robin(reads, 6)
        chunk_hap += [hap] * 6
    return eng, wl, chunks, np.asarray(chunk_hap, np.uint8)


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


def _records(rec):
    """device records as oracle tuples, in device order"""
    out = []
    for i in range(len(rec["read"])):
        a = (int(rec["id1"][i]), int(rec["start1"][i]), int(rec["pos1"][i]))
        b = (int(rec["id2"][i]), int(rec["start2"][i]), int(rec["pos2"][i]))
        d = abs(b[2] - a[2]) - (b[1] - a[1])
        out.append((int(rec["read"][i]), int(rec["contig"][i]), a, b, d, "longer" if d >= 0 else "shorter"))
    return out


def _runs(rn):
    return [tuple(int(rn[c][i]) for c in ("contig", "start", "end", "spans", "longer", "shorter")) for i in range(len(rn["contig"]))]


def _oracle(eng, contig_len):
    kept = eng.rows(1)
    rows = list(zip(*(kept[c].astype(np.int64).tolist() for c in ("read", "pos", "contig", "start", "group"))))
    gt = eng.groups()
    groups = set(zip(gt["contig"].tolist(), gt["group"].tolist()))
    bad = {(int(gt["contig"][i]), int(gt["group"][i])) for i in eng.bad_list().tolist()}
    pr = eng.pairs()
    validated = set(zip(pr["read"].tolist(), pr["group"].tolist()))
    sp = O.spans(rows, bad, validated)
    contigs = [(str(i), int(l)) for i, l in enumerate(contig_len)]
    return sp, O.records(sp), O.runs(sp, groups, contigs)


def _check_known_answers(recs, rn, sp, gaps):
    """one call per event, of the right kind, whose peak holds the edit, with the size near +-EVENT; no other call; no
    gap at either event"""
    cl = O.calls(recs, rn)
    at_p = [c for c in cl if c[0] == 0 and c[4] <= P < c[5]]
    at_q = [c for c in cl if c[0] == 1 and c[4] <= Q < c[5]]
    assert len(at_p) == 1 and len(at_q) == 1 and len(cl) == 2, cl
    for c, kind, want in ((at_p[0], "collapse", EVENT), (at_q[0], "expansion", -EVENT)):
        assert c[3] == kind and abs(c[8] - want) <= 100 + 0.03 * EVENT, c
    for ctg, x in ((0, P), (1, Q)):
        assert sum(1 for s in sp if s[1] == ctg and s[2][0] <= x < s[3][0]) >= 5
    for c, s, e in zip(gaps["contig"].tolist(), gaps["start"].tolist(), gaps["end"].tolist()):
        assert not (c == 0 and s <= P <= e + 1) and not (c == 1 and s <= Q + EVENT and e >= Q), (c, s, e)


@pytest.fixture(scope="module")
def planted():
    eng, wl, chunks, chunk_hap = _planted()
    return dict(eng=eng, wl=wl, chunks=chunks, chunk_hap=chunk_hap, oracle={})


@pytest.mark.parametrize("split", SPLITS)
def test_records_and_runs_equal_oracle(planted, split):
    eng, wl = planted["eng"], planted["wl"]
    eng.run_batches(_binds(_host_batches(planted["chunks"], planted["chunk_hap"], split)), wl.contig_hap, min_read_len=MINLEN)
    got = _records(eng.spans())
    rn = _runs(eng.discordance(wl.contig_len))
    if "want" not in planted["oracle"]:
        planted["oracle"]["want"] = _oracle(eng, wl.contig_len)
    sp, recs, want_rn = planted["oracle"]["want"]
    assert got == recs and rn == want_rn
    gaps, _ = eng.gaps(wl.contig_len)
    _check_known_answers(recs, rn, sp, gaps)


def test_two_contexts_equal_one(planted):
    """two contexts on one GPU, half of the batches each, exchanging through parallel.ThreadExchange: the runs (summed
    difference arrays) are the single context's on both, and the records of the two concatenate to its records"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    from gavisunk_b200 import workload as W
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], [[0, 1, 2], [3], [4, 5, 6], [7, 8, 9, 10, 11]])
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
    want = _records(eng.spans())
    want_rn = _runs(eng.discordance(wl.contig_len))
    eng2 = Engine(20)
    W.build_db(eng2, wl)
    engines = [eng, eng2]
    xch = ThreadExchange(engines)
    out, errs = [None, None], []

    def work(i):
        try:
            cx = xch.for_rank(i)
            part = hb[:2] if i == 0 else hb[2:]
            engines[i].run_batches(_binds(part), wl.contig_hap, min_read_len=MINLEN, allreduce_hist=cx.allreduce_hist,
                                   gather_forests=cx.gather_forests)
            rec = engines[i].spans()
            out[i] = (rec, engines[i].discordance(wl.contig_len, allreduce=cx.allreduce_hist))
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    assert _runs(out[0][1]) == want_rn and _runs(out[1][1]) == want_rn
    rec = {c: np.concatenate([out[0][0][c], out[1][0][c] + (np.uint32(hb[2][4]) if c == "read" else np.uint32(0))]) for c in out[0][0]}
    assert _records(rec) == want and len(want) > 0
    eng2.close()


def test_unedited_reads_make_no_call():
    eng, wl, chunks, chunk_hap = _planted(edit=False)
    eng.run_batches(_binds(_host_batches(chunks, chunk_hap, SPLITS[0])), wl.contig_hap, min_read_len=MINLEN)
    recs = _records(eng.spans())
    rn = _runs(eng.discordance(wl.contig_len))
    assert sum(r[3] for r in rn) > 0
    assert O.calls(recs, rn) == []
    eng.close()


def test_spans_before_validate_raises():
    from gavisunk_b200.engine import Engine
    from gavisunk_b200._lib import GavisunkError
    e2 = Engine(20)
    with pytest.raises(GavisunkError):
        e2.spans()
    e2.close()


# ------------------------------------------------------------------------------------------------
# hand-set rows (gvs_rows_set(1), no database: groups in first-appearance order, the rank is computed)
# ------------------------------------------------------------------------------------------------
def _hand_engine(rows, n_reads, lens):
    from gavisunk_b200.engine import Engine
    eng = Engine(20)
    eng.set_reads_meta(np.asarray(lens, np.uint32))
    cols = [np.asarray([r[k] for r in rows], np.uint32) for k in range(5)]
    eng.set_rows(1, *cols, n_contigs=2)
    eng.set_contigs([0, 0])
    return eng


def _hand_rows(seed=7):
    """read 0: 1500 groups of one contig, +strand with a 1 kb insertion in the middle, its rows in a shuffled order
    (non-monotone starts); read 1: the same groups on the - strand with one repeated ID; read 2: a short clean read"""
    rng = np.random.default_rng(seed)
    ids = np.arange(1500) * 200 + 1000
    rows = []
    order = rng.permutation(len(ids))
    for k in order:
        s = int(ids[k]) + 3
        rows.append((0, 5000 + s + (1000 if s > 150000 else 0) + int(rng.integers(0, 3)), 0, s, int(ids[k])))
    for k in range(len(ids)):
        s = int(ids[k]) + 7
        rows.append((1, 700000 - s - (1000 if s > 150000 else 0), 0, s, int(ids[k])))
        if k == 300:  # a second row of the group, 1 kb off: kept, its spans would be discordant
            rows.append((1, 700000 - s - 2 - 1000, 0, s + 2, int(ids[k])))
    for k in range(20):
        s = int(ids[k]) + 1
        rows.append((2, 10 + s, 0, s, int(ids[k])))
    # read 3: groups 2000 apart, +360 after the 10th and -360 after the 15th: two spans exactly on the default bound
    # (1000 * 360 = 1000 * 300 + 30 * 2000)
    for m in range(20):
        s = 1000 + 2000 * m + 1
        rows.append((3, 10 + s + (360 if 10 <= m < 15 else 0), 0, s, s - 1))
    return rows


def _hand_check(eng, rows, contig_len, bad=frozenset()):
    eng.validate(MINLEN)
    pr = eng.pairs()
    validated = set(zip(pr["read"].tolist(), pr["group"].tolist()))
    gt = eng.groups()
    groups = set(zip(gt["contig"].tolist(), gt["group"].tolist()))
    sp = O.spans(rows, set(bad), validated)
    got = _records(eng.spans())
    rn = _runs(eng.discordance(contig_len))
    assert got == O.records(sp)
    assert rn == O.runs(sp, groups, [(str(i), l) for i, l in enumerate(contig_len)])
    return sp, validated


def test_hand_set_rows_long_non_monotone_read_and_repeated_ids():
    rows = _hand_rows()
    eng = _hand_engine(rows, 4, [400000, 400000, 20000, 50000])
    sp, validated = _hand_check(eng, rows, [400000, 1000])
    assert [(s[4], s[5]) for s in sp if s[0] == 3 and s[5]] == [(360, "longer"), (-360, "shorter")]
    assert sum(1 for s in sp if s[0] == 0) > 1024 and any(s[5] == "longer" for s in sp if s[0] == 0)
    gid = 300 * 200 + 1000
    assert (1, gid) in validated
    assert not any(s[0] == 1 and gid in (s[2][0], s[3][0]) for s in sp)  # the repeated ID is skipped
    assert any(s[0] == 1 and s[3][0] - s[2][0] == 400 for s in sp)         # and its neighbours span across it
    eng.close()


def test_hand_set_rows_all_bad():
    rows = _hand_rows()
    eng = _hand_engine(rows, 4, [400000, 400000, 20000, 50000])
    eng.validate(MINLEN)
    gids = sorted({r[4] for r in rows})
    eng.bad_set([0] * len(gids), gids)
    assert _records(eng.spans()) == []
    assert _runs(eng.discordance([400000, 1000])) == [(0, 0, 400000, 0, 0, 0), (1, 0, 1000, 0, 0, 0)]
    eng.close()


# ------------------------------------------------------------------------------------------------
# the reference's bundled samples (BASELINE configs 1-2)
# ------------------------------------------------------------------------------------------------
FILES = ("discordance.reads.tsv", "discordance.tsv", "discordance.bed")


def _fused_argv(case, asm, chunks):
    return ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1]]


@pytest.fixture(scope="module", params=["j1_amy_pseudodip", "j1_amy_hg02723"])
def runs(request, tmp_path_factory):
    from gavisunk_b200 import cli
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_discordance")
    asm, fai, chunks = _materialise(case, tmp)
    out = {}
    from gavisunk_b200.engine import Engine
    real = (Engine.spans, Engine.discordance)

    def refuse(*a, **kw):
        raise AssertionError("fused without --discordance ran a discordance stage")
    for name, extra in (("plain", []), ("dc", ["--discordance"]), ("two", ["--discordance", "--devices", "0,0", "--batch-files", "3"])):
        out[name] = tmp / name
        Engine.spans, Engine.discordance = (refuse, refuse) if not extra else real
        try:
            assert cli.main(_fused_argv(case, asm, chunks) + ["--outdir", str(out[name])] + extra) == 0, name
        finally:
            Engine.spans, Engine.discordance = real
    return dict(name=request.param, case=case, tmp=tmp, asm=asm, fai=fai, out=out)


def _files(root):
    got = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            got[os.path.relpath(p, root)] = open(p, "rb").read()
    return got


def test_flag_adds_only_its_six_files(runs):
    plain, dc = _files(runs["out"]["plain"]), _files(runs["out"]["dc"])
    new = {os.path.join("final_out", f"hap{h}.{t}") for h in (1, 2) for t in FILES}
    assert set(dc) == set(plain) | new and not (set(plain) & new)
    for k, v in plain.items():
        assert dc[k] == v, k
    two = _files(runs["out"]["two"])
    for k in new:
        assert two[k] == dc[k], k


def _oracle_files(d, h, fai_p, validated_from):
    """the oracle's three files of haplotype h from fused's sunkpos / rlen / bad_sunks.txt, reads keyed by (contig, name),
    validated = the (contig, read, ID) rows of `validated_from` ({stem: inter_outs text})"""
    from gavisunk_b200 import io as gio
    rd = lambda *p: open(os.path.join(d, *p)).read()
    fai = [(l.split("\t")[0], int(l.split("\t")[1])) for l in open(fai_p).read().splitlines()]
    cidx = {n: i for i, (n, _) in enumerate(fai)}
    rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in rd("sunkpos", f"hap{h}.rlen").splitlines()}
    bad = {(cidx[b.split(":")[0]], int(b.split(":")[1])) for b in rd("sunkpos", "bad_sunks.txt").split() if b.split(":")[0] in cidx}
    rows = [((cidx[c], n), p, cidx[c], s, g) for n, p, c, s, g in dict.fromkeys(gio.read_sunkpos(os.path.join(d, "sunkpos", f"hap{h}.sunkpos")))]
    stem_of = {n.replace("#", "_") + f"_hap{h}": i for i, (n, _) in enumerate(fai)}
    validated = set()
    for stem, txt in validated_from.items():
        if stem not in stem_of:
            continue
        for l in txt.splitlines():
            p = l.split("\t")
            if len(p) == 2:
                validated.add(((stem_of[stem], p[1]), int(p[0])))
    groups = {(r[2], r[4]) for r in rows}
    sp = O.spans(rows, bad, validated)
    recs = O.records(sp)
    rn = O.runs(sp, groups, fai)
    return O.texts(recs, rn, fai, range(len(fai)), lambda r: r[1], lambda r: rlen.get(r[1], 0)), recs, rn


def test_files_equal_oracle_on_reference_validated_reads(runs):
    d = runs["out"]["dc"]
    n_calls = 0
    for h in (1, 2):
        want, _, _ = _oracle_files(d, h, runs["fai"][h - 1], runs["case"]["inter_outs"])
        for t, w in zip(FILES, want):
            assert open(d / "final_out" / f"hap{h}.{t}").read() == w, (h, t)
        n_calls += len(want[2].splitlines())
    print(f"{runs['name']}: {n_calls} calls")


def test_shim_reproduces_fused(runs):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["dc"], runs["tmp"]
    for h in (1, 2):
        outs = [str(tmp / f"shim_hap{h}.{t}") for t in FILES]
        assert cli.main(["discordance", str(d / "sunkpos" / f"hap{h}.sunkpos"), str(d / "sunkpos" / f"hap{h}.rlen"),
                         str(d / "sunkpos" / "bad_sunks.txt"), runs["fai"][h - 1], *outs]) == 0
        for t, o in zip(FILES, outs):
            assert open(o, "rb").read() == open(d / "final_out" / f"hap{h}.{t}", "rb").read(), (h, t)


def test_shim_missing_input_writes_nothing(runs, capsys):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["dc"], runs["tmp"]
    outs = [str(tmp / f"missing.{t}") for t in FILES]
    rc = cli.main(["discordance", str(d / "sunkpos" / "hap1.sunkpos"), str(tmp / "no.rlen"), str(d / "sunkpos" / "bad_sunks.txt"),
                   runs["fai"][0], *outs])
    assert rc == 1 and "no.rlen" in capsys.readouterr().err
    assert not any(os.path.exists(o) for o in outs)


REAL_INSERT = 2000


def test_planted_insertion_on_the_bundled_sample(runs):
    """a 2 kb insertion at the midpoint of the plain run's longest hap-1 interval, reads simulated with the sample's own
    lengths and seed from the edited haplotype, fused against the unedited assembly: no new gap, and a collapse call
    whose peak holds the insertion point"""
    if runs["name"] != "j1_amy_hg02723":
        pytest.skip("one sample is enough")
    from gavisunk_b200 import cli
    case, tmp = runs["case"], runs["tmp"]
    iv = [(p[0], int(p[1]), int(p[2])) for p in (l.split("\t") for l in open(runs["out"]["plain"] / "final_out" / "hap1.valid.bed").read().splitlines())]
    contig, s, e = max(iv, key=lambda t: t[2] - t[1])
    x = (s + e) // 2
    rng = np.random.default_rng(case["seed"])
    haps = [[(n, q.encode()) for n, q in h] for h in case["asm"]]
    haps[0] = [(n, q[:x] + np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, REAL_INSERT)].tobytes() + q[x:] if n == contig else q)
               for n, q in haps[0]]
    forbid = None
    if case["forbid"]:
        fn, lo, hi = case["forbid"]
        shift = lambda v: v + REAL_INSERT if (fn == contig and v >= x) else v
        forbid = (fn, shift(lo), shift(hi))
    work = tmp / "planted"
    os.makedirs(work, exist_ok=True)
    chunks = [[], []]
    for hi_ in range(2):
        reads = S.simulate(haps[hi_], case["lengths"][hi_], case["seed"] + hi_, f"h{hi_ + 1}r",
                           forbid=forbid if hi_ == 0 else (tuple(case["forbid"]) if case["forbid"] else None), skip=case["skip"])
        for ci, part in enumerate(S.split_round_robin(reads, case["nchunks"])):
            p = work / f"hap{hi_ + 1}_{ci + 1}.fq"
            p.write_bytes(S.fastq_text(part))
            chunks[hi_].append(str(p))
    out = work / "results"
    assert cli.main(_fused_argv(case, runs["asm"], chunks) + ["--outdir", str(out), "--discordance"]) == 0
    gaps = [(p[0], int(p[1]), int(p[2])) for p in (l.split("\t") for l in open(out / "final_out" / "hap1.gaps.bed").read().splitlines())]
    assert not any(g[0] == contig and g[1] < x <= g[2] + 1 for g in gaps), (x, gaps)
    calls = [l.split("\t") for l in open(out / "final_out" / "hap1.discordance.bed").read().splitlines()]
    hit = [c for c in calls if c[0] == contig and int(c[4]) <= x < int(c[5])]
    assert len(hit) == 1 and hit[0][3] == "collapse", (x, calls)
    assert abs(int(hit[0][8]) - REAL_INSERT) <= 100 + 0.03 * REAL_INSERT, hit


def test_no_new_launches_without_the_flag(planted):
    """run_batches without spans() launches exactly what it launches with spans() taken out: the feature only adds launches
    of its own, and fused without --discordance never calls it (the bundled-sample runs above patch it to fail)"""
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], SPLITS[1])
    counts = []
    for _ in range(2):
        l0 = eng.launches
        eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
        counts.append(eng.launches - l0)
        l0 = eng.launches
        eng.spans()
        eng.discordance(wl.contig_len)
        assert eng.launches - l0 > 0
    assert counts[0] == counts[1]

"""Strand switches and inversion calls (Engine.strand_switches, csrc/inversions.cu; `fused --inversions`, `cli inversions`):
records against the CPU oracle (tests/inversions_oracle.py) on an assembly with a planted 20 kb and 80 kb inversion and
fold-back reads, one vs several batches and contexts, hand-set rows, and the reference's bundled samples.  No reference
counterpart."""
import os
import sys
import threading

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

import inversions_oracle as O

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

SPLITS = [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]]
MINLEN = 3000
CONTIGS = (300000, 200000)
NC = len(CONTIGS)
INV = [(0, 150000, 170000), (NC + 1, 60000, 140000)]  # (contig, x, y): [x, y) reverse-complemented in the reads' sequence
MEDIAN_LEN, MAX_LEN = 30000, 120000  # the 80 kb inversion is longer than most reads
N_FOLD = 20
TOL = 5000


def _revcomp(s: bytes) -> bytes:
    return S._COMP[np.frombuffer(s, np.uint8)[::-1]].tobytes()


def _planted(seed=71, cov_per_hap=15.0, edit=True):
    """a synthetic diploid assembly (database built from it unedited) and 12 chunks of reads (6 per haplotype) simulated
    from its contigs, with the two inversions planted when `edit`, plus N_FOLD fold-back reads (a read followed by its
    reverse complement) from contigs without an inversion"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    eng = Engine(20)
    wl = W.make_assembly(eng, list(CONTIGS), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    W.build_db(eng, wl)
    asm = wl.asm.cpu().numpy()
    off = wl.contig_off.cpu().numpy()
    seqs = [asm[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(wl.contig_names))]
    if edit:
        for c, x, y in INV:
            seqs[c] = seqs[c][:x] + _revcomp(seqs[c][x:y]) + seqs[c][y:]
    chunks, chunk_hap = [], []
    rng = np.random.default_rng(seed + 1)
    for hap in range(2):
        contigs = [(wl.contig_names[hap * NC + i], seqs[hap * NC + i]) for i in range(NC)]
        want = cov_per_hap * sum(len(s) for _, s in contigs)
        lengths = []
        while sum(lengths) < want:
            lengths.append(int(min(MAX_LEN, max(1000, rng.lognormal(np.log(MEDIAN_LEN), 0.6)))))
        reads = S.simulate(contigs, lengths, seed + 10 + hap, f"h{hap + 1}_")
        chunks += S.split_round_robin(reads, 6)
        chunk_hap += [hap] * 6
    for k in range(N_FOLD):
        hap = k % 2
        c = hap * NC + (1 if hap == 0 else 0)  # hap-1 contig 1, hap-2 contig 0: no inversion
        l = int(rng.integers(8000, 25000))
        st = int(rng.integers(0, len(seqs[c]) - l))
        r = S.mutate(rng, np.frombuffer(seqs[c][st:st + l], np.uint8)).tobytes()
        r = r + _revcomp(S.mutate(rng, np.frombuffer(seqs[c][st:st + l], np.uint8)).tobytes())
        chunks[hap * 6 + k % 6].append((f"fold{k:03d}", r))
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
        out.append((seq, off, cf, chunk_hap[g], r0, lens, [n for n, _ in reads]))
        r0 += len(reads)
    return out


def _binds(hb):
    return [(lambda e, b=b: e.set_reads(b[0], b[1], b[2], b[3])) for b in hb]


def _records(sw):
    """device records as oracle tuples, in device order"""
    out = []
    for i in range(len(sw["read"])):
        side = lambda k: (int(sw["strand" + k][i]), int(sw["ids" + k][i]), int(sw["lo" + k][i]), int(sw["hi" + k][i]),
                          (int(sw["id" + k][i]), int(sw["start" + k][i]), int(sw["pos" + k][i])))
        out.append((int(sw["read"][i]), int(sw["contig"][i]), side("1"), side("2")))
    return out


def _bad(eng):
    gt = eng.groups()
    return {(int(gt["contig"][i]), int(gt["group"][i])) for i in eng.bad_list().tolist()}


def _oracle(eng, lens):
    kept = eng.rows(1)
    rows = list(zip(*(kept[c].astype(np.int64).tolist() for c in ("read", "pos", "contig", "start", "group"))))
    return O.switches(rows, dict(enumerate(lens.tolist())), _bad(eng), MINLEN)


def _check_known_answers(recs, names, gaps):
    """one call per inversion with both ends within TOL, no other call, fold-back reads give fold-back records only, and
    no gap at the 20 kb inversion"""
    cl = O.calls(recs)
    errs = []
    for c, x, y in INV:
        hit = [t for t in cl if t[0] == c and abs(t[1] - x) <= TOL and abs(t[2] - y) <= TOL]
        near = [t for t in cl if t[0] == c]
        errs.append([(t[1] - x, t[2] - y) for t in near])
        assert len(hit) == 1, (c, x, y, near)
    print("call end errors (start - x, end - y) per inversion:", errs)
    assert len(cl) == len(INV), cl
    fold = [r for r in recs if names[r[0]].startswith("fold")]
    assert len({r[0] for r in fold}) >= N_FOLD // 2 and all(O.kind(r) == "foldback" for r in fold)
    c, x, y = INV[0]
    for gc, s, e in zip(gaps["contig"].tolist(), gaps["start"].tolist(), gaps["end"].tolist()):
        assert not (gc == c and s < y and e >= x), (gc, s, e)


@pytest.fixture(scope="module")
def planted():
    eng, wl, chunks, chunk_hap = _planted()
    return dict(eng=eng, wl=wl, chunks=chunks, chunk_hap=chunk_hap, oracle={})


def _names_lens(hb):
    return [n for b in hb for n in b[6]], np.concatenate([b[5] for b in hb]).astype(np.uint32)


@pytest.mark.parametrize("split", SPLITS)
def test_records_equal_oracle_and_calls_are_right(planted, split):
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], split)
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
    got = _records(eng.strand_switches(MINLEN))
    names, lens = _names_lens(hb)
    if "want" not in planted["oracle"]:
        planted["oracle"]["want"] = _oracle(eng, lens)
    want = planted["oracle"]["want"]
    assert got == want
    gaps, _ = eng.gaps(wl.contig_len)
    _check_known_answers(want, names, gaps)


def test_two_contexts_equal_one(planted):
    """two contexts on one GPU, half of the batches each, exchanging through parallel.ThreadExchange: the records of the
    two concatenate to the single context's"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    from gavisunk_b200 import workload as W
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], [[0, 1, 2], [3], [4, 5, 6], [7, 8, 9, 10, 11]])
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
    want = _records(eng.strand_switches(MINLEN))
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
            out[i] = engines[i].strand_switches(MINLEN)
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    rec = {c: np.concatenate([out[0][c], out[1][c] + (np.uint32(hb[2][4]) if c == "read" else np.uint32(0))]) for c in out[0]}
    assert _records(rec) == want and len(want) > 0
    eng2.close()


def test_unedited_reads_make_no_call():
    eng, wl, chunks, chunk_hap = _planted(edit=False)
    hb = _host_batches(chunks, chunk_hap, SPLITS[0])
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
    recs = _records(eng.strand_switches(MINLEN))
    names, _ = _names_lens(hb)
    assert any(names[r[0]].startswith("fold") for r in recs)
    assert O.calls(recs) == []
    eng.close()


def test_stage_before_kept_rows_raises():
    from gavisunk_b200.engine import Engine
    from gavisunk_b200._lib import GavisunkError
    e2 = Engine(20)
    with pytest.raises(GavisunkError):
        e2.strand_switches()
    e2.close()


def test_no_launch_and_no_stage_time_without_the_call(planted):
    """run_batches without strand_switches() launches exactly what it launches when the stage follows it, and the stage's
    timer never runs; the stage itself adds launches of its own"""
    from gavisunk_b200._lib import GavisunkError
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], SPLITS[1])
    eng.set_profiling(True)
    counts = []
    try:
        for k in range(2):
            l0 = eng.launches
            eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
            counts.append(eng.launches - l0)
            if k == 0:
                with pytest.raises(GavisunkError):
                    eng.stage_ms("switches")
            l0 = eng.launches
            eng.strand_switches(MINLEN)
            assert eng.launches - l0 > 0 and eng.stage_ms("switches") > 0
    finally:
        eng.set_profiling(False)
    assert counts[0] == counts[1]


# ------------------------------------------------------------------------------------------------
# hand-set rows (gvs_rows_set(1), no database)
# ------------------------------------------------------------------------------------------------
def _across(read, segs, step, pos0=0):
    rows, p = [], pos0
    for lo, hi, d in segs:
        ss = list(range(lo, hi, step)) if d == 0 else list(range(hi - step, lo - step, -step))
        rows += [(read, p + k * step, 0, s, s) for k, s in enumerate(ss)]
        p += hi - lo
    return rows


def _hand_rows(seed=5):
    """read 0: 1300 rows across two inversions; read 1: a read spanning an inversion, rows shuffled (not in pos order);
    reads 2 / 3: monotone on + and -; read 4: a far-away inverted run of exactly 2 IDs; read 5: of exactly 3 IDs; read 6:
    short; read 7: rows on the other contig after its first row"""
    rng = np.random.default_rng(seed)
    rows = _across(0, [(0, 40000, 0), (40000, 60000, 1), (60000, 90000, 0), (90000, 100000, 1), (100000, 130000, 0)], 100)
    r1 = _across(1, [(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)], 500)
    rows += [r1[i] for i in rng.permutation(len(r1))]
    rows += _across(2, [(1000, 61000, 0)], 300) + _across(3, [(1000, 61000, 1)], 300)
    for rd, n_mid in ((4, 2), (5, 3)):
        rows += _across(rd, [(10000, 15000, 0)], 500)
        rows += [(rd, 5000 + k * 500, 0, 100000 + (n_mid - 1 - k) * 500, 100000 + (n_mid - 1 - k) * 500) for k in range(n_mid)]
        rows += _across(rd, [(15000, 25000, 0)], 500, pos0=5000 + n_mid * 500)
    rows += _across(6, [(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)], 500)
    r7 = _across(7, [(10000, 20000, 0), (20000, 30000, 1), (30000, 45000, 0)], 500)
    rows += r7[:1] + [(7, 100 + k, 1, 90000 - 700 * k, 90000 - 700 * k) for k in range(30)] + r7[1:]
    lens = [200000, 60000, 70000, 70000, 30000, 30000, MINLEN - 1, 60000]
    return rows, lens


def _hand_engine(rows, lens):
    from gavisunk_b200.engine import Engine
    eng = Engine(20)
    eng.set_reads_meta(np.asarray(lens, np.uint32))
    cols = [np.asarray([r[k] for r in rows], np.uint32) for k in range(5)]
    eng.set_rows(1, *cols, n_contigs=2)
    eng.set_contigs([0, 0])
    return eng


def test_hand_set_rows_equal_oracle():
    rows, lens = _hand_rows()
    eng = _hand_engine(rows, lens)
    got = _records(eng.strand_switches(MINLEN))
    want = O.switches(rows, dict(enumerate(lens)), minlen=MINLEN)
    assert got == want
    per = {}
    for r in want:
        per[r[0]] = per.get(r[0], 0) + 1
    # read 0 has 8: each of its inverted pieces is shorter than the flanks, whose pairs turn the piece's centre back to '+'
    # (the reflection maps the centre onto itself), so the centre is a '+' block between two '-' blocks
    assert per == {0: 8, 1: 2, 5: 2, 7: 2}, per
    assert sum(1 for r in rows if r[0] == 0) > 1024
    eng.validate(MINLEN)  # the validation's segments are current now: the same records through them
    assert _records(eng.strand_switches(MINLEN)) == want
    eng.close()


def test_hand_set_rows_all_bad():
    rows, lens = _hand_rows()
    eng = _hand_engine(rows, lens)
    keys = sorted({(r[2], r[4]) for r in rows})
    eng.bad_set([c for c, _ in keys], [g for _, g in keys])
    assert _records(eng.strand_switches(MINLEN)) == []
    eng.close()


# ------------------------------------------------------------------------------------------------
# the reference's bundled samples (BASELINE configs 1-2)
# ------------------------------------------------------------------------------------------------
FILES = ("inversions.reads.tsv", "inversions.bed")


def _fused_argv(case, asm, chunks):
    return ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1]]


@pytest.fixture(scope="module", params=["j1_amy_pseudodip", "j1_amy_hg02723"])
def runs(request, tmp_path_factory):
    from gavisunk_b200 import cli
    from gavisunk_b200.engine import Engine
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_inversions")
    asm, fai, chunks = _materialise(case, tmp)
    out = {}
    real = Engine.strand_switches

    def refuse(*a, **kw):
        raise AssertionError("fused without --inversions ran the strand-switch stage")
    for name, extra in (("plain", []), ("inv", ["--inversions"]), ("two", ["--inversions", "--devices", "0,0", "--batch-files", "3"])):
        out[name] = tmp / name
        Engine.strand_switches = refuse if not extra else real
        try:
            assert cli.main(_fused_argv(case, asm, chunks) + ["--outdir", str(out[name])] + extra) == 0, name
        finally:
            Engine.strand_switches = real
    return dict(name=request.param, case=case, tmp=tmp, asm=asm, fai=fai, chunks=chunks, out=out)


def _files(root):
    got = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            got[os.path.relpath(p, root)] = open(p, "rb").read()
    return got


def test_flag_adds_only_its_four_files(runs):
    plain, inv = _files(runs["out"]["plain"]), _files(runs["out"]["inv"])
    new = {os.path.join("final_out", f"hap{h}.{t}") for h in (1, 2) for t in FILES}
    assert set(inv) == set(plain) | new and not (set(plain) & new)
    for k, v in plain.items():
        assert inv[k] == v, k
    two = _files(runs["out"]["two"])
    for k in new:
        assert two[k] == inv[k], k


def _oracle_files(d, h, fai_p):
    """the oracle's two files of haplotype h from fused's sunkpos / rlen / bad_sunks.txt, reads keyed by (contig, name)"""
    from gavisunk_b200 import io as gio
    rd = lambda *p: open(os.path.join(d, *p)).read()
    fai = [(l.split("\t")[0], int(l.split("\t")[1])) for l in open(fai_p).read().splitlines()]
    cidx = {n: i for i, (n, _) in enumerate(fai)}
    rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in rd("sunkpos", f"hap{h}.rlen").splitlines()}
    bad = {(cidx[b.split(":")[0]], int(b.split(":")[1])) for b in rd("sunkpos", "bad_sunks.txt").split() if b.split(":")[0] in cidx}
    rows = [((cidx[c], n), p, cidx[c], s, g) for n, p, c, s, g in dict.fromkeys(gio.read_sunkpos(os.path.join(d, "sunkpos", f"hap{h}.sunkpos")))]
    recs = O.switches(rows, {k: rlen.get(k[1], 0) for k in {r[0] for r in rows}}, bad, 10000)
    return O.texts(recs, fai, range(len(fai)), lambda r: r[1], lambda r: rlen.get(r[1], 0)), recs


def test_files_equal_oracle(runs):
    d = runs["out"]["inv"]
    n = [0, 0]
    for h in (1, 2):
        want, recs = _oracle_files(d, h, runs["fai"][h - 1])
        for t, w in zip(FILES, want):
            assert open(d / "final_out" / f"hap{h}.{t}").read() == w, (h, t)
        n[0] += len(recs)
        n[1] += len(want[1].splitlines())
    print(f"{runs['name']}: {n[0]} records, {n[1]} calls")


def test_shim_reproduces_fused(runs):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["inv"], runs["tmp"]
    for h in (1, 2):
        outs = [str(tmp / f"shim_hap{h}.{t}") for t in FILES]
        assert cli.main(["inversions", str(d / "sunkpos" / f"hap{h}.sunkpos"), str(d / "sunkpos" / f"hap{h}.rlen"),
                         str(d / "sunkpos" / "bad_sunks.txt"), runs["fai"][h - 1], *outs]) == 0
        for t, o in zip(FILES, outs):
            assert open(o, "rb").read() == open(d / "final_out" / f"hap{h}.{t}", "rb").read(), (h, t)


def test_shim_missing_input_writes_nothing(runs, capsys):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["inv"], runs["tmp"]
    outs = [str(tmp / f"missing.{t}") for t in FILES]
    rc = cli.main(["inversions", str(d / "sunkpos" / "hap1.sunkpos"), str(tmp / "no.rlen"), str(d / "sunkpos" / "bad_sunks.txt"),
                   runs["fai"][0], *outs])
    assert rc == 1 and "no.rlen" in capsys.readouterr().err
    assert not any(os.path.exists(o) for o in outs)


REAL_INV = 30000


def test_planted_inversion_on_the_bundled_sample(runs):
    """a 30 kb inversion centred in the plain run's longest hap-1 interval, reads simulated with the sample's own lengths
    and seed from the edited haplotype, fused against the unedited assembly: one call with both ends within TOL"""
    if runs["name"] != "j1_amy_hg02723":
        pytest.skip("one sample is enough")
    from gavisunk_b200 import cli
    case, tmp = runs["case"], runs["tmp"]
    iv = [(p[0], int(p[1]), int(p[2])) for p in (l.split("\t") for l in open(runs["out"]["plain"] / "final_out" / "hap1.valid.bed").read().splitlines())]
    contig, s, e = max(iv, key=lambda t: t[2] - t[1])
    x = (s + e) // 2 - REAL_INV // 2
    y = x + REAL_INV
    haps = [[(n, q.encode()) for n, q in h] for h in case["asm"]]
    haps[0] = [(n, q[:x] + _revcomp(q[x:y]) + q[y:] if n == contig else q) for n, q in haps[0]]
    work = tmp / "planted"
    os.makedirs(work, exist_ok=True)
    chunks = [[], []]
    forbid = tuple(case["forbid"]) if case["forbid"] else None
    for hi_ in range(2):
        reads = S.simulate(haps[hi_], case["lengths"][hi_], case["seed"] + hi_, f"h{hi_ + 1}r", forbid=forbid, skip=case["skip"])
        for ci, part in enumerate(S.split_round_robin(reads, case["nchunks"])):
            p = work / f"hap{hi_ + 1}_{ci + 1}.fq"
            p.write_bytes(S.fastq_text(part))
            chunks[hi_].append(str(p))
    out = work / "results"
    assert cli.main(_fused_argv(case, runs["asm"], chunks) + ["--outdir", str(out), "--inversions"]) == 0
    calls = [l.split("\t") for l in open(out / "final_out" / "hap1.inversions.bed").read().splitlines()]
    print("planted", (contig, x, y), "calls", calls)
    hit = [c for c in calls if c[0] == contig and abs(int(c[1]) - x) <= TOL and abs(int(c[2]) - y) <= TOL]
    assert len(hit) == 1, (contig, x, y, calls)

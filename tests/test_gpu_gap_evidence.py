"""Gap evidence (Engine.gap_evidence, csrc/gap_evidence.cu; `fused --gap-evidence`, `cli gap_evidence`): records against
the CPU oracle (tests/gap_evidence_oracle.py) on assemblies with planted insertions and deletions, one vs several
batches and contexts, and on the reference's bundled samples.  No reference counterpart (viz.py only plots)."""
import os
import sys
import threading

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

import gap_evidence_oracle as O

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

SPLITS = [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]]
MINLEN = 3000
CONTIGS = (300000, 200000)
P, Q, EVENT = 150000, 100000, 6000  # EVENT random bases inserted into contig 0 at P, deleted from contig 1 at Q
# reads stay below 10 x EVENT: a pair of SUNKs across the event then always fails the ratio test, so no read validates
# across it and the event leaves a gap
MAX_LEN = 50000


def _tol(size):
    return 250 + 0.03 * size


def _rname(i):
    return f"r{int(i):08d}"  # bytewise order == read index order


def _planted(seed=51, cov_per_hap=15.0):
    """a synthetic diploid assembly (database built from it unedited) and 12 chunks of reads (6 per haplotype)
    simulated from its hap-1 contigs with the two events planted"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    eng = Engine(20)
    wl = W.make_assembly(eng, list(CONTIGS), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    W.build_db(eng, wl)
    asm = wl.asm.cpu().numpy()
    off = wl.contig_off.cpu().numpy()
    seqs = [asm[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(wl.contig_names))]
    rng = np.random.default_rng(seed)
    seqs[0] = seqs[0][:P] + np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, EVENT)].tobytes() + seqs[0][P:]
    seqs[1] = seqs[1][:Q] + seqs[1][Q + EVENT:]
    nc = len(CONTIGS)
    chunks, chunk_hap = [], []
    for hap in range(2):
        contigs = [(wl.contig_names[hap * nc + i], seqs[hap * nc + i]) for i in range(nc)]
        want = cov_per_hap * sum(len(s) for _, s in contigs)
        lengths = []
        while sum(lengths) < want:
            lengths.append(int(min(MAX_LEN, max(1000, rng.lognormal(np.log(14000), 0.6)))))
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


def _records(ev, gaps):
    """device records as oracle tuples"""
    out = []
    for i in range(len(ev["read"])):
        ds = int(ev["right_start"][i]) - int(ev["left_start"][i])
        dp = abs(int(ev["right_pos"][i]) - int(ev["left_pos"][i]))
        out.append((int(ev["gap"][i]), _rname(ev["read"][i]), (int(ev["left_id"][i]), int(ev["left_start"][i]), int(ev["left_pos"][i])),
                    (int(ev["right_id"][i]), int(ev["right_start"][i]), int(ev["right_pos"][i])), dp - ds, 9 * ds < 10 * dp < 11 * ds))
    return sorted(out, key=lambda t: (t[0], t[1]))


def _oracle(eng, rlen, gaps):
    kept = eng.rows(1)
    rows = [(_rname(r), int(p), int(c), int(s), int(g)) for r, p, c, s, g in
            zip(kept["read"], kept["pos"], kept["contig"], kept["start"], kept["group"])]
    gt = eng.groups()
    bad = {(int(gt["contig"][i]), int(gt["group"][i])) for i in eng.bad_list().tolist()}
    gl = [(int(c), int(s), int(e)) for c, s, e in zip(gaps["contig"], gaps["start"], gaps["end"])]
    return O.gap_evidence(rows, rlen, bad, gl, MINLEN), gl


@pytest.fixture(scope="module")
def planted():
    eng, wl, chunks, chunk_hap = _planted()
    hb = _host_batches(chunks, chunk_hap, SPLITS[0])
    rlen = {_rname(i): int(l) for i, l in enumerate(hb[0][5])}
    return dict(eng=eng, wl=wl, chunks=chunks, chunk_hap=chunk_hap, rlen=rlen, oracle={})


def _check_known_answers(recs, gl):
    summ = O.summary(recs, gl)
    at_p = [s for s in summ if s[0] == 0 and s[1] < P <= s[2] + 1]
    at_q = [s for s in summ if s[0] == 1 and s[1] < Q + EVENT and s[2] >= Q]
    assert len(at_p) == 1 and len(at_q) == 1, (at_p, at_q, gl)
    for s, want in ((at_p[0], EVENT), (at_q[0], -EVENT)):
        assert s[3] >= 3 and s[4] == 0, s
        assert abs(s[6] - want) <= _tol(EVENT), s


@pytest.mark.parametrize("split", SPLITS)
def test_records_equal_oracle(planted, split):
    eng, wl = planted["eng"], planted["wl"]
    eng.run_batches(_binds(_host_batches(planted["chunks"], planted["chunk_hap"], split)), wl.contig_hap, min_read_len=MINLEN)
    gaps, _ = eng.gaps(wl.contig_len)
    got = _records(eng.gap_evidence(MINLEN), gaps)
    if "want" not in planted["oracle"]:
        planted["oracle"]["want"] = _oracle(eng, planted["rlen"], gaps)
    want, gl = planted["oracle"]["want"]
    assert [(int(c), int(s), int(e)) for c, s, e in zip(gaps["contig"], gaps["start"], gaps["end"])] == gl
    assert got == want
    _check_known_answers(got, gl)


def test_two_contexts_equal_one(planted):
    """two contexts on one GPU, half of the batches each, exchanging through parallel.ThreadExchange: every context has
    the same gaps, and the records of the two concatenate to the single context's"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    from gavisunk_b200 import workload as W
    eng, wl = planted["eng"], planted["wl"]
    hb = _host_batches(planted["chunks"], planted["chunk_hap"], [[0, 1, 2], [3], [4, 5, 6], [7, 8, 9, 10, 11]])
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
    gaps, _ = eng.gaps(wl.contig_len)
    want = _records(eng.gap_evidence(MINLEN), gaps)
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
            g, _ = engines[i].gaps(wl.contig_len)
            out[i] = (g, engines[i].gap_evidence(MINLEN))
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    for c in gaps:
        assert (out[0][0][c] == gaps[c]).all() and (out[1][0][c] == gaps[c]).all()
    ev = {c: np.concatenate([out[0][1][c], out[1][1][c] + (np.uint32(hb[2][4]) if c == "read" else np.uint32(0))]) for c in out[0][1]}
    assert _records(ev, gaps) == want and len(want) > 0
    eng2.close()


def test_gap_evidence_before_gaps_raises():
    from gavisunk_b200.engine import Engine
    from gavisunk_b200._lib import GavisunkError
    from gavisunk_b200 import workload as W
    eng = Engine(20)
    wl = W.make_assembly(eng, [90000], snp_rate=2e-3, dup_frac=0.02, seed=45)
    W.build_db(eng, wl)
    W.add_reads(eng, wl, coverage=4.0, n50=14000, sigma=0.6, len_min=200, len_max=300000, seed=46, nchunks=1)
    W.bind_reads(eng, wl)
    eng.run_all(wl.contig_hap, min_read_len=MINLEN)
    with pytest.raises(GavisunkError):
        eng.gap_evidence(MINLEN)
    eng.gaps(wl.contig_len)
    eng.gap_evidence(MINLEN)
    e2 = Engine(20)
    with pytest.raises(GavisunkError):
        e2.gap_evidence()
    e2.close()
    eng.close()


# ------------------------------------------------------------------------------------------------
# the reference's bundled samples (BASELINE configs 1-2)
# ------------------------------------------------------------------------------------------------
FILES = ("gaps.reads.tsv", "gaps.evidence.tsv")


def _fused_argv(case, asm, chunks):
    return ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1]]


@pytest.fixture(scope="module", params=["j1_amy_pseudodip", "j1_amy_hg02723"])
def runs(request, tmp_path_factory):
    from gavisunk_b200 import cli
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_gapev")
    asm, fai, chunks = _materialise(case, tmp)
    out = {}
    for name, extra in (("plain", []), ("ev", ["--gap-evidence"]), ("two", ["--gap-evidence", "--devices", "0,0", "--batch-files", "3"])):
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
    plain, ev = _files(runs["out"]["plain"]), _files(runs["out"]["ev"])
    new = {os.path.join("final_out", f"hap{h}.{t}") for h in (1, 2) for t in FILES}
    assert set(ev) == set(plain) | new and not (set(plain) & new)
    for k, v in plain.items():
        assert ev[k] == v, k
    two = _files(runs["out"]["two"])
    for k in new:
        assert two[k] == ev[k], k


def _read_files(d, h):
    rd = lambda *p: open(os.path.join(d, *p)).read()
    gaps = [(p[0], int(p[1]), int(p[2])) for p in (l.split("\t") for l in rd("final_out", f"hap{h}.gaps.bed").splitlines())]
    rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in rd("sunkpos", f"hap{h}.rlen").splitlines()}
    bad = {(b.split(":")[0], int(b.split(":")[1])) for b in rd("sunkpos", "bad_sunks.txt").split()}
    from gavisunk_b200 import io as gio
    rows = gio.read_sunkpos(os.path.join(d, "sunkpos", f"hap{h}.sunkpos"))
    return gaps, rlen, bad, rows, rd


def _check_against_oracle(d, h):
    gaps, rlen, bad, rows, rd = _read_files(d, h)
    recs = O.gap_evidence(rows, rlen, bad, gaps)
    reads = rd("final_out", f"hap{h}.gaps.reads.tsv").splitlines()
    assert reads[0].split("\t") == ["contig", "gap_start", "gap_end", "read", "read_len", "left_id", "left_start", "left_pos", "right_id",
                                    "right_start", "right_pos", "delta", "consistent"]
    assert reads[1:] == O.reads_tsv_lines(recs, gaps, rlen)
    ev = [l.split("\t") for l in rd("final_out", f"hap{h}.gaps.evidence.tsv").splitlines()]
    assert ev[0] == ["contig", "start", "end", "bridging_reads", "consistent_reads", "min_delta", "median_delta", "max_delta"]
    assert ev[1:] == [[str(x) if x is not None else "." for x in s] for s in O.summary(recs, gaps)]
    return gaps, recs


def test_files_equal_oracle(runs):
    for h in (1, 2):
        _check_against_oracle(runs["out"]["ev"], h)
    if runs["name"] == "j1_amy_hg02723":  # README.md:36-37: nothing reaches both sides of the desert
        ev = open(runs["out"]["ev"] / "final_out" / "hap1.gaps.evidence.tsv").read()
        assert "AMY_h1\t284861\t324275\t0\t0\t.\t.\t.\n" in ev


def test_shim_reproduces_fused(runs):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["ev"], runs["tmp"]
    for h in (1, 2):
        outs = [str(tmp / f"shim_hap{h}.{t}") for t in FILES]
        assert cli.main(["gap_evidence", str(d / "sunkpos" / f"hap{h}.sunkpos"), str(d / "sunkpos" / f"hap{h}.rlen"),
                         str(d / "sunkpos" / "bad_sunks.txt"), runs["fai"][h - 1], str(d / "final_out" / f"hap{h}.valid.bed"), *outs]) == 0
        for t, o in zip(FILES, outs):
            assert open(o, "rb").read() == open(d / "final_out" / f"hap{h}.{t}", "rb").read(), (h, t)


def test_shim_missing_input_writes_nothing(runs, capsys):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["ev"], runs["tmp"]
    outs = [str(tmp / f"missing.{t}") for t in FILES]
    rc = cli.main(["gap_evidence", str(d / "sunkpos" / "hap1.sunkpos"), str(tmp / "no.rlen"), str(d / "sunkpos" / "bad_sunks.txt"),
                   runs["fai"][0], str(d / "final_out" / "hap1.valid.bed"), *outs])
    assert rc == 1 and "no.rlen" in capsys.readouterr().err
    assert not any(os.path.exists(o) for o in outs)


# the bundled sample's reads reach 523 kb: an insertion is only left unvalidated (a gap) when it exceeds a tenth of the
# assembly span of every read across it (the ratio test then fails for every pair of SUNKs across it)
REAL_INSERT = 60000


def test_planted_insertion_on_the_bundled_sample(runs):
    """an insertion at the midpoint of the plain run's longest hap-1 interval, reads simulated with the sample's own
    lengths and seed from the edited haplotype, fused against the unedited assembly: a new gap holds the insertion
    point and its reads recover the size"""
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
    assert cli.main(_fused_argv(case, runs["asm"], chunks) + ["--outdir", str(out), "--gap-evidence"]) == 0
    gaps, recs = _check_against_oracle(out, 1)
    summ = O.summary(recs, gaps)
    hit = [g for g in summ if g[0] == contig and g[1] < x <= g[2] + 1]
    assert len(hit) == 1, (x, gaps)
    assert hit[0][3] >= 3 and hit[0][4] == 0, hit
    assert abs(hit[0][6] - REAL_INSERT) <= _tol(REAL_INSERT), hit

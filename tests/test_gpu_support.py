"""Support tracks of the validated reads (Engine.placements / Engine.support, csrc/support.cu; `fused --support-tracks`,
`cli support_tracks`): placements and depth runs against the oracle, one vs several batches and contexts, and on the
reference's bundled samples against the committed inter_outs goldens.  No reference counterpart (viz.py only plots)."""
import os
import threading

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

import support_oracle as O

SPLITS = [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]]
MINLEN = 3000


def _setup(seed=41, contig_lens=(350000, 120000), cov=18.0, n50=14000, nchunks=6, k=20):
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    eng = Engine(k)
    wl = W.make_assembly(eng, list(contig_lens), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    W.build_db(eng, wl)
    W.add_reads(eng, wl, coverage=cov, n50=n50, sigma=0.6, len_min=200, len_max=300000, seed=seed + 1, nchunks=nchunks)
    return eng, wl


def _host_batches(wl, groups):
    reads = wl.reads.cpu().numpy()
    off = wl.read_off.cpu().numpy().astype(np.uint64)
    cf = wl.chunk_first.astype(np.int64)
    out = []
    for g in groups:
        r0, r1 = int(cf[g[0]]), int(cf[g[-1] + 1])
        o = (off[r0:r1 + 1] - off[r0]).astype(np.uint64)
        out.append((reads[int(off[r0]):int(off[r1])].copy(), o, (cf[g[0]:g[-1] + 2] - r0).astype(np.uint64),
                    wl.chunk_hap[g[0]:g[-1] + 1].copy(), r0))
    return out


def _binds(hb):
    return [(lambda e, b=b: e.set_reads(b[0], b[1], b[2], b[3])) for b in hb]


def _rname(i):
    return f"r{int(i):08d}"  # bytewise order == read index order


def _tuples(pl, runs):
    p = sorted((int(c), int(s), int(e), _rname(r), int(n), "-" if st else "+")
               for c, s, e, r, n, st in zip(pl["contig"], pl["start"], pl["end"], pl["read"], pl["n_ids"], pl["strand"]))
    r = [(int(c), int(s), int(e), int(d)) for c, s, e, d in zip(runs["contig"], runs["start"], runs["end"], runs["depth"])]
    return p, r


_ORACLE = {}


def _oracle(eng, wl, key):
    """oracle placements / runs from the engine's kept rows and bad groups (the same for every split of one workload)"""
    if key in _ORACLE:
        return _ORACLE[key]
    kept = eng.rows(1)
    rlen = np.diff(wl.read_off.cpu().numpy().astype(np.int64))
    rows = [(_rname(r), int(p), int(c), int(s), int(g)) for r, p, c, s, g in
            zip(kept["read"], kept["pos"], kept["contig"], kept["start"], kept["group"])]
    gt = eng.groups()
    bad = {(int(gt["contig"][i]), int(gt["group"][i])) for i in eng.bad_list().tolist()}
    fai = [(c, int(L)) for c, L in enumerate(wl.contig_len)]
    pls, runs = O.support_tracks(rows, {_rname(i): int(L) for i, L in enumerate(rlen)}, bad, fai, minlen=MINLEN)
    _ORACLE[key] = (sorted(pls), runs)
    return _ORACLE[key]


def _check_identities(pl, runs, iv, contig_len):
    ln = runs["end"].astype(np.int64) - runs["start"].astype(np.int64)
    assert (ln > 0).all()
    assert int((runs["depth"].astype(np.int64) * ln).sum()) == int((pl["end"].astype(np.int64) - pl["start"]).sum())
    for c, L in enumerate(contig_len):  # every contig tiled exactly by maximal runs
        m = runs["contig"] == c
        s, e, d = runs["start"][m], runs["end"][m], runs["depth"][m]
        assert s[0] == 0 and e[-1] == L and (s[1:] == e[:-1]).all() and (d[1:] != d[:-1]).all()
    for c, a, b in zip(iv["contig"], iv["start"], iv["end"]):  # validated intervals are supported at every base
        m = (runs["contig"] == c) & (runs["end"] > a) & (runs["start"] < b)
        assert m.any() and runs["depth"][m].min() >= 1, (c, a, b)


@pytest.mark.parametrize("split", SPLITS)
def test_support_equals_oracle(split):
    eng, wl = _setup()
    iv, _ = eng.run_batches(_binds(_host_batches(wl, split)), wl.contig_hap, min_read_len=MINLEN)
    pl = eng.placements()
    runs = eng.support(wl.contig_len)
    got_p, got_r = _tuples(pl, runs)
    want_p, want_r = _oracle(eng, wl, 41)
    assert len(want_p) > 50 and {p[5] for p in want_p} == {"+", "-"}
    assert got_p == want_p
    assert got_r == want_r
    _check_identities(pl, runs, iv, wl.contig_len)
    # the same run in one batch gives the same tracks
    from gavisunk_b200 import workload as W
    W.bind_reads(eng, wl)
    eng.run_all(wl.contig_hap, min_read_len=MINLEN)
    assert _tuples(eng.placements(), eng.support(wl.contig_len)) == (got_p, got_r)


def test_two_contexts_equal_one():
    """two contexts on one GPU, half of the batches each, exchanging through parallel.ThreadExchange: the difference
    arrays are summed by the callable that sums the bad-SUNK histogram"""
    from gavisunk_b200.engine import Engine
    from gavisunk_b200.parallel import ThreadExchange
    from gavisunk_b200 import workload as W
    eng, wl = _setup(seed=43, nchunks=4)
    hb = _host_batches(wl, [[0, 1, 2], [3], [4, 5], [6, 7]])
    eng.run_batches(_binds(hb), wl.contig_hap, min_read_len=MINLEN)
    want = _tuples(eng.placements(), eng.support(wl.contig_len))
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
            pl = engines[i].placements()
            out[i] = (pl, engines[i].support(wl.contig_len, allreduce=cx.allreduce_hist))
        except BaseException as ex:  # noqa: BLE001
            errs.append(ex)
            xch.abort()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errs, errs
    pl = {c: np.concatenate([out[0][0][c], out[1][0][c] + (np.uint32(hb[2][4]) if c == "read" else 0)]) for c in out[0][0]}
    for i in range(2):
        assert _tuples(pl, out[i][1]) == want
    eng2.close()


def test_placements_before_validate_raises():
    from gavisunk_b200.engine import Engine
    from gavisunk_b200._lib import GavisunkError
    eng, wl = _setup(seed=45, contig_lens=(90000,), cov=4.0, nchunks=1)
    with pytest.raises(GavisunkError):
        eng.placements()
    e2 = Engine(20)
    with pytest.raises(GavisunkError):
        e2.support([1000])
    e2.close()


# ------------------------------------------------------------------------------------------------
# the reference's bundled samples (BASELINE configs 1-2)
# ------------------------------------------------------------------------------------------------
TRACKS = ("reads.bed", "support.bedgraph", "support.tsv")


@pytest.fixture(scope="module", params=["j1_amy_pseudodip", "j1_amy_hg02723"])
def runs(request, tmp_path_factory):
    from gavisunk_b200 import cli
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_support")
    asm, fai, chunks = _materialise(case, tmp)
    base = ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1]]
    out = {}
    for name, extra in (("plain", []), ("tracks", ["--support-tracks"]), ("two", ["--support-tracks", "--devices", "0,0"])):
        out[name] = tmp / name
        assert cli.main(base + ["--outdir", str(out[name])] + extra) == 0, name
    return dict(name=request.param, case=case, tmp=tmp, fai=fai, out=out)


def _files(root):
    got = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            got[os.path.relpath(p, root)] = open(p, "rb").read()
    return got


def test_fused_tracks_leave_other_outputs_unchanged(runs):
    plain, tracks = _files(runs["out"]["plain"]), _files(runs["out"]["tracks"])
    new = {os.path.join("final_out", f"hap{h}.{t}") for h in (1, 2) for t in TRACKS}
    assert set(tracks) == set(plain) | new and not (set(plain) & new)
    for k, v in plain.items():
        assert tracks[k] == v, k
    two = _files(runs["out"]["two"])
    for k in new:
        assert two[k] == tracks[k], k


def test_placements_match_reference_inter_outs(runs):
    """start / end / n_ids of every placement = min / max / count of the read's IDs in the reference's own inter_outs"""
    case, d = runs["case"], runs["out"]["tracks"]
    got = {}
    for h in (1, 2):
        for l in open(d / "final_out" / f"hap{h}.reads.bed").read().splitlines():
            c, s, e, r, n, st, rl = l.split("\t")
            assert st in "+-" and int(rl) >= 10000
            got[(c.replace("#", "_") + f"_hap{h}", r)] = (int(s), int(e), int(n))
    want = {}
    for stem, txt in case["inter_outs"].items():
        ids = {}
        for l in txt.splitlines():
            p = l.split("\t")
            if len(p) == 2:
                ids.setdefault(p[1], []).append(int(p[0]))
        for r, v in ids.items():
            if len(set(v)) >= 2:
                want[(stem, r)] = (min(v), max(v), len(set(v)))
    assert len(want) > 10 and got == want


def test_track_identities(runs):
    d = runs["out"]["tracks"]
    for h in (1, 2):
        fai = [l.split("\t")[:2] for l in open(runs["fai"][h - 1]).read().splitlines()]
        bg = [l.split("\t") for l in open(d / "final_out" / f"hap{h}.support.bedgraph").read().splitlines()]
        bed = [l.split("\t") for l in open(d / "final_out" / f"hap{h}.reads.bed").read().splitlines()]
        valid = [l.split("\t") for l in open(d / "final_out" / f"hap{h}.valid.bed").read().splitlines()]
        tsv = [l.split("\t") for l in open(d / "final_out" / f"hap{h}.support.tsv").read().splitlines()]
        assert tsv[0] == ["contig", "length", "reads", "validated_bases", "covered_bases", "depth_bases", "max_depth", "min_valid_depth"]
        assert [t[:2] for t in tsv[1:]] == fai and [r[0] for r in bg] == sorted([r[0] for r in bg], key=[f[0] for f in fai].index)
        assert sum(int(t[5]) for t in tsv[1:]) == sum(int(b[2]) - int(b[1]) for b in bed)
        for c, s, e in valid:
            depth = [int(r[3]) for r in bg if r[0] == c and int(r[2]) > int(s) and int(r[1]) < int(e)]
            assert depth and min(depth) >= 1
        for t in tsv[1:]:
            rows = [r for r in bg if r[0] == t[0]]
            assert int(rows[0][1]) == 0 and int(rows[-1][2]) == int(t[1])
            assert int(t[4]) == sum(int(r[2]) - int(r[1]) for r in rows if int(r[3]) > 0)
            assert int(t[2]) == sum(1 for b in bed if b[0] == t[0])
            assert (t[7] == ".") == (not any(v[0] == t[0] for v in valid))
    if runs["name"] == "j1_amy_hg02723":  # README's gap: no placement inside it, else the two intervals would be joined
        bg = [l.split("\t") for l in open(d / "final_out" / "hap1.support.bedgraph").read().splitlines()]
        cover = [r for r in bg if r[0] == "AMY_h1" and int(r[1]) <= 284861 and int(r[2]) >= 324276]
        assert len(cover) == 1 and cover[0][3] == "0"


def test_shim_reproduces_fused_tracks(runs):
    """the per-rule shim on fused's own sunkpos / rlen / bad_sunks.txt / valid.bed (groups in first-appearance order: the
    rank is computed, not the identity)"""
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["tracks"], runs["tmp"]
    for h in (1, 2):
        outs = [str(tmp / f"shim_hap{h}.{t}") for t in TRACKS]
        assert cli.main(["support_tracks", str(d / "sunkpos" / f"hap{h}.sunkpos"), str(d / "sunkpos" / f"hap{h}.rlen"),
                         str(d / "sunkpos" / "bad_sunks.txt"), runs["fai"][h - 1], str(d / "final_out" / f"hap{h}.valid.bed"),
                         *outs]) == 0
        for t, o in zip(TRACKS, outs):
            assert open(o, "rb").read() == open(d / "final_out" / f"hap{h}.{t}", "rb").read(), (h, t)


def test_shim_missing_input_writes_nothing(runs, capsys):
    from gavisunk_b200 import cli
    d, tmp = runs["out"]["tracks"], runs["tmp"]
    outs = [str(tmp / f"missing.{t}") for t in TRACKS]
    rc = cli.main(["support_tracks", str(d / "sunkpos" / "hap1.sunkpos"), str(tmp / "no.rlen"), str(d / "sunkpos" / "bad_sunks.txt"),
                   runs["fai"][0], str(d / "final_out" / "hap1.valid.bed"), *outs])
    assert rc == 1 and "no.rlen" in capsys.readouterr().err
    assert not any(os.path.exists(o) for o in outs)

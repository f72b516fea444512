"""Read haplotypes (Engine.diag_filter(read_haps=True) / Engine.read_haps, csrc/diag.cu haplotype mode; `fused --reads`,
`fused --read-haplotypes`): records and kept rows against the CPU oracle (tests/read_haps_oracle.py) on a synthetic
diploid with chunks binned right, binned wrong, mixed and unbinned, over several batch splits and two contexts; hand-set
rows with segments of more than 1024 rows and Table ties; binned runs unchanged by the flag; unbinned runs of the
bundled samples.  No reference counterpart."""
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

import read_haps_oracle as O

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

CONTIGS = (200000, 150000, 120000)  # per haplotype
ANY = 2
# chunk i: (true haplotype of its reads ('m': both), chunk haplotype given to the filter)
CHUNKS = [(0, 0), (1, 1), (1, 0), ("m", ANY), (0, ANY), ("m", 1), (1, ANY), ("m", 0)]
SPLITS = [[list(range(8))], [[0, 1, 2], [3], [4, 5, 6, 7]], [[i] for i in range(8)]]
NONE = 0xFFFFFFFF


def _rname(i):
    return f"r{int(i):08d}"  # bytewise order == run-wide index order


@pytest.fixture(scope="module")
def diploid():
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    tmp = Engine(20)
    wl = W.make_assembly(tmp, list(CONTIGS), snp_rate=2e-3, dup_frac=0.02, seed=71)
    asm, off = wl.asm.cpu().numpy(), wl.contig_off.cpu().numpy()
    names = list(wl.contig_names)
    seqs = [asm[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(names))]
    tmp.close()
    nc = len(CONTIGS)
    rng = np.random.default_rng(71)
    per_hap = []
    for hap in range(2):
        contigs = [(names[hap * nc + i], seqs[hap * nc + i]) for i in range(nc)]
        want = 12.0 * sum(len(s) for _, s in contigs)
        lengths = []
        while sum(lengths) < want:
            lengths.append(int(min(60000, max(1000, rng.lognormal(np.log(12000), 0.7)))))
        per_hap.append(S.split_round_robin(S.simulate(contigs, lengths, 80 + hap, f"h{hap + 1}_"), 8))
    chunks, chunk_hap = [], []
    for i, (truth, given) in enumerate(CHUNKS):
        chunks.append(per_hap[0][i][::2] + per_hap[1][i][1::2] if truth == "m" else per_hap[truth][i])
        chunk_hap.append(given)
    truth = [int(n.startswith("h2_")) for ch in chunks for n, _ in ch]
    eng = Engine(20)
    eng.build_db(list(zip(names, seqs)))
    contig_hap = np.asarray([0] * nc + [1] * nc, np.uint8)
    return dict(eng=eng, names=names, db=list(zip(names, seqs)), contig_hap=contig_hap, chunks=chunks,
                chunk_hap=np.asarray(chunk_hap, np.uint8), truth=truth)


def _host_batches(chunks, chunk_hap, groups):
    out = []
    for g in groups:
        reads = [r for c in g for r in chunks[c]]
        off = np.zeros(len(reads) + 1, np.uint64)
        off[1:] = np.cumsum([len(s) for _, s in reads])
        cf = np.cumsum([0] + [len(chunks[c]) for c in g]).astype(np.uint64)
        out.append((np.frombuffer(b"".join(s for _, s in reads), np.uint8), off, cf, chunk_hap[g]))
    return out


def _run(eng, d, groups, read_haps=True):
    """run_batches over the chunks grouped as `groups` (its intervals left in d["iv"]); -> (engine, match rows per chunk
    as oracle rows)"""
    hb = _host_batches(d["chunks"], d["chunk_hap"], groups)
    names = d["names"]
    per_chunk = []

    def on_batch(e, b, base):
        r = e.rows(0)
        rows = list(zip((_rname(x + base) for x in r["read"].tolist()), r["pos"].tolist(), (names[c] for c in r["contig"].tolist()),
                        r["start"].tolist(), r["group"].tolist()))
        cf = hb[b][2]
        for c in range(len(cf) - 1):
            lo, hi = _rname(int(cf[c]) + base), _rname(int(cf[c + 1]) + base)
            per_chunk.append([x for x in rows if lo <= x[0] < hi])
    iv, _ = eng.run_batches([(lambda e, b=b: e.set_reads(b[0], b[1], b[2], b[3])) for b in hb], d["contig_hap"], min_read_len=3000,
                            on_batch=on_batch, read_haps=read_haps)
    d["iv"] = iv
    return eng, per_chunk


def _records(rh, names):
    sd = "+-"
    vote = lambda i, k: None if int(rh["contig" + k][i]) == NONE else (names[int(rh["contig" + k][i])], int(rh["n" + k][i]),
                                                                       sd[int(rh["strand" + k][i])])
    hap = {0: 0, 1: 1, 2: "tie"}
    return [(_rname(rh["read"][i]), vote(i, "1"), vote(i, "2"), hap[int(rh["hap"][i])]) for i in range(len(rh["read"]))]


def _kept(eng, names):
    k = eng.rows(1)
    return list(zip((_rname(x) for x in k["read"].tolist()), k["pos"].tolist(), (names[c] for c in k["contig"].tolist()),
                    k["start"].tolist(), k["group"].tolist()))


def _oracle(d, per_chunk):
    hap_sets = [{n for n, h in zip(d["names"], d["contig_hap"]) if h == k} for k in range(2)]
    return O.read_haps(list(zip(d["chunk_hap"].tolist(), per_chunk)), hap_sets)


@pytest.mark.parametrize("split", range(len(SPLITS)))
def test_records_and_kept_rows_equal_oracle(diploid, split):
    eng, per_chunk = _run(diploid["eng"], diploid, SPLITS[split])
    want = _oracle(diploid, per_chunk)
    got = _records(eng.read_haps(), diploid["names"])
    assert len(want["records"]) > 100
    assert got == want["records"]
    assert sorted(_kept(eng, diploid["names"])) == sorted(want["kept"])
    if split == 0:
        diploid["want"] = want


def test_two_contexts_equal_one(diploid):
    """a second context, batches split differently: the same records"""
    from gavisunk_b200.engine import Engine
    e2 = Engine(20)
    try:
        e2.build_db(diploid["db"])
        _, per_chunk = _run(e2, diploid, SPLITS[1])
        assert _records(e2.read_haps(), diploid["names"]) == _oracle(diploid, per_chunk)["records"]
    finally:
        e2.close()


def test_assignment_against_truth(diploid, capsys):
    eng, _ = _run(diploid["eng"], diploid, SPLITS[0])
    rh = eng.read_haps()
    truth = np.asarray(diploid["truth"])
    a = rh["hap"] <= 1
    wrong = int((rh["hap"][a] != truth[rh["read"][a]]).sum())
    voted = len(rh["read"])
    with capsys.disabled():
        print(f"\nsynthetic diploid: {voted} voted reads of {len(truth)}, {int(a.sum())} assigned, {wrong} to the wrong "
              f"haplotype, {int((rh['hap'] == 2).sum())} ties")
    assert wrong <= 0.005 * voted


def test_binned_flag_changes_nothing(diploid):
    """read_haps on binned input: kept rows, best rows, pairs, intervals and gaps as without it; without it the
    haplotype kernels never run"""
    d = dict(diploid, chunk_hap=np.asarray([h if h != ANY else 0 for h in diploid["chunk_hap"]], np.uint8))
    eng = d["eng"]
    cl = np.asarray([CONTIGS[i % len(CONTIGS)] for i in range(2 * len(CONTIGS))], np.uint32)
    out = []
    for flag in (False, True):
        l0 = eng.launches
        _run(eng, d, SPLITS[1], read_haps=flag)
        n = eng.launches - l0
        kept = eng.rows(1)
        pairs, iv = eng.pairs(), d["iv"]
        gaps, nodata = eng.gaps(cl)
        out.append((n, [kept[c].tolist() for c in eng.ROW_COLUMNS], [pairs[c].tolist() for c in eng.PAIR_COLUMNS],
                    [iv[c].tolist() for c in iv], [gaps[c].tolist() for c in gaps], nodata.tolist()))
        if not flag:
            from gavisunk_b200.engine import GavisunkError
            with pytest.raises(GavisunkError):
                eng.read_haps()
    assert out[0][1:] == out[1][1:]
    assert out[1][0] > out[0][0]


def test_best_rows_unchanged_by_flag(diploid):
    eng = diploid["eng"]
    hb = _host_batches(diploid["chunks"], np.asarray([1 if h == 1 else 0 for h in diploid["chunk_hap"]], np.uint8), [list(range(8))])
    best = []
    for flag in (False, True):
        eng.set_reads(*hb[0])
        eng.match()
        eng.diag_filter(diploid["contig_hap"], read_haps=flag)
        b = eng.best()
        best.append([b[c].tolist() for c in ("read", "contig", "ngood", "dir")])
    assert best[0] == best[1]


# ---- hand-set rows: big segments, Table ties decided by the other haplotype's contigs ----
def _hand_chunks():
    X, Y = "h1tg000000l", "h1tg000001l"  # Nim hash slots 29 < 36 at capacity 64, 93 > 36 at capacity 128
    step = 3000
    run = lambda r, c, n, first, pos0=0, rev=False: [(r, pos0 + k * step, c, i, i) for k, i in
                                                      enumerate(sorted((first + j * step for j in range(n)), reverse=rev))]
    filler = lambda r, n1, n2: (run(r, "A", 3, 100000) + [(r, 5000000 + k, f"f1_{k}", 0, 0) for k in range(n1)]
                                + [(r, 6000000 + k, f"f2_{k}", 0, 0) for k in range(n2)])
    tie = lambda r: run(r, "C", 2, 900000) + run(r, X, 3, 100000) + run(r, Y, 3, 300000, 9000)
    big = lambda r, na, nc: run(r, "A", na, 100000) + run(r, "C", nc, 200000, 10 ** 7, rev=True)
    chunks = [
        (ANY, filler("a0", 10, 32) + tie("a1") + big("a2", 1500, 1200)),
        (ANY, filler("b0", 10, 33) + tie("b1") + big("b2", 1100, 1100) + tie("b3")),
        (0, big("c0", 1030, 1300) + filler("c1", 10, 33) + tie("c2")),
        (1, tie("d0") + big("d1", 2000, 10)),
    ]
    hap = [{"A", "B", X, Y} | {f"f1_{k}" for k in range(10)}, {"C", "D"} | {f"f2_{k}" for k in range(34)}]
    return chunks, hap


def test_hand_set_rows_equal_oracle():
    from gavisunk_b200.engine import Engine
    chunks, hap = _hand_chunks()
    want = O.read_haps(chunks, hap)
    cnames, cidx, rnames = [], {}, []
    cols = ([], [], [], [], [])
    cf, chap = [0], []
    for h, rows in chunks:
        for r, p, c, s, g in rows:
            if c not in cidx:
                cidx[c] = len(cnames)
                cnames.append(c)
            if not rnames or rnames[-1] != r:
                rnames.append(r)
            for col, v in zip(cols, (len(rnames) - 1, p, cidx[c], s, g)):
                col.append(v)
        cf.append(len(rnames))
        chap.append(h)
    eng = Engine(20)
    try:
        eng.contig_names = cnames
        eng.set_reads_meta(np.full(len(rnames), 20000, np.uint32), cf, chap)
        eng.set_rows(0, *cols)
        eng.diag_filter([0 if c in hap[0] else 1 for c in cnames], read_haps=True)
        rh, kept = eng.read_haps(), eng.rows(1)
    finally:
        eng.close()
    sd, hp = "+-", {0: 0, 1: 1, 2: "tie"}
    vote = lambda i, k: None if int(rh["contig" + k][i]) == NONE else (cnames[int(rh["contig" + k][i])], int(rh["n" + k][i]),
                                                                       sd[int(rh["strand" + k][i])])
    got = [(rnames[int(rh["read"][i])], vote(i, "1"), vote(i, "2"), hp[int(rh["hap"][i])]) for i in range(len(rh["read"]))]
    assert got == want["records"]
    assert ("b1", ("h1tg000001l", 3, "+"), ("C", 2, "+"), 0) in got and ("a1", ("h1tg000000l", 3, "+"), ("C", 2, "+"), 0) in got
    got_kept = list(zip((rnames[x] for x in kept["read"].tolist()), kept["pos"].tolist(), (cnames[c] for c in kept["contig"].tolist()),
                        kept["start"].tolist(), kept["group"].tolist()))
    assert got_kept == want["kept"]


# ---- the bundled samples, unbinned ----
SAMPLES = ["j1_amy_pseudodip", "j1_amy_hg02723"]


@pytest.fixture(scope="module", params=SAMPLES)
def j1u(request, tmp_path_factory):
    """the sample's chunk files, a binned run of them, and the same reads re-chunked into 7 mixed files"""
    from test_j1_configs import _materialise
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param + "_unbinned")
    asm, fai, chunks = _materialise(case, tmp)
    haps = [[(n, s.encode()) for n, s in h] for h in case["asm"]]
    forbid = tuple(case["forbid"]) if case["forbid"] else None
    reads = [S.simulate(haps[hi], case["lengths"][hi], case["seed"] + hi, f"h{hi + 1}r", forbid=forbid, skip=case["skip"])
             for hi in range(2)]
    per_file = [part for hi in range(2) for part in S.split_round_robin(reads[hi], case["nchunks"])]
    mixed_parts = S.split_round_robin(reads[0][::2] + reads[1] + reads[0][1::2], 7)
    mixed = []
    for i, part in enumerate(mixed_parts):
        p = tmp / f"mixed_{i + 1}-of-7.fq"
        p.write_bytes(S.fastq_text(part))
        mixed.append(str(p))
    j = dict(name=request.param, case=case, tmp=tmp, asm=asm, chunks=chunks[0] + chunks[1], per_file=per_file, mixed=mixed,
             mixed_parts=mixed_parts, haps=haps)
    from gavisunk_b200 import cli
    argv = ["fused", "--k", str(case["k"]), "--hap1-asm", asm[0], "--hap2-asm", asm[1], "--hap1-reads", *chunks[0],
            "--hap2-reads", *chunks[1], "--outdir", str(tmp / "binned")]
    assert cli.main(argv) == 0
    j["binned"] = _tree(tmp / "binned")
    return j


def _fused(j, outdir, files, *extra):
    from gavisunk_b200 import cli
    argv = ["fused", "--k", str(j["case"]["k"]), "--hap1-asm", j["asm"][0], "--hap2-asm", j["asm"][1], "--reads", *files,
            "--outdir", str(outdir), *extra]
    assert cli.main(argv) == 0
    return _tree(outdir)


def _tree(d):
    out = {}
    for dp, _, fns in os.walk(d):
        for fn in fns:
            p = os.path.join(dp, fn)
            out[os.path.relpath(p, d)] = open(p, "rb").read()
    return out


def _oracle_unbinned(j, parts):
    """match rows of every chunk (one chunk per batch, GVS_HAP_ANY) through the oracle's read haplotypes"""
    from gavisunk_b200.engine import Engine
    eng = Engine(j["case"]["k"])
    try:
        db = [c for h in j["haps"] for c in h]
        eng.build_db(db)
        names = [n for n, _ in db]
        chunks = []
        for part in parts:
            off = np.zeros(len(part) + 1, np.uint64)
            off[1:] = np.cumsum([len(s) for _, s in part])
            eng.set_reads(np.frombuffer(b"".join(s for _, s in part), np.uint8), off, [0, len(part)], [ANY])
            eng.match()
            r = eng.rows(0)
            chunks.append((ANY, list(zip((part[x][0] for x in r["read"].tolist()), r["pos"].tolist(),
                                         (names[c] for c in r["contig"].tolist()), r["start"].tolist(), r["group"].tolist()))))
        hap_sets = [{n for n, _ in h} for h in j["haps"]]
        want = O.read_haps(chunks, hap_sets)
        read_names = [n for part in parts for n, _ in part]
        fh = O.file_haps(read_names, [ANY] * len(read_names), want["assigned"])
        return want, dict(zip(read_names, fh))
    finally:
        eng.close()


def _check_unbinned(j, got, parts):
    want, fh = _oracle_unbinned(j, parts)
    rows = lambda t: sorted(l for l in t.decode().splitlines())
    kept = rows(got["sunkpos/hap1.sunkpos"] + got["sunkpos/hap2.sunkpos"])
    assert kept == sorted("\t".join(map(str, r)) for r in want["kept"])
    for hn in (1, 2):
        rl = [l.split("\t")[0] for l in got[f"sunkpos/hap{hn}.rlen"].decode().splitlines()]
        assert rl and all(fh[n] == hn - 1 for n in rl)
    assert sum(len(got[f"sunkpos/hap{hn}.rlen"].decode().splitlines()) for hn in (1, 2)) == len(fh)
    # against the true haplotype (read names h1r... / h2r...)
    voted = wrong = 0
    for hn in (1, 2):
        for l in got[f"final_out/hap{hn}.haplotype.reads.tsv"].decode().splitlines()[1:]:
            f = l.split("\t")
            voted += 1
            wrong += f[-1] in ("hap1", "hap2") and f[-1][-1] != f[0][1]
    return voted, wrong, _check_oracle_pipeline(j, got)


def _check_oracle_pipeline(j, got):
    """bad SUNKs, inter_outs, bed_files, valid.bed, gaps and nodata of the run equal the oracle's Python stages run on
    the run's own hap{N}.sunkpos rows and hap{N}.rlen lengths (the file-haplotype split); -> the oracle's hap-1 mode"""
    import gavisunk_oracle as G
    from gavisunk_b200 import io as gio
    txt = lambda p: got.get(p, b"").decode()
    rows = {h: gio.parse_sunkpos(txt(f"sunkpos/hap{h}.sunkpos")) for h in ("1", "2")}
    fai = {h: [(l.split("\t")[0], int(l.split("\t")[1])) for l in j["case"][f"fai{h}"].splitlines()] for h in ("1", "2")}
    _, mode1 = G.bad_sunks_one_hap(rows["1"], {n for n, _ in fai["1"]})
    bad = G.bad_sunks(rows["1"], {n for n, _ in fai["1"]}, rows["2"], {n for n, _ in fai["2"]})
    assert {f"{c}:{g}" for c, g in bad} == set(txt("sunkpos/bad_sunks.txt").split())
    for h in ("1", "2"):
        rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in txt(f"sunkpos/hap{h}.rlen").splitlines()}
        byc, beds, valid = {}, {}, []
        for r in rows[h]:
            byc.setdefault(r[2], []).append(r)
        for ctg, rr in byc.items():
            inter, bed = G.process_by_contig(rr, rlen, bad, ctg)
            stem = f"{ctg}_hap{h}"
            assert txt(f"inter_outs/{stem}.tsv") == ("".join(f"{g}\t{n}\n" for g, n in inter) if inter else ctg + "\n"), stem
            assert txt(f"bed_files/{stem}.bed") == "".join(f"{c}\t{s}\t{e}\n" for c, s, e in (bed or [])), stem
            if bed is not None:
                beds[ctg] = [(s, e) for _, s, e in bed]
                valid += [f"{c}\t{s}\t{e}" for c, s, e in bed]
        assert sorted(txt(f"final_out/hap{h}.valid.bed").splitlines()) == sorted(valid)
        gaps, nodata = G.get_gaps(fai[h], beds)
        assert txt(f"final_out/hap{h}.gaps.bed") == "".join(f"{c}\t{s}\t{e}\n" for c, s, e in gaps)
        assert txt(f"final_out/hap{h}.nodata.bed") == "".join(f"{c}\t{s}\t{e}\n" for c, s, e in nodata)
    return mode1


def test_unbinned_run_of_the_bundled_samples(j1u, capsys):
    """`fused --reads` on the hap1 and hap2 chunk files as they are: every file of the binned run and the two read
    haplotype files per haplotype; kept rows equal the oracle's, reads split into the .rlen files by file haplotype, bad
    SUNKs / inter_outs / intervals / gaps equal the oracle's Python stages on those rows; two contexts and
    --batch-files 3 write the same bytes"""
    got = _fused(j1u, j1u["tmp"] / "unbinned", j1u["chunks"])
    extra = {f"final_out/hap{hn}.haplotype{s}.tsv" for hn in (1, 2) for s in ("", ".reads")}
    assert set(got) == set(j1u["binned"]) | extra
    voted, wrong, mode1 = _check_unbinned(j1u, got, j1u["per_file"])
    if j1u["name"] == "j1_amy_hg02723":  # README.md:36-37
        # Binned, the README gap is found.  Unbinned, 4 hap-2 reads without a hap-2 vote have 2 votes each on the hap-1
        # decoy contig `nonuniq_kmers` and are assigned to hap 1: their 8 single-row groups tie the 8 groups of the true
        # mode (100 rows), badsunks_AR.py's smallest mode becomes 1 (limit 5), and every AMY_h1 group is bad: the oracle's
        # own stages above then give no interval on hap 1 (nodata), so no gap.
        assert b"AMY_h1\t284861\t324275\n" in j1u["binned"]["final_out/hap1.gaps.bed"]
        assert mode1 == 1 and got["final_out/hap1.gaps.bed"] == b""
    two = _fused(j1u, j1u["tmp"] / "unbinned_n2", j1u["chunks"], "--devices", "0,0", "--batch-files", "3")
    assert two == got
    with capsys.disabled():
        print(f"\n{j1u['name']} unbinned: {voted} voted reads, {wrong} assigned to the wrong haplotype; hap-1 mode {mode1}")
    assert wrong <= 0.005 * voted


def test_unbinned_mixed_chunks(j1u):
    got = _fused(j1u, j1u["tmp"] / "mixed", j1u["mixed"])
    _check_unbinned(j1u, got, j1u["mixed_parts"])


def test_binned_run_with_read_haplotypes_adds_only_its_files(j1u):
    from gavisunk_b200 import cli
    case, tmp = j1u["case"], j1u["tmp"]
    n = case["nchunks"]
    argv = ["fused", "--k", str(case["k"]), "--hap1-asm", j1u["asm"][0], "--hap2-asm", j1u["asm"][1], "--hap1-reads",
            *j1u["chunks"][:n], "--hap2-reads", *j1u["chunks"][n:], "--outdir", str(tmp / "binned_rh"), "--read-haplotypes"]
    assert cli.main(argv) == 0
    got = _tree(tmp / "binned_rh")
    extra = {f"final_out/hap{hn}.haplotype{s}.tsv" for hn in (1, 2) for s in ("", ".reads")}
    assert set(got) == set(j1u["binned"]) | extra
    assert {k: v for k, v in got.items() if k not in extra} == j1u["binned"]

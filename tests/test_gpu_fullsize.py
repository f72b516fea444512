"""BASELINE.json config 3 at FULL size (150 Mbp x2 diploid assembly, 30x ONT-like reads, k=20: 5.9 M SUNKs,
124 k reads / 4.45 Gbp, 2.9 M sunkpos rows) -- too large for the pure-Python oracle, so parity is checked
through (i) the reference's match / diag lines for a sample of the reads against the FULL database (stored in
tests/golden/fullsize_sample.json.gz), (ii) size-independent properties the reference's algorithm guarantees,
(iii) invariance under the engine's own batching choices (chunk split, host copy pipeline), (iv) idempotence."""
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K = 20
# the sample of the reference comparison: the first SAMPLE_READS reads of one chunk file per haplotype
SAMPLE_CHUNKS = ((0, 3), (1, 14))  # (haplotype, chunk)
SAMPLE_READS = 40


def build_full():
    """config 3 on cuda:0, run once through the fused path; returns (engine, workload, results)"""
    from gavisunk_b200 import workload as W
    from gavisunk_b200.engine import Engine
    eng = Engine(K)
    wl = W.make_assembly(eng, [150_000_000], snp_rate=1e-3, dup_frac=0.01, seed=1001, name="s150")
    W.build_db(eng, wl)
    W.add_reads(eng, wl, coverage=30.0, n50=50000.0, sigma=0.8, len_min=1000, len_max=1000000, seed=2001, nchunks=10)
    W.bind_reads(eng, wl)
    iv = eng.run_all(wl.contig_hap, min_read_len=10000)
    gaps, nodata = eng.gaps(wl.contig_len.astype(np.uint32))
    res = dict(rows=eng.rows(0), kept=eng.rows(1), best=eng.best(), pairs=eng.pairs(), bad=eng.bad_list(), iv=iv, gaps=gaps,
               nodata=nodata, off=wl.read_off.cpu().numpy().astype(np.int64))
    return eng, wl, res


def sample_texts(wl, res, r0, r1):
    """{hap}.sunkpos, {hap}_diag.sunkpos and {hap}_diag2.sunkpos lines of reads [r0, r1) as the reference's
    kmerpos_annot3 / diag_filter_v3 / diag_filter_step2 write them (reads named r%09d by their index)"""
    names = wl.contig_names
    fmt = lambda rows: "".join(
        f"r{rd:09d}\t{p}\t{names[c]}\t{s}\t{g}\n"
        for rd, p, c, s, g in zip(rows["read"].tolist(), rows["pos"].tolist(), rows["contig"].tolist(), rows["start"].tolist(),
                                  rows["group"].tolist()) if r0 <= rd < r1)
    b = res["best"]
    sel = (b["read"] >= r0) & (b["read"] < r1)
    diag = "".join(f"r{rd:09d}\t{names[c]}\t{g}\t{'+' if d else '-'}\t{g}\n"
                   for rd, c, g, d in zip(b["read"][sel].tolist(), b["contig"][sel].tolist(), b["ngood"][sel].tolist(), b["dir"][sel].tolist()))
    return dict(sunkpos=fmt(res["rows"]), diag=diag, diag2=fmt(res["kept"]))


def sample_reads(wl, res, r0, r1):
    """[(name, bases)] of reads [r0, r1), named r%09d by their index"""
    off = res["off"]
    seq = wl.reads[int(off[r0]):int(off[r1])].cpu().numpy()
    return [("r%09d" % i, seq[off[i] - off[r0]:off[i + 1] - off[r0]].tobytes()) for i in range(r0, r1)]


def bases_sha256(reads):
    return hashlib.sha256(b"".join(s for _, s in reads)).hexdigest()


def sample_loc(wl, db, reads):
    """indices of the exported database rows that a window of the reads hits, and their kmer.loc lines"""
    import gavisunk_oracle as O
    from gavisunk_b200 import cli
    order = np.argsort(db["kmer"], kind="stable")
    keys = db["kmer"][order]
    assert np.all(keys[1:] != keys[:-1]), "a SUNK is one row of the database"
    hits = []
    for _, s in reads:
        canon = O.canonical_windows(O.codes_of(s), K)
        idx = np.minimum(np.searchsorted(keys, canon), len(keys) - 1)
        hits.append(order[idx[keys[idx] == canon]])
    sub = np.unique(np.concatenate(hits))
    kmers = cli.decode_kmers(db["kmer"][sub], K)
    text = "".join(f"{wl.contig_names[c]}\t{s}\t{km}\t{g}\n"
                   for c, s, km, g in zip(db["contig"][sub].tolist(), db["start"][sub].tolist(), kmers, db["group"][sub].tolist()))
    return sub, text


@pytest.fixture(scope="module")
def full():
    import torch
    eng, wl, res = build_full()
    yield eng, wl, res
    eng.close()
    del wl
    torch.cuda.empty_cache()


def _sub_batch(wl, r0, r1):
    """reads [r0, r1) as their own 16-byte aligned device batch"""
    import torch
    off = wl.read_off[r0:r1 + 1].clone()
    b0, b1 = int(off[0]), int(off[-1])
    seq = torch.zeros(b1 - b0 + 64, dtype=torch.uint8, device=wl.reads.device)
    seq[:b1 - b0] = wl.reads[b0:b1]
    return seq, (off - b0).contiguous()


def test_sizes_are_config3(full):
    eng, wl, res = full
    n_sunks, n_groups = eng.db_size()
    assert 5_000_000 < n_sunks < 7_000_000 and 250_000 < n_groups < 320_000
    assert wl.total_bases > 4_000_000_000 and len(res["rows"]["read"]) > 2_000_000
    assert len(res["pairs"]["read"]) > 2_000_000 and len(res["iv"]["start"]) >= 1


def test_properties_of_the_reference_algorithm(full):
    check_properties(*full)


def check_properties(eng, wl, res):
    rows, kept, best, pairs = res["rows"], res["kept"], res["best"], res["pairs"]
    rd, pos, ctg, st, grp = (rows[c].astype(np.int64) for c in ("read", "pos", "contig", "start", "group"))
    lens = np.diff(res["off"])
    # rows come read by read, positions never decrease inside a read and stay inside it (kmerpos_annot3.nim:88-96)
    assert np.all(np.diff(rd) >= 0)
    same = np.diff(rd) == 0
    assert np.all(np.diff(pos)[same] >= 0)
    assert np.all(pos <= lens[rd] - K)
    # curLoc != prevLoc (nim:92): two consecutive rows of a chunk never name the same (contig, group)
    chunk = np.searchsorted(wl.chunk_first.astype(np.int64), rd, side="right") - 1
    same_chunk = np.diff(chunk) == 0
    assert not np.any(same_chunk & (np.diff(ctg) == 0) & (np.diff(grp) == 0))
    # a row's SUNK lies inside its group's run: group start <= start (bedtools merge, defineSUNKs.smk:125)
    assert np.all(grp <= st)
    # diag_filter_step2: kept rows = the rows on the best contig of their read, in order (nim:40-62)
    bc = np.full(wl.n_reads, -1, np.int64)
    bc[best["read"]] = best["contig"]
    m = bc[rd] == ctg
    for c in ("read", "pos", "contig", "start", "group"):
        assert np.array_equal(rows[c][m], kept[c])
    # diag_filter_v3: best contig belongs to the read's own haplotype assembly, n >= 2 (nim:82,141)
    hap_of_read = wl.chunk_hap[np.searchsorted(wl.chunk_first.astype(np.int64), best["read"].astype(np.int64), side="right") - 1]
    assert np.array_equal(wl.contig_hap[best["contig"]], hap_of_read)
    assert best["ngood"].min() >= 2
    # validated pairs: only reads >= 10 kb (:106), never a bad group (:70-72), every pair is a kept row of that read,
    # IDs distinct inside a read (graph vertices)
    pr, pg, pgi = pairs["read"].astype(np.int64), pairs["group"].astype(np.int64), pairs["gidx"].astype(np.int64)
    assert lens[pr].min() >= 10000
    assert not np.isin(pgi, res["bad"]).any()
    key_kept = np.unique(kept["read"].astype(np.int64) << 32 | kept["group"].astype(np.int64))
    key_pair = pr << 32 | pg
    assert np.isin(key_pair, key_kept).all()
    assert len(np.unique(key_pair)) == len(key_pair)
    # an edge has two ends: a read reports >= 2 IDs, or a single ID that sits on >= 2 of its rows (a self-loop
    # of the ID graph: the same group hit at two consistent positions)
    ur, cnt = np.unique(pr, return_counts=True)
    single = key_pair[np.isin(pr, ur[cnt == 1])]
    kk, kc = np.unique(kept["read"].astype(np.int64) << 32 | kept["group"].astype(np.int64), return_counts=True)
    assert np.all(kc[np.searchsorted(kk, single)] >= 2)
    # intervals: >= 3 groups means start < end; sorted by (contig, start) (:248-260)
    iv = res["iv"]
    assert np.all(iv["start"] < iv["end"])
    order = np.lexsort((iv["start"], iv["contig"]))
    assert np.array_equal(order, np.arange(len(order)))
    assert np.isin(iv["start"], pg).all() and np.isin(iv["end"], pg).all()  # [min, max] of validated IDs
    # gaps (get_gaps.py:43-61): exactly the holes between the merged intervals of a contig
    g = res["gaps"]
    want = []
    for c in np.unique(iv["contig"]):
        sel = iv["contig"] == c
        s, e = iv["start"][sel].astype(np.int64), iv["end"][sel].astype(np.int64)
        run_end = np.maximum.accumulate(e)
        new_run = s[1:] > run_end[:-1]
        want += [(int(c), int(a), int(b) - 1) for a, b in zip(run_end[:-1][new_run], s[1:][new_run])]
    assert list(zip(g["contig"].tolist(), g["start"].tolist(), g["end"].tolist())) == want
    assert set(res["nodata"].tolist()) == set(range(len(wl.contig_names))) - set(iv["contig"].tolist())


def test_idempotent(full):
    eng, wl, res = full
    from gavisunk_b200 import workload as W
    W.bind_reads(eng, wl)
    iv = eng.run_all(wl.contig_hap, min_read_len=10000)
    for c in ("read", "pos", "contig", "start", "group"):
        assert np.array_equal(eng.rows(0)[c], res["rows"][c])
        assert np.array_equal(eng.rows(1)[c], res["kept"][c])
    for c in ("read", "group", "gidx"):
        assert np.array_equal(eng.pairs()[c], res["pairs"][c])
    for c in ("contig", "start", "end"):
        assert np.array_equal(iv[c], res["iv"][c])


def test_chunk_split_invariance(full):
    """the prevLoc carry and the Table capacity live inside a chunk file: matching + filtering the chunks in two
    separate batches must give the rows of the single batch"""
    eng, wl, res = full
    cf = wl.chunk_first.astype(np.int64)
    cut_c = 7  # chunk boundary inside haplotype 1
    cut = int(cf[cut_c])
    got = {c: [] for c in ("read", "pos", "contig", "start", "group")}
    for (r0, r1, c0, c1) in ((0, cut, 0, cut_c), (cut, wl.n_reads, cut_c, len(cf) - 1)):
        seq, off = _sub_batch(wl, r0, r1)
        eng.set_reads_device(seq.data_ptr(), off.data_ptr(), r1 - r0, cf[c0:c1 + 1] - r0, wl.chunk_hap[c0:c1])
        eng.match()
        eng.diag_filter(wl.contig_hap)
        k = eng.rows(1)
        for c in got:
            got[c].append(k[c].astype(np.int64) + (r0 if c == "read" else 0))
    for c in got:
        assert np.array_equal(np.concatenate(got[c]), res["kept"][c].astype(np.int64)), c


def test_host_copy_pipeline_equals_resident(full):
    """ASCII reads in pinned HOST memory, copied in 16 segments overlapped with per-segment probe launches"""
    import torch
    eng, wl, res = full
    h = torch.empty(wl.total_bases + 64, dtype=torch.uint8, pin_memory=True)
    h[:wl.total_bases].copy_(wl.reads[:wl.total_bases])
    torch.cuda.synchronize()
    for mode in (eng.PACK_OFF, eng.PACK_ALL, eng.PACK_ADAPTIVE):  # segments as ASCII / 2-bit packed on the host / mixed
        eng.set_host_pack(mode)
        eng.set_reads(h.numpy()[:wl.total_bases], res["off"].astype(np.uint64), wl.chunk_first, wl.chunk_hap)
        eng.match()
        for c in ("read", "pos", "contig", "start", "group"):
            assert np.array_equal(eng.rows(0)[c], res["rows"][c]), (mode, c)
        nbytes, nseg, npk = eng.copy_stats()
        assert nseg > 1 and npk == {eng.PACK_OFF: 0, eng.PACK_ALL: nseg}.get(mode, npk)
        assert wl.total_bases // 4 <= nbytes <= wl.total_bases + 4096 * nseg
    del h


def test_sample_of_reads_against_reference_executables(full, golden):
    """the lines of kmerpos_annot3 / diag_filter_v3 / diag_filter_step2 for the first reads of one chunk per haplotype,
    matched against the FULL 5.9 M-SUNK database (exported): tests/golden/fullsize_sample.json.gz, made by
    tests/golden/make_golden_fullsize.py.  Its "source" field names what wrote them: the reference's executables run
    on the whole exported database, or -- where they are not at hand, as for the stored file -- the oracle's
    restatement of them (pinned to their own output by test_oracle_golden)"""
    eng, wl, res = full
    case = golden("fullsize_sample")
    assert case["k"] == K and [(s["hap"], s["chunk"]) for s in case["sample"]] == list(SAMPLE_CHUNKS)
    off = res["off"]
    db = eng.db_export()
    for s in case["sample"]:
        r0 = int(wl.chunk_first[s["chunk"]])
        r1 = r0 + SAMPLE_READS
        assert wl.chunk_hap[s["chunk"]] == s["hap"] and r0 == s["first_read"]
        reads = sample_reads(wl, res, r0, r1)
        assert np.diff(off[r0:r1 + 1]).tolist() == s["read_len"] and bases_sha256(reads) == s["bases_sha256"], \
            "the workload generator no longer draws the stored sample"
        # the database rows these reads can hit, as the reference reads them from kmer.loc
        loc = sample_loc(wl, db, reads)[1]
        assert hashlib.sha256(loc.encode()).hexdigest() == s["loc_sha256"], s["hap"]
        # the chunk starts at r0, so the prevLoc carry of the full batch restarts exactly there
        got = sample_texts(wl, res, r0, r1)
        for f in ("sunkpos", "diag", "diag2"):
            assert got[f] == s[f], (s["hap"], f)
        assert len(s["sunkpos"].splitlines()) > 500

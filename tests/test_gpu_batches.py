"""The two-phase multi-batch engine (Engine.run_batches, csrc/batches.cu): a run whose chunk files arrive in
several batches gives exactly what one batch holding all of them gives -- the reference gathers every chunk of a
haplotype before the global stages (workflow/Snakefile:23-24, tagONT.smk:112-131, badsunks_AR.py:20-27)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _setup(seed=41, contig_lens=(350000, 120000), cov=18.0, n50=14000, nchunks=6, k=20):
    import torch
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    eng = Engine(k)
    wl = W.make_assembly(eng, list(contig_lens), snp_rate=2e-3, dup_frac=0.02, seed=seed)
    W.build_db(eng, wl)
    W.add_reads(eng, wl, coverage=cov, n50=n50, sigma=0.6, len_min=200, len_max=300000, seed=seed + 1, nchunks=nchunks)
    return eng, wl


def _collect(eng, wl, iv):
    gaps, nodata = eng.gaps(wl.contig_len.astype(np.uint32))
    return dict(iv={c: v.tolist() for c, v in iv.items()}, gaps={c: v.tolist() for c, v in gaps.items()}, nodata=nodata.tolist(),
                bad=sorted(eng.bad_list().tolist()), kept={c: v.tolist() for c, v in eng.rows(1).items()},
                pairs={c: v.tolist() for c, v in eng.pairs().items()})


def _host_batches(wl, groups):
    """chunk groups -> host batches (seq, off, chunk_first, chunk_hap, first read)"""
    reads = wl.reads.cpu().numpy()
    off = wl.read_off.cpu().numpy().astype(np.uint64)
    cf = wl.chunk_first.astype(np.int64)
    out = []
    for g in groups:
        r0, r1 = int(cf[g[0]]), int(cf[g[-1] + 1])
        seq = reads[int(off[r0]):int(off[r1])].copy()
        o = (off[r0:r1 + 1] - off[r0]).astype(np.uint64)
        out.append((seq, o, (cf[g[0]:g[-1] + 2] - r0).astype(np.uint64), wl.chunk_hap[g[0]:g[-1] + 1].copy(), r0))
    return out


@pytest.mark.parametrize("split", [[list(range(12))], [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10, 11]], [[i] for i in range(12)]])
def test_batches_equal_one_batch(split):
    from gavisunk_b200 import workload as W
    eng, wl = _setup()
    W.bind_reads(eng, wl)
    want = _collect(eng, wl, eng.run_all(wl.contig_hap, min_read_len=3000))
    assert len(want["iv"]["contig"]) > 0 and len(want["pairs"]["read"]) > 100 and len(want["bad"]) > 0
    hb = _host_batches(wl, split)
    seen = []
    binds = [(lambda e, b=b: e.set_reads(b[0], b[1], b[2], b[3])) for b in hb]
    iv, bases = eng.run_batches(binds, wl.contig_hap, min_read_len=3000, on_batch=lambda e, b, base: seen.append((b, base, e.n_kept)))
    assert bases == [b[4] for b in hb]  # run-wide read indices count through the batches
    assert [s[:2] for s in seen] == list(enumerate(bases))
    got = _collect(eng, wl, iv)
    assert got == want
    assert eng.n_kept == len(want["kept"]["read"]) == sum(s[2] for s in seen)
    # a second run on the same engine re-uses the stash buffers and starts from a clean histogram / forest
    iv2, _ = eng.run_batches(binds, wl.contig_hap, min_read_len=3000)
    assert _collect(eng, wl, iv2) == want
    # ... and run_all afterwards is unaffected by the batch state
    W.bind_reads(eng, wl)
    assert _collect(eng, wl, eng.run_all(wl.contig_hap, min_read_len=3000)) == want


def test_two_engines_exchange_like_two_ranks():
    """two contexts on one GPU, each with half of the batches; the two exchanges done by hand (sum of the histograms,
    union of the forests) -- the result equals the single-engine run (what NCCL does between ranks, SURVEY 8e)"""
    import torch
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    from gavisunk_b200.parallel import alias_device_array
    eng, wl = _setup(seed=43, nchunks=4)
    W.bind_reads(eng, wl)
    want = _collect(eng, wl, eng.run_all(wl.contig_hap, min_read_len=3000))
    hb = _host_batches(wl, [[0, 1, 2], [3], [4, 5], [6, 7]])
    eng2 = Engine(20)
    W.build_db(eng2, wl)
    dev = torch.device("cuda", 0)
    engines = [eng, eng2]
    parts = [hb[:2], hb[2:]]
    ng = eng.db_groups()
    hp = []
    for e, part in zip(engines, parts):
        e.batches_begin()
        for b in part:
            e.set_reads(b[0], b[1], b[2], b[3])
            e.match()
            e.diag_filter(wl.contig_hap)
            p = e.group_hist(accumulate=True)
            e.batch_stash()
        e.batches_bind()
        e.sync()
        hp.append(alias_device_array(p, ng, "<i4", dev))
    tot = hp[0] + hp[1]
    hp[0].copy_(tot)
    hp[1].copy_(tot)
    torch.cuda.synchronize()
    forests = []
    for e in engines:
        e.bad_groups()
        e.validate(3000)
        forests.append(e.components_local())
        e.sync()
    gathered = torch.stack([alias_device_array(f, ng, "<i4", dev) for f in forests])
    torch.cuda.synchronize()
    res = []
    for i, e in enumerate(engines):
        e.components_merge_all(int(gathered.data_ptr()), 2, i)
        iv = e.intervals()
        gaps, nodata = e.gaps(wl.contig_len.astype(np.uint32))
        res.append((dict(iv={c: v.tolist() for c, v in iv.items()}, gaps={c: v.tolist() for c, v in gaps.items()}, nodata=nodata.tolist(),
                         bad=sorted(e.bad_list().tolist()))))
    for r in res:
        for key in ("iv", "gaps", "nodata", "bad"):
            assert r[key] == want[key], key
    # the validated pairs of the two halves together are the single run's (read indices shifted by the half's first read)
    shift = [0, hb[2][4]]
    reads = np.concatenate([e.pairs()["read"] + np.uint32(s) for e, s in zip(engines, shift)])
    groups = np.concatenate([e.pairs()["group"] for e in engines])
    assert reads.tolist() == want["pairs"]["read"] and groups.tolist() == want["pairs"]["group"]


def test_rank_without_batches():
    """more ranks than batches: the idle rank still has a (zero) histogram and a singleton forest to exchange"""
    eng, wl = _setup(seed=45, contig_lens=(90000,), cov=6.0, nchunks=2)
    iv, bases = eng.run_batches([], wl.contig_hap)
    assert bases == [] and len(iv["contig"]) == 0 and eng.n_pairs == 0 and eng.n_bad == 0
    gaps, nodata = eng.gaps(wl.contig_len.astype(np.uint32))
    assert len(gaps["contig"]) == 0 and sorted(nodata.tolist()) == [0, 1]

"""Host-side multi-GPU logic on CPU: chunk sharding and the two exchanges of the path (histogram
all-reduce, forest all-gather + merge) with world_size 2 over gloo."""
import os
import socket

import numpy as np
import pytest

from gavisunk_b200 import parallel as P


def test_shard_chunks_cover_and_keep_chunks_whole():
    for n, w in [(20, 1), (20, 2), (20, 8), (3, 8), (7, 4)]:
        sh = P.shard_chunks(n, w)
        assert sh[0][0] == 0 and sh[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(sh, sh[1:]))
        sizes = [b - a for a, b in sh]
        assert max(sizes) - min(sizes) <= 1


def test_shard_reads_rebases_chunk_table():
    cf = [0, 5, 9, 9, 14, 20]
    hap = [0, 0, 0, 1, 1]
    seen = []
    for r in range(2):
        r0, r1, lcf, lh = P.shard_reads(cf, hap, r, 2)
        assert lcf[0] == 0 and lcf[-1] == r1 - r0
        seen.append((r0, r1, list(lh)))
    assert seen[0][1] == seen[1][0] and seen[0][0] == 0 and seen[1][1] == 20
    assert seen[0][2] + seen[1][2] == hap
    r0, r1, lcf, lh = P.shard_reads([0, 4], [1], 3, 4)  # more ranks than chunks
    assert r0 == r1 and list(lcf) == [0, 0]


def _find(par, x):
    while par[x] != x:
        par[x] = par[par[x]]
        x = par[x]
    return x


def _forest(n, edges):
    par = np.arange(n, dtype=np.int64)
    for a, b in edges:
        ra, rb = _find(par, a), _find(par, b)
        if ra != rb:
            par[max(ra, rb)] = min(ra, rb)
    return par


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 500
        rng = np.random.default_rng(100 + rank)
        hist = rng.integers(0, 5, n).astype(np.int32)
        edges = [(int(a), int(b)) for a, b in rng.integers(0, n, (120, 2))]
        par = _forest(n, edges)
        x = P.Exchange()
        h = torch.from_numpy(hist.copy())
        x.allreduce_hist(h)
        gathered = x.gather_forests(torch.from_numpy(par.astype(np.int32)))
        assert gathered.shape == (world, n) and gathered[rank].tolist() == par.tolist()
        peers = [gathered[r] for r in range(world) if r != rank]
        merged = par.copy()
        for p in peers:
            pp = p.numpy()
            for g in range(n):
                if pp[g] != g:
                    ra, rb = _find(merged, g), _find(merged, int(pp[g]))
                    if ra != rb:
                        merged[max(ra, rb)] = min(ra, rb)
        roots = np.array([_find(merged, g) for g in range(n)])
        q.put((rank, h.numpy().tolist(), roots.tolist(), len(peers)))
    finally:
        dist.destroy_process_group()


def test_exchanges_world2_gloo():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    n = 500
    hists, all_edges = [], []
    for rank in range(2):
        rng = np.random.default_rng(100 + rank)
        hists.append(rng.integers(0, 5, n).astype(np.int32))
        all_edges += [(int(a), int(b)) for a, b in rng.integers(0, n, (120, 2))]
    exp_hist = (hists[0] + hists[1]).tolist()
    par = _forest(n, all_edges)
    exp_roots = [int(_find(par, g)) for g in range(n)]
    for rank, h, roots, npeers in out:
        assert npeers == 1
        assert h == exp_hist
        assert roots == exp_roots  # replicated result: min index of the component on every rank


def test_parse_cpulist_and_numa_binding_is_best_effort():
    from gavisunk_b200.parallel import parse_cpulist, bind_to_gpu_numa
    assert parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    assert parse_cpulist("") == []
    info = bind_to_gpu_numa(0)  # no GPU here: must not raise, must not change anything
    assert info["device"] == 0 and info["cpus"] is None

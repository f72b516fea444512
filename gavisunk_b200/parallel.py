"""Multi-GPU plumbing of the hot path (SURVEY.md 8e): reads shard by chunk file, the SUNK table is
replicated, and exactly two exchanges cross GPUs:

  1. sum of the per-group hit histogram (badsunks_AR.py:24 counts rows of ALL chunks of a
     haplotype) -- all-reduce of int32[n_groups];
  2. the contig-wide component merge (process-by-contig_lowmem_AR.py:219-237 sees the reads of ALL
     chunks) -- all-gather of the union-find parent arrays uint32[n_groups]; every rank then unions
     all peers' forests into its own in one pass (gvs_components_merge_all), so the result is replicated.

Two adapters give Engine.run_all / run_batches these exchanges: EngineExchange (one process per GPU,
torch.distributed) and ThreadExchange (one process, one host thread per GPU, torch copies between
the devices).  Both follow one convention: allreduce_hist(ptr, n_groups) sums in place, and
gather_forests(ptr, n_groups) returns None with a single rank or no groups, else (pointer of an
int32 [n_ranks][n_groups] array on the engine's device whose row r is rank r's forest -- the own row
may be left unwritten --, n_ranks, own rank), kept alive until the adapter's next gather.

torch.distributed is plumbing only (NCCL on GPUs; gloo in the CPU tests).  The tensors alias the
library's device buffers, so the collectives run in place on them.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np


def shard_chunks(n_chunks: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous blocks of chunk files per rank.  A chunk file is never split: kmerpos_annot3's
    `prevLoc` carry (workflow/src/kmerpos_annot3.nim:82-84, SURVEY Q4) and diag_filter_v3's sticky
    Table capacity (Q9) live inside one chunk file, so whole chunks keep every rank bit-exact."""
    out = []
    base, extra = divmod(n_chunks, world)
    lo = 0
    for r in range(world):
        hi = lo + base + (1 if r < extra else 0)
        out.append((lo, hi))
        lo = hi
    return out


def shard_reads(chunk_first: Sequence[int], chunk_hap: Sequence[int], rank: int, world: int):
    """-> (first read, last read + 1, local chunk_first, local chunk_hap) of this rank's shard"""
    chunk_first = np.asarray(chunk_first, dtype=np.uint64)
    chunk_hap = np.asarray(chunk_hap, dtype=np.uint8)
    lo, hi = shard_chunks(len(chunk_hap), world)[rank]
    r0, r1 = int(chunk_first[lo]), int(chunk_first[hi])
    if hi == lo:  # more ranks than chunks: an empty shard still needs one (empty) chunk
        return r0, r0, np.array([0, 0], dtype=np.uint64), np.array([0], dtype=np.uint8)
    return r0, r1, (chunk_first[lo:hi + 1] - chunk_first[lo]).astype(np.uint64), chunk_hap[lo:hi].copy()


def parse_cpulist(text: str) -> List[int]:
    """'0-3,8,10-11' -> [0, 1, 2, 3, 8, 10, 11] (the format of /sys/devices/system/node/nodeN/cpulist)"""
    out: List[int] = []
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        out.extend(range(int(a), int(b or a) + 1))
    return out


def bind_to_gpu_numa(device_index: int) -> dict:
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, BEFORE any page-locked host
    buffer is allocated: pinned pages are placed on the allocating thread's node, and a shard that
    streams 11 GB per step through the other socket halves the host->device rate once several ranks
    run.  Best effort (no-op when sysfs / NVML do not say); returns what was done."""
    import os
    info = dict(device=device_index, numa_node=None, cpus=None)
    try:
        import pynvml
        pynvml.nvmlInit()
        # NVML enumerates in PCI order; honour CUDA_VISIBLE_DEVICES when it is a plain index list
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = device_index
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if device_index < len(ids) and ids[device_index].isdigit():
                idx = int(ids[device_index])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = parse_cpulist(f.read())
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["cpus"] = len(allowed)
    except Exception as ex:  # containers without sysfs topology, missing NVML, ...
        info["error"] = repr(ex)[:120]
    return info


class Exchange:
    """The two collectives on torch tensors (any device / backend)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0

    def allreduce_hist(self, hist):
        """hist: int32[n_groups] tensor, summed in place across ranks"""
        if self.world > 1 and hist.numel():
            self.dist.all_reduce(hist, op=self.dist.ReduceOp.SUM, group=self.group)
        return hist

    def gather_forests(self, parent):
        """parent: int32-typed view of uint32[n_groups]; returns the gathered [world, n_groups] tensor
        (row r = rank r's array), None with a single rank or no groups"""
        import torch
        if self.world == 1 or parent.numel() == 0:
            return None
        n = parent.numel()
        buf = getattr(self, "_keep", None)  # one gather buffer per run shape, reused (a rank pays this once per run)
        if buf is None or buf.numel() != self.world * n or buf.dtype != parent.dtype or buf.device != parent.device:
            buf = torch.empty(self.world * n, dtype=parent.dtype, device=parent.device)
        self.dist.all_gather_into_tensor(buf, parent, group=self.group) if parent.is_cuda else \
            self.dist.all_gather(list(buf.view(self.world, n).unbind(0)), parent, group=self.group)
        self._keep = buf
        return buf.view(self.world, n)


_ALIASES: dict = {}


def alias_device_array(ptr: int, n: int, typestr: str, device):
    """torch tensor over a raw device pointer owned by libgavisunk_b200.so (CUDA array interface); the wrapper of a
    given (pointer, length) is built once -- the library's histogram / forest buffers keep their place from run to run"""
    import torch
    key = (int(ptr), int(n), typestr, str(device))
    t = _ALIASES.get(key)
    if t is not None:
        return t
    if len(_ALIASES) > 64:
        _ALIASES.clear()

    class _A:
        pass
    a = _A()
    a.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)
    t = torch.as_tensor(a, device=device)
    _ALIASES[key] = t
    return t


class EngineExchange:
    """Adapters with the signatures Engine.run_all / run_batches expect (raw device pointers).

    The aliased buffers are written and read by kernels queued on the engine's stream, while
    ProcessGroupNCCL orders its work against torch's CURRENT stream only.  Give the engine
    (`eng=`) and every collective is bracketed by stream dependencies in both directions, whichever
    stream the engine was created on; without it the caller must run the engine on torch's current
    stream."""

    def __init__(self, device, group=None, eng=None):
        self.x = Exchange(group)
        self.device = device
        self.eng_stream = None
        if eng is not None and self.x.world > 1:
            import torch
            self.eng_stream = (torch.cuda.ExternalStream(eng.stream_ptr, device=device) if eng.stream_ptr
                               else torch.cuda.default_stream(device))

    def _before(self):
        if self.eng_stream is not None:
            import torch
            torch.cuda.current_stream(self.device).wait_stream(self.eng_stream)

    def _after(self):
        if self.eng_stream is not None:
            import torch
            self.eng_stream.wait_stream(torch.cuda.current_stream(self.device))

    def allreduce_hist(self, ptr: int, n_groups: int):
        if self.x.world > 1 and n_groups:
            self._before()
            self.x.allreduce_hist(alias_device_array(ptr, n_groups, "<i4", self.device))
            self._after()

    def gather_forests(self, ptr: int, n_groups: int):
        if self.x.world == 1 or not n_groups:
            return None
        self._before()
        gathered = self.x.gather_forests(alias_device_array(ptr, n_groups, "<i4", self.device))
        self._after()
        return int(gathered.data_ptr()), self.x.world, self.x.rank


class ThreadExchange:
    """The two exchanges between the engines of one process (one host thread per GPU): the histogram is summed by
    rank 0 and the forests are gathered with torch copies between the devices (plumbing).  for_rank(r) gives the
    adapter of engine r; abort() releases the peers of a thread that failed."""

    def __init__(self, engines):
        import threading
        self.engines = engines
        self.n = len(engines)
        self.bar = threading.Barrier(self.n)
        self.slots = [None] * self.n  # rank r's aliased device array of the current exchange
        self.keep = [None] * self.n   # rank r's gather buffer, reused while the shape holds

    def abort(self):
        self.bar.abort()

    def for_rank(self, r: int) -> "_ThreadRank":
        return _ThreadRank(self, r)


class _ThreadRank:
    def __init__(self, x: ThreadExchange, r: int):
        self.x, self.r = x, r

    def _publish(self, ptr: int, n_groups: int):
        """waits for the engine's work on the array, then for every rank to have published its own"""
        import torch
        x, r = self.x, self.r
        dev = torch.device("cuda", x.engines[r].device)
        x.engines[r].sync()
        x.slots[r] = alias_device_array(ptr, n_groups, "<i4", dev)
        x.bar.wait()
        return dev

    def allreduce_hist(self, ptr: int, n_groups: int):
        x, r = self.x, self.r
        if x.n == 1 or not n_groups:
            return
        import torch
        self._publish(ptr, n_groups)
        if r == 0:
            tot = x.slots[0].clone()
            for p in range(1, x.n):
                tot += x.slots[p].to(tot.device)
            for p in range(x.n):
                x.slots[p].copy_(tot.to(x.slots[p].device))
            for p in range(x.n):
                torch.cuda.synchronize(x.slots[p].device)
        x.bar.wait()

    def gather_forests(self, ptr: int, n_groups: int):
        x, r = self.x, self.r
        if x.n == 1 or not n_groups:
            return None
        import torch
        dev = self._publish(ptr, n_groups)
        buf = x.keep[r]
        if buf is None or buf.shape != (x.n, n_groups):
            buf = x.keep[r] = torch.empty(x.n, n_groups, dtype=torch.int32, device=dev)
        for p in range(x.n):
            if p != r:
                buf[p].copy_(x.slots[p])
        torch.cuda.synchronize(dev)
        x.bar.wait()  # nobody unions into its own forest while a peer still copies it
        return int(buf.data_ptr()), x.n, r

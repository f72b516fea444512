"""Host-side driver of libgavisunk_b200.so: one Engine per GPU.

The methods mirror the reference's stages one to one (names of the reference programs in the
docstrings; file:line relative to the reference repository).  Everything here is plumbing --
array marshalling, the scalar arithmetic the reference does in Python, name <-> index maps; all
per-base / per-row work happens in the CUDA library.  No CPU fallback exists.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import GavisunkError, GavisunkKeyError

GVS_HAP_ANY = 2  # chunk haplotype of unbinned reads: the diag filter assigns each read from its SUNK votes

_LUT = np.zeros(256, dtype=np.uint64)
for _ch, _v in (("A", 0), ("C", 1), ("G", 2), ("T", 3), ("U", 3)):
    _LUT[ord(_ch)] = _v
    _LUT[ord(_ch.lower())] = _v
_LUT[1], _LUT[2], _LUT[3] = 1, 2, 3


def encode_kmers(lines: Sequence[bytes], k: Optional[int] = None) -> np.ndarray:
    """kmer.encode of every text k-mer (workflow/src/kmerpos_annot3.nim:24,68): 2-bit big-endian,
    first base most significant.  Vectorised over equal-length k-mers."""
    if len(lines) == 0:
        return np.zeros(0, dtype=np.uint64)
    if k is None:
        k = len(lines[0])
    if all(len(l) == k for l in lines):
        a = np.frombuffer(b"".join(lines), dtype=np.uint8).reshape(len(lines), k)
        codes = _LUT[a]
        sh = (np.uint64(2) * np.arange(k - 1, -1, -1, dtype=np.uint64))
        return np.bitwise_or.reduce(codes << sh, axis=1) if k else np.zeros(len(lines), dtype=np.uint64)
    out = np.zeros(len(lines), dtype=np.uint64)
    for i, l in enumerate(lines):  # ragged input: per line, wrapping like the reference's uint64
        v = 0
        for b in l:
            v = ((v << 2) | int(_LUT[b])) & 0xFFFFFFFFFFFFFFFF
        out[i] = v
    return out


def revcomp_kmers(km: np.ndarray, k: int) -> np.ndarray:
    """reverse complement of 2-bit big-endian k-mers (vectorised)"""
    x = ~np.ascontiguousarray(km, np.uint64)
    m = [(0x3333333333333333, 2), (0x0F0F0F0F0F0F0F0F, 4), (0x00FF00FF00FF00FF, 8), (0x0000FFFF0000FFFF, 16), (0x00000000FFFFFFFF, 32)]
    for mask, sh in m:
        mk = np.uint64(mask)
        x = ((x >> np.uint64(sh)) & mk) | ((x & mk) << np.uint64(sh))
    return x >> np.uint64(64 - 2 * k)


def pack_2bit(seq: np.ndarray, threads: int = 0, out: Optional[np.ndarray] = None) -> np.ndarray:
    """kmer.encode's byte map applied to a whole batch on the host (gvs_pack_2bit): uint8[n] -> uint32[ceil(n/16)]"""
    import os
    seq = _c(seq, np.uint8)
    nw = (len(seq) + 15) // 16
    if out is None:
        out = np.zeros(nw, np.uint32)
    assert out.dtype == np.uint32 and len(out) >= nw
    rc = _lib.load().gvs_pack_2bit(_ptr(seq), len(seq), _ptr(out), threads or (os.cpu_count() or 1))
    if rc != 0:
        raise GavisunkError(rc, "gvs_pack_2bit failed")
    return out


def murmur3_32(data: bytes, seed: int = 0) -> int:
    """MurmurHash3_x86_32 == Nim's `hash(string)` (workflow/src/diag_filter_v3.nim:54 Table keys)."""
    c1, c2 = 0xCC9E2D51, 0x1B873593
    h = seed & 0xFFFFFFFF
    n = len(data)
    nb = n // 4
    for i in range(nb):
        kk = int.from_bytes(data[4 * i:4 * i + 4], "little")
        kk = (kk * c1) & 0xFFFFFFFF
        kk = ((kk << 15) | (kk >> 17)) & 0xFFFFFFFF
        kk = (kk * c2) & 0xFFFFFFFF
        h ^= kk
        h = ((h << 13) | (h >> 19)) & 0xFFFFFFFF
        h = (h * 5 + 0xE6546B64) & 0xFFFFFFFF
    tail = data[4 * nb:]
    kk = 0
    if len(tail) >= 3:
        kk ^= tail[2] << 16
    if len(tail) >= 2:
        kk ^= tail[1] << 8
    if len(tail) >= 1:
        kk ^= tail[0]
        kk = (kk * c1) & 0xFFFFFFFF
        kk = ((kk << 15) | (kk >> 17)) & 0xFFFFFFFF
        kk = (kk * c2) & 0xFFFFFFFF
        h ^= kk
    h ^= n
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & 0xFFFFFFFF
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & 0xFFFFFFFF
    h ^= h >> 16
    return h


def nim_hash(name: str) -> int:
    h = murmur3_32(name.encode("utf-8"))
    return 314159265 if h == 0 else h  # tables.nim remaps a zero hash code


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


class Engine:
    """One GPU context (gvs_ctx)."""

    def __init__(self, k: int, device: int = 0, stream: Optional[int] = None):
        self.lib = _lib.load()
        self.k = int(k)
        self.device = device
        self.ctx = self.lib.gvs_create(device, self.k)
        if not self.ctx:
            raise GavisunkError(-1, f"gvs_create(device={device}, k={k}) failed: no CUDA device or bad k "
                                    "(gavisunk_b200 has no CPU fallback)")
        self.contig_names: List[str] = []
        self._keep = []  # host arrays that must outlive async copies
        self._pool: Dict[str, Tuple[int, int]] = {}  # page-locked result buffers: name -> (pointer, bytes)
        self._retired: List[int] = []                # outgrown page-locked buffers (freed by close())
        self.stream_ptr = int(stream) if stream else 0  # cudaStream_t all work of this context is queued on (0 = legacy default)
        if stream is not None:
            self._ck(self.lib.gvs_set_stream(self.ctx, C.c_void_p(stream)))

    # ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "ctx", None):
            for ptr in [p for p, _ in getattr(self, "_pool", {}).values()] + list(getattr(self, "_retired", [])):
                self.lib.gvs_host_free(C.c_void_p(ptr))
            self._pool, self._retired = {}, []
            self.lib.gvs_destroy(self.ctx)
            self.ctx = None

    def _out(self, name: str, n: int, dtype, pinned: bool) -> np.ndarray:
        """result array of n elements: a fresh numpy array, or (pinned=True) a view of a page-locked buffer
        owned by this engine that the next call with the same name overwrites (the device->host copy then
        runs at PCIe speed instead of being staged page by page)"""
        dt = np.dtype(dtype)
        if not pinned:
            return np.zeros(n, dt)
        need = max(n * dt.itemsize, 16)
        ptr, cap = self._pool.get(name, (0, 0))
        if cap < need:
            if ptr:
                # views handed out by earlier rows(pinned=True) / pairs(pinned=True) calls still point into the old
                # buffer: it is retired, not freed, and lives until close()
                self._retired.append(ptr)
            p = C.c_void_p()
            cap = need + need // 2
            self._ck(self.lib.gvs_host_alloc(cap, C.byref(p)))
            ptr = int(p.value)
            self._pool[name] = (ptr, cap)
        buf = (C.c_uint8 * need).from_address(ptr)
        return np.frombuffer(buf, dtype=dt, count=n)

    def _table(self, name: str, get, n: int, cols: Sequence[Optional[str]], lead=(), dtypes=None, counts=None,
               pinned: bool = False) -> Dict[str, np.ndarray]:
        """Host columns of table `name` from get(ctx, *lead, one pointer per entry of cols): n entries each (counts[c]
        for a column given there), uint32 unless dtypes[c] says otherwise; a None in cols passes a null pointer.
        pinned: views of page-locked buffers keyed "name.column" (see _out)."""
        dtypes, counts = dtypes or {}, counts or {}
        out = {c: self._out(f"{name}.{c}", counts.get(c, n), dtypes.get(c, np.uint32), pinned) for c in cols if c is not None}
        self._ck(get(self.ctx, *lead, *[_ptr(out.get(c)) for c in cols]))
        return out

    def _runs(self, name: str, run, get, cols: Sequence[str], diff: str, contig_len, allreduce):
        """support() / discordance(): runs (contig, start, end, one column per value) tiling every contig, after the
        optional in-place all-reduce of the int32 difference arrays (one per value column) at the pointer attribute `diff`"""
        if allreduce is not None:
            allreduce(getattr(self, diff), (len(cols) - 3) * self.db_groups())
        cl = _c(contig_len, np.uint32)
        n = C.c_uint64()
        self._ck(run(self.ctx, _ptr(cl), C.byref(n)))
        return self._table(name, get, int(n.value), cols)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc: int):
        if rc != 0:
            msg = self.lib.gvs_last_error(self.ctx).decode("utf-8", "replace")
            if rc == _lib.GVS_E_KEYERROR:
                raise GavisunkKeyError(rc, msg)
            raise GavisunkError(rc, msg)

    def sync(self):
        self._ck(self.lib.gvs_sync(self.ctx))

    def set_profiling(self, on: bool):
        self._ck(self.lib.gvs_set_profiling(self.ctx, 1 if on else 0))

    def stage_ms(self, stage: str) -> float:
        ms = C.c_float()
        self._ck(self.lib.gvs_stage_ms(self.ctx, _lib.STAGES[stage], C.byref(ms)))
        return float(ms.value)

    @property
    def launches(self) -> int:
        return int(self.lib.gvs_launch_count(self.ctx))

    # ------------------------------------------------------------------------------------
    # database
    # ------------------------------------------------------------------------------------
    def load_loc(self, db_kmer, loc_kmer, loc_contig, loc_start, loc_group, contig_names: Sequence[str]):
        """kmerpos_annot3's table load (workflow/src/kmerpos_annot3.nim:20-26,57-69)."""
        db_kmer = _c(db_kmer, np.uint64)
        loc_kmer = _c(loc_kmer, np.uint64)
        loc_contig = _c(loc_contig, np.uint32)
        loc_start = _c(loc_start, np.uint32)
        loc_group = _c(loc_group, np.uint32)
        self.contig_names = list(contig_names)
        self._ck(self.lib.gvs_db_load_loc(self.ctx, _ptr(db_kmer), len(db_kmer), _ptr(loc_kmer), _ptr(loc_contig),
                                          _ptr(loc_start), _ptr(loc_group), len(loc_kmer), len(self.contig_names)))

    def load_loc_text(self, db_lines: Sequence[bytes], loc_rows: Sequence[Tuple[str, int, bytes, int]],
                      contig_names: Optional[Sequence[str]] = None):
        """db_lines: lines of jellyfish.db; loc_rows: (contig, start, kmer, group) of kmer.loc."""
        names = list(contig_names) if contig_names is not None else []
        idx: Dict[str, int] = {n: i for i, n in enumerate(names)}
        ci = np.zeros(len(loc_rows), dtype=np.uint32)
        for i, r in enumerate(loc_rows):
            j = idx.get(r[0])
            if j is None:
                j = idx[r[0]] = len(names)
                names.append(r[0])
            ci[i] = j
        self.load_loc(encode_kmers(list(db_lines)), encode_kmers([r[2] for r in loc_rows]), ci,
                      np.array([r[1] for r in loc_rows], dtype=np.uint32),
                      np.array([r[3] for r in loc_rows], dtype=np.uint32), names)

    def build_db(self, contigs: Sequence[Tuple[str, bytes]]):
        """defineSUNKs.smk:1-127 on the GPU; contigs in ref.fa order (hap1 then hap2)."""
        self.contig_names = [n for n, _ in contigs]
        off = np.zeros(len(contigs) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(s) for _, s in contigs], dtype=np.uint64)
        seq = np.frombuffer(b"".join(s for _, s in contigs), dtype=np.uint8)
        self._ck(self.lib.gvs_db_build(self.ctx, _ptr(seq), _ptr(off), len(contigs), 0))

    def build_db_device(self, seq_dev_ptr: int, contig_off_dev_ptr: int, contig_names: Sequence[str]):
        self.contig_names = list(contig_names)
        self._ck(self.lib.gvs_db_build(self.ctx, C.c_void_p(seq_dev_ptr), C.c_void_p(contig_off_dev_ptr),
                                       len(self.contig_names), 1))

    def db_size(self) -> Tuple[int, int]:
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.gvs_db_size(self.ctx, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def db_export(self) -> Dict[str, np.ndarray]:
        n, _ = self.db_size()
        return self._table("db", self.lib.gvs_db_export, n, ("kmer", "contig", "start", "group", "gidx"),
                           dtypes=dict(kmer=np.uint64))

    # ------------------------------------------------------------------------------------
    # reads
    # ------------------------------------------------------------------------------------
    def set_reads(self, seq: np.ndarray, read_off: np.ndarray, chunk_first=None, chunk_hap=None):
        """Host batch: concatenated ASCII reads + offsets (+ chunk table)."""
        seq = _c(seq, np.uint8)
        read_off = _c(read_off, np.uint64)
        n = len(read_off) - 1
        chunk_first = _c([0, n] if chunk_first is None else chunk_first, np.uint64)
        chunk_hap = _c([0] * (len(chunk_first) - 1) if chunk_hap is None else chunk_hap, np.uint8)
        self._keep = [seq, read_off]
        self.n_reads = n
        self._ck(self.lib.gvs_reads_set(self.ctx, _ptr(seq), _ptr(read_off), n, _ptr(chunk_first), _ptr(chunk_hap),
                                        len(chunk_hap), 0))

    def set_reads_packed(self, words: np.ndarray, read_off: np.ndarray, chunk_first=None, chunk_hap=None):
        """Host batch whose bases are already 2-bit packed (pack_2bit / NativeReads.pack()): a quarter of
        the bytes of set_reads() on the PCIe link, identical results."""
        words = _c(words, np.uint32)
        read_off = _c(read_off, np.uint64)
        n = len(read_off) - 1
        assert len(words) * 16 >= int(read_off[-1])
        chunk_first = _c([0, n] if chunk_first is None else chunk_first, np.uint64)
        chunk_hap = _c([0] * (len(chunk_first) - 1) if chunk_hap is None else chunk_hap, np.uint8)
        self._keep = [words, read_off]
        self.n_reads = n
        self._ck(self.lib.gvs_reads_set_packed(self.ctx, _ptr(words), _ptr(read_off), n, _ptr(chunk_first), _ptr(chunk_hap),
                                               len(chunk_hap), 0))

    def set_copy_pipeline(self, min_bytes: int = 256 << 20, segments: int = 16):
        """Host batches >= min_bytes are copied in `segments` pieces overlapped with the match."""
        self._ck(self.lib.gvs_set_copy_pipeline(self.ctx, int(min_bytes), int(segments)))

    PACK_OFF, PACK_ADAPTIVE, PACK_ALL, PACK_ALTERNATE = 0, 1, 2, 3

    def set_probe_variant(self, variant: int = 0):
        """0: probe instantiation by database size, 1: small-database, 2: large-database (call before the
        database is loaded / built; results are identical)."""
        self._ck(self.lib.gvs_set_probe_variant(self.ctx, int(variant)))

    def set_db_passes(self, n: int = 0):
        """Count passes of build_db / build_db_device: 0 (default) as few as the free device memory allows, 1..64
        exactly n (the database is the same; call before the build)."""
        self._ck(self.lib.gvs_set_db_passes(self.ctx, int(n)))

    def set_host_pack(self, mode: int = 1, threads: int = 0):
        """How the segments of a pipelined ASCII host batch travel: as they are (PACK_OFF), 2-bit packed by
        `threads` host threads (PACK_ALL), or whichever keeps both the PCIe link and the cores busy
        (PACK_ADAPTIVE, the default).  Results do not depend on it."""
        self._ck(self.lib.gvs_set_host_pack(self.ctx, int(mode), int(threads)))

    def copy_stats(self):
        """(sequence bytes copied host->device, segments, segments sent packed) of the last host batch."""
        b, n, k = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
        self._ck(self.lib.gvs_copy_stats(self.ctx, C.byref(b), C.byref(n), C.byref(k)))
        return int(b.value), int(n.value), int(k.value)

    def set_reads_device(self, seq_ptr: int, off_ptr: int, n_reads: int, chunk_first, chunk_hap):
        chunk_first = _c(chunk_first, np.uint64)
        chunk_hap = _c(chunk_hap, np.uint8)
        self.n_reads = n_reads
        self._ck(self.lib.gvs_reads_set(self.ctx, C.c_void_p(seq_ptr), C.c_void_p(off_ptr), n_reads, _ptr(chunk_first),
                                        _ptr(chunk_hap), len(chunk_hap), 1))

    def set_reads_packed_device(self, words_ptr: int, off_ptr: int, n_reads: int, chunk_first, chunk_hap):
        """batch resident in HBM as 2-bit words (device pointers; see set_reads_packed)"""
        chunk_first = _c(chunk_first, np.uint64)
        chunk_hap = _c(chunk_hap, np.uint8)
        self.n_reads = n_reads
        self._ck(self.lib.gvs_reads_set_packed(self.ctx, C.c_void_p(words_ptr), C.c_void_p(off_ptr), n_reads, _ptr(chunk_first),
                                               _ptr(chunk_hap), len(chunk_hap), 1))

    def set_reads_meta(self, read_len, chunk_first=None, chunk_hap=None):
        """Read table without sequences ({hap}.rlen, workflow/src/rlen.nim:13-14)."""
        read_len = _c(read_len, np.uint32)
        n = len(read_len)
        chunk_first = _c([0, n] if chunk_first is None else chunk_first, np.uint64)
        chunk_hap = _c([0] * (len(chunk_first) - 1) if chunk_hap is None else chunk_hap, np.uint8)
        self.n_reads = n
        self._ck(self.lib.gvs_reads_meta(self.ctx, _ptr(read_len), n, _ptr(chunk_first), _ptr(chunk_hap), len(chunk_hap)))

    def set_rows(self, which: int, read, pos, contig, start, group, n_contigs: Optional[int] = None):
        """Rows parsed from a .sunkpos file (input of diag_filter_v3 / badsunks / process-by-contig)."""
        cols = [_c(a, np.uint32) for a in (read, pos, contig, start, group)]
        n = len(cols[0])
        nc = len(self.contig_names) if n_contigs is None else n_contigs
        self._ck(self.lib.gvs_rows_set(self.ctx, which, *[_ptr(a) for a in cols], n, nc))
        if which == 0:
            self.n_rows = n
        else:
            self.n_kept = n

    # ------------------------------------------------------------------------------------
    # stages
    # ------------------------------------------------------------------------------------
    def match(self) -> int:
        """kmerpos_annot3 main loop (workflow/src/kmerpos_annot3.nim:81-97)."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_match(self.ctx, C.byref(n)))
        self.n_rows = int(n.value)
        return self.n_rows

    ROW_COLUMNS = ("read", "pos", "contig", "start", "group")

    def rows(self, which: int = 0, n: Optional[int] = None, pinned: bool = False) -> Dict[str, np.ndarray]:
        if n is None:
            n = self.n_rows if which == 0 else self.n_kept
        return self._table(f"rows{which}", self.lib.gvs_rows_get, n, self.ROW_COLUMNS, lead=(which,), pinned=pinned)

    def diag_filter(self, contig_hap: Sequence[int], read_haps: bool = False) -> Tuple[int, int]:
        """diag_filter_v3 + diag_filter_step2 (workflow/src/diag_filter_v3.nim:18-229,
        workflow/src/diag_filter_step2.nim:13-66).  contig_hap[c] = haplotype whose .fai lists
        contig c (255 = neither).  read_haps: also vote on the other haplotype and keep the records for
        read_haps() (include/gavisunk_b200.h gvs_diag_filter_haps); always on for a batch with GVS_HAP_ANY chunks,
        whose reads keep their rows on the haplotype their votes assign."""
        ch = _c(contig_hap, np.uint8)
        hh = np.array([nim_hash(n) for n in self.contig_names], dtype=np.uint32)
        assert len(ch) == len(self.contig_names)
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.gvs_diag_filter_haps(self.ctx, _ptr(ch), _ptr(hh), 1 if read_haps else 0, C.byref(a), C.byref(b)))
        self.n_best, self.n_kept = int(a.value), int(b.value)
        return self.n_best, self.n_kept

    READ_HAP_COLUMNS = ("read", "contig1", "n1", "strand1", "contig2", "n2", "strand2", "hap")

    def read_haps(self, pinned: bool = False) -> Dict[str, np.ndarray]:
        """Read haplotypes (no reference counterpart; include/gavisunk_b200.h gvs_diag_filter_haps): one record per read
        with a vote on either haplotype, of the last diag filter in haplotype mode, or of the run after run_batches --
        read (run-wide index), per haplotype the voted contig (0xFFFFFFFF: none), its votes n (0: none) and strand
        (0 '+', 1 '-'), and the assignment hap (0, 1, 2 = tie)."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_read_haps(self.ctx, C.byref(n)))
        return self._table("read_haps", self.lib.gvs_read_haps_get, int(n.value), self.READ_HAP_COLUMNS, pinned=pinned)

    def best(self) -> Dict[str, np.ndarray]:
        return self._table("best", self.lib.gvs_best_get, self.n_best, ("read", "contig", "ngood", "dir"),
                           dtypes=dict(dir=np.uint8))

    def filter_best(self, best_contig_of_read) -> int:
        """diag_filter_step2 (workflow/src/diag_filter_step2.nim:13-66) with the best contigs given."""
        b = _c(best_contig_of_read, np.uint32)
        n = C.c_uint64()
        self._ck(self.lib.gvs_filter_best(self.ctx, _ptr(b), C.byref(n)))
        self.n_kept = int(n.value)
        return self.n_kept

    def set_contigs(self, contig_hap: Sequence[int]):
        ch = _c(contig_hap, np.uint8)
        hh = np.array([nim_hash(n) for n in self.contig_names], dtype=np.uint32)
        self._ck(self.lib.gvs_contigs_set(self.ctx, _ptr(ch), _ptr(hh) if len(hh) == len(ch) else None, len(ch)))

    def run_all(self, contig_hap: Sequence[int], min_read_len: int = 10000, allreduce_hist=None, gather_forests=None):
        """The fused hot path on the reads bound to this engine: match -> diag filter -> bad-SUNK
        histogram -> validation -> contig-wide components -> intervals.  With several GPUs
        `allreduce_hist(ptr, n_groups)` sums the int32 histogram across ranks in place and
        `gather_forests(ptr, n_groups)` gathers the parent arrays: None with a single rank, else
        (pointer of the [n_ranks][n_groups] array on this device, n_ranks, own rank)."""
        self.match()
        self.diag_filter(contig_hap)
        return self._global_stages(self.group_hist(), min_read_len, allreduce_hist, gather_forests)

    def _global_stages(self, hist_ptr: int, min_read_len: int, allreduce_hist, gather_forests):
        """everything after the histogram: its all-reduce, bad groups, validation, local forest, forest
        merge, intervals"""
        if allreduce_hist is not None:
            allreduce_hist(hist_ptr, self.db_groups())
        self.bad_groups()
        self.validate(min_read_len)
        pp = self.components_local()
        gathered = gather_forests(pp, self.db_groups()) if gather_forests is not None else None
        if gathered is not None:
            self.components_merge_all(*gathered)
        return self.intervals()

    # ------------------------------------------------------------------------------------
    # several batches of one run (two phases; csrc/batches.cu)
    # ------------------------------------------------------------------------------------
    def batches_begin(self):
        self._ck(self.lib.gvs_batches_begin(self.ctx))

    def batch_stash(self) -> int:
        """keeps the batch's kept rows + read lengths resident; returns the run-wide index of its first read"""
        b = C.c_uint64()
        self._ck(self.lib.gvs_batch_stash(self.ctx, C.byref(b)))
        return int(b.value)

    def batches_bind(self) -> Tuple[int, int]:
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.gvs_batches_bind(self.ctx, C.byref(a), C.byref(b)))
        self.n_kept, self.n_reads = int(a.value), int(b.value)
        return self.n_kept, self.n_reads

    def run_batches(self, binds, contig_hap: Sequence[int], min_read_len: int = 10000, allreduce_hist=None,
                    gather_forests=None, on_batch=None, junctions: bool = False, read_haps: bool = False,
                    sunk_depth: bool = False, allele_support: bool = False):
        """The hot path over a run whose reads come in several batches (a sample's chunk files, or the shard of
        them this GPU owns).  The reference gathers all chunks of a haplotype before the global stages
        (workflow/Snakefile:23-24, workflow/rules/tagONT.smk:112-131; badsunks_AR.py:20-27 counts over every
        row), so the run has two phases:
          1. per batch: bind(self) registers the batch's reads (set_reads / set_reads_packed /
             set_reads_device ...), then match -> diag filter -> histogram (accumulated) -> stash of the kept rows;
             on_batch(self, b, read_base) may fetch the batch's rows (rows(0) / rows(1), best()) for file egress;
          2. ONE histogram all-reduce (`allreduce_hist`), bad groups, validation of all stashed rows, local
             forest, ONE forest all-gather (`gather_forests`), intervals.
        Results equal run_all() on the concatenation of the batches; read indices of rows(1) / pairs() count
        through the batches in order.  junctions: also screen every batch after its diag filter (junction_screen),
        so that junctions() reports the run's records afterwards.  read_haps: run every diag filter in haplotype mode,
        so that read_haps() reports the run's records afterwards (batches with GVS_HAP_ANY chunks always are).  sunk_depth:
        also count every batch's match rows (sunk_depth, accumulated), so that depth() reports the run's SUNK hit depth.
        allele_support: also count every batch's match rows by read haplotype after its diag filter (allele_support,
        accumulated; unbinned reads take the haplotype that filter assigns), so that alleles() reports the run's counts.
        Returns (intervals, [read_base of every batch])."""
        self.batches_begin()
        bases, hp = [], 0
        rows = best = 0
        for b, bind in enumerate(binds):
            bind(self)
            rows += self.match()
            if sunk_depth:
                self.sunk_depth(accumulate=True)
            best += self.diag_filter(contig_hap, read_haps)[0]
            if allele_support:
                self.allele_support(accumulate=True)
            if junctions:
                self.junction_screen(min_read_len)
            hp = self.group_hist(accumulate=True)
            base = self.batch_stash()
            if on_batch is not None:
                on_batch(self, b, base)
            bases.append(base)
        self.batches_bind()
        self.n_rows, self.n_best = rows, best
        if not bases:  # a rank without a batch still takes part in both exchanges (and in depth()'s and alleles()')
            self.set_contigs(contig_hap)
            hp = self.group_hist(accumulate=True)
            if sunk_depth:
                self.sunk_depth(accumulate=True)
            if allele_support:
                self.allele_support(accumulate=True)
        return self._global_stages(hp, min_read_len, allreduce_hist, gather_forests), bases

    def db_groups(self) -> int:
        a, b = C.c_uint64(), C.c_uint64()
        rc = self.lib.gvs_db_size(self.ctx, C.byref(a), C.byref(b))
        return int(b.value) if rc == 0 else 0

    def group_hist(self, accumulate: bool = False) -> int:
        """badsunks_AR.py:20-27 histogram; returns the device pointer of the int32[n_groups] array."""
        p = C.c_void_p()
        self._ck(self.lib.gvs_group_hist(self.ctx, 1 if accumulate else 0, C.byref(p)))
        return int(p.value or 0)

    def bad_groups(self) -> int:
        """badsunks_AR.py:43-52: mode per haplotype on the device, limit = m + 4*sqrt(m) in float64
        on the host exactly as the reference computes it, threshold test on the device."""
        mode = (C.c_int64 * 2)()
        self._ck(self.lib.gvs_hist_mode(self.ctx, mode))
        lim = (C.c_int64 * 2)()
        self.modes = [int(mode[0]), int(mode[1])]
        for h in range(2):
            m = int(mode[h])
            lim[h] = int(math.floor(m + (np.int64(m) ** 0.5) * 4)) if m > 0 else (1 << 62)
        n = C.c_uint64()
        self._ck(self.lib.gvs_bad_groups(self.ctx, lim, C.byref(n)))
        self.n_bad = int(n.value)
        return self.n_bad

    def bad_list(self) -> np.ndarray:
        out = np.zeros(self.n_bad, np.uint32)
        self._ck(self.lib.gvs_bad_get(self.ctx, _ptr(out)))
        return out

    def bad_set(self, contig, group) -> int:
        """bad groups from a bad_sunks.txt (process-by-contig_lowmem_AR.py:66-72): (contig id, group) pairs."""
        c = _c(contig, np.uint32)
        g = _c(group, np.uint32)
        n = C.c_uint64()
        self._ck(self.lib.gvs_bad_set(self.ctx, _ptr(c), _ptr(g), len(c), C.byref(n)))
        self.n_bad = int(n.value)
        return self.n_bad

    def groups(self, with_hist: bool = False) -> Dict[str, np.ndarray]:
        """group table behind every group index: (contig, group start[, row count of group_hist])"""
        n = C.c_uint64()
        self._ck(self.lib.gvs_groups_count(self.ctx, C.byref(n)))
        return self._table("groups", self.lib.gvs_groups_get, int(n.value), ("contig", "group", "count" if with_hist else None),
                           dtypes=dict(count=np.int32))

    def validate(self, min_read_len: int = 10000) -> int:
        """process-by-contig_lowmem_AR.py:50-207 (per-read part)."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_validate(self.ctx, min_read_len, C.byref(n)))
        self.n_pairs = int(n.value)
        return self.n_pairs

    def validate_empty_reads(self) -> int:
        """reads of the last validate() whose multipos clean-up dropped every oriented edge (they validate nothing)"""
        n = C.c_uint64()
        self._ck(self.lib.gvs_validate_stats(self.ctx, C.byref(n)))
        return int(n.value)

    PAIR_COLUMNS = ("read", "contig", "group", "gidx")

    def pairs(self, pinned: bool = False) -> Dict[str, np.ndarray]:
        return self._table("pairs", self.lib.gvs_pairs_get, self.n_pairs, self.PAIR_COLUMNS, pinned=pinned)

    PLACEMENT_COLUMNS = ("read", "contig", "start", "end", "n_ids", "strand")

    def placements(self, pinned: bool = False) -> Dict[str, np.ndarray]:
        """Support placements of the validated reads (no reference counterpart): one per read with >= 2 validated
        IDs -- read (run-wide index), contig, start / end (smallest / largest validated ID), n_ids, strand (0 '+',
        1 '-').  Also leaves the per-rank difference array on the device for support()."""
        n, p = C.c_uint64(), C.c_void_p()
        self._ck(self.lib.gvs_placements(self.ctx, C.byref(n), C.byref(p)))
        self._diff_ptr = int(p.value or 0)
        return self._table("placements", self.lib.gvs_placements_get, int(n.value), self.PLACEMENT_COLUMNS,
                           dtypes=dict(strand=np.uint8), pinned=pinned)

    SUPPORT_COLUMNS = ("contig", "start", "end", "depth")

    def support(self, contig_len: Sequence[int], allreduce=None) -> Dict[str, np.ndarray]:
        """Support depth after placements(): runs (contig, start, end, depth) tiling every contig.  With several GPUs
        `allreduce(ptr, n_groups)` sums the int32 difference array across ranks in place first (the callable that
        sums the bad-SUNK histogram)."""
        return self._runs("support", self.lib.gvs_support, self.lib.gvs_support_get, self.SUPPORT_COLUMNS, "_diff_ptr",
                          contig_len, allreduce)

    SPAN_COLUMNS = ("read", "contig", "id1", "start1", "pos1", "id2", "start2", "pos2")

    def spans(self, min_delta: int = 300, rel_permille: int = 30) -> Dict[str, np.ndarray]:
        """Distance discordance of the validated reads (no reference counterpart; include/gavisunk_b200.h gvs_spans), after
        validate(): one record per non-concordant span between consecutive usable rows of a read -- read (run-wide
        index), contig, and the (ID, start, pos) of both rows; delta = |pos2 - pos1| - (start2 - start1), longer when
        delta >= 0.  Also leaves the per-rank difference arrays (spans, longer, shorter) on the device for discordance()."""
        n, p = C.c_uint64(), C.c_void_p()
        self._ck(self.lib.gvs_spans(self.ctx, int(min_delta), int(rel_permille), C.byref(n), C.byref(p)))
        self._dc_diff_ptr = int(p.value or 0)
        return self._table("spans", self.lib.gvs_spans_get, int(n.value), self.SPAN_COLUMNS)

    DISCORDANCE_COLUMNS = ("contig", "start", "end", "spans", "longer", "shorter")

    def discordance(self, contig_len: Sequence[int], allreduce=None) -> Dict[str, np.ndarray]:
        """Discordance runs after spans(): (contig, start, end, spans, longer, shorter) tiling every contig.  With several
        GPUs `allreduce(ptr, n)` sums the int32 difference arrays (n = 3 * n_groups) across ranks in place first (the
        callable that sums the bad-SUNK histogram)."""
        return self._runs("discordance", self.lib.gvs_discordance, self.lib.gvs_discordance_get, self.DISCORDANCE_COLUMNS,
                          "_dc_diff_ptr", contig_len, allreduce)

    def sunk_depth(self, accumulate: bool = False) -> int:
        """SUNK hit depth of the current match rows (after match() or set_rows(0); no reference counterpart;
        include/gavisunk_b200.h gvs_sunk_depth): adds every row to hits[g] and every distinct (read, group) to reads[g].
        accumulate: add to the previous counts (run_batches starts from zero at its batches_begin).  Returns the device
        pointer of the int32[2][n_groups] array."""
        p = C.c_void_p()
        self._ck(self.lib.gvs_sunk_depth(self.ctx, 1 if accumulate else 0, C.byref(p)))
        self._dp_ptr = int(p.value or 0)
        self._dp_summed = False
        return self._dp_ptr

    def _n_groups(self) -> int:
        n = C.c_uint64()
        self._ck(self.lib.gvs_groups_count(self.ctx, C.byref(n)))
        return int(n.value)

    def depth(self, allreduce=None) -> Dict[str, np.ndarray]:
        """Per group index (the table of groups()): hits, reads (int32, of sunk_depth), sunks (.loc rows) and kept (the
        int32 histogram of group_hist).  With several GPUs `allreduce(ptr, n)` sums the hits and reads (n = 2 * n_groups)
        across ranks in place first (the callable that sums the bad-SUNK histogram), once per sunk_depth(): a later call
        reads the counts summed already."""
        ng = self._n_groups()
        if allreduce is not None and not getattr(self, "_dp_summed", False):
            allreduce(self._dp_ptr, 2 * ng)
            self._dp_summed = True
        out = self._table("depth", self.lib.gvs_sunk_depth_get, ng, ("hits", "reads", "sunks"), dtypes=dict(hits=np.int32, reads=np.int32))
        out["kept"] = self.groups(with_hist=True)["count"]
        return out

    DEPTH_COLUMNS = ("contig", "start", "end", "hits", "reads", "kept")

    def depth_runs(self, contig_len: Sequence[int]) -> Dict[str, np.ndarray]:
        """SUNK hit depth runs after sunk_depth() (and depth()'s all-reduce) and group_hist(): (contig, start, end, hits,
        reads, kept) tiling every contig in segment space."""
        return self._runs("depth_runs", self.lib.gvs_depth_runs, self.lib.gvs_depth_runs_get, self.DEPTH_COLUMNS, "_dp_ptr",
                          contig_len, None)

    def allele_support(self, accumulate: bool = False) -> int:
        """Allele support of the current match rows (after match() or set_rows(0), and after the diag filter of a batch
        with unbinned chunks; no reference counterpart; include/gavisunk_b200.h gvs_allele_support): adds every distinct
        (read, group) to own[g] when the read's file haplotype is the group's, else to other[g].  accumulate: add to the
        previous counts (run_batches starts from zero at its batches_begin).  Returns the device pointer of the
        int32[2][n_groups] array."""
        p = C.c_void_p()
        self._ck(self.lib.gvs_allele_support(self.ctx, 1 if accumulate else 0, C.byref(p)))
        self._al_ptr = int(p.value or 0)
        self._al_summed = False
        return self._al_ptr

    def alleles(self, allreduce=None) -> Dict[str, np.ndarray]:
        """Per group index (the table of groups()): own, other (int32, of allele_support), sunks (.loc rows) and end (last
        SUNK start + k).  With several GPUs `allreduce(ptr, n)` sums own and other (n = 2 * n_groups) across ranks in place
        first (the callable that sums the bad-SUNK histogram), once per allele_support(): a later call reads the counts
        summed already."""
        ng = self._n_groups()
        if allreduce is not None and not getattr(self, "_al_summed", False):
            allreduce(self._al_ptr, 2 * ng)
            self._al_summed = True
        return self._table("alleles", self.lib.gvs_allele_support_get, ng, ("own", "other", "sunks", "end"),
                           dtypes=dict(own=np.int32, other=np.int32))

    ALLELE_COLUMNS = ("contig", "start", "end", "own", "other")

    def allele_runs(self, contig_len: Sequence[int]) -> Dict[str, np.ndarray]:
        """Allele support runs after allele_support() (and alleles()' all-reduce): (contig, start, end, own, other) tiling
        every contig in segment space."""
        return self._runs("allele_runs", self.lib.gvs_allele_runs, self.lib.gvs_allele_runs_get, self.ALLELE_COLUMNS, "_al_ptr",
                          contig_len, None)

    def components_local(self) -> int:
        """this GPU's forest of the validated pairs; returns the device pointer of its uint32[n_groups] parent array"""
        p = C.c_void_p()
        self._ck(self.lib.gvs_components_local(self.ctx, C.byref(p)))
        return int(p.value or 0)

    def components_merge_all(self, gathered_ptr: int, n_ranks: int, own_rank: int):
        """unions in every peer's forest in one pass (gathered = [n_ranks][n_groups] parent arrays on this device)"""
        self._ck(self.lib.gvs_components_merge_all(self.ctx, C.c_void_p(gathered_ptr), int(n_ranks), int(own_rank)))

    def intervals(self) -> Dict[str, np.ndarray]:
        """process-by-contig_lowmem_AR.py:215-260 -> rows of bed_files/*.bed."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_intervals(self.ctx, C.byref(n)))
        return self._table("intervals", self.lib.gvs_intervals_get, int(n.value), ("contig", "start", "end"))

    def set_intervals(self, contig, start, end, n_contigs: int):
        """rows of bed_files/*.bed as the input of gaps() (get_gaps.py:30)."""
        c, s, e = _c(contig, np.uint32), _c(start, np.uint32), _c(end, np.uint32)
        self._ck(self.lib.gvs_intervals_set(self.ctx, _ptr(c), _ptr(s), _ptr(e), len(c), int(n_contigs)))

    def gaps(self, contig_len: Sequence[int]):
        """get_gaps.py:17-123."""
        cl = _c(contig_len, np.uint32)
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.gvs_gaps(self.ctx, _ptr(cl), C.byref(a), C.byref(b)))
        g = self._table("gaps", self.lib.gvs_gaps_get, int(a.value), ("contig", "start", "end", "nodata"),
                        counts=dict(nodata=int(b.value)))
        nd = g.pop("nodata")
        return g, nd

    GAP_EVIDENCE_COLUMNS = ("read", "gap", "left_id", "left_start", "left_pos", "right_id", "right_start", "right_pos")

    def gap_evidence(self, min_read_len: int = 10000) -> Dict[str, np.ndarray]:
        """The reads that bridge each gap of gaps() (no reference counterpart; include/gavisunk_b200.h gvs_gap_evidence):
        one record per bridging (read, gap) of the kept rows minus the bad groups, reads of length >= min_read_len --
        read (run-wide index), gap (index into the gaps() arrays), and the (ID, start, pos) of its left and right flank
        rows.  Call gaps() on this engine first."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_gap_evidence(self.ctx, int(min_read_len), C.byref(n)))
        return self._table("gap_evidence", self.lib.gvs_gap_evidence_get, int(n.value), self.GAP_EVIDENCE_COLUMNS)

    JUNCTION_COLUMNS = ("read", "contig1", "strand1", "ids1", "id1", "start1", "pos1", "contig2", "strand2", "ids2", "id2",
                        "start2", "pos2")

    def junction_screen(self, min_read_len: int = 10000) -> Tuple[int, int]:
        """Junction screen of the current match rows (after match() or set_rows(0); in run_batches before the batch's
        stash): the anchored rows of qualifying contigs of reads with >= 2 of them join the run's junction stash
        (include/gavisunk_b200.h gvs_junction_screen).  -> (rows, reads) in the stash"""
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.gvs_junction_screen(self.ctx, int(min_read_len), C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def junctions(self) -> Dict[str, np.ndarray]:
        """Reads whose SUNKs jump from one contig to another (no reference counterpart; include/gavisunk_b200.h
        gvs_junctions): one record per pair of consecutive blocks of a screened read, with the bad groups of this engine
        (or none) -- read (run-wide index), then per side contig, strand (0 '+', 1 '-'), distinct IDs of the block and
        the (ID, start, pos) of its row next to the junction."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_junctions(self.ctx, C.byref(n)))
        return self._table("junctions", self.lib.gvs_junctions_get, int(n.value), self.JUNCTION_COLUMNS)

    SWITCH_COLUMNS = ("read", "contig", "strand1", "ids1", "lo1", "hi1", "id1", "start1", "pos1", "strand2", "ids2", "lo2", "hi2",
                      "id2", "start2", "pos2")

    def strand_switches(self, min_read_len: int = 10000, pinned: bool = False) -> Dict[str, np.ndarray]:
        """Reads whose SUNKs switch strand inside one contig (no reference counterpart; include/gavisunk_b200.h
        gvs_strand_switches), from the kept rows minus the bad groups, reads of length >= min_read_len: one record per pair
        of consecutive blocks of one strand -- read (run-wide index), contig, then per block its strand (0 '+', 1 '-'),
        distinct IDs, smallest / largest start and the (ID, start, pos) of its row next to the switch."""
        n = C.c_uint64()
        self._ck(self.lib.gvs_strand_switches(self.ctx, int(min_read_len), C.byref(n)))
        return self._table("switches", self.lib.gvs_strand_switches_get, int(n.value), self.SWITCH_COLUMNS, pinned=pinned)

    def covprob_table(self, kbp, cnt, genome_kbp: float, pn: float) -> np.ndarray:
        """covprob.py:56-100."""
        kbp = _c(kbp, np.int64)
        cnt = _c(cnt, np.int64)
        out = np.zeros(3500, np.float64)
        self._ck(self.lib.gvs_covprob_table(self.ctx, _ptr(kbp), _ptr(cnt), len(kbp), float(genome_kbp), float(pn),
                                            _ptr(out)))
        return out


    def covprob_gaps(self, grp_contig, grp_id, gap_contig, gap_start, gap_end, table):
        """covprob.py:109-131: per gap (max_gap, covprob)."""
        gc, gi = _c(grp_contig, np.uint32), _c(grp_id, np.uint32)
        pc, ps, pe = _c(gap_contig, np.uint32), _c(gap_start, np.int64), _c(gap_end, np.int64)
        tb = _c(table, np.float64)
        assert len(tb) == 3500
        mg, pr = np.zeros(len(pc), np.int64), np.zeros(len(pc), np.float64)
        self._ck(self.lib.gvs_covprob_gaps(self.ctx, _ptr(gc), _ptr(gi), len(gc), _ptr(pc), _ptr(ps), _ptr(pe), len(pc),
                                           _ptr(tb), _ptr(mg), _ptr(pr)))
        return mg, pr

    def slop(self, contig, start, end, contig_len, b: int = 200000):
        """slop_gaps (workflow/rules/tagONT.smk:249)."""
        c = _c(contig, np.uint32)
        s, e = np.array(start, dtype=np.int64), np.array(end, dtype=np.int64)
        cl = _c(contig_len, np.uint32)
        self._ck(self.lib.gvs_slop(self.ctx, _ptr(c), _ptr(s), _ptr(e), len(c), _ptr(cl), len(cl), int(b)))
        return s, e


# ----------------------------------------------------------------------------------------------
# covprob host scalars (workflow/scripts/covprob.py:63-81): the reference solves
# 1 - x + q p^r x^(r+1) = 0 with sympy and keeps the positive real root that is NOT 1/p; pn is the
# probability of at least one error-free run of r bases in a window of n = 30 (Feller).  Two
# scalars per run: computed on the host in float64, the 3500-entry table is the GPU kernel.
# ----------------------------------------------------------------------------------------------
def covprob_root(r: int, p: float = 0.94) -> float:
    q = 1.0 - p
    a = q * p ** r

    def f(x):
        return 1.0 - x + a * x ** (r + 1)

    def df(x):
        return -1.0 + a * (r + 1) * x ** r

    xs = ((r + 1) * a) ** (-1.0 / r)  # minimiser of the convex f on x > 0; the two roots bracket it
    pinv = 1.0 / p
    if pinv > xs:
        lo, hi = 1.0, xs
    else:
        lo, hi = xs, max(2.0, 4.0 * xs)
        while f(hi) < 0:
            hi *= 2.0
    flo = f(lo)
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        fm = f(mid)
        if (fm > 0) == (flo > 0):
            lo, flo = mid, fm
        else:
            hi = mid
    x = 0.5 * (lo + hi)
    for _ in range(4):
        x -= f(x) / df(x)
    return x


def covprob_pn(r: int, p: float = 0.94, n: int = 30) -> float:
    q = 1.0 - p
    x = covprob_root(r, p)
    qn = ((1.0 - p * x) / (q * (r + 1 - r * x))) * (1.0 / (x ** (n + 1)))  # covprob.py:79
    return float(1.0 - qn)


def covprob_bins(read_lens):
    """covprob.py:44-53: drop duplicate (name, len) rows, sort by length descending, kbp = int(len/1000),
    value_counts(sort=False) -> bins in order of first appearance."""
    seen, lens = set(), []
    for nm, ln in read_lens:
        if (nm, ln) in seen:
            continue
        seen.add((nm, ln))
        lens.append(int(ln))
    kbp, cnt, idx = [], [], {}
    for ln in sorted(lens, reverse=True):
        b = int(ln / 1000)
        if b not in idx:
            idx[b] = len(kbp)
            kbp.append(b)
            cnt.append(0)
        cnt[idx[b]] += 1
    return np.asarray(kbp, np.int64), np.asarray(cnt, np.int64)

#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: ONT read Gbp/s SUNK-matched + distance-validated.

One "step" = one pass of the whole hot path (match -> best-contig filter -> bad-SUNK histogram ->
inter-SUNK distance validation -> contig-wide components -> intervals -> gaps; SURVEY.md 8d) over
one batch of synthetic reads, against a SUNK database built on the GPU from a synthetic diploid
assembly.  `value` is measured with the reads already resident in HBM; `e2e` goes through the same
public API (gavisunk_b200.engine.Engine) with HOST buffers, host->device copy of the reads and
device->host read of the results inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload s150|h3100|tiny] [--impl reference] [--dump-outputs DIR]

N > 1: launched by torchrun, one rank per GPU; every rank owns its own shard of reads of the same
size (weak scaling), the SUNK table is replicated; NCCL all-reduces the group-hit histogram and
all-gathers the union-find forests (the only two exchanges on the path, SURVEY.md 8e).

--impl reference: the reference's own executables (oracle/_ref: kmerpos_annot3, diag_filter_v3,
diag_filter_step2, unmodified prebuilt binaries) on the host cores, one process per chunk with all
cores busy, followed by the CPU port of the Python stages (oracle/gavisunk_oracle.py; the
reference's scripts need graph_tool / pyranges which are not installed) -- on a bounded sample.

--dump-outputs DIR: after the timed steps of the GPU path (--impl b200), what its last step computed is written to
DIR as .npy files (dump_outputs), so that two builds of the project can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "ont_read_gbp_per_s_sunk_matched_validated"
UNIT = "Gbp/s"
STAGES = ("probe", "emit", "diag", "hist", "validate", "intervals")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="h3100", choices=["tiny", "s150", "h3100"])
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--asm-mbp", type=float, default=None, help="override haploid assembly size (Mbp)")
    ap.add_argument("--coverage", type=float, default=None, help="override read coverage per GPU shard")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-batches", type=int, default=2, help="batches per rank of the end-to-end run (0 = all; page-locked host memory)")
    ap.add_argument("--e2e-headline-only", action="store_true", help="skip the secondary e2e figures (ASCII copies only, packed host input)")
    ap.add_argument("--batches", type=int, default=None, help="override the number of read batches of the run")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the run (all batches) is the same for every N; weak: one batch per rank")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary figures of the N = 1 run (2-bit resident reads, s150 k sweep)")
    ap.add_argument("--resident", default="ascii", choices=["ascii", "packed"],
                    help="form of the HBM-resident reads of `value`: ASCII bases (what the reference consumes) or the 2-bit words the "
                         "ingest emits (gvs_fastx_read_packed)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-mbp", type=float, default=None, help="read Mbp per CPU process of the baseline sample")
    ap.add_argument("--ref-asm-mbp", type=float, default=40.0, help="--impl reference: haploid size of the sample assembly (numpy + oracle set-up)")
    ap.add_argument("--e2e-files-gbp", type=float, default=None, help="read Gbp of the files -> files run (default: 4 at N = 1, skipped at N > 1; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl b200: write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB; "
                         "see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's results (--impl b200)")
    return args


WORKLOADS = {
    "tiny": dict(mbp=2.0, human=False, cov=15.0, batches=2, n50=20000.0,
                 desc="synthetic 2 Mbp x2 diploid + 30x ONT-like reads in 2 batches (smoke size)"),
    "s150": dict(mbp=150.0, human=False, cov=30.0, batches=1, n50=50000.0,
                 desc="synthetic 150 Mbp single-chromosome x2 diploid assembly + 30x simulated ONT reads (N50 ~50 kb), one batch"),
    "h3100": dict(mbp=3100.0, human=True, cov=3.75, batches=8, n50=100000.0,
                  desc="synthetic 3.1 Gbp x2 diploid assembly (23 contigs) + 30x ultra-long ONT-like reads (N50 ~100 kb, 93 Gbp) "
                       "in 8 batches of 3.75x (10 chunk files per haplotype each)"),
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            time.sleep(0.25)  # let the first sample land before the timed region starts
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if t_begin is not None and not (t_begin <= ts <= t_end + 0.06):
                continue
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
                pw.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=(float(np.median(sm)) if sm else None), sm_max_mhz=(max(mx) if mx else None),
                    power_w_max=(max(pw) if pw else None), reasons=sorted(reasons), samples=len(sm))


def shard_batches(n_batches: int, world: int):
    """contiguous blocks of batches per rank (a batch is a group of whole chunk files, SURVEY 8e)"""
    from gavisunk_b200.parallel import shard_chunks
    return shard_chunks(n_batches, world)


def build_workload(args, eng, rank, world=1, with_reads=True):
    """assembly + SUNK database on this GPU and the read batches this rank owns.  The run is the SAME for every
    N (batch b always has seed 2001 + 16 b): rank r owns a contiguous block of the batches (strong scaling), or --
    --scaling weak -- every rank owns batch `rank` only, a run N times as large as at N = 1."""
    from gavisunk_b200 import workload as W
    spec = dict(WORKLOADS[args.workload])
    if args.asm_mbp is not None:
        spec["mbp"] = args.asm_mbp
    if args.coverage is not None:
        spec["cov"] = args.coverage
    if args.batches is not None:
        spec["batches"] = args.batches
    L = int(spec["mbp"] * 1e6)
    contigs = W.human_contigs(spec["mbp"]) if spec["human"] else [L]
    t0 = time.time()
    wl = W.make_assembly(eng, contigs, snp_rate=1e-3, dup_frac=0.01, seed=1001, name=args.workload)
    eng.set_profiling(True)
    W.build_db(eng, wl)
    db_ms = eng.stage_ms("dbbuild")
    nb = int(spec["batches"])
    if args.scaling == "weak":
        mine, nb_total = [rank], world
    else:
        lo, hi = shard_batches(nb, world)[rank]
        mine, nb_total = list(range(lo, hi)), nb
    wl.batch_ids, wl.batches, wl.n_batches_total = mine, [], nb_total
    wl.batch_args = dict(coverage=spec["cov"], n50=spec["n50"], sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    if with_reads:
        for b in mine:
            nbt = W.new_batch(eng, wl, seed=2001 + 16 * b, **wl.batch_args)
            if args.resident == "packed":
                W.pack_batch_on_device(nbt, drop_ascii=False)
            wl.batches.append(nbt)
    wl.meta.update(db_build_ms=db_ms, setup_s=time.time() - t0, desc=spec["desc"], asm_mbp=spec["mbp"], n50=spec["n50"], sigma=0.8,
                   cov_per_batch=spec["cov"], n_batches=nb_total)
    return wl


def run_step(eng, wl, binds, coll):
    """one pass of the hot path over this rank's batches (two phases, gavisunk_b200.engine.Engine.run_batches);
    returns the result sizes (rows / best / kept / validated pairs are this rank's, the rest is global)"""
    iv, bases = eng.run_batches(binds, wl.contig_hap, min_read_len=10000, allreduce_hist=coll.allreduce_hist,
                                gather_forests=coll.gather_forests)
    gaps, nodata = eng.gaps(wl.contig_len.astype(np.uint32))
    return dict(rows=eng.n_rows, best=eng.n_best, kept=eng.n_kept, bad_groups=eng.n_bad, validated_pairs=eng.n_pairs,
                intervals=int(len(iv["contig"])), gaps=int(len(gaps["contig"])), nodata=int(len(nodata))), iv, gaps


def result_digest(iv, gaps, eng):
    """sha256 over the run's global results: validated intervals, gaps, bad SUNK groups"""
    import hashlib
    h = hashlib.sha256()
    for d in (iv, gaps):
        for c in ("contig", "start", "end"):
            h.update(np.ascontiguousarray(d[c], dtype=np.uint32).tobytes())
    h.update(np.sort(eng.bad_list()).astype(np.uint32).tobytes())
    return h.hexdigest()


# --dump-outputs: rows kept per array (a fixed, seeded sample of larger results); together at most DUMP_LIMIT bytes
DUMP_ROWS = dict(intervals=1 << 18, gaps=1 << 18, bad_groups=1 << 18, pairs=1 << 20)
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, sizes, iv, gaps, eng, seed=0):
    """What the last timed step handed its caller, as DIR/<name>.npy in float64 (every value is an integer below
    2**53, so the conversion is exact):
      size_<name>  one result size of the step as run_step reports it (rows, best, kept, bad_groups,
                   validated_pairs, intervals, gaps, nodata), as an array of one element
      intervals    validated intervals (contig, start, end)         gaps        gaps between them (contig, start, end)
      bad_groups   bad SUNK groups (group index), sorted            pairs       this rank's validated pairs (read,
                                                                                contig, group, gidx) in engine order
    An array longer than DUMP_ROWS[name] rows is replaced by the rows at a sorted random sample of its indices
    (numpy default_rng(seed)), written beside it as <name>_index.npy.  The inputs of a run are fixed by its
    arguments, so two builds can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    pairs = eng.pairs()
    tables = dict(intervals=[iv[c] for c in ("contig", "start", "end")], gaps=[gaps[c] for c in ("contig", "start", "end")],
                  bad_groups=[np.sort(eng.bad_list())], pairs=[pairs[c] for c in ("read", "contig", "group", "gidx")])
    out = {f"size_{k}": np.array([v], np.float64) for k, v in sizes.items()}
    for name, cols in tables.items():
        n, cap = len(cols[0]), DUMP_ROWS[name]
        if n > cap:
            idx = np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))
            out[name + "_index"] = idx.astype(np.float64)
            cols = [c[idx] for c in cols]
        out[name] = np.stack([np.asarray(c, np.float64) for c in cols], axis=1)
    assert sum(a.nbytes for a in out.values()) <= DUMP_LIMIT
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main_b200(args):
    import torch
    import torch.distributed as dist
    from gavisunk_b200 import workload as W
    from gavisunk_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from gavisunk_b200.parallel import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local) if world > 1 else dict(numa_node=None)  # pinned read buffers on the GPU's own socket
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng = Engine(args.k, device=local, stream=torch.cuda.current_stream().cuda_stream)
    wl = build_workload(args, eng, rank, world)
    n_sunks, n_groups = eng.db_size()
    from gavisunk_b200.parallel import EngineExchange
    coll = EngineExchange(dev, eng=eng)
    my_bases = int(sum(b.total_bases for b in wl.batches))
    my_reads = int(sum(b.n_reads for b in wl.batches))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allsum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def allmax(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in wl.batches]
    # ---- HBM-resident timing ----
    for _ in range(max(args.warmup, 3)):
        res, iv, gaps = run_step(eng, wl, binds, coll)
    launches0 = eng.launches
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms = {}
    tb = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        res, iv, gaps = run_step(eng, wl, binds, coll)
    e1.record()
    barrier()
    te = time.perf_counter()
    clocks = sampler.stop(tb, te)
    ms = e0.elapsed_time(e1)
    launches = eng.launches - launches0
    ms_max = allmax(ms)
    total_bases = allsum(my_bases)
    value = total_bases * args.steps / (ms_max * 1e-3) / 1e9
    digest = result_digest(iv, gaps, eng)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, iv, gaps, eng)

    # ---- per-stage device times (CUDA events of the library around each stage, on its stream): one extra pass with
    #      the stage times read after every batch / phase-2 stage (reading them waits for the stage, so it is kept out
    #      of the timed region above) ----
    per_batch = {st: [] for st in ("probe", "emit", "diag", "hist")}

    def on_batch(e, b, base):
        for st in per_batch:
            per_batch[st].append(e.stage_ms(st))
    for _ in range(2):
        for st in per_batch:
            per_batch[st].clear()
        eng.run_batches(binds, wl.contig_hap, allreduce_hist=coll.allreduce_hist, gather_forests=coll.gather_forests, on_batch=on_batch)
    phase2 = {}
    for st in ("mode", "bad", "validate", "components", "merge", "intervals"):  # the once-per-run stages (merge: N > 1 only)
        try:
            phase2[st] = eng.stage_ms(st) if wl.batches else 0.0
        except Exception:
            pass
    stage_ms = {st: float(np.sum(v)) for st, v in per_batch.items()}
    stage_ms.update(phase2)

    # ---- roofline of the dominant kernel (k_probe2): one launch per batch ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    k = args.k
    roofline = None
    if wl.batches:
        windows = 0
        for b in wl.batches:
            lens = np.diff(b.read_off.cpu().numpy())
            windows += int(np.maximum(lens - k + 1, 0).sum())
        nbm = len(wl.batches)
        probe_bytes = (float(my_bases) * 1.0 + windows * 16.0) / nbm  # SURVEY 8d: 1 B/base in + one 16 B slot per window, per launch
        probe_ms = float(np.mean(per_batch["probe"]))
        achieved = probe_bytes / (probe_ms * 1e-3) / 1e9
        traffic = None
        if k == 20 and args.asm_mbp is None and args.coverage is None:  # the ncu capture is of the default shapes
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "probe_traffic.json"))).get(args.workload)
            except Exception:
                pass
        roofline = dict(bound="hbm", kernel=f"k_probe2<{k}>", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                        traffic=traffic, traffic_unit="DRAM bytes per launch (ncu --set full, profiles/probe_traffic.json)",
                        traffic_gbs=(traffic / (probe_ms * 1e-3) / 1e9 if traffic else None),
                        traffic_frac_of_peak=(traffic / (probe_ms * 1e-3) / 1e9 / peak if traffic else None),
                        peak_source="MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650",
                        alg_bytes_per_launch=probe_bytes, kernel_ms=probe_ms, launches_per_step=nbm,
                        kernel_share_of_step=probe_ms * nbm * args.steps / ms,
                        whole_path_alg_gbs=(probe_bytes * nbm + 24.0 * res["rows"]) * args.steps / (ms * 1e-3) / 1e9,
                        note=("algorithmic bytes follow SURVEY.md 8d (1 B per base + one 16 B table slot per window); the "
                              "two-level filter answers ~99 % of the windows without touching their slot, so `achieved` may "
                              "exceed the DRAM peak -- `traffic_gbs` is what the kernel really moves"))

    # ---- N ranks == 1 rank: the same run on rank 0 alone (all batches, no exchange), outside the timed region ----
    parity_check = None
    if world > 1 and not args.no_parity_check:
        pairs_total = allsum(res["validated_pairs"])
        kept_total = allsum(res["kept"])
        ok, single = None, None
        if rank == 0:
            class _NoColl:
                allreduce_hist = None
                gather_forests = None
            eng1 = eng
            mine = {b: wl.batches[i] for i, b in enumerate(wl.batch_ids)}
            cache = {}

            def bind_any(e, b):
                if b in mine:
                    W.bind_batch(e, mine[b])
                else:  # a peer's batch: regenerated here from its seed (one at a time, the buffer is reused)
                    cache.clear()
                    cache[b] = W.new_batch(e, wl, seed=2001 + 16 * b, **wl.batch_args)
                    W.bind_batch(e, cache[b])
            all_ids = list(range(wl.n_batches_total))
            iv1, _ = eng1.run_batches([(lambda e, b=b: bind_any(e, b)) for b in all_ids], wl.contig_hap)
            gaps1, _nd1 = eng1.gaps(wl.contig_len.astype(np.uint32))
            single = dict(digest=result_digest(iv1, gaps1, eng1), intervals=int(len(iv1["contig"])), gaps=int(len(gaps1["contig"])),
                          bad_groups=eng1.n_bad, validated_pairs=eng1.n_pairs, kept=eng1.n_kept)
            cache.clear()
            ok = (single["digest"] == digest and single["validated_pairs"] == int(pairs_total) and single["kept"] == int(kept_total)
                  and single["bad_groups"] == res["bad_groups"])
        flag = torch.tensor([1.0 if (ok or rank != 0) else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        # every rank holds the replicated global result: their digests must agree as well
        dg = torch.tensor([int(digest[:15], 16)], dtype=torch.int64, device=dev)
        dmin, dmax = dg.clone(), dg.clone()
        dist.all_reduce(dmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(dmax, op=dist.ReduceOp.MAX)
        if rank == 0:
            parity_check = dict(n_ranks=world, ok=bool(ok and int(dmin.item()) == int(dmax.item())), replicated_result_agrees=int(dmin.item()) == int(dmax.item()),
                                intervals=res["intervals"], gaps=res["gaps"], bad_groups=res["bad_groups"], validated_pairs=int(pairs_total),
                                kept_rows=int(kept_total), digest=digest, single_rank=single,
                                what="rank 0 re-ran ALL batches of the run alone (no exchange) after the timed region: intervals, gaps and bad "
                                     "SUNK groups (sha256), validated pairs and kept rows equal the N-rank run's")
        if float(flag.item()) == 0.0 or int(dmin.item()) != int(dmax.item()):
            if rank == 0:
                print(json.dumps({"metric": METRIC, "error": "parity_check failed: N-rank result differs from the single-rank run",
                                  "parity_check": parity_check}))
            if world > 1:
                dist.destroy_process_group()
            sys.exit(3)
        # the re-run left rank 0's engine holding the single-rank results; restore the distributed state for what follows
        res, iv, gaps = run_step(eng, wl, binds, coll)

    # ---- end to end through the public API with HOST buffers ----
    e2e = None
    if args.e2e_steps > 0:
        e2e = measure_e2e(args, eng, wl, coll, dev, world, rank, numa, barrier, allmax, allsum)
        # files -> files: by default at N = 1 only (a rank that failed in there would leave its peers waiting in a collective)
        if (args.e2e_files_gbp is None and world == 1) or (args.e2e_files_gbp or 0) > 0:
            try:
                ef = measure_e2e_files(args, eng, wl, coll, dev, world, rank, barrier, allmax, allsum)
            except Exception as ex:  # a secondary figure must never take the bench down
                import traceback
                ef = dict(error=repr(ex)[:300], where=traceback.format_exc()[-400:])
            if e2e is not None:
                e2e["from_files"] = ef
            res, iv, gaps = run_step(eng, wl, binds, coll)  # back to the resident state of the run

    # ---- secondary figures (N = 1): the same run with the reads resident as the ingest's 2-bit words, and BASELINE
    #      configs 3 / 5 (150 Mbp, SUNK_len sweep) ----
    secondary = None
    if world == 1 and not args.no_secondary and args.workload == "h3100":
        secondary = {}
        try:
            secondary["resident_2bit"] = measure_packed_resident(args, eng, wl, coll, run_step)
        except Exception as ex:
            secondary["resident_2bit"] = dict(error=repr(ex)[:300])
        try:
            secondary["s150_k_sweep"] = measure_k_sweep(args, local)
        except Exception as ex:
            secondary["s150_k_sweep"] = dict(error=repr(ex)[:300])
        res, iv, gaps = run_step(eng, wl, binds, coll)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu_baseline = cpu_reference_sample(args, wl, eng, per_proc_mbp=args.cpu_sample_mbp or 12.0)
        except Exception as ex:  # the baseline must never take the bench down
            cpu_baseline = dict(error=repr(ex)[:300])

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": wl.meta["desc"], "k": k, "asm_haploid_mbp": wl.meta["asm_mbp"], "resident_reads": args.resident,
                       "read_gbp_per_step": total_bases / 1e9, "batches_per_step": wl.n_batches_total,
                       "read_gbp_rank0": my_bases / 1e9, "reads_rank0": my_reads, "batches_rank0": len(wl.batches),
                       "n_sunks": n_sunks, "n_groups": n_groups, "results_per_step": res,
                       "l2": "inputs larger than L2 (every batch's reads >> 126 MB)",
                       "stages": ["match", "diag_filter", "bad_sunks", "validate", "components", "intervals", "gaps"],
                       "phases": "per batch: match -> diag filter -> histogram (accumulated) -> stash; once: all-reduce, bad groups, "
                                 "validation, components, all-gather, intervals, gaps",
                       "db_build_ms": wl.meta["db_build_ms"], "stage_ms_per_step_rank0": stage_ms,
                       "parallelism": f"batches of chunk files sharded over {world} GPU(s), SUNK table replicated; 2 collectives per run"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "parity_check": parity_check, "secondary": secondary,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def measure_packed_resident(args, eng, wl, coll, run_step, steps=5):
    """`value` again with every batch resident in HBM as 2-bit words -- the form gvs_fastx_read_packed delivers and
    cli.run_reads feeds to the GPU (the PACKED instantiation of the probe; 2.9 GB instead of 11.5 GB per batch stream
    through L2).  Results must equal the ASCII-resident run's."""
    import torch
    from gavisunk_b200 import workload as W
    want, _, _ = run_step(eng, wl, [(lambda e, b=b: W.bind_batch(e, b)) for b in wl.batches], coll)
    for b in wl.batches:
        W.pack_batch_on_device(b, drop_ascii=False)
    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in wl.batches]
    try:
        got, _, _ = run_step(eng, wl, binds, coll)
        assert got == want, "2-bit resident reads must give the ASCII run's results"
        run_step(eng, wl, binds, coll)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            run_step(eng, wl, binds, coll)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        probe = []
        eng.run_batches(binds, wl.contig_hap, on_batch=lambda e, b, base: probe.append(e.stage_ms("probe")))
        bases = sum(b.total_bases for b in wl.batches)
        return dict(value=bases / (ms * 1e-3) / 1e9, unit=UNIT, ms_per_step=ms, steps=steps, probe_ms_per_launch=float(np.mean(probe)),
                    note="reads resident as 2-bit words (kmer.encode's byte map; what the ingest emits); identical results")
    finally:
        for b in wl.batches:
            b.words = None


def measure_k_sweep(args, device, steps=8):
    """BASELINE configs 3 and 5: synthetic 150 Mbp x2 assembly + 30x reads (N50 ~50 kb, 4.5 Gbp, one batch), SUNK_len
    16 / 20 / 24 / 31, reads resident in HBM; one engine per SUNK_len"""
    import copy
    import torch
    from gavisunk_b200.engine import Engine
    from gavisunk_b200 import workload as W
    out = {}
    for k in (16, 20, 24, 31):
        a2 = copy.copy(args)
        a2.workload, a2.k, a2.asm_mbp, a2.coverage, a2.batches, a2.resident, a2.scaling = "s150", k, None, None, None, "ascii", "strong"
        e2 = Engine(k, device=device, stream=torch.cuda.current_stream().cuda_stream)
        try:
            w2 = build_workload(a2, e2, 0, 1)

            class _NoColl:
                allreduce_hist = None
                gather_forests = None
            binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in w2.batches]
            for _ in range(3):
                r2, _, _ = run_step(e2, w2, binds, _NoColl)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                run_step(e2, w2, binds, _NoColl)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            bases = sum(b.total_bases for b in w2.batches)
            ns, ng = e2.db_size()
            out[f"k{k}"] = dict(value=bases / (ms * 1e-3) / 1e9, unit=UNIT, ms_per_step=ms, read_gbp=bases / 1e9, n_sunks=ns, n_groups=ng,
                                rows=r2["rows"], probe_ms=e2.stage_ms("probe"), db_build_ms=w2.meta["db_build_ms"])
            del w2, binds
        finally:
            e2.close()
            torch.cuda.empty_cache()
    out["workload"] = WORKLOADS["s150"]["desc"]
    return out


def measure_e2e(args, eng, wl, coll, dev, world, rank, numa, barrier, allmax, allsum):
    """The same run through Engine.run_batches with HOST buffers: every batch's reads start in page-locked host
    memory as ASCII (what the reference's readfq loop consumes), cross PCIe inside the timed region (as they are or
    2-bit packed on the way by the library's host threads) and the results (validated pairs, intervals, gaps) come
    back to the host.  Page-locked memory for the whole run may exceed the host (30x human = 93 GB): the run is then
    timed over the first `--e2e-batches` batches of every rank (same path, same per-batch sizes; stated)."""
    import torch
    from gavisunk_b200 import workload as W
    nb_e2e = len(wl.batches) if args.e2e_batches <= 0 else min(len(wl.batches), args.e2e_batches)
    sub = wl.batches[:nb_e2e]
    sub_bases = int(sum(b.total_bases for b in sub))
    sub_reads = int(sum(b.n_reads for b in sub))
    total_sub = allsum(sub_bases)
    # resident run on the same subset = what the host path must reproduce
    binds_res = [(lambda e, b=b: W.bind_batch(e, b)) for b in sub]
    res, _, _ = run_step(eng, wl, binds_res, coll)
    host = []
    for b in sub:
        h_reads = torch.empty(b.total_bases + 64, dtype=torch.uint8, pin_memory=True)
        h_reads[:b.total_bases].copy_(b.reads[:b.total_bases])
        h_off = torch.empty(b.n_reads + 1, dtype=torch.int64, pin_memory=True)
        h_off.copy_(b.read_off)
        host.append((h_reads, h_off, h_reads.numpy()[:b.total_bases], h_off.numpy().view(np.uint64), b))
    torch.cuda.synchronize()
    binds_h = [(lambda e, h=h: e.set_reads(h[2], h[3], h[4].chunk_first, h[4].chunk_hap)) for h in host]

    def time_host_path(binds):
        r0, _, _ = run_step(eng, wl, binds, coll)
        assert r0 == res, "the host path must reproduce the resident path"
        eng.pairs(pinned=True)  # warm-up also sizes the page-locked result and staging buffers
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        f0.record()
        d2h = h2d = 0
        for _ in range(args.e2e_steps):
            h2d = [0]

            def on_batch(e, b, base):
                h2d[0] += e.copy_stats()[0] + 8 * (sub[b].n_reads + 1)
            iv2, _ = eng.run_batches(binds, wl.contig_hap, allreduce_hist=coll.allreduce_hist, gather_forests=coll.gather_forests,
                                     on_batch=on_batch)
            gaps2, _nd = eng.gaps(wl.contig_len.astype(np.uint32))   # intervals + gaps come back to the host
            pairs = eng.pairs(pinned=True)                            # inter_outs rows (group, read) into page-locked memory
            d2h = sum(a.nbytes for a in pairs.values()) + sum(a.nbytes for a in iv2.values()) + sum(a.nbytes for a in gaps2.values())
        f1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        return allmax(max(f0.elapsed_time(f1), wall_ms)), d2h, h2d[0]

    n_cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    pack_threads = max(1, min(16, n_cores // max(local_world, 1)))
    # Ranks that share one host share its memory bandwidth between the DMA reads and the packers (profiles/README.md): the
    # adaptive packing is used where a rank has at least 12 cores to itself.
    pack_mode = eng.PACK_ADAPTIVE if (local_world == 1 or pack_threads >= 12) else eng.PACK_OFF
    eng.set_host_pack(pack_mode, pack_threads)
    e2e = None
    if sub:
        ems, d2h, h2d = time_host_path(binds_h)
        seq_bytes, n_seg, n_seg_packed = eng.copy_stats()
        e2e = dict(value=total_sub * args.e2e_steps / (ems * 1e-3) / 1e9, unit=UNIT,
                   h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                   steps=args.e2e_steps, ms_per_step=ems / args.e2e_steps, host_numa_node=numa.get("numa_node"),
                   batches_per_step_per_rank=nb_e2e, read_gbp_per_step=total_sub / 1e9,
                   host_input_bytes_per_step=int(sub_bases + 8 * (sub_reads + nb_e2e)),
                   scope=(f"the first {nb_e2e} of this rank's {len(wl.batches)} batches (page-locked host memory for the whole run "
                          f"would be {sum(b.total_bases for b in wl.batches) / 1e9:.0f} GB); same two-phase path, results checked against "
                          "the resident run on the same batches") if nb_e2e < len(wl.batches) else "all batches of the run",
                   transfer=dict(mode="adaptive" if pack_mode == eng.PACK_ADAPTIVE else "ascii copies only (host cores shared by the ranks)",
                                 host_pack_threads=pack_threads, segments_last_batch=n_seg, segments_packed_last_batch=n_seg_packed,
                                 note="input = ASCII bases in page-locked host memory; a segment crosses PCIe as ASCII or 2-bit "
                                      "packed by the host threads (kmer.encode's byte map), chosen at run time"))
        if pack_mode != eng.PACK_OFF and not args.e2e_headline_only:
            try:  # the same call with the host cores idle (every segment as ASCII): the transfer-bound figure
                eng.set_host_pack(eng.PACK_OFF, pack_threads)
                ems0, _, h2d0 = time_host_path(binds_h)
                e2e["ascii_copy_only"] = dict(value=total_sub * args.e2e_steps / (ems0 * 1e-3) / 1e9, unit=UNIT,
                                              ms_per_step=ems0 / args.e2e_steps, h2d_bytes_per_step=int(h2d0))
            except Exception as ex:
                e2e["ascii_copy_only"] = dict(error=repr(ex)[:200])
            eng.set_host_pack(pack_mode, pack_threads)
        if not args.e2e_headline_only:
            # secondary: host batches that the ingest delivered 2-bit packed (gvs_fastx_read's native output /
            # gvs_pack_2bit; the packing is outside the timed region like the parse that produces the ASCII buffers)
            try:
                from gavisunk_b200.engine import pack_2bit
                packed = []
                for h in host:
                    nw = (h[4].total_bases + 15) // 16
                    hw = torch.zeros(nw + 16, dtype=torch.int32, pin_memory=True)
                    npw = hw.numpy().view(np.uint32)
                    pack_2bit(h[2], threads=pack_threads, out=npw)
                    packed.append((hw, npw[:nw], h[3], h[4]))
                binds_p = [(lambda e, q=q: e.set_reads_packed(q[1], q[2], q[3].chunk_first, q[3].chunk_hap)) for q in packed]
                emsp, _, h2dp = time_host_path(binds_p)
                e2e["packed_host_input"] = dict(value=total_sub * args.e2e_steps / (emsp * 1e-3) / 1e9, unit=UNIT,
                                                h2d_bytes_per_step=int(h2dp), ms_per_step=emsp / args.e2e_steps,
                                                note="2-bit words (kmer.encode's byte map, lossless for this path) as the library's ingest "
                                                     "emits them; packing is part of the ingest, outside the timed region")
                del packed
            except Exception as ex:
                e2e["packed_host_input"] = dict(error=repr(ex)[:200])
    del host
    return e2e


def measure_e2e_files(args, eng, wl, coll, dev, world, rank, barrier, allmax, allsum):
    """The reference's REAL boundary: chunk FASTQ files in, result files out.  The reads of (a part of) this rank's
    first batch are written as the 2 x 10 chunk files split_ONT would leave (4-line FASTQ, quality '#';
    page-cache warm: they sit in tmpfs) -- untimed set-up.  Timed: gavisunk_b200.cli.run_reads (parse + 2-bit pack
    on the host threads, H2D of the words, every kernel of the path, the two exchanges) + cli.write_outputs
    (sunkpos/, breaks/*.sunkpos, inter_outs/, bed_files/, final_out/ formatted natively and written to disk; the
    exports of the database itself are left out, they belong to the database build).  A second pass times the
    same files gzip-compressed (.fq.gz, what the rule really writes) on a tenth of the reads: zlib inflate bound."""
    import gzip
    import torch
    from concurrent.futures import ThreadPoolExecutor
    from gavisunk_b200 import cli
    if not wl.batches:
        return dict(skipped="this rank owns no batch")
    b = wl.batches[0]
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    base_dir = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else tempfile.gettempdir()
    free = shutil.disk_usage(base_dir).free
    want_gbp = args.e2e_files_gbp if args.e2e_files_gbp is not None else 4.0
    cap_gbp = free * 0.45 / max(local_world, 1) / 2.1 / 1e9  # FASTQ = 2 bytes per base (+ names)
    gbp = min(want_gbp, cap_gbp, b.total_bases / 1e9)
    if gbp < 0.05:
        return dict(skipped=f"no room for the chunk files under {base_dir} ({free / 1e9:.0f} GB free)")
    root = tempfile.mkdtemp(prefix=f"gvs_e2e_r{rank}_", dir=base_dir)
    try:
        off = b.read_off.cpu().numpy().astype(np.int64)
        cf = b.chunk_first.astype(np.int64)
        frac = gbp * 1e9 / b.total_bases
        files, file_hap, n_sel_reads, n_sel_bases, gz_files = [], [], 0, 0, []

        def write_chunk(c):
            r0, r1 = int(cf[c]), int(cf[c + 1])
            r1 = r0 + max(1, int(round((r1 - r0) * frac)))  # the first part of every chunk
            seq = b.reads[int(off[r0]):int(off[r1])].cpu().numpy()
            lens = (off[r0 + 1:r1 + 1] - off[r0:r1]).astype(np.int64)
            names = [b"@r%09d\n" % i for i in range(r0, r1)]
            nl = np.fromiter((len(x) for x in names), np.int64, len(names))
            rec = nl + 2 * lens + 4  # name line, seq, '\n+\n', quality, '\n'
            out = np.full(int(rec.sum()), ord("#"), np.uint8)
            o = np.concatenate([[0], np.cumsum(rec)[:-1]])
            so = off[r0:r1] - off[r0]
            for i in range(r1 - r0):
                p0 = int(o[i])
                out[p0:p0 + int(nl[i])] = np.frombuffer(names[i], np.uint8)
                p1 = p0 + int(nl[i])
                L = int(lens[i])
                out[p1:p1 + L] = seq[int(so[i]):int(so[i]) + L]
                out[p1 + L:p1 + L + 3] = (10, 43, 10)
                out[p1 + 2 * L + 3] = 10
            hap = int(b.chunk_hap[c])
            idx = c - (0 if hap == 0 else int(np.sum(b.chunk_hap == 0)))
            fp = os.path.join(root, f"hap{hap + 1}_{idx + 1}-of-10.fq")
            out.tofile(fp)
            gzp = None
            if idx == 0:  # one chunk file per haplotype also as .fq.gz
                gzp = fp + ".gz"
                with gzip.open(gzp, "wb", compresslevel=1) as f:
                    f.write(out.data)
            return fp, hap, r1 - r0, int(lens.sum()), gzp
        with ThreadPoolExecutor(max_workers=min(8, len(cf) - 1)) as ex:
            for fp, hap, nr, nb, gzp in ex.map(write_chunk, range(len(cf) - 1)):
                files.append(fp)
                file_hap.append(hap)
                n_sel_reads += nr
                n_sel_bases += nb
                if gzp:
                    gz_files.append((gzp, hap, nb))
        file_bytes = sum(os.path.getsize(f) for f in files)
        clen = wl.contig_len.astype(np.uint32)

        def one_pass(fl, fh, outdir, batch_gbp):
            t0 = time.perf_counter()
            results = cli.run_reads([eng], wl.contig_hap, fl, fh, batch_gbp=batch_gbp, coll=coll if world > 1 else None)
            gaps, nodata = eng.gaps(clen)
            t1 = time.perf_counter()
            cli.write_outputs(args.k, eng, results, clen, wl.contig_hap, wl.contig_names, results[0]["iv"], gaps, nodata, outdir, db_files=False)
            t2 = time.perf_counter()
            return t2 - t0, t1 - t0, t2 - t1, results
        outdir = os.path.join(root, "results")
        one_pass(files, file_hap, outdir, 12.0)  # warm-up: buffers, page-locked pools
        barrier()
        times, split = [], [0.0, 0.0]
        for _ in range(max(1, args.e2e_steps)):
            shutil.rmtree(outdir, ignore_errors=True)
            barrier()
            t, t_run, t_write, results = one_pass(files, file_hap, outdir, 12.0)
            times.append(t)
            split[0] += t_run / max(1, args.e2e_steps)
            split[1] += t_write / max(1, args.e2e_steps)
        t_files = allmax(float(np.mean(times)))
        total = allsum(n_sel_bases)
        out_bytes = sum(os.path.getsize(os.path.join(dp, f)) for dp, _, fs in os.walk(outdir) for f in fs)
        kept_rows = int(len(results[0]["kept"]["read"]))
        n_lines = sum(1 for _ in open(os.path.join(outdir, "sunkpos", "hap1.sunkpos"), "rb")) + \
            sum(1 for _ in open(os.path.join(outdir, "sunkpos", "hap2.sunkpos"), "rb"))
        assert n_lines == kept_rows, "every kept row must be a line of {hap}.sunkpos"
        res = dict(value=total / t_files / 1e9, unit=UNIT, read_gbp=total / 1e9, s_per_pass=t_files, input_file_bytes_rank0=int(file_bytes),
                   output_file_bytes_rank0=int(out_bytes), host_split_s=dict(ingest_and_gpu=round(split[0], 3), format_and_write=round(split[1], 3)),
                   files=f"{len(files)} chunk FASTQ files per rank under {base_dir} (page-cache warm), one batch, ingest threads = "
                         f"{max(1, (len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else os.cpu_count()))}",
                   kept_rows_rank0=kept_rows, note="files -> files: parse + 2-bit pack (gvs_fastx_read_packed), H2D, kernels, D2H, native formatting "
                                                   "(gvs_format_rows) and writes inside the timed region; database exports excluded")
        if gz_files:
            gl, gh = [g[0] for g in gz_files], [g[1] for g in gz_files]
            gb = sum(g[2] for g in gz_files)
            one_pass(gl, gh, os.path.join(root, "results_gz"), 12.0)
            barrier()
            tg, _, _, _ = one_pass(gl, gh, os.path.join(root, "results_gz"), 12.0)
            res["fq_gz"] = dict(value=allsum(gb) / allmax(tg) / 1e9, unit=UNIT, read_gbp=allsum(gb) / 1e9, files=f"{len(gl)} .fq.gz chunk files per rank (gzip level 1)",
                                note="same path from gzip-compressed chunk files: bound by zlib inflate, one host thread per file")
        return res
    finally:
        shutil.rmtree(root, ignore_errors=True)


# --------------------------------------------------------------------------------------------
# CPU reference (oracle/_ref executables + oracle port of the Python stages) on a bounded sample
# --------------------------------------------------------------------------------------------
def _write_db_files(eng, wl, workdir, contig_sel=None):
    """jellyfish.db / kmer.loc / .fai text files in the reference's formats from the GPU-built db
    (contig_sel: only the .loc rows of these contigs -- the sample of a database too large for the
    reference's 278 B/SUNK hash tables and ~2 us/SUNK text load)"""
    import pandas as pd
    db = eng.db_export()
    if contig_sel is not None:
        m = np.isin(db["contig"], np.asarray(sorted(contig_sel), dtype=np.uint32))
        db = {c: v[m] for c, v in db.items()}
    k = eng.k
    km = db["kmer"]
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    codes = ((km[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    kmers = letters.view(f"S{k}").ravel().astype(str)
    names = np.asarray(wl.contig_names)
    dbp, locp = os.path.join(workdir, "jellyfish.db"), os.path.join(workdir, "kmer.loc")
    pd.DataFrame({"k": kmers}).to_csv(dbp, header=False, index=False)
    pd.DataFrame({"c": names[db["contig"]], "s": db["start"], "k": kmers, "g": db["group"]}).to_csv(
        locp, sep="\t", header=False, index=False)
    nc = len(wl.contig_names) // 2
    fais = []
    for hap in range(2):
        fp = os.path.join(workdir, f"hap{hap + 1}.fai")
        with open(fp, "w") as f:
            for c in range(hap * nc, (hap + 1) * nc):
                f.write(f"{wl.contig_names[c]}\t{int(wl.contig_len[c])}\t0\t60\t61\n")
        fais.append(fp)
    return dbp, locp, fais


def _prepare_reference_sample(args, wl, eng, per_proc_mbp, cores):
    """writes the sample's input files; returns what the timed part needs"""
    workdir = tempfile.mkdtemp(prefix="gvs_cpu_")
    if True:
        n_sunks, _ = eng.db_size()
        contig_sel, sample_note = None, ""
        if n_sunks > 8_000_000:
            # whole-genome database: the reference would need ~33 GB and ~4 min of text parsing per process.
            # Sample = a contiguous run of contigs of ~150 Mbp per haplotype: their .loc rows + reads drawn
            # from them by the same generator (same length / error model).
            import copy
            from gavisunk_b200 import workload as W
            nc = len(wl.contig_names) // 2
            lens = wl.contig_len[:nc].astype(np.int64)
            best = (0, 1)
            for lo in range(nc):
                for hi in range(lo + 1, nc + 1):
                    if abs(int(lens[lo:hi].sum()) - 150_000_000) < abs(int(lens[best[0]:best[1]].sum()) - 150_000_000):
                        best = (lo, hi)
            lo, hi = best
            sub_len = int(lens[lo:hi].sum())
            swl = copy.copy(wl)
            swl.meta = dict(wl.meta)
            cov = per_proc_mbp * 1e6 * cores * 1.15 / sub_len
            W.add_reads(eng, swl, coverage=cov, n50=wl.meta.get("n50", 50000.0), sigma=wl.meta.get("sigma", 0.8), len_min=1000,
                        len_max=1000000, seed=777, nchunks=1, contig_range=(lo, hi))
            contig_sel = set(range(lo, hi)) | set(range(nc + lo, nc + hi))
            sample_note = (f"database restricted to contigs {wl.contig_names[lo]}..{wl.contig_names[hi - 1]} of both haplotypes "
                           f"({sub_len / 1e6:.0f} Mbp x2; the full {n_sunks / 1e6:.0f} M-SUNK table needs ~33 GB and minutes of text "
                           "parsing per reference process), reads drawn from them by the same generator; ")
            wl = swl
        else:  # small database: the sample is cut from the run's first batch
            import copy
            from gavisunk_b200 import workload as W
            if not wl.batches:
                wl.batches.append(W.new_batch(eng, wl, seed=2001, **wl.batch_args))
            b0 = wl.batches[0]
            swl = copy.copy(wl)
            swl.reads, swl.read_off, swl.n_reads, swl.total_bases = b0.reads, b0.read_off, b0.n_reads, b0.total_bases
            wl = swl
        dbp, locp, fais = _write_db_files(eng, wl, workdir, contig_sel)
        off = wl.read_off.cpu().numpy()
        nph = wl.n_reads // 2
        per_hap_procs = max(1, cores // 2)
        jobs, sample_bases, sample_reads, rlen = [], 0, 0, {}
        want = int(per_proc_mbp * 1e6)
        for hap in range(2):
            r = hap * nph
            for c in range(per_hap_procs):
                r0 = r
                while r < (hap + 1) * nph and off[r] - off[r0] < want:
                    r += 1
                if r == r0:
                    break
                seq = wl.reads[int(off[r0]):int(off[r])].cpu().numpy()
                fp = os.path.join(workdir, f"hap{hap + 1}_{c}.fa")
                with open(fp, "wb") as f:
                    for i in range(r0, r):
                        f.write(b">r%09d\n" % i)
                        f.write(seq[int(off[i] - off[r0]):int(off[i + 1] - off[r0])].tobytes())
                        f.write(b"\n")
                        rlen["r%09d" % i] = int(off[i + 1] - off[i])
                jobs.append(dict(workdir=workdir, tag=f"hap{hap + 1}_{c}", reads=fp, db=dbp, loc=locp, fai=fais[hap]))
                sample_bases += int(off[r] - off[r0])
                sample_reads += r - r0
        return dict(workdir=workdir, jobs=jobs, dbp=dbp, locp=locp, rlen=rlen, sample_note=sample_note, sample_bases=sample_bases,
                    sample_reads=sample_reads, wl=wl)


_SAMPLE_CACHE = {}


def _cleanup_samples():
    for prep in _SAMPLE_CACHE.values():
        shutil.rmtree(prep["workdir"], ignore_errors=True)
    _SAMPLE_CACHE.clear()


def _prepare_numpy_sample(args, per_proc_mbp, cores, asm_mbp=40.0):
    """The reference arm's own inputs, made WITHOUT libgavisunk_b200.so: numpy generator of the same recipe (SURVEY
    8d: i.i.d. haplotype 1 with 1 % segmental duplications in 10-100 kb blocks, haplotype 2 = SNPs at 1e-3, reads
    log-normal N50 ~100 kb, 3 % substitutions + 2 % deletions + 1 % insertions, both strands), the oracle's
    restatement of defineSUNKs.smk for jellyfish.db / kmer.loc (jellyfish, mrsfast, bedtools are not installed)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import gavisunk_oracle as O
    import j1_sim as S
    from concurrent.futures import ThreadPoolExecutor
    workdir = tempfile.mkdtemp(prefix="gvs_ref_")
    k = args.k
    L = int(asm_mbp * 1e6)
    rng = np.random.default_rng(1001)
    alpha = np.frombuffer(b"ACGT", np.uint8)
    h1 = alpha[rng.integers(0, 4, L)]
    done = 0
    while done < L // 100:
        ln = int(rng.integers(10000, 100000))
        a, b = int(rng.integers(0, L - ln)), int(rng.integers(0, L - ln))
        h1[b:b + ln] = h1[a:a + ln]
        done += ln
    h2 = h1.copy()
    snp = rng.random(L) < 1e-3
    h2[snp] = alpha[(O.BASE_LUT[h1[snp]] + rng.integers(1, 4, int(snp.sum()))) % 4]
    n_ctg = 8  # contigs per haplotype: process_by_contig is one job per contig in the reference (tagONT.smk:170-191)
    cuts = [L * i // n_ctg for i in range(n_ctg + 1)]
    haps = [[(f"synH{h + 1}_chr{i + 1}", (h1, h2)[h][cuts[i]:cuts[i + 1]].tobytes()) for i in range(n_ctg)] for h in range(2)]
    names = [n for h in haps for n, _ in h]
    db = O.build_sunk_db(haps[0] + haps[1], k)
    kms = np.asarray(db["kmer"], np.uint64)
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    letters = alpha[((kms[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)].view(f"S{k}").ravel().astype(str)
    import pandas as pd
    dbp, locp = os.path.join(workdir, "jellyfish.db"), os.path.join(workdir, "kmer.loc")
    pd.DataFrame({"k": letters}).to_csv(dbp, header=False, index=False)
    pd.DataFrame({"c": np.asarray(names)[db["contig"]], "s": db["start"], "k": letters, "g": db["group"]}).to_csv(
        locp, sep="\t", header=False, index=False)
    fais = []
    for hap in range(2):
        fp = os.path.join(workdir, f"hap{hap + 1}.fai")
        open(fp, "w").write("".join(f"{n}\t{len(sq)}\t0\t60\t61\n" for n, sq in haps[hap]))
        fais.append(fp)
    n50, sigma = 100000.0, 0.8
    mu = math.log(n50) - sigma * sigma
    per_hap_procs = max(1, cores // 2)
    want = int(per_proc_mbp * 1e6)
    jobs, rlen, sample_bases, sample_reads = [], {}, 0, 0

    def make_chunk(hc):
        hap, c = hc
        r = np.random.default_rng(7000 + 100 * hap + c)
        lens, tot = [], 0
        while tot < want:
            ln = int(min(max(r.lognormal(mu, sigma), 1000), 1000000))  # (clipped to its contig by the simulator)
            lens.append(ln)
            tot += ln
        reads = S.simulate(haps[hap], lens, 9000 + 100 * hap + c, f"h{hap + 1}c{c}r")
        fp = os.path.join(workdir, f"hap{hap + 1}_{c}.fa")
        with open(fp, "wb") as f:
            for n, sq in reads:
                f.write(b">" + n.encode() + b"\n" + sq + b"\n")
        return dict(workdir=workdir, tag=f"hap{hap + 1}_{c}", reads=fp, db=dbp, loc=locp, fai=fais[hap]), {n: len(sq) for n, sq in reads}
    with ThreadPoolExecutor(max_workers=cores) as ex:
        for job, rl in ex.map(make_chunk, [(h, c) for h in range(2) for c in range(per_hap_procs)]):
            jobs.append(job)
            rlen.update(rl)
            sample_bases += sum(rl.values())
            sample_reads += len(rl)
    note = (f"inputs made without libgavisunk_b200.so: numpy generator of the workload's recipe on a {asm_mbp:.0f} Mbp x2 diploid sample "
            f"assembly ({len(kms)} SUNKs; jellyfish.db / kmer.loc from the oracle's restatement of defineSUNKs.smk), ")
    return dict(workdir=workdir, jobs=jobs, dbp=dbp, locp=locp, rlen=rlen, sample_note=note, sample_bases=sample_bases,
                sample_reads=sample_reads, hap_contigs=[{n for n, _ in haps[0]}, {n for n, _ in haps[1]}],
                fai=[[(n, len(sq)) for n, sq in haps[h]] for h in range(2)])


def _port_contig(task):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gavisunk_oracle as O
    rr, rlen, bad, ctg = task
    inter, bed = O.process_by_contig(rr, rlen, bad, ctg)
    return ctg, bed


def run_reference_pipeline(prep, cores):
    """one timed pass of the reference pipeline over a prepared sample: kmerpos_annot3 -> diag_filter_v3 ->
    diag_filter_step2 (the reference's ELFs), one process chain per chunk file with all cores busy (snakemake --cores
    N), then the CPU port of badsunks_AR.py / process-by-contig_lowmem_AR.py / get_gaps.py on ALL chunks."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_runner as RR
    import gavisunk_oracle as O
    from gavisunk_b200 import io as gio
    workdir, jobs, dbp, locp, rlen = (prep[k2] for k2 in ("workdir", "jobs", "dbp", "locp", "rlen"))
    for fn in os.listdir(workdir):  # outputs of an earlier step
        if fn.endswith(".sunkpos"):
            os.remove(os.path.join(workdir, fn))
    t_load = RR.table_load_seconds(workdir, dbp, locp)
    res, wall_elf = RR.run_chunks_parallel(jobs, cores)
    t0 = time.perf_counter()
    rows_h = [[], []]
    for j, r in zip(jobs, res):
        rows_h[0 if j["tag"].startswith("hap1") else 1] += gio.read_sunkpos(r["diag2"])
    hapc = prep["hap_contigs"]
    bad = O.bad_sunks(rows_h[0], hapc[0], rows_h[1], hapc[1])
    beds, n_iv = {}, 0
    tasks = []
    for hap in range(2):
        byc = {}
        for row in rows_h[hap]:
            byc.setdefault(row[2], []).append(row)
        for ctg, rr in byc.items():
            names_c = {r[0] for r in rr}
            tasks.append((rr, {n: rlen[n] for n in names_c if n in rlen}, bad, ctg))
    # one process_by_contig job per contig, `cores` at once, as snakemake runs the rule (tagONT.smk:170-191)
    import multiprocessing as mp
    with mp.get_context("fork").Pool(min(cores, max(1, len(tasks)))) as pool:
        for ctg, bed in pool.map(_port_contig, tasks):
            if bed is not None:
                beds[ctg] = [(s, e) for _, s, e in bed]
                n_iv += len(bed)
    for hap in range(2):
        O.get_gaps(prep["fai"][hap], beds)
    t_py = time.perf_counter() - t0
    wall = wall_elf + t_py
    sample_bases = prep["sample_bases"]
    # every reference process first parses jellyfish.db + kmer.loc from text (kmerpos_annot3.nim:20-69); for a bounded sample that
    # load would dominate (at the reference's real chunk size of ~9 Gbp it is < 30 %), so `value` leaves it out and it is
    # reported beside it
    wall_noload = max(wall - t_load, 1e-9)
    return dict(value=sample_bases / wall_noload / 1e9, unit=UNIT, cores=cores, kind="reference",
                sample=(prep["sample_note"] + f"{prep['sample_reads']} reads / {sample_bases / 1e6:.0f} Mbp of the same workload in {len(jobs)} "
                        f"chunk files; reference ELFs kmerpos_annot3+diag_filter_v3+diag_filter_step2 one process per chunk, {cores} at "
                        f"once (wall {wall_elf:.1f} s, of which {t_load:.1f} s is every process loading the SUNK table from text: left out of "
                        f"`value`, see value_incl_table_load), then the CPU port of badsunks / process-by-contig (one process per contig, {cores} at once) / get_gaps on "
                        f"all chunks ({t_py:.1f} s; the reference's Python needs graph_tool/pyranges)"),
                wall_s=wall, elf_wall_s=wall_elf, table_load_s=t_load, python_port_s=t_py,
                value_incl_table_load=sample_bases / wall / 1e9,
                scan_only_value=sample_bases / max(wall_elf - t_load, 1e-9) / 1e9, sample_intervals=n_iv)


def cpu_reference_sample(args, wl, eng, per_proc_mbp=12.0):
    """cpu_baseline leg of the b200 arm (rank 0, N = 1): the reference pipeline on a sample cut from THIS run's workload
    (database exported from the engine, reads from the same generator).  The sample's input files are written once and
    reused by later calls; only the pipeline itself is timed."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_runner as RR
    cores = os.cpu_count() or 1
    if not RR.available():
        return dict(error="oracle/_ref executables missing", cores=cores)
    key = (id(wl), float(per_proc_mbp))
    if key not in _SAMPLE_CACHE:
        import atexit
        if not _SAMPLE_CACHE:
            atexit.register(_cleanup_samples)
        prep = _prepare_reference_sample(args, wl, eng, per_proc_mbp, cores)
        swl = prep["wl"]
        nc = len(swl.contig_names) // 2
        prep["hap_contigs"] = [set(swl.contig_names[:nc]), set(swl.contig_names[nc:])]
        prep["fai"] = [[(swl.contig_names[c], int(swl.contig_len[c])) for c in range(h * nc, (h + 1) * nc)] for h in range(2)]
        _SAMPLE_CACHE[key] = prep
    return run_reference_pipeline(_SAMPLE_CACHE[key], cores)


def main_reference(args):
    """--impl reference: only rank 0 works, on the host cores; no GPU and no libgavisunk_b200.so is involved: the
    sample's inputs come from numpy + the oracle (_prepare_numpy_sample, untimed set-up), every timed step runs
    the reference executables + the CPU port of its Python stages."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_runner as RR
    cores = os.cpu_count() or 1
    if not RR.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref executables missing"}))
        return
    import atexit
    atexit.register(_cleanup_samples)
    t_setup = time.perf_counter()
    prep = _prepare_numpy_sample(args, args.cpu_sample_mbp or 24.0, cores, asm_mbp=args.ref_asm_mbp)
    _SAMPLE_CACHE["ref"] = prep
    t_setup = time.perf_counter() - t_setup
    vals, last = [], None
    for i in range(min(args.warmup, 1) + args.steps):
        last = run_reference_pipeline(prep, cores)
        if i >= min(args.warmup, 1):
            vals.append(last["value"])
    steps = len(vals)
    v = float(np.mean(vals))
    spec = WORKLOADS[args.workload]
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": steps,
           "warmup": min(args.warmup, 1), "ms_per_step": (last["wall_s"] - last["table_load_s"]) * 1e3, "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": None, "dtype": "u64", "data": "synthetic",
           "config": {"workload": spec["desc"], "k": args.k, "asm_haploid_mbp": spec["mbp"], "setup_s": round(t_setup, 1),
                      "native_so_loaded": "gavisunk_b200" in sys.modules and getattr(sys.modules.get("gavisunk_b200._lib"), "_lib", None) is not None},
           "cpu_baseline": dict(last, value=v),
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    a = parse_args()
    # stdout carries exactly ONE line, the JSON: libraries that write to fd 1 on their own (NCCL prints its
    # version banner there at the first communicator) are pointed at stderr, the JSON goes to the real stdout
    sys.stdout.flush()
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _json_out
    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)

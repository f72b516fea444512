"""Device time of the distance discordance (GVS_ST_DISCORDANCE: Engine.spans = gvs_spans, then Engine.discordance =
gvs_discordance), on bench.py's default workload (h3100: 3.1 Gbp x2 synthetic diploid assembly, 8 batches of 3.75x
ONT-like reads, k = 20, one GPU) after run_batches.

  python profiles/discordance_stage.py [--reps 30]

Both calls are repeated --reps times after the run (stage timer of each).  The workload's reads are drawn from the
assembly itself, so every call in the bed file is a false positive.  Prints one JSON line with the card's name and power
limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception as ex:  # noqa: BLE001
        out = f"nvidia-smi unavailable: {ex}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    from gavisunk_b200 import cli, io as gio, workload as W
    from gavisunk_b200.engine import Engine
    if not torch.cuda.is_available():
        raise SystemExit("discordance_stage.py measures on a GPU; none found")
    eng = Engine(20)
    contigs = W.human_contigs(3100.0)
    wl = W.make_assembly(eng, contigs, snp_rate=1e-3, dup_frac=0.01, seed=1001, name="h3100")
    W.build_db(eng, wl)
    batch_args = dict(coverage=3.75, n50=100000.0, sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    batches = [W.new_batch(eng, wl, seed=2001 + 16 * b, **batch_args) for b in range(8)]
    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in batches]
    eng.set_profiling(True)
    eng.run_batches(binds, wl.contig_hap, min_read_len=10000)
    validate_ms = eng.stage_ms("validate")
    spans_ms, runs_ms = [], []
    for i in range(a.warmup + a.reps):
        rec = eng.spans()
        t_spans = eng.stage_ms("discordance")
        runs = eng.discordance(wl.contig_len)
        if i >= a.warmup:
            spans_ms.append(t_spans)
            runs_ms.append(eng.stage_ms("discordance"))
    spans_ms, runs_ms = np.array(spans_ms), np.array(runs_ms)
    lens = np.concatenate([np.diff(b.read_off.cpu().numpy()) for b in batches]).astype(np.uint32)
    n_reads = eng.n_reads
    rtab = gio.NameTable([f"read{i}" for i in range(n_reads)])
    calls = []
    for hap in range(2):
        _, _, bed = cli.discordance_texts(np.flatnonzero(wl.contig_hap == hap).tolist(), wl.contig_names, rec, runs, rtab, lens,
                                          np.arange(n_reads, dtype=np.int64))
        calls += [l.split(b"\t") for l in bed.splitlines()]
    print(json.dumps(dict(
        metric="discordance_stage_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
        gpu=gpu_info(), reps=a.reps, kept_rows=int(eng.n_kept), reads=int(n_reads), validated_pairs=int(eng.n_pairs),
        validate_ms=float(validate_ms), spans_ms_median=float(np.median(spans_ms)), spans_ms_min=float(spans_ms.min()),
        spans_ms_max=float(spans_ms.max()), runs_ms_median=float(np.median(runs_ms)), runs_ms_min=float(runs_ms.min()),
        runs_ms_max=float(runs_ms.max()), records=int(len(rec["read"])), spans_total=int(runs["spans"].astype(np.int64).sum()),
        runs=int(len(runs["contig"])), calls=len(calls), calls_collapse=sum(1 for c in calls if c[3] == b"collapse"),
        calls_expansion=sum(1 for c in calls if c[3] == b"expansion"))))
    eng.close()


if __name__ == "__main__":
    main()

"""Device time of the support-track stage (GVS_ST_SUPPORT: Engine.placements + Engine.support) and the host egress of
the three track files, on bench.py's default workload (h3100: 3.1 Gbp x2 synthetic diploid assembly, 8 batches of
3.75x ONT-like reads, k = 20, one GPU).

  python profiles/support_stage.py [--reps 30] [--out DIR]

Runs the whole path once (as bench.py does), then times the stage over --reps repetitions with CUDA events (the stage
timer of the library) and the formatting + writing of the three files per haplotype into a temporary directory.
Prints one JSON line with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

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
        raise SystemExit("support_stage.py measures on a GPU; none found")
    eng = Engine(20)
    contigs = W.human_contigs(3100.0)
    wl = W.make_assembly(eng, contigs, snp_rate=1e-3, dup_frac=0.01, seed=1001, name="h3100")
    W.build_db(eng, wl)
    batch_args = dict(coverage=3.75, n50=100000.0, sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    batches = [W.new_batch(eng, wl, seed=2001 + 16 * b, **batch_args) for b in range(8)]
    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in batches]
    eng.set_profiling(True)
    iv, _ = eng.run_batches(binds, wl.contig_hap, min_read_len=10000)
    clen = wl.contig_len.astype(np.uint32)
    ms = []
    for i in range(a.warmup + a.reps):
        pl = eng.placements()
        t_pl = eng.stage_ms("support")
        runs = eng.support(clen)
        t_sup = eng.stage_ms("support")
        if i >= a.warmup:
            ms.append((t_pl, t_sup, t_pl + t_sup))
    tot = np.array([m[2] for m in ms])
    # host egress: names / lengths of every read as the fused rule holds them, then the three files per haplotype
    n_reads = eng.n_reads
    rnames = [f"read{i}" for i in range(n_reads)]
    rtab = gio.NameTable(rnames)
    lens = np.concatenate([np.diff(b.read_off.cpu().numpy()) for b in batches]).astype(np.uint32)
    name_rank = cli.bytewise_rank(rtab)
    egress = []
    with tempfile.TemporaryDirectory() as td:
        for _ in range(3):
            t0 = time.perf_counter()
            for hap in range(2):
                texts = cli.support_texts(np.flatnonzero(wl.contig_hap == hap).tolist(), clen, wl.contig_names, pl, runs, iv, rtab,
                                          lens, name_rank)
                cli._write_all([os.path.join(td, f"hap{hap + 1}.{ext}") for ext in cli.EVIDENCE_PRODUCTS["support_tracks"].suffixes],
                               texts)
            egress.append((time.perf_counter() - t0) * 1e3)
    print(json.dumps(dict(
        metric="support_stage_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
        gpu=gpu_info(), reps=a.reps, placements=int(len(pl["read"])), validated_pairs=int(eng.n_pairs), groups=int(eng.db_groups()),
        runs=int(len(runs["contig"])), reads=int(n_reads),
        stage_ms_median=float(np.median(tot)), stage_ms_min=float(tot.min()), stage_ms_max=float(tot.max()),
        placements_ms_median=float(np.median([m[0] for m in ms])), support_ms_median=float(np.median([m[1] for m in ms])),
        egress_ms=[round(x, 1) for x in egress])))
    eng.close()


if __name__ == "__main__":
    main()

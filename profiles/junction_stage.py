"""Device time of the junction screen (GVS_ST_SCREEN: Engine.junction_screen, once per batch) and of the resolve
(GVS_ST_JUNCTIONS: Engine.junctions), on bench.py's default workload (h3100: 3.1 Gbp x2 synthetic diploid assembly,
8 batches of 3.75x ONT-like reads, k = 20, one GPU) run with run_batches(junctions=True).

  python profiles/junction_stage.py [--reps 30]

The screen time of every batch is the stage timer read in on_batch; the resolve is repeated --reps times after the run.
The workload's reads are drawn from the assembly itself, so every record is a false positive: the record count should be
near zero.  Prints one JSON line with the card's name and power limit."""
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
        raise SystemExit("junction_stage.py measures on a GPU; none found")
    eng = Engine(20)
    contigs = W.human_contigs(3100.0)
    wl = W.make_assembly(eng, contigs, snp_rate=1e-3, dup_frac=0.01, seed=1001, name="h3100")
    W.build_db(eng, wl)
    batch_args = dict(coverage=3.75, n50=100000.0, sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    batches = [W.new_batch(eng, wl, seed=2001 + 16 * b, **batch_args) for b in range(8)]
    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in batches]
    eng.set_profiling(True)
    screen_ms, stash = [], []
    real = eng.junction_screen

    def screen(min_read_len):  # run_batches' call, keeping the stash size it returns
        stash.append(real(min_read_len))
        return stash[-1]
    eng.junction_screen = screen
    eng.run_batches(binds, wl.contig_hap, min_read_len=10000, on_batch=lambda e, b, base: screen_ms.append(e.stage_ms("screen")),
                    junctions=True)
    del eng.junction_screen
    ms = []
    for i in range(a.warmup + a.reps):
        jn = eng.junctions()
        if i >= a.warmup:
            ms.append(eng.stage_ms("junctions"))
    screen_ms, ms = np.array(screen_ms), np.array(ms)
    lens = np.concatenate([np.diff(b.read_off.cpu().numpy()) for b in batches]).astype(np.uint32)
    n_reads = eng.n_reads
    rtab = gio.NameTable([f"read{i}" for i in range(n_reads)])
    name_rank = np.arange(n_reads, dtype=np.int64)
    _, clusters = cli.junction_texts(jn, np.arange(len(jn["read"])), wl.contig_names, wl.contig_len, wl.contig_hap, rtab, lens, name_rank)
    cl = clusters.splitlines()
    print(json.dumps(dict(
        metric="junction_stage_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
        gpu=gpu_info(), reps=a.reps, match_rows=int(eng.n_rows), reads=int(n_reads),
        screen_ms_per_batch=[round(float(x), 4) for x in screen_ms], screen_ms_median=float(np.median(screen_ms)),
        screen_ms_max=float(screen_ms.max()), resolve_ms_median=float(np.median(ms)), resolve_ms_min=float(ms.min()),
        resolve_ms_max=float(ms.max()), stash_rows=int(stash[-1][0]), stash_reads=int(stash[-1][1]), records=int(len(jn["read"])),
        records_cross_hap=int((wl.contig_hap[jn["contig1"]] != wl.contig_hap[jn["contig2"]]).sum()),
        records_link=int((cli.junction_columns(jn, wl.contig_len)[4] == 0).sum()),
        clusters=len(cl) - 1, clusters_3plus=sum(1 for l in cl[1:] if int(l.split(b"\t")[8]) >= 3))))
    eng.close()


if __name__ == "__main__":
    main()

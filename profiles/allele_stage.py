"""Device time of the allele support (GVS_ST_ALLELES: Engine.allele_support = gvs_allele_support per batch,
Engine.allele_runs = gvs_allele_runs once per run) on bench.py's default workload (h3100: 3.1 Gbp x2 synthetic diploid
assembly, 8 batches of 3.75x ONT-like reads, k = 20, one GPU), in run_batches(allele_support=True).

  python profiles/allele_stage.py [--reps 30]

The per-batch stage time is read after every batch (its stage timer); the runs are repeated --reps times after the run.
How many read segments of the match rows take the non-monotone path of k_al_count is counted on the host from each
batch's match rows (the kernel does not report it).  The workload's reads are drawn from the assembly itself, so every
call is a false positive; the calls per kind, error_eligible and the baselines of own are reported.  Prints one JSON line
with the card's name and power limit."""
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


def paths(read, key):
    """(segments, non-monotone segments, their rows, largest) of one batch's match rows: read indices and the key
    k_al_count tests (the group index)"""
    read, key = read.astype(np.int64), key.astype(np.int64)
    n = len(read)
    if n == 0:
        return 0, 0, 0, 0
    head = np.ones(n, bool)
    head[1:] = read[1:] != read[:-1]
    seg = np.cumsum(head) - 1
    n_seg = int(seg[-1]) + 1
    same = ~head[1:]
    d = np.diff(key)[same]
    s = seg[1:][same]
    up = np.bincount(s[d < 0], minlength=n_seg) == 0
    down = np.bincount(s[d > 0], minlength=n_seg) == 0
    rest = ~(up | down)
    size = np.bincount(seg, minlength=n_seg)
    return n_seg, int(rest.sum()), int(size[rest].sum()), int(size[rest].max()) if rest.any() else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    from gavisunk_b200 import cli, workload as W
    from gavisunk_b200.engine import Engine
    if not torch.cuda.is_available():
        raise SystemExit("allele_stage.py measures on a GPU; none found")
    eng = Engine(20)
    contigs = W.human_contigs(3100.0)
    wl = W.make_assembly(eng, contigs, snp_rate=1e-3, dup_frac=0.01, seed=1001, name="h3100")
    W.build_db(eng, wl)
    batch_args = dict(coverage=3.75, n50=100000.0, sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    batches = [W.new_batch(eng, wl, seed=2001 + 16 * b, **batch_args) for b in range(8)]
    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in batches]
    eng.set_profiling(True)
    per_batch, stats = [], []
    gt = eng.groups()
    gkey = (gt["contig"].astype(np.int64) << 32) | gt["group"].astype(np.int64)
    gorder = np.argsort(gkey)

    def on_batch(e, b, base):
        per_batch.append(e.stage_ms("alleles"))
        r0 = e.rows(0)
        k = (r0["contig"].astype(np.int64) << 32) | r0["group"].astype(np.int64)
        stats.append(paths(r0["read"], gorder[np.searchsorted(gkey[gorder], k)]))  # the group index of every row
    eng.run_batches(binds, wl.contig_hap, min_read_len=10000, on_batch=on_batch, allele_support=True)
    al = eng.alleles()
    ms = []
    for i in range(a.warmup + a.reps):
        rn = eng.allele_runs(wl.contig_len)
        if i >= a.warmup:
            ms.append(eng.stage_ms("alleles"))
    ms = np.array(ms)
    calls, summary = [], []
    for hap in range(2):
        hc = np.flatnonzero(wl.contig_hap == hap).tolist()
        cl, per, base = cli.allele_calls(gt["contig"], gt["group"], al["end"], al["own"], al["other"], al["sunks"], hc)
        calls += [(hap + 1, wl.contig_names[c], s, e, kind, ng, nm, o, t) for c, s, e, kind, ng, nm, o, t in cl]
        tot = [int(sum(v[i] for v in per)) for i in range(8)]
        summary.append(dict(zip(("groups", "assessed", "flipped", "flips", "switches", "errors", "error_eligible", "shared"), tot),
                            baselines=[b[2] for b in base]))
    seg, rest, rest_rows, rest_max = (int(sum(s[i] for s in stats)) if i < 3 else int(max(s[i] for s in stats)) for i in range(4))
    print(json.dumps(dict(
        metric="allele_stage_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
        gpu=gpu_info(), reps=a.reps, groups=int(len(gt["contig"])), distinct_read_groups=int(al["own"].sum() + al["other"].sum()),
        per_batch_ms=[round(float(x), 4) for x in per_batch], per_batch_ms_median=float(np.median(per_batch)),
        per_batch_ms_min=float(min(per_batch[1:] or per_batch)), per_batch_ms_max=float(max(per_batch[1:] or per_batch)),
        runs_ms_median=float(np.median(ms)), runs_ms_min=float(ms.min()), runs_ms_max=float(ms.max()), runs=int(len(rn["contig"])),
        segments=seg, non_monotone_segments=rest, non_monotone_share=float(rest / max(1, seg)), non_monotone_rows=rest_rows,
        non_monotone_rows_max=rest_max, calls=len(calls), calls_flip=sum(1 for c in calls if c[4] == "flip"),
        calls_switch=sum(1 for c in calls if c[4] == "switch"), calls_error=sum(1 for c in calls if c[4] == "error"),
        summary=summary, first_calls=[list(map(str, c)) for c in calls[:20]])))
    eng.close()


if __name__ == "__main__":
    main()

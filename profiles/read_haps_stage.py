"""Device time of the diag filter (GVS_ST_DIAG: gvs_diag_filter / gvs_diag_filter_haps, once per batch) in three modes, on
bench.py's default workload (h3100: 3.1 Gbp x2 synthetic diploid assembly, 8 batches of 3.75x ONT-like reads, k = 20,
one GPU) run with run_batches:

  off        read_haps=False, chunks binned by the haplotype the reads were drawn from (today's filter)
  binned     read_haps=True on the same chunks (both votes, the records; rows as with the flag off)
  unbinned   every chunk rebound as GVS_HAP_ANY (rows kept on the assigned haplotype)

  python profiles/read_haps_stage.py [--out FILE]

Per batch the stage timers are read in on_batch (GVS_ST_READHAPS: the haplotype-mode part of the filter).  The
assignments of the unbinned run are counted against the true haplotype of every read (the workload draws a batch's
first half of reads from hap 1's contigs and the second half from hap 2's).  Prints one JSON line with the card's name
and power limit."""
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
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    from gavisunk_b200 import workload as W
    from gavisunk_b200.engine import GVS_HAP_ANY, Engine
    if not torch.cuda.is_available():
        raise SystemExit("read_haps_stage.py measures on a GPU; none found")
    eng = Engine(20)
    wl = W.make_assembly(eng, W.human_contigs(3100.0), snp_rate=1e-3, dup_frac=0.01, seed=1001, name="h3100")
    W.build_db(eng, wl)
    batch_args = dict(coverage=3.75, n50=100000.0, sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    batches = [W.new_batch(eng, wl, seed=2001 + 16 * b, **batch_args) for b in range(8)]
    truth = np.concatenate([np.repeat(b.chunk_hap, np.diff(b.chunk_first.astype(np.int64))) for b in batches])
    eng.set_profiling(True)
    res = {}
    for mode in ("off", "binned", "unbinned", "off"):  # "off" again last: its spread against the first
        hap = (lambda b: np.full(len(b.chunk_hap), GVS_HAP_ANY, np.uint8)) if mode == "unbinned" else (lambda b: b.chunk_hap)
        binds = [(lambda e, b=b: e.set_reads_device(W._dev_ptr(b.reads), W._dev_ptr(b.read_off), b.n_reads, b.chunk_first, hap(b)))
                 for b in batches]
        diag, rh_ms = [], []

        def on_batch(e, b, base):
            diag.append(e.stage_ms("diag"))
            if mode != "off":
                rh_ms.append(e.stage_ms("readhaps"))
        eng.run_batches(binds, wl.contig_hap, min_read_len=10000, on_batch=on_batch, read_haps=mode != "off")
        r = dict(diag_ms_per_batch=[round(float(x), 4) for x in diag], diag_ms_median=float(np.median(diag)), kept_rows=int(eng.n_kept))
        if mode != "off":
            rec = eng.read_haps()
            hp = rec["hap"]
            tr = truth[rec["read"]]
            r.update(readhaps_ms_median=float(np.median(rh_ms)), records=int(len(hp)), reads=int(eng.n_reads),
                     assigned_right=int(((hp <= 1) & (hp == tr)).sum()), assigned_wrong=int(((hp <= 1) & (hp != tr)).sum()),
                     ties=int((hp == 2).sum()), no_vote=int(eng.n_reads - len(hp)),
                     other_hap_votes=int(np.where(tr == 0, rec["n2"] > 0, rec["n1"] > 0).sum()))
        res[mode if mode not in res else mode + "_again"] = r
    line = json.dumps(dict(metric="read_haps_diag_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
                           gpu=gpu_info(), **res))
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()

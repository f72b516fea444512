"""Device time of the gap-evidence stage (GVS_ST_EVIDENCE: Engine.gap_evidence) and the host egress of its four files,
on bench.py's default workload (h3100: 3.1 Gbp x2 synthetic diploid assembly, 8 batches of 3.75x ONT-like reads,
k = 20, one GPU).

  python profiles/gap_evidence_stage.py [--reps 30]

Runs the whole path once (as bench.py does) and the gaps, then times the stage over --reps repetitions with CUDA events
(the stage timer of the library) and the formatting + writing of the two files per haplotype into a temporary
directory.  The candidate count (read segments x gaps they could bridge, what the second kernel resolves) is recounted
on the host from the kept rows with the first kernel's rule.  Prints one JSON line with the card's name and power
limit."""
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


def count_candidates(eng, read_len, gaps, min_read_len):
    """(segment, gap) pairs with min ID <= gs and max ID > ge over the non-bad kept rows of reads >= min_read_len"""
    kept = eng.rows(1)
    gt = eng.groups()
    bad = eng.bad_list()
    bad_key = np.sort((gt["contig"][bad].astype(np.int64) << 32) | gt["group"][bad].astype(np.int64))
    key = (kept["contig"].astype(np.int64) << 32) | kept["group"].astype(np.int64)
    ok = ~np.isin(key, bad_key, assume_unique=False) & (read_len[kept["read"]] >= min_read_len)
    rd, key = kept["read"][ok], key[ok]
    if len(rd) == 0:
        return 0
    first = np.flatnonzero(np.concatenate([[True], rd[1:] != rd[:-1]]))
    mn, mx = np.minimum.reduceat(key, first), np.maximum.reduceat(key, first)
    gc = gaps["contig"].astype(np.int64) << 32
    i0 = np.searchsorted(gc | gaps["start"].astype(np.int64), mn, side="left")
    i1 = np.searchsorted(gc | gaps["end"].astype(np.int64), mx, side="left")
    return int(np.maximum(i1 - i0, 0).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    from gavisunk_b200 import cli, io as gio, workload as W
    from gavisunk_b200.engine import Engine
    if not torch.cuda.is_available():
        raise SystemExit("gap_evidence_stage.py measures on a GPU; none found")
    eng = Engine(20)
    contigs = W.human_contigs(3100.0)
    wl = W.make_assembly(eng, contigs, snp_rate=1e-3, dup_frac=0.01, seed=1001, name="h3100")
    W.build_db(eng, wl)
    batch_args = dict(coverage=3.75, n50=100000.0, sigma=0.8, len_min=1000, len_max=1000000, nchunks=10)
    batches = [W.new_batch(eng, wl, seed=2001 + 16 * b, **batch_args) for b in range(8)]
    binds = [(lambda e, b=b: W.bind_batch(e, b)) for b in batches]
    eng.set_profiling(True)
    eng.run_batches(binds, wl.contig_hap, min_read_len=10000)
    clen = wl.contig_len.astype(np.uint32)
    gaps, _ = eng.gaps(clen)
    ms = []
    for i in range(a.warmup + a.reps):
        ev = eng.gap_evidence(10000)
        if i >= a.warmup:
            ms.append(eng.stage_ms("evidence"))
    ms = np.array(ms)
    lens = np.concatenate([np.diff(b.read_off.cpu().numpy()) for b in batches]).astype(np.uint32)
    n_cand = count_candidates(eng, lens, gaps, 10000)
    # host egress: names of every read as the fused rule holds them, then the two files per haplotype
    n_reads = eng.n_reads
    rtab = gio.NameTable([f"read{i}" for i in range(n_reads)])
    name_rank = cli.bytewise_rank(rtab)
    chap = wl.contig_hap
    egress = []
    with tempfile.TemporaryDirectory() as td:
        for _ in range(3):
            t0 = time.perf_counter()
            for hap in range(2):
                gsel = np.flatnonzero(chap[gaps["contig"]] == hap)
                texts = cli.gap_evidence_texts(gsel, gaps, wl.contig_names, ev, rtab, lens, name_rank)
                cli._write_all([os.path.join(td, f"hap{hap + 1}.{ext}") for ext in cli.EVIDENCE_PRODUCTS["gap_evidence"].suffixes],
                               texts)
            egress.append((time.perf_counter() - t0) * 1e3)
    print(json.dumps(dict(
        metric="gap_evidence_stage_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
        gpu=gpu_info(), reps=a.reps, gaps=int(len(gaps["contig"])), kept_rows=int(eng.n_kept), reads=int(n_reads),
        candidates=n_cand, records=int(len(ev["read"])),
        stage_ms_median=float(np.median(ms)), stage_ms_min=float(ms.min()), stage_ms_max=float(ms.max()),
        egress_ms=[round(x, 1) for x in egress])))
    eng.close()


if __name__ == "__main__":
    main()

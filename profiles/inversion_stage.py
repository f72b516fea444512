"""Device time of the strand switches (GVS_ST_SWITCHES: Engine.strand_switches = gvs_strand_switches) on bench.py's default
workload (h3100: 3.1 Gbp x2 synthetic diploid assembly, 8 batches of 3.75x ONT-like reads, k = 20, one GPU) after
run_batches.

  python profiles/inversion_stage.py [--reps 30]

The stage is repeated --reps times after the run (its stage timer).  How many read segments leave at each exit of
k_sw_resolve is counted on the host from the kept rows, bad groups and read lengths (the kernel does not report it):
too short, fewer than 6 usable rows, monotone (pos non-decreasing in row order and starts monotone along it), and the
rest, which take the O(m^2) path.  The workload's reads are drawn from the assembly itself, so every call in the bed file
is a false positive; the first calls are listed.  Prints one JSON line with the card's name and power limit."""
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


def exits(kept, bad_keys, lens, min_len=10000):
    """per exit of k_sw_resolve, the number of read segments that take it"""
    read = kept["read"].astype(np.int64)
    n = len(read)
    if n == 0:
        return dict(segments=0)
    head = np.ones(n, bool)
    head[1:] = read[1:] != read[:-1]
    seg = np.cumsum(head) - 1
    first = np.flatnonzero(head)
    c0 = kept["contig"][first][seg]
    key = (kept["contig"].astype(np.int64) << 32) | kept["group"].astype(np.int64)
    use = (kept["contig"] == c0) & ~np.isin(key, bad_keys)
    n_seg = len(first)
    nu = np.bincount(seg[use], minlength=n_seg)
    u = np.flatnonzero(use)
    su = seg[u]
    same = su[1:] == su[:-1]
    p, s = kept["pos"][u].astype(np.int64), kept["start"][u].astype(np.int64)
    dp, ds = np.diff(p)[same], np.diff(s)[same]
    sg = su[1:][same]
    viol = lambda m: np.bincount(sg[m], minlength=n_seg) > 0
    unsorted, not_up, not_down = viol(dp < 0), viol(ds < 0), viol(ds > 0)
    short = lens[read[first]] < min_len
    few = ~short & (nu < 6)
    mono = ~short & ~few & ~unsorted & (~not_up | ~not_down)
    rest = ~short & ~few & ~mono
    return dict(segments=int(n_seg), exit_short=int(short.sum()), exit_few_rows=int(few.sum()), exit_monotone=int(mono.sum()),
                resolved=int(rest.sum()), resolved_unsorted=int((rest & unsorted).sum()),
                resolved_rows=int(nu[rest].sum()), resolved_rows_max=int(nu[rest].max()) if rest.any() else 0,
                monotone_share_of_long_reads=float(mono.sum() / max(1, (~short).sum())))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    from gavisunk_b200 import cli, io as gio, workload as W
    from gavisunk_b200.engine import Engine
    if not torch.cuda.is_available():
        raise SystemExit("inversion_stage.py measures on a GPU; none found")
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
    ms = []
    for i in range(a.warmup + a.reps):
        rec = eng.strand_switches(10000)
        if i >= a.warmup:
            ms.append(eng.stage_ms("switches"))
    ms = np.array(ms)
    lens = np.concatenate([np.diff(b.read_off.cpu().numpy()) for b in batches]).astype(np.uint32)
    n_reads = eng.n_reads
    gt = eng.groups()
    bad = eng.bad_list()
    bad_keys = np.sort((gt["contig"][bad].astype(np.int64) << 32) | gt["group"][bad].astype(np.int64))
    ex = exits(eng.rows(1), bad_keys, lens)
    rtab = gio.NameTable([f"read{i}" for i in range(n_reads)])
    calls = []
    kinds = cli.switch_kinds(rec)
    for hap in range(2):
        _, bed = cli.inversion_texts(np.flatnonzero(wl.contig_hap == hap).tolist(), wl.contig_names, rec, rtab, lens,
                                     np.arange(n_reads, dtype=np.int64))
        calls += [l.decode() for l in bed.splitlines()]
    print(json.dumps(dict(
        metric="inversion_stage_ms", workload="h3100 (bench.py default: 3.1 Gbp x2, 8 batches of 3.75x, k 20), 1 GPU",
        gpu=gpu_info(), reps=a.reps, kept_rows=int(eng.n_kept), reads=int(n_reads), validate_ms=float(validate_ms),
        switches_ms_median=float(np.median(ms)), switches_ms_min=float(ms.min()), switches_ms_max=float(ms.max()), **ex,
        records=int(len(rec["read"])), records_foldback=int(kinds.sum()), records_inversion=int(len(kinds) - kinds.sum()),
        reads_with_records=int(len(np.unique(rec["read"]))), calls=len(calls), first_calls=calls[:20])))
    eng.close()


if __name__ == "__main__":
    main()

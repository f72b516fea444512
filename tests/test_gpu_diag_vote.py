"""GPU parity of the diag filter's vote (csrc/diag.cu) with the oracle (diag_filter_v3 + diag_filter_step2) at every
size tier of the vote and on adversarial diagonals.

A (read, contig) candidate is voted on by one of three code paths, chosen by its row count: 2-48 rows rank all pairs
in k_cand_vote_warp, 49-256 rows bisect on the value in the same kernel (select2), and larger candidates go to
k_cand_vote<1024>, one block per candidate over a grid-stride loop.  The golden cases of test_gpu_diag.py never exceed
23 rows per candidate, so this file builds rows from the generator of test_oracle_diag_big.py (which pins the oracle
itself at these sizes) and compares best() and rows(1) byte for byte with the oracle, chunk by chunk.
"""
import random

import numpy as np
import pytest

import gavisunk_oracle as O
from conftest import format_rows
from test_oracle_diag_big import (RANK_MAX, WARP_MAX, ZOO, candidate_zoo, chimera, designed, diag, is_sorted, one_strand,
                                  set_groups, strand_flip, tie_both)

pytestmark = pytest.mark.gpu


# ---- running both sides -------------------------------------------------------------------------
# A case is a list of reads (name, [(contig, pos, start, group), ...]), the first read index of every chunk, every
# chunk's haplotype (0 / 1) and the haplotype of every contig (contigs missing from it are in neither .fai).
def _fmt_best(best, read_names, contig_names, lo, hi):
    return "".join(f"{read_names[r]}\t{contig_names[c]}\t{g}\t{'+' if d else '-'}\t{g}\n"
                   for r, c, g, d in zip(best["read"], best["contig"], best["ngood"], best["dir"]) if lo <= r < hi)


def run_gpu(reads, chunk_first, chunk_hap, contig_hap):
    from gavisunk_b200.engine import Engine
    cnames, cidx = [], {}
    cols = ([], [], [], [], [])
    for i, (_, rows) in enumerate(reads):
        for c, p, s, g in rows:
            if c not in cidx:
                cidx[c] = len(cnames)
                cnames.append(c)
            for col, v in zip(cols, (i, p, cidx[c], s, g)):
                col.append(v)
    eng = Engine(20)
    try:
        eng.contig_names = cnames
        eng.set_reads_meta(np.full(len(reads), 20000, np.uint32), chunk_first, chunk_hap)
        eng.set_rows(0, *cols)
        eng.diag_filter([contig_hap.get(c, 255) for c in cnames])
        best, kept = eng.best(), eng.rows(1)
    finally:
        eng.close()
    rnames = [n for n, _ in reads]
    return [(_fmt_best(best, rnames, cnames, chunk_first[i], chunk_first[i + 1]),
             format_rows(kept, rnames, cnames, chunk_first[i], chunk_first[i + 1])) for i in range(len(chunk_hap))]


def oracle_rows(reads, lo, hi):
    return [(n, p, c, s, g) for n, rows in reads[lo:hi] for c, p, s, g in rows]


def run_oracle(reads, chunk_first, chunk_hap, contig_hap):
    """the reference chain, once per chunk with that chunk's haplotype contigs"""
    out = []
    for i, h in enumerate(chunk_hap):
        rows = oracle_rows(reads, chunk_first[i], chunk_first[i + 1])
        best = O.diag_filter_v3(rows, {c for c, hh in contig_hap.items() if hh == h})
        kept = O.diag_filter_step2(rows, best)
        out.append(("".join(f"{r}\t{c}\t{n}\t{d}\t{n2}\n" for r, c, n, d, n2 in best),
                    "".join(f"{r}\t{p}\t{c}\t{s}\t{g}\n" for r, p, c, s, g in kept)))
    return out


def check(reads, chunk_first, chunk_hap, contig_hap):
    got = run_gpu(reads, chunk_first, chunk_hap, contig_hap)
    want = run_oracle(reads, chunk_first, chunk_hap, contig_hap)
    for i, ((gb, gk), (wb, wk)) in enumerate(zip(got, want)):
        for what, g, w in (("best", gb, wb), ("kept rows", gk, wk)):
            if g != w:
                gl, wl = g.splitlines(), w.splitlines()
                j = next((j for j, (a, b) in enumerate(zip(gl, wl)) if a != b), min(len(gl), len(wl)))
                pytest.fail(f"chunk {i} {what}: {len(gl)} lines, oracle {len(wl)}; first difference at line {j}: "
                            f"gpu {gl[j] if j < len(gl) else None!r}, oracle {wl[j] if j < len(wl) else None!r}")
    return want


def candidates(reads, chunk_first, chunk_hap, contig_hap):
    """rows of every voting candidate: contig in the chunk's haplotype, at least 2 rows in the read"""
    out = []
    for i, h in enumerate(chunk_hap):
        for _, rows in reads[chunk_first[i]:chunk_first[i + 1]]:
            by = {}
            for c, p, s, g in rows:
                by.setdefault(c, []).append((p, s, g))
            out += [r for c, r in by.items() if len(r) >= 2 and contig_hap.get(c) == h]
    return out


def read_of(name, contig, cand):
    return (name, [(contig, p, s, g) for p, s, g in cand])


def n_blocks_big():
    """blocks of k_cand_vote<1024>: 2 per SM"""
    import torch
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count


def tie_names(prefix, cap_lo, cap_hi=None):
    """two contig names (first, second); inserted in that order into an empty Table of cap_lo slots, the second
    takes the earlier slot, and with cap_hi slots (if given) the later one"""
    names = [f"{prefix}{i}" for i in range(400)]
    h = [O.nim_hash(n) for n in names]
    for i in range(len(names)):
        for j in range(len(names)):
            if (h[i] & (cap_lo - 1)) <= (h[j] & (cap_lo - 1)):
                continue
            if cap_hi is None or (h[i] & (cap_hi - 1)) < (h[j] & (cap_hi - 1)):
                return names[i], names[j]
    raise AssertionError("no such pair")


# ---- cases --------------------------------------------------------------------------------------
def test_zoo_every_tier():
    """every shape of the generator at sizes 2 ... 5000, one read per candidate"""
    reads = [read_of(label, f"h1#c{i % 7}", rows) for i, (label, rows) in enumerate(ZOO)]
    cf, ch, hap = [0, len(reads)], [0], {f"h1#c{i}": 0 for i in range(7)}
    cands = candidates(reads, cf, ch, hap)
    assert any(len(r) > RANK_MAX and not is_sorted(diag(r, 0)) and not is_sorted(diag(r, 1)) for r in cands)
    assert any(RANK_MAX < len(r) <= WARP_MAX and is_sorted(diag(r, 0)) != is_sorted(diag(r, 1)) for r in cands)
    assert any(RANK_MAX < len(r) <= WARP_MAX and not is_sorted(diag(r, 0)) and not is_sorted(diag(r, 1)) for r in cands)
    assert any(len(r) > WARP_MAX and not is_sorted(diag(r, 0)) and not is_sorted(diag(r, 1)) for r in cands)
    assert sum(len(r) > WARP_MAX for r in cands) > 100
    want = check(reads, cf, ch, hap)
    assert sum(1 for l in want[0][0].splitlines() if l.startswith("tie_both_")) == sum(1 for l, _ in ZOO if l.startswith("tie_both_"))
    assert all(l.split("\t")[3] == "-" for l in want[0][0].splitlines() if l.startswith("tie_both_"))


def test_grid_stride():
    """more candidates of more than 256 rows than k_cand_vote<1024> has blocks"""
    nb = n_blocks_big()
    rng = random.Random(11)
    shapes = [lambda n: one_strand(rng, n, True), lambda n: one_strand(rng, n, False), lambda n: strand_flip(rng, n),
              lambda n: chimera(rng, n), lambda n: designed(rng, n, 1, -40_001, 2001, 3),
              lambda n: designed(rng, n, 0, 9_000_001, 1001, (n - 1) // 2)]
    reads = [read_of(f"g{i}", f"h1#g{i % 5}", shapes[i % len(shapes)](WARP_MAX + 1 + i % 40)) for i in range(nb + 37)]
    cf, ch, hap = [0, len(reads)], [0], {f"h1#g{i}": 0 for i in range(5)}
    assert sum(len(r) > WARP_MAX for r in candidates(reads, cf, ch, hap)) > nb
    want = check(reads, cf, ch, hap)
    assert len(want[0][0].splitlines()) == len(reads)


def test_decisions():
    rng = random.Random(5)
    reads, hap = [], {}
    winner = {}
    for n in (60, 257, 1025):
        # cross-contig tie on (good, hitlen): the Table's slot order decides, against and along insertion order
        for flip in (True, False):
            a, b = tie_names(f"h1#t{n}{'f' if flip else 'k'}_", 64)
            winner[f"tie_{n}_{flip}"] = b
            if not flip:
                a, b = b, a
            cand = designed(rng, n, 1, 3_000_001, 1999, 2)
            reads.append((f"tie_{n}_{flip}", [(a, p, s, g) for p, s, g in cand] + [(b, p, s, g) for p, s, g in cand]))
            hap[a] = hap[b] = 0
        # equal good, different hitlen: the contig with fewer rows wins though it comes second
        cand = one_strand(rng, n, False)
        # two rows below and two above every other row on both diagonals: same medians, same good, 4 more rows
        far = [(10, 10, 1), (20, 5, 2), (10, (1 << 32) - 10, 3), (30, (1 << 32) - 40, 4)]
        reads.append((f"hitlen_{n}", [("h1#long", p, s, g) for p, s, g in cand + far] + [("h1#short", p, s, g) for p, s, g in cand]))
        # maxgood <= 1: one group only, or rows far apart in both orientations
        one = [(p, s, 77) for p, s, _ in one_strand(rng, n, True)]
        reads.append((f"onegroup_{n}", [("h1#short", p, s, g) for p, s, g in one]))
        apart = [(i * 50_000, 3_000_000_000 - i * 120_000 + (i % 2) * 9_000_000, i) for i in range(n)]
        reads.append((f"apart_{n}", [("h1#long", p, s, g) for p, s, g in apart]))
    hap["h1#long"] = hap["h1#short"] = 0
    cf, ch = [0, len(reads)], [0]
    want = check(reads, cf, ch, hap)
    best = {l.split("\t")[0]: l.split("\t") for l in want[0][0].splitlines()}
    for n in (60, 257, 1025):
        assert best[f"hitlen_{n}"][1] == "h1#short"
        assert f"onegroup_{n}" not in best and f"apart_{n}" not in best
    assert all(best[r][1] == c for r, c in winner.items())


def test_read_shapes():
    rng = random.Random(9)
    reads = []
    # contigs interleaved A, B, A, B, ...: k_row_first scans back, k_cand_gather collects rows that are apart
    for n in (50, 300, 1100):
        a, b = one_strand(rng, n, True), strand_flip(rng, n - 7)
        rows = []
        for i in range(n):
            rows.append(("h1#A", *a[i]))
            if i < len(b):
                rows.append(("h1#B", *b[i]))
            if i % 97 == 0:
                rows.append(("h1#C", *a[i]))
        reads.append((f"interleaved_{n}", rows))
    # contigs outside the read's haplotype with many rows enter the Table but do not vote
    for n in (40, 400):
        strong = one_strand(rng, 2000, False)
        weak = set_groups(designed(rng, n, 0, 5_000_001, 3, 1), "dup", rng)
        reads.append((f"offhap_{n}", [("h2#X", p, s, g) for p, s, g in strong[:1000]] + [("h1#A", p, s, g) for p, s, g in weak]
                      + [("nofai#Y", p, s, g) for p, s, g in strong[1000:]]))
    # single-row contigs: 70 of them grow the Table to 128 slots, around a tie that the slot order decides
    a, b = tie_names("h1#one_", 128)
    cand = one_strand(rng, 300, True)
    rows = [(f"h1#s{i}", 100 * i, 5000 + 100 * i, i) for i in range(35)]
    rows += [(a, p, s, g) for p, s, g in cand] + [(f"h1#s{i}", 100 * i, 5000 + 100 * i, i) for i in range(35, 70)]
    rows += [(b, p, s, g) for p, s, g in cand]
    reads.append(("singles", rows))
    hap = {c: 0 for _, rr in reads for c, *_ in rr if c.startswith("h1#")}
    hap["h2#X"] = 1
    check(reads, [0, len(reads)], [0], hap)


def _chunk_reads(rng):
    """reads of both haplotypes, alternating, whose ties are decided by a Table that an earlier read of the chunk grew
    to 128 slots"""
    per_hap, hap = [], {}
    for h in (0, 1):
        a, b = tie_names(f"h{h + 1}#cap_", 64, 128)
        reads = [(f"grow{h}", [(f"h{h + 1}#m{i}", 1000 * i, 7000 + 1000 * i + (i % 3) * 5, i) for i in range(80)])]
        for n in (2, 49, 257, 1025):
            cand = tie_both(rng, n) if n < 49 else one_strand(rng, n, n % 2 == 1)
            reads.append((f"tie{h}_{n}", [(a, p, s, g) for p, s, g in cand] + [(b, p, s, g) for p, s, g in cand]))
            reads.append((f"vote{h}_{n}", [(f"h{h + 1}#m{n % 80}", p, s, g) for p, s, g in designed(rng, max(n, 8), h, 6_000_001, 2001, 1)]))
        hap.update({c: h for _, rr in reads for c, *_ in rr})
        per_hap.append(reads)
    return [r for pair in zip(*per_hap) for r in pair], hap


@pytest.mark.parametrize("n_chunks", [1, 2, 5])
@pytest.mark.parametrize("first_hap", [0, 1])
def test_chunk_splits(n_chunks, first_hap):
    """the same rows in 1, 2 and 5 chunks of alternating haplotype: Table capacity is sticky within a chunk only"""
    reads, hap = _chunk_reads(random.Random(3))
    cf = [len(reads) * i // n_chunks for i in range(n_chunks + 1)]
    ch = [(first_hap + i) % 2 for i in range(n_chunks)]
    want = check(reads, cf, ch, hap)
    assert sum(len(b.splitlines()) for b, _ in want) > 4


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_fuzz(seed):
    rng = random.Random(seed)
    zoo = candidate_zoo(100 + seed)
    contigs = [f"h1#f{i}" for i in range(6)] + [f"h2#f{i}" for i in range(5)] + ["other#0"]
    hap = {c: 0 if c.startswith("h1") else 1 for c in contigs if not c.startswith("other")}
    reads = []
    for r in range(60):
        rows = []
        for c in rng.sample(contigs, rng.randrange(1, 5)):
            label, cand = zoo[rng.randrange(len(zoo))]
            rows.append([(c, p, s, g) for p, s, g in cand])
        if rng.random() < 0.3 and len(rows) > 1:  # a tie: the same candidate on a second contig
            c2 = rows[1][0][0]
            rows[1] = [(c2, p, s, g) for _, p, s, g in rows[0]]
        if rng.random() < 0.5:  # interleave the contigs' rows
            flat = [x for i in range(max(map(len, rows))) for rr in rows if i < len(rr) for x in [rr[i]]]
        else:
            flat = [x for rr in rows for x in rr]
        reads.append((f"fz{seed}_{r}", flat))
    cf, ch = [0, 20, 45, 60], [0, 1, 0]
    assert any(len(c) > WARP_MAX for c in candidates(reads, cf, ch, hap))
    check(reads, cf, ch, hap)


def _adversarial_reads():
    rng = random.Random(4)
    reads = [read_of(label, f"h1#c{i % 3}", rows) for i, (label, rows) in enumerate(ZOO)
             if label.startswith(("odd_gap", "min_at_lo", "ties_below", "spread", "flip")) and len(rows) > RANK_MAX]
    a, b = tie_names("h1#shim_", 64)
    cand = one_strand(rng, 300, False)
    reads.append(("shimtie", [(a, p, s, g) for p, s, g in cand] + [(b, p, s, g) for p, s, g in cand]))
    return reads + _dup_name_reads()[0]  # the shims group and key reads by name, as the reference does


def test_shims(tmp_path, capsys):
    """`cli diag_filter_v3` and `cli diag_filter_step2` on an adversarial set, with reads that share a name, write
    the oracle's text"""
    from gavisunk_b200 import cli
    reads = _adversarial_reads()
    rows = oracle_rows(reads, 0, len(reads))
    contigs = sorted({r[2] for r in rows})
    sp, fai, dg = tmp_path / "a.sunkpos", tmp_path / "asm.fai", tmp_path / "a_diag.sunkpos"
    sp.write_text("".join(f"{r}\t{p}\t{c}\t{s}\t{g}\n" for r, p, c, s, g in rows))
    fai.write_text("".join(f"{c}\t1000000\t0\t60\t61\n" for c in contigs))
    best = O.diag_filter_v3(rows, set(contigs))
    want_best = "".join(f"{r}\t{c}\t{n}\t{d}\t{n2}\n" for r, c, n, d, n2 in best)
    want_kept = "".join(f"{r}\t{p}\t{c}\t{s}\t{g}\n" for r, p, c, s, g in O.diag_filter_step2(rows, best))
    capsys.readouterr()
    assert cli.main(["diag_filter_v3", str(sp), str(fai)]) == 0
    got_best = capsys.readouterr().out
    assert got_best == want_best
    dg.write_text(got_best)
    assert cli.main(["diag_filter_step2", str(sp), str(dg)]) == 0
    assert capsys.readouterr().out == want_kept


def _dup_name_reads():
    """records sharing a name: 'a' twice in a row, 'b' twice with another read between; every record has its own
    best contig"""
    rng = random.Random(8)
    c1 = [("h1#d1", p, s, g) for p, s, g in one_strand(rng, 300, True)]
    c2 = [("h1#d2", p, s, g) for p, s, g in one_strand(rng, 60, False)]
    c3 = [("h1#d1", p, s, g) for p, s, g in one_strand(rng, 40, False)]
    c4 = [("h1#d2", p, s, g) for p, s, g in one_strand(rng, 270, True)]
    return [("a", c1), ("a", c2), ("b", c3), ("x", c1), ("b", c4)], {"h1#d1": 0, "h1#d2": 0}


def test_duplicate_read_names():
    """The fused filter takes every record as its own read; the reference chain takes consecutive equal names as one
    read and keys the best contig by name (DESIGN.md §9).  The fused result is the oracle's on names made unique per
    record, and it differs from the reference chain's on this input."""
    reads, hap = _dup_name_reads()
    cf, ch = [0, len(reads)], [0]
    got = run_gpu(reads, cf, ch, hap)
    uniq = [(f"{n}@{i}", rows) for i, (n, rows) in enumerate(reads)]
    per_record = [tuple("".join(l.split("@")[0] + l[l.index("\t"):] + "\n" for l in t.splitlines()) for t in chunk)
                  for chunk in run_oracle(uniq, cf, ch, hap)]
    assert got == per_record
    reference = run_oracle(reads, cf, ch, hap)
    assert got[0][0] != reference[0][0] and got[0][1] != reference[0][1]

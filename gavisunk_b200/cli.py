"""Command-line shims with the reference's argv (SURVEY.md 8b) on top of the GPU engine.

  python -m gavisunk_b200.cli kmerpos_annot3 <reads.fa|fq[.gz]> <db.txt> <kmer.loc> <out.sunkpos>
  python -m gavisunk_b200.cli rlen <reads> <out.rlen>
  python -m gavisunk_b200.cli diag_filter_v3 <sunkpos> <asm.fai>            (stdout)
  python -m gavisunk_b200.cli diag_filter_step2 <sunkpos[.gz]> <diag[.gz]>  (stdout)
  python -m gavisunk_b200.cli badsunks_AR <fai1> <fai2> <sunkpos1> <sunkpos2> <out>
  python -m gavisunk_b200.cli process_by_contig <locs> <sunkpos> <rlen> <badsunks> <out.tsv> <out.bed> [--minlen N] [--opt_filt]
  python -m gavisunk_b200.cli get_gaps <fai1> <fai2> <sample> <indir/> <outdir/>
  python -m gavisunk_b200.cli slop_gaps <gaps.bed> <asm.fai> <out.bed>
  python -m gavisunk_b200.cli covprob --bed B --locs L --rlen R --fai F --sunk-len K --tsv OUT
  python -m gavisunk_b200.cli split_locs --ont-pos P --kmer-loc L --flag results/S/breaks/hapN_splits_pos.done --hap hapN
  python -m gavisunk_b200.cli split_ont --reads R.. --out temp/S/reads/hapN_1-of-10.fq.gz ..   (seqtk seq -F '#' | rustybam fastq-split)
  python -m gavisunk_b200.cli combine_ont_nofilt <chunk.sunkpos>.. <hapN_detailed.sunkpos>
  python -m gavisunk_b200.cli fused --sample S --k K --hap1-asm .. --hap2-asm .. (--hap1-reads f.. --hap2-reads f.. | --reads f..)
                                    --outdir D [--devices 0,1,..] [--batch-files N] [--detailed] [--support-tracks]
                                    [--gap-evidence] [--junctions] [--discordance] [--read-haplotypes]
  python -m gavisunk_b200.cli support_tracks <sunkpos> <rlen> <bad_sunks.txt> <fai> <valid.bed> <out.reads.bed> <out.bedgraph> <out.tsv>
  python -m gavisunk_b200.cli gap_evidence <sunkpos> <rlen> <bad_sunks.txt> <fai> <valid.bed> <out.gaps.reads.tsv> <out.gaps.evidence.tsv>
  python -m gavisunk_b200.cli junctions <hapN_detailed.sunkpos> <hapN.rlen> <bad_sunks.txt> <fai1> <fai2> <out.junctions.reads.tsv> <out.junctions.tsv>
  python -m gavisunk_b200.cli discordance <sunkpos> <rlen> <bad_sunks.txt> <fai> <out.discordance.reads.tsv> <out.discordance.tsv> <out.discordance.bed>

The first four replace workflow/scripts/{kmerpos_annot3,rlen,diag_filter_v3,diag_filter_step2}
(workflow/rules/tagONT.smk:36,73,92,110) one to one; the next six replace badsunks_AR.py,
process-by-contig_lowmem_AR.py, get_gaps.py, `bedtools slop`, covprob.py and split_locs.py with the
argv of their rules (tagONT.smk:150,189,230,249; the two `script:` rules take their snakemake.input /
.output / .config values as options, and `covprob_script(snakemake)` / `split_locs_script(snakemake)`
accept the snakemake object itself); `fused` replaces the rules from jellyfish_count
to get_gaps and writes the same files under results/{sample}/.  `fused --support-tracks` and `support_tracks`
add per-read placements, support depth and a per-contig summary of the validated reads (no reference
counterpart: the reference only plots them, viz.py).  `fused --gap-evidence` and `gap_evidence` report, per gap, the
reads that reach both of its sides and the size change their SUNK distances imply (no reference counterpart either).
`fused --junctions` and `junctions` report the reads whose SUNKs jump from one contig to another, and cluster them into
contig links and breakpoints (no reference counterpart: the diag filter keeps one contig per read).
`fused --discordance` and `discordance` report collapses and expansions inside validated intervals, from the SUNK spacing
of the validated reads across them (no reference counterpart).
`fused --read-haplotypes` reports each read's SUNK vote on both haplotypes and the haplotype it assigns; `fused --reads`
takes unbinned chunk files and keeps each read's rows on the haplotype its votes assign (no reference counterpart: the
reference needs the reads binned by haplotype).
Text parsing / formatting is host
plumbing; all per-base and per-row work runs in libgavisunk_b200.so.  Errors exit non-zero with a
message on stderr and never leave a partial output file behind.
"""
from __future__ import annotations

import argparse
import os
import sys
from collections import defaultdict
from typing import Dict, List, NamedTuple, Sequence, Tuple

import numpy as np

from . import io as gio
from .engine import GVS_HAP_ANY, Engine, encode_kmers
from .parallel import ThreadExchange, shard_chunks


def _atomic_write(path: str, text: str):
    tmp = path + ".tmp%d" % os.getpid()
    with open(tmp, "w") as f:
        f.write(text)
    os.replace(tmp, path)


def _fmt_rows(rows, read_names, contig_names) -> str:
    out = []
    for r, p, c, s, g in zip(rows["read"].tolist(), rows["pos"].tolist(), rows["contig"].tolist(), rows["start"].tolist(),
                             rows["group"].tolist()):
        out.append(f"{read_names[r]}\t{p}\t{contig_names[c]}\t{s}\t{g}\n")
    return "".join(out)


def _k_from_db(db_lines: Sequence[bytes]) -> int:
    return len(db_lines[0]) if db_lines else 0  # kmerpos_annot3.nim:28-38: k = length of the first db line


def cmd_kmerpos_annot3(argv):
    reads_p, db_p, loc_p, out_p = argv
    db_lines = [l.encode() for l in gio.read_db(db_p)]
    sys.stderr.write("FINISHED READING KMERS\n")
    contig, start, kmer, group = gio.read_loc(loc_p)
    sys.stderr.write("FINISHED READING LOCS\n")
    k = _k_from_db(db_lines)
    eng = Engine(k if 1 <= k <= 32 else 20)
    eng.load_loc_text(db_lines, list(zip(contig, start, [km.encode() for km in kmer], group)))
    reads = gio.NativeReads([reads_p], packed=True)  # parse + 2-bit pack in one pass into page-locked memory (csrc/fastx.cu)
    eng.set_reads_packed(reads.words, reads.read_off)
    eng.match()
    rows = eng.rows(0)
    rtab, ctab = gio.NameTable(blob=reads.name_blob, off=reads.name_off), gio.NameTable(eng.contig_names)
    _write_bytes(out_p, gio.format_rows([("name", rows["read"], rtab), ("u32", rows["pos"]), ("name", rows["contig"], ctab),
                                         ("u32", rows["start"]), ("u32", rows["group"])]))


def cmd_rlen(argv):
    reads_p, out_p = argv
    reads = gio.NativeReads([reads_p], pin=False, packed=True)
    rtab = gio.NameTable(blob=reads.name_blob, off=reads.name_off)
    _write_bytes(out_p, gio.format_rows([("name", np.arange(reads.n_reads, dtype=np.uint32), rtab), ("u64", reads.lengths())]))


def _rows_from_sunkpos(path):
    rows = gio.read_sunkpos(path)
    cnames, cidx, rnames, ridx, prev = [], {}, [], [], None
    for r in rows:
        if r[2] not in cidx:
            cidx[r[2]] = len(cnames)
            cnames.append(r[2])
        if r[0] != prev:  # consecutive rows with equal names form a read (diag_filter_v3.nim:64)
            rnames.append(r[0])
            prev = r[0]
        ridx.append(len(rnames) - 1)
    cols = (np.asarray(ridx, np.uint32), np.asarray([r[1] for r in rows], np.uint32),
            np.asarray([cidx[r[2]] for r in rows], np.uint32), np.asarray([r[3] for r in rows], np.uint32),
            np.asarray([r[4] for r in rows], np.uint32))
    return rows, cnames, rnames, cols


def cmd_diag_filter_v3(argv):
    sunkpos_p, fai_p = argv
    rows, cnames, rnames, cols = _rows_from_sunkpos(sunkpos_p)
    fai = {n for n, _ in gio.read_fai(fai_p)}
    eng = Engine(20)
    eng.contig_names = cnames
    eng.set_reads_meta(np.zeros(len(rnames), np.uint32))
    eng.set_rows(0, *cols)
    eng.diag_filter([0 if n in fai else 255 for n in cnames])
    b = eng.best()
    out = sys.stdout
    for r, c, g, d in zip(b["read"].tolist(), b["contig"].tolist(), b["ngood"].tolist(), b["dir"].tolist()):
        out.write(f"{rnames[r]}\t{cnames[c]}\t{g}\t{'+' if d else '-'}\t{g}\n")


def cmd_diag_filter_step2(argv):
    sunkpos_p, diag_p = argv
    rows, cnames, rnames, cols = _rows_from_sunkpos(sunkpos_p)
    best: Dict[str, str] = {}
    with gio.open_maybe_gz(diag_p) as f:
        for l in f.read().decode().splitlines():
            p = l.split("\t")
            if len(p) >= 2:
                best[p[0]] = p[1]  # later rows of a read name overwrite earlier ones (nim:17-22)
    cidx = {n: i for i, n in enumerate(cnames)}
    table = np.array([cidx.get(best.get(n, ""), 0xFFFFFFFF) for n in rnames], dtype=np.uint32)
    eng = Engine(20)
    eng.contig_names = cnames
    eng.set_reads_meta(np.zeros(len(rnames), np.uint32))
    eng.set_rows(0, *cols)
    eng.filter_best(table)
    sys.stdout.write(_fmt_rows(eng.rows(1), rnames, cnames))



# ------------------------------------------------------------------------------------------------
# per-rule shims of the Python stages (SURVEY.md 8b)
# ------------------------------------------------------------------------------------------------
def _index_names(names: Sequence[str], known: Dict[str, int] = None):
    idx = dict(known or {})
    out = np.zeros(len(names), np.uint32)
    for i, n in enumerate(names):
        j = idx.get(n)
        if j is None:
            j = idx[n] = len(idx)
        out[i] = j
    return out, idx


def _engine_with_rows(rows, contig_order: Sequence[str] = ()):
    """kept-row engine from parsed sunkpos rows: reads = distinct names in sorted order (pandas groupby
    order), each read's rows contiguous in file order."""
    rnames = sorted({r[0] for r in rows})
    ridx = {n: i for i, n in enumerate(rnames)}
    rows = sorted(rows, key=lambda r: ridx[r[0]])  # stable: file order inside a read
    cidx = {n: i for i, n in enumerate(contig_order)}
    ccol, cidx = _index_names([r[2] for r in rows], cidx)
    cnames = [None] * len(cidx)
    for n, i in cidx.items():
        cnames[i] = n
    eng = Engine(20)
    eng.contig_names = cnames
    cols = (np.asarray([ridx[r[0]] for r in rows], np.uint32), np.asarray([r[1] for r in rows], np.uint32), ccol,
            np.asarray([r[3] for r in rows], np.uint32), np.asarray([r[4] for r in rows], np.uint32))
    return eng, rows, rnames, cnames, cols


def bad_sunks_of_hap(sunkpos_p: str, fai_p: str, hap: int):
    """badsunks_AR.py:20-52 (hap1) / :56-93 (hap2) -> set of 'contig:ID'"""
    rows = gio.read_sunkpos(sunkpos_p)
    fai = {n for n, _ in gio.read_fai(fai_p)}
    eng, rows, rnames, cnames, cols = _engine_with_rows(rows)
    if not any(c in fai for c in cnames):
        raise IndexError("index 0 is out of bounds for axis 0 with size 0 (mode of no correct-haplotype counts, badsunks_AR.py:43)")
    eng.set_reads_meta(np.zeros(len(rnames), np.uint32), [0, len(rnames)], [hap])
    eng.set_rows(1, *cols)
    # contigs of this haplotype's .fai are "correct"; the others only get the upper limit (:48-51)
    eng.set_contigs([hap if c in fai else 2 + hap for c in cnames])
    eng.group_hist()
    eng.bad_groups()
    sys.stdout.write(f"mean coverage {eng.modes[hap]}\n")
    g = eng.groups()
    return {f"{cnames[g['contig'][i]]}:{g['group'][i]}" for i in eng.bad_list().tolist()}


def cmd_badsunks(argv):
    fai1, fai2, sp1, sp2, out_p = argv
    bad = bad_sunks_of_hap(sp1, fai1, 0) | bad_sunks_of_hap(sp2, fai2, 1)
    sys.stdout.write(f"{len(bad)}\n")
    _atomic_write(out_p, "".join(b + "\n" for b in sorted(bad)))  # the reference writes set order (SURVEY Q18)


def _read_rlen(path) -> Dict[str, int]:
    """{hap}.rlen: read name -> length (the first row of a name wins)"""
    rlen = {}
    with gio.open_maybe_gz(path) as f:
        for l in f.read().decode().splitlines():
            p = l.split("\t")
            if len(p) >= 2:
                rlen.setdefault(p[0], int(p[1]))
    return rlen


def _read_badsunks(path) -> set:
    with open(path) as f:
        return set(f.read().splitlines())


def _read_lens(rlen: Dict[str, int], rnames) -> np.ndarray:
    """u32 length of every read name ({hap}.rlen; 0 when missing, clipped to u32)"""
    return np.asarray([min(rlen.get(n, 0), 0xFFFFFFFF) for n in rnames], np.uint32)


def bytewise_rank(rtab) -> np.ndarray:
    """Rank of every name of a NameTable in bytewise order, equal names in table order: the order in which
    `for rname, g in grouped` visits reads (groupby sorts the names, process-by-contig_lowmem_AR.py:135-136) and in which
    every per-read file lists them"""
    rank = np.empty(len(rtab), np.int64)
    rank[np.argsort(rtab.as_bytes_array(), kind="stable")] = np.arange(len(rtab))
    return rank


def _set_bad(eng, badset, cnames):
    """bad groups of a bad_sunks.txt ('contig:ID' lines) on the engine's contigs"""
    bc, bg = [], []
    cidx = {n: i for i, n in enumerate(cnames)}
    for b in badset:
        c, _, g = b.partition(":")  # ID2 = chrom + ":" + ID (process-by-contig_lowmem_AR.py:68)
        if c in cidx and g.isdigit() and int(g) <= 0xFFFFFFFF:
            bc.append(cidx[c])
            bg.append(int(g))
    eng.bad_set(bc, bg)


def _keyed_hap(sunkpos_p, rlen_p, badsunks_p, fai_p, valid_p=None):
    """One haplotype of the per-rule path ({hap}.sunkpos, {hap}.rlen, bad_sunks.txt, the .fai[, {hap}.valid.bed]) on a
    kept-row engine with one read per (contig, read name), as process_by_contig groups the reads per contig, and the
    read lengths and bad groups set.  -> (engine, contig names, contig lengths, validated intervals (None without
    valid_p), (name table, lengths, bytewise name rank) of the reads)"""
    fai = gio.read_fai(fai_p)
    names = [n for n, _ in fai]
    rlen = _read_rlen(rlen_p)
    badset = _read_badsunks(badsunks_p)
    valid = _read_bed3(valid_p) if valid_p is not None else []
    rows = list(dict.fromkeys(gio.read_sunkpos(sunkpos_p)))  # drop_duplicates (process-by-contig_lowmem_AR.py:104)
    cidx = {n: i for i, n in enumerate(names)}
    for r in rows:
        if r[2] not in cidx:
            raise KeyError(f"contig {r[2]} of {sunkpos_p} is not in {fai_p}")
    for c, _, _ in valid:
        if c not in cidx:
            raise KeyError(f"contig {c} of {valid_p} is not in {fai_p}")
    # one engine read per (contig, read name): key the rows by both, the name stays the read's; every contig is in the
    # .fai, so the engine's contigs are its contigs in its order
    keyed = [(f"{r[2]}\t{r[0]}",) + tuple(r[1:]) for r in rows]
    eng, keyed, keys, _, cols = _engine_with_rows(keyed, names)
    rnames = [k.split("\t", 1)[1] for k in keys]
    lens = _read_lens(rlen, rnames)
    eng.set_reads_meta(lens)
    eng.set_rows(1, *cols)
    _set_bad(eng, badset, names)
    iv = None if valid_p is None else dict(contig=np.asarray([cidx[c] for c, _, _ in valid], np.uint32),
                                           start=np.asarray([s for _, s, _ in valid], np.uint32),
                                           end=np.asarray([e for _, _, e in valid], np.uint32))
    rtab = gio.NameTable(rnames)
    return eng, names, [l for _, l in fai], iv, (rtab, lens, bytewise_rank(rtab))


def process_by_contig(locs_p, sunkpos_p, rlen_p, badsunks_p, out_tsv, out_bed):
    """process-by-contig_lowmem_AR.py:30-260 for one breaks/{contig}_{hap}.sunkpos"""
    rlen = _read_rlen(rlen_p)
    open(locs_p).close()  # the reference reads it (:54-57) but none of its outputs depend on it
    rows = gio.read_sunkpos(sunkpos_p)
    if not rows:
        raise ValueError("No columns to parse from file (empty sunkpos, process-by-contig_lowmem_AR.py:60)")
    contig = rows[0][2]  # sunkposcat['chrom'].unique()[0] (:62)
    badset = _read_badsunks(badsunks_p)
    rows = list(dict.fromkeys(rows))  # drop_duplicates (:104) keeps the first of identical rows
    eng, rows, rnames, cnames, cols = _engine_with_rows(rows)
    eng.set_reads_meta(_read_lens(rlen, rnames))
    eng.set_rows(1, *cols)
    eng.set_contigs([0] * len(cnames))
    _set_bad(eng, badset, cnames)
    eng.validate(10000)  # the reference overwrites --minlen with 10000 (:106, SURVEY Q13)
    if eng.n_pairs == 0:  # :92-94, :202-204: contig name only, no bed (the rule touches it)
        _atomic_write(out_tsv, contig + "\n")
        return None
    pairs = eng.pairs()
    _atomic_write(out_tsv, "".join(f"{g}\t{rnames[r]}\n" for g, r in zip(pairs["group"].tolist(), pairs["read"].tolist())))
    eng.components_local()
    iv = eng.intervals()
    _atomic_write(out_bed, "".join(f"{contig}\t{s}\t{e}\n" for s, e in sorted(zip(iv["start"].tolist(), iv["end"].tolist()))))
    return iv


def cmd_process_by_contig(argv):
    ap = argparse.ArgumentParser(prog="gavisunk_b200.cli process_by_contig")
    for a in ("SUNKs", "sunkpos", "rlen", "badsunks", "outputfile", "outputbed"):
        ap.add_argument(a)
    ap.add_argument("--minlen", default=10000, type=int)
    ap.add_argument("--opt_filt", action="store_true")
    a = ap.parse_args(argv)
    process_by_contig(a.SUNKs, a.sunkpos, a.rlen, a.badsunks, a.outputfile, a.outputbed)


# ------------------------------------------------------------------------------------------------
# support tracks of the validated reads (no reference counterpart; DESIGN.md section 5)
# ------------------------------------------------------------------------------------------------
SUPPORT_TSV_HEADER = "contig\tlength\treads\tvalidated_bases\tcovered_bases\tdepth_bases\tmax_depth\tmin_valid_depth\n"
_STRAND = gio.NameTable(["+", "-"])


def support_texts(hap_contigs, contig_len, names, pl, runs, iv, rtab, read_len, name_rank):
    """The three support files of one haplotype: hap_contigs = its contig ids in .fai order; pl = Engine.placements()
    with run-wide read indices, runs = Engine.support(), iv = validated intervals (rows of valid.bed); rtab / read_len /
    name_rank = name table, length and bytewise name rank of every run-wide read.  -> (reads.bed, bedGraph, tsv) bytes"""
    ctab = gio.NameTable(names)
    inhap = np.zeros(len(names), bool)
    inhap[np.asarray(hap_contigs, np.int64)] = True
    p = np.flatnonzero(inhap[pl["contig"]])
    p = p[np.lexsort((name_rank[pl["read"][p]], pl["end"][p], pl["start"][p], pl["contig"][p]))]
    reads_bed = gio.format_rows([("name", pl["contig"], ctab), ("u32", pl["start"]), ("u32", pl["end"]), ("name", pl["read"], rtab),
                                 ("u32", pl["n_ids"]), ("name", pl["strand"], _STRAND), ("u32", read_len[pl["read"]])], sel=p)
    r = np.flatnonzero(inhap[runs["contig"]])
    bedgraph = gio.format_rows([("name", runs["contig"], ctab), ("u32", runs["start"]), ("u32", runs["end"]), ("u32", runs["depth"])], sel=r)
    rc = runs["contig"][r].astype(np.int64)
    rs, re_, rd = (runs[c][r].astype(np.int64) for c in ("start", "end", "depth"))
    ln = re_ - rs
    cs, first = np.unique(rc, return_index=True)  # runs come in contig order and tile every contig
    hi = np.append(first[1:], len(rc))
    at = {int(c): i for i, c in enumerate(cs)}
    covered = np.add.reduceat(np.where(rd > 0, ln, 0), first) if len(first) else []
    depth_b = np.add.reduceat(rd * ln, first) if len(first) else []
    max_d = np.maximum.reduceat(rd, first) if len(first) else []
    n_reads = np.bincount(pl["contig"][p], minlength=len(names))
    ivs = defaultdict(list)
    for c, a, b in zip(iv["contig"].tolist(), iv["start"].tolist(), iv["end"].tolist()):
        ivs[c].append((a, b))
    out = [SUPPORT_TSV_HEADER]
    for c in hap_contigs:
        i = at[int(c)]
        lo, up = int(first[i]), int(hi[i])
        valid, mvd, cur_s, cur_e = 0, None, -1, -1
        for a, b in sorted(ivs.get(int(c), [])):
            if a >= b:
                continue
            if a > cur_e:  # union of the intervals: a new block starts
                valid += cur_e - cur_s
                cur_s, cur_e = a, b
            else:
                cur_e = max(cur_e, b)
            j0 = lo + int(np.searchsorted(re_[lo:up], a, side="right"))
            j1 = lo + int(np.searchsorted(rs[lo:up], b, side="left"))
            m = int(rd[j0:j1].min())
            mvd = m if mvd is None else min(mvd, m)
        valid += cur_e - cur_s
        out.append(f"{names[c]}\t{int(contig_len[c])}\t{int(n_reads[c])}\t{valid}\t{int(covered[i])}\t{int(depth_b[i])}\t{int(max_d[i])}\t"
                   f"{'.' if mvd is None else mvd}\n")
    return reads_bed, bedgraph, "".join(out).encode("latin-1")


def support_tracks(sunkpos_p, rlen_p, badsunks_p, fai_p, valid_p, out_reads_bed, out_bedgraph, out_tsv):
    """Support tracks of one haplotype from the files of the per-rule path ({hap}.sunkpos, {hap}.rlen, bad_sunks.txt,
    the .fai, {hap}.valid.bed): the whole haplotype is validated in one pass, reads grouped by (contig, read name) as
    process_by_contig groups them per contig."""
    eng, names, clen, iv, reads = _keyed_hap(sunkpos_p, rlen_p, badsunks_p, fai_p, valid_p)
    eng.validate(10000)  # the reference's fixed minimum read length (process-by-contig_lowmem_AR.py:106, SURVEY Q13)
    texts = support_texts(list(range(len(names))), clen, names, eng.placements(), eng.support(clen), iv, *reads)
    _write_all((out_reads_bed, out_bedgraph, out_tsv), texts)


def cmd_support_tracks(argv):
    support_tracks(*argv)


# ------------------------------------------------------------------------------------------------
# gap evidence: the reads that bridge each gap (no reference counterpart; DESIGN.md section 5.5b)
# ------------------------------------------------------------------------------------------------
GAP_EVIDENCE_HEADER = "contig\tstart\tend\tbridging_reads\tconsistent_reads\tmin_delta\tmedian_delta\tmax_delta\n"
GAP_READS_HEADER = ("contig\tgap_start\tgap_end\tread\tread_len\tleft_id\tleft_start\tleft_pos\tright_id\tright_start\tright_pos\t"
                    "delta\tconsistent\n")
_BIT = gio.NameTable(["0", "1"])


def span_delta(start1, pos1, start2, pos2) -> np.ndarray:
    """Size change a read implies between two SUNKs it carries (gap evidence, discordant spans): |pos2 - pos1| -
    (start2 - start1) in int64, > 0 when the read holds more bases between them than the assembly"""
    return np.abs(pos2.astype(np.int64) - pos1.astype(np.int64)) - (start2.astype(np.int64) - start1.astype(np.int64))


def gap_evidence_texts(gsel, gaps, names, ev, rtab, read_len, name_rank):
    """The two gap-evidence files of one haplotype: gsel = indices into the gap arrays of its rows of hap{N}.gaps.bed, in
    that file's order; ev = Engine.gap_evidence() with run-wide read indices; rtab / read_len / name_rank = name table,
    length and bytewise name rank of every run-wide read.  delta = |right_pos - left_pos| - (right_start - left_start);
    consistent = 9*ds < 10*dp < 11*ds.  -> (gaps.reads.tsv, gaps.evidence.tsv) bytes"""
    ctab = gio.NameTable(names)
    gsel = np.asarray(gsel, np.int64)
    slot_of = np.full(len(gaps["contig"]), -1, np.int64)
    slot_of[gsel] = np.arange(len(gsel))
    slot = slot_of[ev["gap"].astype(np.int64)]
    r = np.flatnonzero(slot >= 0)
    r = r[np.lexsort((name_rank[ev["read"][r]], slot[r]))]
    ds = ev["right_start"].astype(np.int64) - ev["left_start"].astype(np.int64)
    delta = span_delta(ev["left_start"], ev["left_pos"], ev["right_start"], ev["right_pos"])
    dp = delta + ds
    cons = ((9 * ds < 10 * dp) & (10 * dp < 11 * ds)).astype(np.uint32)
    g = ev["gap"]
    reads_tsv = GAP_READS_HEADER.encode() + gio.format_rows(
        [("name", gaps["contig"][g], ctab), ("u32", gaps["start"][g]), ("u32", gaps["end"][g]), ("name", ev["read"], rtab),
         ("u32", read_len[ev["read"]])] + [("u32", ev[c]) for c in ("left_id", "left_start", "left_pos", "right_id", "right_start", "right_pos")]
        + [("i64", delta), ("name", cons, _BIT)], sel=r)
    n = np.bincount(slot[r], minlength=len(gsel))
    n_cons = np.bincount(slot[r], weights=cons[r], minlength=len(gsel)).astype(np.int64)
    lo = np.concatenate([[0], np.cumsum(n)])
    d_r = delta[r]
    out = [GAP_EVIDENCE_HEADER]
    for i, gi in enumerate(gsel.tolist()):
        head = f"{names[gaps['contig'][gi]]}\t{int(gaps['start'][gi])}\t{int(gaps['end'][gi])}\t{int(n[i])}\t{int(n_cons[i])}"
        if n[i] == 0:
            out.append(head + "\t.\t.\t.\n")
            continue
        d = np.sort(d_r[lo[i]:lo[i + 1]])
        out.append(head + f"\t{int(d[0])}\t{int(d[(len(d) - 1) // 2])}\t{int(d[-1])}\n")
    return reads_tsv, "".join(out).encode("latin-1")


def gap_evidence(sunkpos_p, rlen_p, badsunks_p, fai_p, valid_p, out_reads_tsv, out_evidence_tsv):
    """Gap evidence of one haplotype from the files of the per-rule path ({hap}.sunkpos, {hap}.rlen, bad_sunks.txt, the
    .fai, {hap}.valid.bed): gaps from the validated intervals as get_gaps finds them, reads grouped by (contig, read name)
    as process_by_contig groups them per contig, the reference's fixed minimum read length."""
    eng, names, clen, iv, reads = _keyed_hap(sunkpos_p, rlen_p, badsunks_p, fai_p, valid_p)
    eng.set_intervals(iv["contig"], iv["start"], iv["end"], len(names))
    gaps, _ = eng.gaps(clen)
    ev = eng.gap_evidence(10000)  # the reference's fixed minimum read length (process-by-contig_lowmem_AR.py:106, SURVEY Q13)
    texts = gap_evidence_texts(np.arange(len(gaps["contig"])), gaps, names, ev, *reads)
    _write_all((out_reads_tsv, out_evidence_tsv), texts)


def cmd_gap_evidence(argv):
    gap_evidence(*argv)


# ------------------------------------------------------------------------------------------------
# junctions: reads whose SUNKs jump from one contig to another (no reference counterpart; DESIGN.md section 5.5c)
# ------------------------------------------------------------------------------------------------
JUNCTION_READS_HEADER = ("read\tread_len\tcontig1\tstrand1\tids1\tid1\tstart1\tpos1\tcontig2\tstrand2\tids2\tid2\tstart2\tpos2\t"
                         "read_gap\tleave1\tenter2\timplied_gap\tclass\n")
JUNCTION_CLUSTERS_HEADER = ("contig1\tstrand1\thap1\tstart1\tcontig2\tstrand2\thap2\tstart2\trecords\tlinks\tmedian_implied_gap\t"
                            "class\n")
_CLASS = gio.NameTable(["link", "breakpoint"])
JUNCTION_CHAIN = 10000  # start distance that still chains two records into one cluster


def junction_columns(jn, contig_len):
    """Host columns of junction records (Engine.junctions()): read_gap = pos2 - pos1; leave1 = distance from flank 1 to
    the end of contig1 the read leaves through (len1 - start1 on '+', start1 on '-'); enter2 = distance from the end of
    contig2 the read enters through to flank 2 (start2 on '+', len2 - start2 on '-'); implied_gap = read_gap - leave1 -
    enter2; link (class 0) when leave1 + enter2 <= read_gap + read_gap // 10 + 1000, else breakpoint (1).  The class is
    a heuristic: a link is a read that leaves one contig near an end and enters the other near an end, within the
    read gap plus 10 % and 1 kb of slack."""
    clen = np.asarray(contig_len, np.int64)
    s1, s2 = jn["start1"].astype(np.int64), jn["start2"].astype(np.int64)
    read_gap = jn["pos2"].astype(np.int64) - jn["pos1"].astype(np.int64)
    leave1 = np.where(jn["strand1"] == 0, clen[jn["contig1"]] - s1, s1)
    enter2 = np.where(jn["strand2"] == 0, s2, clen[jn["contig2"]] - s2)
    cls = (leave1 + enter2 > read_gap + read_gap // 10 + 1000).astype(np.uint32)
    return read_gap, leave1, enter2, read_gap - leave1 - enter2, cls


def junction_texts(jn, sel, names, contig_len, contig_hap, rtab, read_len, name_rank):
    """The two junction files of one haplotype: jn = Engine.junctions() with run-wide read indices, sel = its records of
    this haplotype's reads; contig_hap[c] = 0 / 1 (hap1 / hap2 .fai), anything else: neither; rtab / read_len /
    name_rank = name table, length and bytewise name rank of every run-wide read.  -> (junctions.reads.tsv,
    junctions.tsv) bytes.  Clusters: each record is canonicalised (sides swapped and both strands flipped when
    (contig2, start2) < (contig1, start1)), keyed by (contig1, strand1, contig2, strand2), chained by start1 and then by
    start2 (consecutive starts at most JUNCTION_CHAIN apart); a cluster reports lower medians and is a link when more
    than half of its records are."""
    ctab = gio.NameTable(names)
    sel = np.asarray(sel, np.int64)
    r = sel[np.lexsort((sel, name_rank[jn["read"][sel]]))]
    read_gap, leave1, enter2, implied, cls = junction_columns(jn, contig_len)
    cols = [("name", jn["read"], rtab), ("u32", read_len[jn["read"]])]
    for side in "12":
        cols += [("name", jn["contig" + side], ctab), ("name", jn["strand" + side], _STRAND)] + [("u32", jn[c + side]) for c in ("ids", "id", "start", "pos")]
    cols += [("i64", read_gap), ("i64", leave1), ("i64", enter2), ("i64", implied), ("name", cls, _CLASS)]
    reads_tsv = JUNCTION_READS_HEADER.encode() + gio.format_rows(cols, sel=r)
    keyed = defaultdict(list)
    for i in sel.tolist():
        a = (int(jn["contig1"][i]), int(jn["strand1"][i]), int(jn["start1"][i]))
        b = (int(jn["contig2"][i]), int(jn["strand2"][i]), int(jn["start2"][i]))
        if (b[0], b[2]) < (a[0], a[2]):
            a, b = (b[0], 1 - b[1], b[2]), (a[0], 1 - a[1], a[2])
        keyed[(a[0], a[1], b[0], b[1])].append((a[2], b[2], int(implied[i]), int(cls[i]) == 0))

    def chains(items, at):
        items = sorted(items, key=lambda t: t[at])
        out = [[items[0]]]
        for t in items[1:]:
            if t[at] - out[-1][-1][at] <= JUNCTION_CHAIN:
                out[-1].append(t)
            else:
                out.append([t])
        return out
    lower_median = lambda v: sorted(v)[(len(v) - 1) // 2]
    clusters = []
    for (c1, d1, c2, d2), items in keyed.items():
        for ch in chains(items, 0):
            for cl in chains(ch, 1):
                links = sum(t[3] for t in cl)
                clusters.append((c1, lower_median([t[0] for t in cl]), c2, lower_median([t[1] for t in cl]), d1, d2, len(cl), links,
                                 lower_median([t[2] for t in cl])))
    clusters.sort()
    hap = lambda c: str(int(contig_hap[c]) + 1) if int(contig_hap[c]) in (0, 1) else "."
    sd = "+-"
    out = [JUNCTION_CLUSTERS_HEADER]
    for c1, s1, c2, s2, d1, d2, n, links, gap in clusters:
        out.append(f"{names[c1]}\t{sd[d1]}\t{hap(c1)}\t{s1}\t{names[c2]}\t{sd[d2]}\t{hap(c2)}\t{s2}\t{n}\t{links}\t{gap}\t"
                   f"{'link' if 2 * links > n else 'breakpoint'}\n")
    return reads_tsv, "".join(out).encode("latin-1")


def junctions(sunkpos_p, rlen_p, badsunks_p, fai1_p, fai2_p, out_reads_tsv, out_clusters_tsv):
    """Junctions of one haplotype from the files of the per-rule path: {hap}_detailed.sunkpos (combine_ont_nofilt: every
    match row, before the diag filter), {hap}.rlen, bad_sunks.txt and both .fai files (contigs in fai1-then-fai2 order).
    A read is a run of consecutive rows with one name (diag_filter_v3.nim:64); the reference's fixed minimum read
    length."""
    fai = [gio.read_fai(fai1_p), gio.read_fai(fai2_p)]
    names = [n for f in fai for n, _ in f]
    clen = [l for f in fai for _, l in f]
    chap = [0] * len(fai[0]) + [1] * len(fai[1])
    rlen = _read_rlen(rlen_p)
    badset = _read_badsunks(badsunks_p)
    rows, cnames, rnames, cols = _rows_from_sunkpos(sunkpos_p)
    cidx = {}
    for i, n in enumerate(names):
        cidx.setdefault(n, i)
    for c in cnames:
        if c not in cidx:
            raise KeyError(f"contig {c} of {sunkpos_p} is in neither {fai1_p} nor {fai2_p}")
    remap = np.asarray([cidx[c] for c in cnames] + [0], np.uint32)
    cols = (cols[0], cols[1], remap[cols[2]], cols[3], cols[4])
    eng = Engine(20)
    eng.contig_names = names
    lens = _read_lens(rlen, rnames)
    eng.set_reads_meta(lens)
    eng.set_rows(0, *cols)
    _set_bad(eng, badset, names)
    eng.junction_screen(10000)  # the reference's fixed minimum read length (process-by-contig_lowmem_AR.py:106, SURVEY Q13)
    jn = eng.junctions()
    rtab = gio.NameTable(rnames)
    texts = junction_texts(jn, np.arange(len(jn["read"])), names, clen, chap, rtab, lens, bytewise_rank(rtab))
    _write_all((out_reads_tsv, out_clusters_tsv), texts)


def cmd_junctions(argv):
    junctions(*argv)


# ------------------------------------------------------------------------------------------------
# distance discordance: collapses and expansions inside validated intervals (no reference counterpart; DESIGN.md 5.5d)
# ------------------------------------------------------------------------------------------------
DISCORDANCE_READS_HEADER = "contig\tread\tread_len\tid1\tstart1\tpos1\tid2\tstart2\tpos2\tdelta\tkind\n"
DISCORDANCE_RUNS_HEADER = "contig\tstart\tend\tspans\tlonger\tshorter\n"
DISCORDANCE_MIN_READS = 3  # supporting spans of a called segment (with a majority of all spans covering it)
_SPAN_KIND = gio.NameTable(["longer", "shorter"])


def discordance_calls(rec, runs, sel_runs, min_reads=DISCORDANCE_MIN_READS):
    """Calls from the runs of Engine.discordance() (indices sel_runs, in run order) and the records of Engine.spans(): a run
    is `collapse` when longer >= min_reads and 2*longer > spans, `expansion` likewise with shorter; adjacent runs of a
    contig with the same call merge.  Peak = the run with the most supporting spans (ties: larger fraction, then the first);
    size = lower median delta of the call's kind among the records that cover the peak's first base x (id1 <= x < id2: runs
    start at group IDs, so these are the spans that cover the peak's segments).
    -> list of (contig, start, end, kind, peak_start, peak_end, spans, supporting, size or None)"""
    delta = span_delta(rec["start1"], rec["pos1"], rec["start2"], rec["pos2"])
    calls, cur = [], None
    for i in np.asarray(sel_runs, np.int64).tolist():
        c, sp, lo, sh = (int(runs[k][i]) for k in ("contig", "spans", "longer", "shorter"))
        kind = "collapse" if lo >= min_reads and 2 * lo > sp else ("expansion" if sh >= min_reads and 2 * sh > sp else None)
        if cur is not None and (kind is None or cur[0] != c or cur[1] != kind):
            calls.append(cur)
            cur = None
        if kind is None:
            continue
        sup = lo if kind == "collapse" else sh
        if cur is None:
            cur = [c, kind, int(runs["start"][i]), 0, i, sp, sup]
        elif sup > cur[6] or (sup == cur[6] and sup * cur[5] > cur[6] * sp):
            cur[4:7] = [i, sp, sup]
        cur[3] = int(runs["end"][i])
    if cur is not None:
        calls.append(cur)
    out = []
    for c, kind, a, b, pk, sp, sup in calls:
        x = int(runs["start"][pk])
        m = (rec["contig"] == c) & (rec["id1"] <= x) & (rec["id2"] > x) & ((delta >= 0) if kind == "collapse" else (delta < 0))
        d = np.sort(delta[m])
        out.append((c, a, b, kind, x, int(runs["end"][pk]), sp, sup, int(d[(len(d) - 1) // 2]) if len(d) else None))
    return out


def discordance_texts(hap_contigs, names, rec, runs, rtab, read_len, name_rank):
    """The three discordance files of one haplotype: hap_contigs = its contig ids; rec = Engine.spans() with run-wide read
    indices, runs = Engine.discordance(); rtab / read_len / name_rank = name table, length and bytewise name rank of every
    run-wide read.  -> (discordance.reads.tsv, discordance.tsv, discordance.bed) bytes"""
    ctab = gio.NameTable(names)
    inhap = np.zeros(len(names), bool)
    inhap[np.asarray(hap_contigs, np.int64)] = True
    r = np.flatnonzero(inhap[rec["contig"]])
    r = r[np.lexsort((name_rank[rec["read"][r]], rec["start2"][r], rec["start1"][r], rec["contig"][r]))]
    delta = span_delta(rec["start1"], rec["pos1"], rec["start2"], rec["pos2"])
    reads_tsv = DISCORDANCE_READS_HEADER.encode() + gio.format_rows(
        [("name", rec["contig"], ctab), ("name", rec["read"], rtab), ("u32", read_len[rec["read"]])]
        + [("u32", rec[c]) for c in ("id1", "start1", "pos1", "id2", "start2", "pos2")]
        + [("i64", delta), ("name", (delta < 0).astype(np.uint32), _SPAN_KIND)], sel=r)
    q = np.flatnonzero(inhap[runs["contig"]])
    runs_tsv = DISCORDANCE_RUNS_HEADER.encode() + gio.format_rows(
        [("name", runs["contig"], ctab)] + [("u32", runs[c]) for c in ("start", "end", "spans", "longer", "shorter")], sel=q)
    bed = "".join(f"{names[c]}\t{a}\t{b}\t{kind}\t{ps}\t{pe}\t{sp}\t{sup}\t{'.' if size is None else size}\n"
                  for c, a, b, kind, ps, pe, sp, sup, size in discordance_calls(rec, runs, q))
    return reads_tsv, runs_tsv, bed.encode("latin-1")


def discordance(sunkpos_p, rlen_p, badsunks_p, fai_p, out_reads_tsv, out_runs_tsv, out_bed):
    """Distance discordance of one haplotype from the files of the per-rule path ({hap}.sunkpos, {hap}.rlen,
    bad_sunks.txt, the .fai): the whole haplotype is validated in one pass, reads grouped by (contig, read name) as
    process_by_contig groups them per contig, the reference's fixed minimum read length."""
    eng, names, clen, _, reads = _keyed_hap(sunkpos_p, rlen_p, badsunks_p, fai_p)
    eng.validate(10000)  # the reference's fixed minimum read length (process-by-contig_lowmem_AR.py:106, SURVEY Q13)
    texts = discordance_texts(list(range(len(names))), names, eng.spans(), eng.discordance(clen), *reads)
    _write_all((out_reads_tsv, out_runs_tsv, out_bed), texts)


def cmd_discordance(argv):
    discordance(*argv)


# ------------------------------------------------------------------------------------------------
# read haplotypes: every read's SUNK vote on both haplotypes (no reference counterpart; DESIGN.md section 5.5e)
# ------------------------------------------------------------------------------------------------
READ_HAP_READS_HEADER = "read\tread_len\tbin\tcontig1\tn1\tstrand1\tcontig2\tn2\tstrand2\thap\n"
_BIN = gio.NameTable(["hap1", "hap2", "unbinned"])
_ASSIGNED = gio.NameTable(["hap1", "hap2", "tie"])
_STRAND_OR_NONE = gio.NameTable(["+", "-", "."])
_NO_VOTE = 0xFFFFFFFF


def file_haps(read_bin, rh) -> np.ndarray:
    """File haplotype (0 / 1) of every run-wide read: its chunk's haplotype (read_bin 0 / 1); for an unbinned read
    (GVS_HAP_ANY) the one its votes assign (rh = Engine.read_haps() with run-wide read indices), and for a tie or a read
    without a vote the parity of its index (even: hap1), so that each haplotype's read-length library gets half of the
    reads SUNKs cannot place."""
    read_bin = np.asarray(read_bin, np.uint8)
    fh = read_bin.copy()
    un = np.flatnonzero(read_bin == GVS_HAP_ANY)
    fh[un] = (un & 1).astype(np.uint8)
    if len(rh["read"]):
        a = (rh["hap"] <= 1) & (read_bin[rh["read"]] == GVS_HAP_ANY)
        fh[rh["read"][a]] = rh["hap"][a].astype(np.uint8)
    return fh


def read_hap_texts(hap, names, contig_hap, rh, read_bin, read_hap, rtab, read_len, name_rank):
    """The two read-haplotype files of haplotype `hap`: rh = Engine.read_haps() with run-wide read indices; read_bin /
    read_hap = chunk haplotype (0, 1, GVS_HAP_ANY) and file haplotype (file_haps) of every run-wide read; rtab / read_len /
    name_rank = name table, length and bytewise name rank of every run-wide read.  -> (haplotype.reads.tsv: one row per
    record of a read of file haplotype `hap`, in name order; haplotype.tsv: per contig of `hap` the reads whose vote on
    `hap` lands on it, by assignment, and a totals row that also counts the reads of file haplotype `hap` without a vote
    and their bases) bytes"""
    hn, on = hap + 1, 2 - hap
    ctab = gio.NameTable(list(names) + ["."])
    sel = np.flatnonzero(read_hap[rh["read"]] == hap) if len(rh["read"]) else np.zeros(0, np.int64)
    r = sel[np.lexsort((sel, name_rank[rh["read"][sel]]))]
    cols = [("name", rh["read"], rtab), ("u32", read_len[rh["read"]]), ("name", read_bin[rh["read"]].astype(np.uint32), _BIN)]
    for side in "12":
        c = rh["contig" + side]
        none = c == _NO_VOTE
        cols += [("name", np.where(none, len(names), c).astype(np.uint32), ctab), ("u32", rh["n" + side]),
                 ("name", np.where(none, 2, rh["strand" + side]).astype(np.uint32), _STRAND_OR_NONE)]
    cols.append(("name", rh["hap"], _ASSIGNED))
    reads_tsv = READ_HAP_READS_HEADER.encode() + gio.format_rows(cols, sel=r)
    c = rh[f"contig{hn}"]
    v = np.flatnonzero(c != _NO_VOTE)
    nc = len(names)
    count = lambda m: np.bincount(c[v][m], minlength=nc).astype(np.int64)
    a = rh["hap"][v]
    same, other, tie = count(a == hap), count(a == 1 - hap), count(a == 2)
    out = [f"contig\treads\tassigned_hap{hn}\tassigned_hap{on}\ttie\tno_vote_reads\tno_vote_bases\n"]
    for ci in np.flatnonzero(np.asarray(contig_hap) == hap).tolist():
        out.append(f"{names[ci]}\t{same[ci] + other[ci] + tie[ci]}\t{same[ci]}\t{other[ci]}\t{tie[ci]}\t.\t.\n")
    voted = np.zeros(len(read_hap), bool)
    voted[rh["read"]] = True
    nv = np.flatnonzero(~voted & (read_hap == hap))
    hc = np.asarray(contig_hap) == hap
    out.append(f"total\t{(same + other + tie)[hc].sum()}\t{same[hc].sum()}\t{other[hc].sum()}\t{tie[hc].sum()}\t{len(nv)}\t"
               f"{int(read_len[nv].astype(np.int64).sum())}\n")
    return reads_tsv, "".join(out).encode("latin-1")


def cmd_get_gaps(argv):
    """get_gaps.py: paths are string-concatenated, so indir / outdir need their trailing slash (:30,70)"""
    fai1, fai2, sample, indir, outdir = argv
    fais = [gio.read_fai(fai1), gio.read_fai(fai2)]
    names, lens, hap_of = [], [], []
    for hap in range(2):
        for n, l in fais[hap]:
            names.append(n)
            lens.append(l)
            hap_of.append(hap)
    ic, is_, ie = [], [], []
    for ci, n in enumerate(names):
        bp = indir + n.replace("#", "_") + f"_hap{hap_of[ci] + 1}.bed"
        if not os.path.exists(bp):
            sys.stdout.write(f"No bed for {n}\n")
            continue
        with open(bp) as f:
            for l in f:
                p = l.rstrip("\n").split("\t")
                if len(p) >= 3:
                    ic.append(ci)
                    is_.append(int(p[1]))
                    ie.append(int(p[2]))
    eng = Engine(20)
    eng.contig_names = names
    eng.set_intervals(ic, is_, ie, len(names))
    gaps, nodata = eng.gaps(np.asarray(lens, np.uint32))
    for hap in range(2):
        g = [(names[c], s, e) for c, s, e in zip(gaps["contig"].tolist(), gaps["start"].tolist(), gaps["end"].tolist()) if hap_of[c] == hap]
        nd = [(names[c], 0, lens[c]) for c in nodata.tolist() if hap_of[c] == hap]
        sys.stdout.write(f"hap{hap + 1}\nbreaks:  {len(g)} {sum(e + 1 - s for _, s, e in g)}\nno data:  {len(nd)} {sum(l for _, _, l in nd)}\n")
        _atomic_write(outdir + f"hap{hap + 1}.nodata.bed", "".join(f"{a}\t{s}\t{e}\n" for a, s, e in nd))
        _atomic_write(outdir + f"hap{hap + 1}.gaps.bed", "".join(f"{a}\t{s}\t{e}\n" for a, s, e in g))


def _read_bed3(path):
    out = []
    with open(path) as f:
        for l in f:
            p = l.rstrip("\n").split("\t")
            if len(p) >= 3:
                out.append((p[0], int(p[1]), int(p[2])))
    return out


def cmd_slop_gaps(argv):
    """bedtools slop -i gaps -g fai -b 200000 (tagONT.smk:249)"""
    bed_p, fai_p, out_p = argv
    fai = gio.read_fai(fai_p)
    cidx = {n: i for i, (n, _) in enumerate(fai)}
    rows = _read_bed3(bed_p)
    for c, _, _ in rows:
        if c not in cidx:
            raise KeyError(f"chromosome {c} is not in the genome file")
    eng = Engine(20)
    s, e = eng.slop([cidx[c] for c, _, _ in rows], [r[1] for r in rows], [r[2] for r in rows], [l for _, l in fai], 200000)
    _atomic_write(out_p, "".join(f"{c}\t{a}\t{b}\n" for (c, _, _), a, b in zip(rows, s.tolist(), e.tolist())))


def _natural_key(s: str):
    import re
    return [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", s)]


def covprob(bed_p, locs_p, rlen_p, fai_p, sunk_len: int, tsv_p):
    """covprob.py:14-134"""
    from .engine import covprob_bins, covprob_pn
    genome_kbp = sum(l for _, l in gio.read_fai(fai_p)) / 1000
    gaps = _read_bed3(bed_p)
    contig, start, kmer, group = gio.read_loc(locs_p)
    seen_k, seen_g, gc, gi = set(), set(), [], []
    cidx: Dict[str, int] = {}
    for c, km, g in zip(contig, kmer, group):  # drop_duplicates(kmer) then drop_duplicates(ID2) (:36-38)
        if km in seen_k:
            continue
        seen_k.add(km)
        if (c, g) in seen_g:
            continue
        seen_g.add((c, g))
        gc.append(cidx.setdefault(c, len(cidx)))
        gi.append(g)
    lens = []
    with gio.open_maybe_gz(rlen_p) as f:
        for l in f.read().decode().splitlines():
            p = l.split("\t")
            if len(p) >= 2:
                lens.append((p[0], int(p[1])))
    kbp, cnt = covprob_bins(lens)
    eng = Engine(int(sunk_len) if 1 <= int(sunk_len) <= 32 else 20)
    table = eng.covprob_table(kbp, cnt, genome_kbp, covprob_pn(int(sunk_len)))
    # breaks.df: pyranges groups the rows by chromosome (natural order of the names), file order inside
    order = sorted(range(len(gaps)), key=lambda i: (_natural_key(gaps[i][0]), i))
    g_sorted = [gaps[i] for i in order]
    unknown = len(cidx)
    mg, pr = eng.covprob_gaps(gc, gi, [cidx.get(c, unknown) for c, _, _ in g_sorted], [s for _, s, _ in g_sorted],
                              [e for _, _, e in g_sorted], table)
    out = ["index\tChromosome\tStart\tEnd\ttype\tmax_gap\tcovprob\n"]
    for i, (c, s, e), m, p in zip(order, g_sorted, mg.tolist(), pr.tolist()):
        out.append(f"{i}\t{c}\t{s}\t{e}\tgap\t{m}\t{p!r}\n")
    _atomic_write(tsv_p, "".join(out))
    return table


def covprob_script(snakemake):
    """drop-in body for `script: ../scripts/covprob.py` (tagONT.smk:211-231)"""
    covprob(snakemake.input.bed, snakemake.input.locs, snakemake.input.rlen, snakemake.input.fai,
            int(snakemake.config["SUNK_len"]), snakemake.output.tsv)


def cmd_covprob(argv):
    ap = argparse.ArgumentParser(prog="gavisunk_b200.cli covprob")
    for a in ("bed", "locs", "rlen", "fai", "tsv"):
        ap.add_argument("--" + a, required=True)
    ap.add_argument("--sunk-len", type=int, required=True)
    a = ap.parse_args(argv)
    covprob(a.bed, a.locs, a.rlen, a.fai, a.sunk_len, a.tsv)


def split_locs(ont_pos_p, kmer_loc_p, flag_p, hap: str):
    """split_locs.py:5-22: byte-level partition by contig, no arithmetic (host only)"""
    dirname = os.path.dirname(flag_p)
    os.makedirs(dirname or ".", exist_ok=True)
    by_c: Dict[str, List[str]] = defaultdict(list)
    with gio.open_maybe_gz(ont_pos_p) as f:
        for l in f.read().decode().splitlines():
            p = l.split("\t")
            if len(p) >= 5:
                by_c[p[2]].append(l + "\n")
    loc_c: Dict[str, List[str]] = defaultdict(list)
    with open(kmer_loc_p) as f:
        for l in f:
            c = l.split("\t", 1)[0]
            if c in by_c:
                loc_c[c].append(l if l.endswith("\n") else l + "\n")
    for c, lines in by_c.items():
        _atomic_write(f"{dirname}/{c.replace('#', '_')}_{hap}.sunkpos", "".join(lines))
    for c, lines in loc_c.items():
        _atomic_write(f"{dirname}/{c.replace('#', '_')}_{hap}.loc", "".join(lines))


def split_locs_script(snakemake):
    split_locs(snakemake.input.ONT_pos, snakemake.input.kmer_loc, snakemake.output.flag, snakemake.wildcards.hap)


def cmd_split_locs(argv):
    ap = argparse.ArgumentParser(prog="gavisunk_b200.cli split_locs")
    ap.add_argument("--ont-pos", required=True)
    ap.add_argument("--kmer-loc", required=True)
    ap.add_argument("--flag", required=True)
    ap.add_argument("--hap", required=True)
    a = ap.parse_args(argv)
    split_locs(a.ont_pos, a.kmer_loc, a.flag, a.hap)
    open(a.flag, "a").close()  # touch() of the checkpoint rule (tagONT.smk:158)


# ------------------------------------------------------------------------------------------------
# split_ONT (workflow/rules/tagONT.smk:2-18): cat reads | seqtk seq -F '#' | rustybam fastq-split outs
# ------------------------------------------------------------------------------------------------
def split_ont(reads_paths: Sequence[str], out_paths: Sequence[str], threads: int = 0):
    """The scatter step of the reference: every record becomes a 4-line FASTQ record with a fake quality of '#'
    (`seqtk seq -F '#'`) and record i goes to output i mod N (`rustybam fastq-split`), outputs gzip-compressed when
    they end in .gz.  seqtk and rustybam are not installed here, so this step is PARITY UNPINNED: the round-robin
    distribution is rustybam's documented behaviour, and the header comment seqtk would keep is dropped (no
    consumer reads past the name: kmerpos_annot3.nim:85, rlen.nim:13).  Outputs that depend on the chunking (the
    prevLoc carry and the Table capacity of a chunk, SURVEY Q4/Q9) are identical to the reference's whenever
    the chunk files are."""
    import gzip
    from concurrent.futures import ThreadPoolExecutor
    reads = gio.NativeReads(list(reads_paths), pin=False)
    n_out = len(out_paths)
    off = reads.read_off
    seq = reads.seq
    nt = gio.NameTable(blob=reads.name_blob, off=reads.name_off)
    no = nt.off.tolist()

    def write(c):
        opener = (lambda p: gzip.open(p, "wb", compresslevel=1)) if out_paths[c].endswith(".gz") else (lambda p: open(p, "wb"))
        tmp = out_paths[c] + ".tmp%d" % os.getpid()
        with opener(tmp) as f:
            for r in range(c, reads.n_reads, n_out):
                a, b = int(off[r]), int(off[r + 1])
                f.write(b"@" + nt.blob[no[r]:no[r + 1]] + b"\n")
                f.write(seq[a:b].tobytes())
                f.write(b"\n+\n" + b"#" * (b - a) + b"\n")
        os.replace(tmp, out_paths[c])
    with ThreadPoolExecutor(max_workers=threads or min(n_out, os.cpu_count() or 1)) as ex:
        list(ex.map(write, range(n_out)))
    reads.close()


def cmd_split_ont(argv):
    ap = argparse.ArgumentParser(prog="gavisunk_b200.cli split_ont")
    ap.add_argument("--reads", nargs="+", required=True)
    ap.add_argument("--out", nargs="+", required=True, help="temp/{sample}/reads/{hap}_{i}-of-{N}.fq.gz in scatter order")
    a = ap.parse_args(argv)
    split_ont(a.reads, a.out)


def cmd_combine_ont_nofilt(argv):
    """combine_ont_nofilt (workflow/rules/tagONT.smk:39-55): cat of the unfiltered chunk outputs in gather order"""
    *ins, out_p = argv
    tmp = out_p + ".tmp%d" % os.getpid()
    with open(tmp, "wb") as o:
        for p in ins:
            with open(p, "rb") as f:
                while True:
                    blk = f.read(1 << 24)
                    if not blk:
                        break
                    o.write(blk)
    os.replace(tmp, out_p)


# ------------------------------------------------------------------------------------------------
# fused: defineSUNKs.smk + tagONT.smk (SUNK_annot .. slop_gaps) for one sample, on one or several GPUs
# ------------------------------------------------------------------------------------------------
def decode_kmers(km: np.ndarray, k: int) -> List[str]:
    if len(km) == 0:
        return []
    shifts = (2 * np.arange(k - 1, -1, -1)).astype(np.uint64)
    codes = ((km[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    return letters.view(f"S{k}").ravel().astype(str).tolist()


def _write_bytes(path: str, data):
    tmp = path + ".tmp%d" % os.getpid()
    with open(tmp, "wb") as f:
        f.write(data)
    os.replace(tmp, path)


def _write_all(paths: Sequence[str], texts: Sequence[bytes]):
    for path, data in zip(paths, texts):
        _write_bytes(path, data)


class Evidence(NamedTuple):
    """An optional output of `fused` that the reference does not produce"""
    flag: str
    help: str
    records: str                  # run_reads' result key of its per-engine records, concatenated run-wide
    columns: Tuple[str, ...]      # their columns
    suffixes: Tuple[str, ...]     # final_out/hap{N}.{suffix}, in the order its *_texts returns them


EVIDENCE_PRODUCTS = {
    "support_tracks": Evidence("--support-tracks", "also write final_out/hap{N}.reads.bed, .support.bedgraph and .support.tsv "
                               "(support of the validated reads)", "placements", Engine.PLACEMENT_COLUMNS,
                               ("reads.bed", "support.bedgraph", "support.tsv")),
    "gap_evidence": Evidence("--gap-evidence", "also write final_out/hap{N}.gaps.evidence.tsv and .gaps.reads.tsv (the reads "
                             "that bridge each gap)", "gap_evidence", Engine.GAP_EVIDENCE_COLUMNS,
                             ("gaps.reads.tsv", "gaps.evidence.tsv")),
    "junctions": Evidence("--junctions", "also write final_out/hap{N}.junctions.reads.tsv and .junctions.tsv (reads that jump "
                          "between contigs)", "junctions", Engine.JUNCTION_COLUMNS, ("junctions.reads.tsv", "junctions.tsv")),
    "discordance": Evidence("--discordance", "also write final_out/hap{N}.discordance.reads.tsv, .discordance.tsv and "
                            ".discordance.bed (collapses and expansions inside validated intervals)", "spans", Engine.SPAN_COLUMNS,
                            ("discordance.reads.tsv", "discordance.tsv", "discordance.bed")),
    "read_haplotypes": Evidence("--read-haplotypes", "also write final_out/hap{N}.haplotype.reads.tsv and .haplotype.tsv (each "
                                "read's SUNK vote on both haplotypes; implied by --reads)", "read_haps", Engine.READ_HAP_COLUMNS,
                                ("haplotype.reads.tsv", "haplotype.tsv")),
}


def plan_batches(files: Sequence[str], n_devices: int, batch_files: int = 0, batch_gbp: float = 12.0) -> List[List[int]]:
    """groups of consecutive chunk files (scatter order: hap1 chunks, then hap2 chunks).  batch_files > 0 fixes the
    group size; otherwise groups hold about `batch_gbp` Gbp (estimated from the file sizes: FASTQ = 2 bytes per
    base, gzip ~ 4x) and there are at least as many groups as devices when the files allow it."""
    n = len(files)
    if n == 0:
        return []
    if batch_files > 0:
        return [list(range(i, min(n, i + batch_files))) for i in range(0, n, batch_files)]

    def est_bases(p):
        try:
            sz = os.path.getsize(p)
        except OSError:
            return 0
        with open(p, "rb") as f:
            head = f.read(2)
        gz = head == b"\x1f\x8b"
        fq = p.endswith((".fq", ".fastq", ".fq.gz", ".fastq.gz"))
        return sz * (4 if gz else 1) // (2 if fq else 1)
    est = [est_bases(p) for p in files]
    want = max(1.0, min(batch_gbp * 1e9, sum(est) / max(1, n_devices)))
    out, cur, acc = [], [], 0
    for i, e in enumerate(est):
        if cur and acc + e > want * 1.05 and len(out) + 1 + (n - i) >= n_devices:
            out.append(cur)
            cur, acc = [], 0
        cur.append(i)
        acc += e
    if cur:
        out.append(cur)
    return out


def run_reads(engines, contig_hap, files: Sequence[str], file_hap: Sequence[int], batch_files: int = 0, batch_gbp: float = 12.0,
              detailed: bool = False, threads: int = 0, min_read_len: int = 10000, coll=None, products: Sequence[str] = (),
              contig_len=None):
    """The read side of the fused rule on engines whose SUNK database is loaded: the chunk files (scatter order, with
    the haplotype each belongs to) are grouped into batches (plan_batches); engine i owns a contiguous block of the
    batches and runs Engine.run_batches on it (one host thread per GPU, two exchanges per run).  Reads are parsed
    and 2-bit packed in one pass (gio.NativeReads(packed=True)) while the previous batch is on the GPU.
    coll: exchange object of a multi-PROCESS run (gavisunk_b200.parallel.EngineExchange) when `engines` is this rank's
    single engine.  products: names of EVIDENCE_PRODUCTS to compute as well (contig_len: the contig lengths) --
    support_tracks: the support placements of every engine and the support runs, with the difference arrays summed
    across engines by the histogram's exchange; gap_evidence: the gaps of every engine (the same on all: intervals are
    merged across engines) and the gap-evidence records of its own reads; junctions: the junction records of every
    engine's own reads (each batch screened after its diag filter, resolved with the run's bad groups); discordance: the
    discordant spans of every engine's own reads and the discordance runs, with the difference arrays summed like the
    support's; read_haplotypes: every engine's diag filters in haplotype mode and the records of its own reads (file_hap
    GVS_HAP_ANY: unbinned chunks, always filtered in haplotype mode).  -> one result dict per engine (read names /
    lengths / chunk tables, kept rows, validated pairs, intervals[, placements, support runs][, gap evidence][,
    junctions][, spans, discordance runs][, read haplotypes])."""
    import threading
    from concurrent.futures import ThreadPoolExecutor
    for p in files:
        if not os.path.exists(p):
            raise FileNotFoundError(p)
    for p in products:
        if p not in EVIDENCE_PRODUCTS:
            raise ValueError(f"unknown evidence product {p!r}")
    n_dev = len(engines)
    batches = plan_batches(files, n_dev, batch_files, batch_gbp)
    shards = shard_chunks(len(batches), n_dev)
    n_cpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    ingest_threads = threads or max(1, n_cpu // n_dev)
    results = [None] * n_dev
    errors = []
    xch = ThreadExchange(engines)

    def worker(di):
        try:
            eng = engines[di]
            cx = coll if (coll is not None and n_dev == 1) else xch.for_rank(di)
            mine = batches[shards[di][0]:shards[di][1]]
            load = lambda fl: gio.NativeReads([files[i] for i in fl], threads=ingest_threads, packed=True)
            info = dict(names=[], lens=[], chunk_first=[], chunk_hap=[], rows0=[], n_reads=0, n_bases=0)
            with ThreadPoolExecutor(max_workers=1) as pre:
                fut = pre.submit(load, mine[0]) if mine else None
                held = []

                def bind_for(bi):
                    def bind(e):
                        nonlocal fut
                        reads = fut.result()
                        fut = pre.submit(load, mine[bi + 1]) if bi + 1 < len(mine) else None
                        for old in held:  # the previous batch's words: its copies finished with its match
                            old.close()
                        held.clear()
                        held.append(reads)
                        ch = [file_hap[i] for i in mine[bi]]
                        e.set_reads_packed(reads.words, reads.read_off, reads.chunk_first, ch)
                        info["names"].append(gio.NameTable(blob=reads.name_blob, off=reads.name_off))
                        info["lens"].append(reads.lengths().astype(np.uint32))
                        info["chunk_first"].append(reads.chunk_first.astype(np.int64) + info["n_reads"])
                        info["chunk_hap"].append(np.asarray(ch, np.uint8))
                        info["n_reads"] += reads.n_reads
                        info["n_bases"] += reads.total_bases
                    return bind

                def on_batch(e, b, base):
                    if detailed:
                        r0 = e.rows(0)
                        r0["read"] = r0["read"] + np.uint32(base)
                        info["rows0"].append(r0)
                iv, bases = eng.run_batches([bind_for(bi) for bi in range(len(mine))], contig_hap, min_read_len=min_read_len,
                                            allreduce_hist=cx.allreduce_hist, gather_forests=cx.gather_forests, on_batch=on_batch,
                                            junctions="junctions" in products, read_haps="read_haplotypes" in products)
                for old in held:
                    old.close()
            info.update(kept=eng.rows(1, pinned=True), pairs=eng.pairs(pinned=True), iv=iv)
            if "support_tracks" in products:
                info.update(placements=eng.placements(pinned=True), support=eng.support(contig_len, allreduce=cx.allreduce_hist))
            if "gap_evidence" in products:
                eng.gaps(contig_len)
                info.update(gap_evidence=eng.gap_evidence(min_read_len))
            if "junctions" in products:
                info.update(junctions=eng.junctions())
            if "discordance" in products:
                info.update(spans=eng.spans(), discordance=eng.discordance(contig_len, allreduce=cx.allreduce_hist))
            if "read_haplotypes" in products:
                info.update(read_haps=eng.read_haps() if mine else {c: np.zeros(0, np.uint32) for c in Engine.READ_HAP_COLUMNS})
            results[di] = info
        except BaseException as ex:  # noqa: BLE001 -- reported by the caller; peers must not wait for this rank
            errors.append(ex)
            xch.abort()

    if n_dev == 1:
        worker(0)
    else:
        ths = [threading.Thread(target=worker, args=(i,)) for i in range(n_dev)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
    if errors:
        first = [e for e in errors if not isinstance(e, threading.BrokenBarrierError)] or errors
        raise first[0]
    return results


def run_fused(k: int, hap_asm: Sequence[str], hap_reads: Sequence[Sequence[str]], outdir: str, device: int = 0,
              devices: Sequence[int] = None, batch_files: int = 0, batch_gbp: float = 12.0, detailed: bool = False,
              threads: int = 0, mrsfast_palindromes: bool = False, products: Sequence[str] = (), reads: Sequence[str] = ()):
    """hap_asm: two FASTA paths; hap_reads: two lists of chunk files in scatter order, or None and `reads`: chunk files of
    unbinned reads, whose haplotypes their SUNK votes assign (implies the read_haplotypes product).  Builds the SUNK
    database on every GPU of `devices`, runs the reads (run_reads) and writes every file of the rules between
    jellyfish_count and slop_gaps under `outdir`, and the files of the EVIDENCE_PRODUCTS named in `products`.  Returns the
    first device's engine."""
    from concurrent.futures import ThreadPoolExecutor
    devices = list(devices) if devices else [device]
    contigs, contig_hap, fai = [], [], [[], []]
    for hap in range(2):
        for n, s in gio.read_fastx(hap_asm[hap]):
            contigs.append((n, s))
            contig_hap.append(hap)
            fai[hap].append((n, len(s)))
    if (hap_reads is None) == (not reads):
        raise ValueError("give either the two haplotypes' chunk files or unbinned chunk files")
    if reads:
        files, file_hap = list(reads), [GVS_HAP_ANY] * len(reads)
        products = list(products) + ["read_haplotypes"] * ("read_haplotypes" not in products)
    else:
        files = list(hap_reads[0]) + list(hap_reads[1])
        file_hap = [0] * len(hap_reads[0]) + [1] * len(hap_reads[1])
    for p in files:
        if not os.path.exists(p):
            raise FileNotFoundError(p)

    def make(d):
        e = Engine(k, device=d)
        e.build_db(contigs)
        return e
    if len(devices) == 1:
        engines = [make(devices[0])]
    else:
        with ThreadPoolExecutor(max_workers=len(devices)) as ex:
            engines = list(ex.map(make, devices))
    clen = [len(s) for _, s in contigs]
    results = run_reads(engines, contig_hap, files, file_hap, batch_files, batch_gbp, detailed, threads, products=products,
                        contig_len=clen)
    eng = engines[0]
    gaps, nodata = eng.gaps(np.asarray(clen, dtype=np.uint32))
    write_outputs(k, eng, results, clen, contig_hap, eng.contig_names, results[0]["iv"], gaps, nodata, outdir,
                  detailed=detailed, palindromes=mrsfast_palindromes, products=products)
    for e in engines[1:]:
        e.close()
    return eng


def write_outputs(k, eng, results, contig_len, contig_hap, names, iv, gaps, nodata, outdir, detailed=False, palindromes=False,
                  db_files=True, products: Sequence[str] = ()):
    """every file of SURVEY Appendix C that the rules between jellyfish_count and slop_gaps produce (db_files=False:
    without the exports of the database itself -- db/jellyfish.db|.fa, mrsfast/kmer.loc and its per-contig copies
    breaks/*.loc -- which belong to the database build, not to a run over reads), and final_out/hap{N}.{suffix} of every
    product named in `products` (EVIDENCE_PRODUCTS; results of run_reads with the same products)"""
    d = lambda *p: os.path.join(outdir, *p)
    for sub in ("db", "mrsfast", "sunkpos", "breaks", "inter_outs", "bed_files", "final_out"):
        os.makedirs(d(sub), exist_ok=True)
    ctab = gio.NameTable(names)
    safe = lambda n: n.replace("#", "_")
    jobs = []  # (path, columns, options): formatted and written by a small pool at the end (the files are independent)

    def emit(path, cols, **kw):
        jobs.append((path, cols, kw))
    # ---- run-wide read table: devices in order, batches in order ----
    read_base, nreads = [], 0
    for r in results:
        read_base.append(nreads)
        nreads += r["n_reads"]
    rtab = gio.NameTable.concat([t for r in results for t in r["names"]])
    lens = np.concatenate([l for r in results for l in r["lens"]] + [np.zeros(0, np.uint32)])
    chunk_first = np.concatenate([cf[:-1] + read_base[i] for i, r in enumerate(results) for cf in r["chunk_first"]] + [np.array([nreads])])
    chunk_hap = np.concatenate([ch for r in results for ch in r["chunk_hap"]] + [np.zeros(0, np.uint8)])
    read_bin = np.zeros(nreads, np.uint8)
    for c in range(len(chunk_hap)):
        read_bin[int(chunk_first[c]):int(chunk_first[c + 1])] = chunk_hap[c]

    def cat_rows(key, cols):
        out = {}
        for c in cols:
            parts = []
            for i, r in enumerate(results):
                tabs = r[key] if isinstance(r[key], list) else [r[key]]
                for t in tabs:
                    parts.append(t[c] + np.uint32(read_base[i]) if (c == "read" and read_base[i]) else t[c])
            out[c] = parts[0] if len(parts) == 1 else (np.concatenate(parts) if parts else np.zeros(0, np.uint32))
        return out
    # the file haplotype of every read: its chunk's, or for unbinned reads the one its votes assign (file_haps)
    if "read_haplotypes" in products:
        rh = cat_rows("read_haps", Engine.READ_HAP_COLUMNS)
        read_hap = file_haps(read_bin, rh)
    elif (read_bin == GVS_HAP_ANY).any():
        raise ValueError("unbinned reads need the read_haplotypes product")
    else:
        read_hap = read_bin
    kept = cat_rows("kept", Engine.ROW_COLUMNS)
    pairs = cat_rows("pairs", Engine.PAIR_COLUMNS)
    sunk_cols = lambda t: [("name", t["read"], rtab), ("u32", t["pos"]), ("name", t["contig"], ctab), ("u32", t["start"]), ("u32", t["group"])]
    # ---- SUNK database files (defineSUNKs.smk:59-60, 126) ----
    from .engine import revcomp_kmers
    loc_sel, loc_c = None, {}
    if db_files:
        db = eng.db_export()
        loc_cols = [("name", db["contig"], ctab), ("u32", db["start"]), ("kmer", db["kmer"], k), ("u32", db["group"])]
        if palindromes and k % 2 == 0 and len(db["kmer"]):
            # mrsfast reports a k-mer that is its own reverse complement on both strands: two identical rows (SURVEY A.2)
            pal = db["kmer"] == revcomp_kmers(db["kmer"], k)
            loc_sel = np.repeat(np.arange(len(pal), dtype=np.uint64), 1 + pal.astype(np.int64))
        emit(d("db", "jellyfish.db"), [("kmer", db["kmer"], k)])
        emit(d("db", "jellyfish.fa"), [("kmer", db["kmer"], k, dict(prefix=b">", sep=b"\n")), ("kmer", db["kmer"], k)])
        emit(d("mrsfast", "kmer.loc"), loc_cols, sel=loc_sel)
    # ---- per-haplotype row files (combine_ont, combine_ont_nofilt, read_lengths) ----
    khap = read_hap[kept["read"]] if len(kept["read"]) else np.zeros(0, np.uint8)
    all_reads = np.arange(nreads, dtype=np.uint32)
    if detailed:
        rows0 = cat_rows("rows0", Engine.ROW_COLUMNS)
        r0hap = read_hap[rows0["read"]] if len(rows0["read"]) else np.zeros(0, np.uint8)
    for hap in range(2):
        emit(d("sunkpos", f"hap{hap + 1}.sunkpos"), sunk_cols(kept), sel=np.flatnonzero(khap == hap))
        emit(d("sunkpos", f"hap{hap + 1}.rlen"), [("name", all_reads, rtab), ("u32", lens)], sel=np.flatnonzero(read_hap == hap))
        if detailed:  # unfiltered rows for plot_detailed (viz_detailed.py:48)
            emit(d("sunkpos", f"hap{hap + 1}_detailed.sunkpos"), sunk_cols(rows0), sel=np.flatnonzero(r0hap == hap))
    gtab = eng.groups()
    bad = eng.bad_list()
    emit(d("sunkpos", "bad_sunks.txt"), [("name", gtab["contig"][bad], ctab, dict(sep=b":")), ("u32", gtab["group"][bad])])
    # ---- per-contig files: breaks/*.sunkpos|.loc (split_locs.py:5-22), inter_outs/*.tsv, bed_files/*.bed ----
    def by_contig(col, read=None, rank=None):
        """row indices per contig, in row order (rank given: by rank[read] first, stable).  Rows come in runs of one
        read on one contig, so the runs are sorted (a few per read), not the rows."""
        n = len(col)
        if n == 0:
            return {}
        brk = np.ones(n, bool)
        if read is not None:
            brk[1:] = (col[1:] != col[:-1]) | (read[1:] != read[:-1])
        else:
            brk[1:] = col[1:] != col[:-1]
        starts = np.flatnonzero(brk)
        lens = np.diff(np.append(starts, n))
        rc = col[starts].astype(np.int64)
        key = rc if rank is None else rc * np.int64(len(rank) + 1) + rank[read[starts]]
        order = np.argsort(key, kind="stable")
        starts, lens, rc = starts[order], lens[order], rc[order]
        ends = np.cumsum(lens)
        rows = np.repeat(starts - (ends - lens), lens) + np.arange(int(ends[-1]), dtype=np.int64)  # expand the sorted runs
        cs, first = np.unique(rc, return_index=True)
        lo = (ends - lens)[first]
        hi = np.append(lo[1:], ends[-1])
        return {int(c): rows[a:b] for c, a, b in zip(cs, lo, hi)}
    name_rank = bytewise_rank(rtab)
    kept_c = by_contig(kept["contig"], kept["read"])
    # a read lives on one engine: the evidence records of all engines, read indices made run-wide (runs are the same on
    # every engine)
    rec = {p: cat_rows(EVIDENCE_PRODUCTS[p].records, EVIDENCE_PRODUCTS[p].columns) for p in products}
    pair_c = by_contig(pairs["contig"], pairs["read"], name_rank)  # reads in name order, pairs of a read in vertex order
    if db_files:
        loc_c = by_contig(db["contig"])
    iv_c = by_contig(iv["contig"])
    for c, idx in kept_c.items():
        stem = f"{safe(names[c])}_hap{contig_hap[c] + 1}"
        emit(d("breaks", stem + ".sunkpos"), sunk_cols(kept), sel=idx)
        if c in loc_c:
            sel = loc_c[c]
            if loc_sel is not None:
                sel = np.repeat(sel, 1 + (db["kmer"][sel] == revcomp_kmers(db["kmer"][sel], k)).astype(np.int64))
            emit(d("breaks", stem + ".loc"), loc_cols, sel=sel)
        if c in pair_c:
            pidx = pair_c[c]
            emit(d("inter_outs", stem + ".tsv"), [("u32", pairs["group"]), ("name", pairs["read"], rtab)], sel=pidx)
            emit(d("bed_files", stem + ".bed"), [("name", iv["contig"], ctab), ("u32", iv["start"]), ("u32", iv["end"])],
                                                                    sel=iv_c.get(c, np.zeros(0, np.uint64)))
        else:  # "no usable reads": contig name only, bed touched empty by the rule (tagONT.smk:190)
            _write_bytes(d("inter_outs", stem + ".tsv"), (names[c] + "\n").encode("latin-1"))
            _write_bytes(d("bed_files", stem + ".bed"), b"")
    clen = np.asarray(contig_len, dtype=np.uint32)
    chap = np.asarray(contig_hap, np.uint8)
    reads = (rtab, lens, name_rank)
    for hap in range(2):
        hn = hap + 1
        open(d("breaks", f"hap{hn}_splits_pos.done"), "a").close()  # touch() of the checkpoint (tagONT.smk:158)
        bed3 = lambda t: [("name", t["contig"], ctab), ("u32", t["start"]), ("u32", t["end"])]
        emit(d("final_out", f"hap{hn}.valid.bed"), bed3(iv), sel=np.flatnonzero(chap[iv["contig"]] == hap))
        gsel = np.flatnonzero(chap[gaps["contig"]] == hap)
        emit(d("final_out", f"hap{hn}.gaps.bed"), bed3(gaps), sel=gsel)
        nd = nodata[chap[nodata] == hap]
        emit(d("final_out", f"hap{hn}.nodata.bed"), [("name", nd, ctab), ("u32", np.zeros(len(nd), np.uint32)), ("u32", clen[nd])])
        s2, e2 = eng.slop(gaps["contig"][gsel], gaps["start"][gsel], gaps["end"][gsel], clen, 200000)  # bedtools slop -b 200000 (tagONT.smk:249)
        emit(d("final_out", f"hap{hn}.gaps.slop.bed"), [("name", gaps["contig"][gsel], ctab), ("i64", s2), ("i64", e2)])
        hap_contigs = np.flatnonzero(chap == hap).tolist()
        texts = dict(
            support_tracks=lambda r: support_texts(hap_contigs, clen, names, r, results[0]["support"], iv, *reads),
            gap_evidence=lambda r: gap_evidence_texts(gsel, gaps, names, r, *reads),
            junctions=lambda r: junction_texts(r, np.flatnonzero(read_hap[r["read"]] == hap), names, clen, contig_hap, *reads),
            discordance=lambda r: discordance_texts(hap_contigs, names, r, results[0]["discordance"], *reads),
            read_haplotypes=lambda r: read_hap_texts(hap, names, chap, r, read_bin, read_hap, *reads))
        for p in products:
            _write_all([d("final_out", f"hap{hn}.{ext}") for ext in EVIDENCE_PRODUCTS[p].suffixes], texts[p](rec[p]))
    from concurrent.futures import ThreadPoolExecutor
    n_cpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    workers = max(1, min(8, n_cpu // 2))
    per_job = max(1, n_cpu // workers)
    jobs.sort(key=lambda j: -(len(j[2]["sel"]) if j[2].get("sel") is not None else len(j[1][0][1])))  # big files first
    with ThreadPoolExecutor(max_workers=workers) as ex:
        list(ex.map(lambda j: _write_bytes(j[0], gio.format_rows(j[1], threads=per_job, **j[2])), jobs))


def cmd_fused(argv):
    ap = argparse.ArgumentParser(prog="gavisunk_b200.cli fused")
    ap.add_argument("--sample", default="sample")
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--hap1-asm", required=True)
    ap.add_argument("--hap2-asm", required=True)
    ap.add_argument("--hap1-reads", nargs="+")
    ap.add_argument("--hap2-reads", nargs="+")
    ap.add_argument("--reads", nargs="+", help="chunk files of unbinned reads, instead of --hap1-reads / --hap2-reads: each read's "
                    "haplotype is assigned from its SUNK votes (implies --read-haplotypes)")
    ap.add_argument("--outdir", required=True)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--devices", default=None, help="comma-separated GPU indices: the chunk files are sharded over them")
    ap.add_argument("--batch-files", type=int, default=0, help="chunk files per batch (0 = by size, about --batch-gbp each)")
    ap.add_argument("--batch-gbp", type=float, default=12.0)
    ap.add_argument("--detailed", action="store_true", help="also write sunkpos/{hap}_detailed.sunkpos (plot_detailed: true)")
    ap.add_argument("--threads", type=int, default=0, help="ingest threads per GPU")
    ap.add_argument("--mrsfast-palindromes", action="store_true",
                    help="write a palindromic SUNK twice into kmer.loc, as mrsfast reports it on both strands (SURVEY A.2; unpinned)")
    for p, e in EVIDENCE_PRODUCTS.items():
        ap.add_argument(e.flag, dest=p, action="store_true", help=e.help)
    a = ap.parse_args(argv)
    binned = a.hap1_reads is not None or a.hap2_reads is not None
    if (a.reads is not None) == binned or (binned and (a.hap1_reads is None or a.hap2_reads is None)):
        ap.error("give either --reads or both --hap1-reads and --hap2-reads")
    devs = [int(x) for x in a.devices.split(",")] if a.devices else [a.device]
    run_fused(a.k, [a.hap1_asm, a.hap2_asm], [a.hap1_reads, a.hap2_reads] if binned else None, a.outdir, devices=devs,
              batch_files=a.batch_files, batch_gbp=a.batch_gbp, detailed=a.detailed, threads=a.threads,
              mrsfast_palindromes=a.mrsfast_palindromes, products=[p for p in EVIDENCE_PRODUCTS if getattr(a, p)],
              reads=a.reads or ())


COMMANDS = {"kmerpos_annot3": (cmd_kmerpos_annot3, 4), "rlen": (cmd_rlen, 2), "diag_filter_v3": (cmd_diag_filter_v3, 2),
            "diag_filter_step2": (cmd_diag_filter_step2, 2), "badsunks_AR": (cmd_badsunks, 5),
            "process_by_contig": (cmd_process_by_contig, None), "get_gaps": (cmd_get_gaps, 5), "slop_gaps": (cmd_slop_gaps, 3),
            "covprob": (cmd_covprob, None), "split_locs": (cmd_split_locs, None), "fused": (cmd_fused, None),
            "split_ont": (cmd_split_ont, None), "combine_ont_nofilt": (cmd_combine_ont_nofilt, None),
            "support_tracks": (cmd_support_tracks, 8), "gap_evidence": (cmd_gap_evidence, 7),
            "junctions": (cmd_junctions, 7), "discordance": (cmd_discordance, 7)}


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv or argv[0] not in COMMANDS:
        sys.stderr.write(__doc__)
        return 2
    fn, nargs = COMMANDS[argv[0]]
    if nargs is not None and len(argv) - 1 != nargs:
        sys.stderr.write(f"{argv[0]}: expected {nargs} arguments\n")
        return 2
    try:
        fn(argv[1:])
    except Exception as ex:  # non-zero exit + message, nothing partial written (SURVEY section 5)
        sys.stderr.write(f"gavisunk_b200 {argv[0]}: {type(ex).__name__}: {ex}\n")
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())

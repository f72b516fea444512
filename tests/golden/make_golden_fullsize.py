#!/usr/bin/env python
"""tests/golden/fullsize_sample.json.gz: the lines the reference's kmerpos_annot3 / diag_filter_v3 /
diag_filter_step2 write for the sample of tests/test_gpu_fullsize.py -- the first reads of one chunk file per
haplotype of BASELINE config 3, matched against the full 5.9 M-SUNK database.

The reads and the database come from the workload generator on the GPU (seeded, as in the test).  The database is
exported in full as jellyfish.db / kmer.loc, the sample's reads as one FASTA per haplotype, and the reference's
own executables (oracle/_ref, see oracle/Makefile) run on them through oracle/ref_runner.py, as the Snakemake rules
run them.  Their three output files are stored, with the sha256 of the sample's bases and of the kmer.loc lines of
the database rows the sample can hit.  As a cross-check, the GPU's lines and those of the oracle's restatement of
the three executables (oracle/gavisunk_oracle.py) are compared with them and the result printed.

--oracle stores the oracle's lines instead, for a machine without the executables; the file's "source" field says
which of the two wrote the stored lines.

  python tests/golden/make_golden_fullsize.py [--oracle] [OUT]     (needs a CUDA device; default OUT: tests/golden/fullsize_sample.json.gz)
"""
import argparse
import gzip
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import gavisunk_oracle as O  # noqa: E402
import ref_runner as RR  # noqa: E402
from gavisunk_b200 import cli  # noqa: E402
from gavisunk_b200 import io as gio  # noqa: E402
import test_gpu_fullsize as T  # noqa: E402

FILES = ("sunkpos", "diag", "diag2")


def oracle_texts(wl, db, sub, reads, hap):
    """the oracle's restatement of the three executables, given the database rows the reads can hit"""
    names = wl.contig_names
    nc = len(names) // 2
    loc = [(names[c], int(s), int(k), int(g)) for c, s, k, g in
           zip(db["contig"][sub], db["start"][sub], db["kmer"][sub], db["group"][sub])]
    rows = O.match_chunk(reads, db["kmer"][sub], loc, T.K)
    diag = O.diag_filter_v3(rows, set(names[hap * nc:(hap + 1) * nc]))
    return dict(sunkpos=gio.format_sunkpos(rows), diag="".join("\t".join(str(x) for x in d) + "\n" for d in diag),
                diag2=gio.format_sunkpos(O.diag_filter_step2(rows, diag)))


def write_db_files(wl, db, workdir):
    """jellyfish.db / kmer.loc of the whole exported database, in the formats the executables read"""
    import pandas as pd
    kmers = np.asarray(cli.decode_kmers(db["kmer"], T.K))
    names = np.asarray(wl.contig_names)
    dbp, locp = os.path.join(workdir, "jellyfish.db"), os.path.join(workdir, "kmer.loc")
    pd.DataFrame({"k": kmers}).to_csv(dbp, header=False, index=False)
    pd.DataFrame({"c": names[db["contig"]], "s": db["start"], "k": kmers, "g": db["group"]}).to_csv(
        locp, sep="\t", header=False, index=False)
    return dbp, locp


def reference_texts(wl, reads, hap, workdir, dbp, locp):
    """the reference's executables on the reads, with the whole database"""
    nc = len(wl.contig_names) // 2
    fa = os.path.join(workdir, f"hap{hap + 1}.fa")
    with open(fa, "wb") as f:
        for n, s in reads:
            f.write(b">" + n.encode() + b"\n" + s + b"\n")
    fai = os.path.join(workdir, f"hap{hap + 1}.fai")
    with open(fai, "w") as f:
        f.write("".join(f"{wl.contig_names[c]}\t{int(wl.contig_len[c])}\t0\t60\t61\n" for c in range(hap * nc, (hap + 1) * nc)))
    r = RR.run_chunk(workdir, f"hap{hap + 1}", fa, dbp, locp, fai)
    return {f: open(r[f]).read() for f in FILES}


def main(argv):
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default=os.path.join(HERE, "fullsize_sample.json.gz"))
    ap.add_argument("--oracle", action="store_true", help="store the oracle's lines (no reference executables here)")
    args = ap.parse_args(argv)
    if not args.oracle and not RR.available():
        print(f"the reference's executables are not in {RR.REF_DIR} (oracle/Makefile copies them there); "
              "--oracle stores the oracle's lines instead", file=sys.stderr)
        return 2
    eng, wl, res = T.build_full()
    db = eng.db_export()
    off = res["off"]
    sample, agree = [], True
    with tempfile.TemporaryDirectory(prefix="gvs_golden_") as workdir:
        dbp, locp = (None, None) if args.oracle else write_db_files(wl, db, workdir)
        for hap, chunk in T.SAMPLE_CHUNKS:
            assert wl.chunk_hap[chunk] == hap
            r0 = int(wl.chunk_first[chunk])
            r1 = r0 + T.SAMPLE_READS
            reads = T.sample_reads(wl, res, r0, r1)
            sub, loc_text = T.sample_loc(wl, db, reads)
            texts = dict(oracle=oracle_texts(wl, db, sub, reads, hap), gpu=T.sample_texts(wl, res, r0, r1))
            if not args.oracle:
                texts["reference"] = reference_texts(wl, reads, hap, workdir, dbp, locp)
            want = texts["oracle" if args.oracle else "reference"]
            for f in FILES:
                same = {who: t[f] == want[f] for who, t in texts.items()}
                print(f"hap {hap + 1} chunk {chunk} {f}: {len(want[f].splitlines())} lines; equal to the stored lines: {same}")
                agree &= all(same.values())
            sample.append(dict(hap=hap, chunk=chunk, first_read=r0, read_len=np.diff(off[r0:r1 + 1]).tolist(),
                               bases_sha256=T.bases_sha256(reads), loc_sha256=hashlib.sha256(loc_text.encode()).hexdigest(), **want))
    eng.close()
    source = ("oracle/gavisunk_oracle.py (match_chunk, diag_filter_v3, diag_filter_step2)" if args.oracle else
              "the reference's executables kmerpos_annot3, diag_filter_v3, diag_filter_step2 with the full database")
    with gzip.open(args.out, "wt") as f:
        json.dump(dict(k=T.K, source=source, sample=sample), f)
    print("wrote", args.out)
    return 0 if agree else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))

"""BASELINE.json configs 1 and 2 end to end: the reference's bundled samples (.test/config.yaml, .test/data/ont.tsv:2-3;
SUNK_len 20, 10 chunks) through `cli fused` and through the chain of per-rule shims, against what the reference's OWN
executables and Python scripts wrote for the same inputs (tests/golden/j1_*.json.gz, made by tests/golden/make_golden_j1.py
in the build container).  The reads are simulated (the real ONT files are missing from the snapshot) and regenerated here
from the committed assemblies; their digest is checked first.  README.md:36-37's known answer -- the gap
AMY_h1 284861-324275, figure name ..._84861_524275 -- is a row of the reference's own output and of ours."""
import gzip
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, load_golden
from gavisunk_b200 import cli, io as gio

sys.path.insert(0, GOLDEN)
import j1_sim as S  # noqa: E402

SAMPLES = ["j1_amy_pseudodip", "j1_amy_hg02723"]


def _materialise(case, tmp, gz_every=4):
    """assemblies + 10 chunk files per haplotype as split_ONT would leave them (FASTQ, quality '#'; some gzipped)"""
    K = case["k"]
    haps = [[(n, s.encode()) for n, s in h] for h in case["asm"]]
    asm_files, fai_files, chunk_files = [], [], [[], []]
    forbid = tuple(case["forbid"]) if case["forbid"] else None
    for hi in range(2):
        ap = tmp / f"hap{hi + 1}.fa"
        ap.write_bytes(b"".join(b">" + n.encode() + b"\n" + s + b"\n" for n, s in haps[hi]))
        asm_files.append(str(ap))
        fp = tmp / f"hap{hi + 1}.fa.fai"
        fp.write_text(case[f"fai{hi + 1}"])
        fai_files.append(str(fp))
        reads = S.simulate(haps[hi], case["lengths"][hi], case["seed"] + hi, f"h{hi + 1}r", forbid=forbid, skip=case["skip"])
        assert S.digest(reads) == case["reads_sha"][hi], "the simulator no longer reproduces the reads the golden outputs belong to"
        for ci, part in enumerate(S.split_round_robin(reads, case["nchunks"])):
            txt = S.fastq_text(part)
            if ci % gz_every == 1:
                p = tmp / f"hap{hi + 1}_{ci + 1}-of-{case['nchunks']}.fq.gz"
                p.write_bytes(gzip.compress(txt, compresslevel=1))
            else:
                p = tmp / f"hap{hi + 1}_{ci + 1}-of-{case['nchunks']}.fq"
                p.write_bytes(txt)
            chunk_files[hi].append(str(p))
    return asm_files, fai_files, chunk_files


def _sha(text):
    import hashlib
    return hashlib.sha256(text.encode()).hexdigest()


@pytest.fixture(scope="module", params=SAMPLES)
def j1(request, tmp_path_factory):
    case = load_golden(request.param)
    tmp = tmp_path_factory.mktemp(request.param)
    asm_files, fai_files, chunk_files = _materialise(case, tmp)
    return dict(name=request.param, case=case, tmp=tmp, asm=asm_files, fai=fai_files, chunks=chunk_files)


def _check_final(case, rd):
    """files of results/{sample}/ against the reference's (rd(*path) -> text)"""
    assert set(rd("sunkpos", "bad_sunks.txt").split()) == set(case["bad_sunks"])
    for hn in ("1", "2"):
        assert rd("sunkpos", f"hap{hn}.sunkpos") == case["hap"][hn]["sunkpos"]
        assert rd("sunkpos", f"hap{hn}.rlen") == case["hap"][hn]["rlen"]
        fo = case["final_out"]
        assert sorted(rd("final_out", f"hap{hn}.valid.bed").splitlines()) == sorted(fo[f"hap{hn}.valid.bed"].splitlines())  # Q18
        for f in ("gaps.bed", "nodata.bed", "gaps.slop.bed"):
            assert rd("final_out", f"hap{hn}.{f}") == (fo[f"hap{hn}.{f}"] or ""), f
    for stem, txt in case["breaks"].items():
        assert rd("breaks", stem) == txt, stem
    for stem, txt in case["inter_outs"].items():
        assert rd("inter_outs", stem + ".tsv") == txt, stem
    for stem, txt in case["bed_files"].items():
        assert rd("bed_files", stem + ".bed") == (txt or ""), stem  # None: the rule's `touch` leaves it empty


@pytest.mark.gpu
@pytest.mark.parametrize("batch_files", [0, 7])
def test_fused_equals_reference_outputs(j1, batch_files):
    case, tmp = j1["case"], j1["tmp"]
    outdir = tmp / f"results_b{batch_files}"
    argv = ["fused", "--k", str(case["k"]), "--hap1-asm", j1["asm"][0], "--hap2-asm", j1["asm"][1], "--hap1-reads", *j1["chunks"][0],
            "--hap2-reads", *j1["chunks"][1], "--outdir", str(outdir), "--detailed", "--batch-files", str(batch_files)]
    assert cli.main(argv) == 0
    rd = lambda *p: open(os.path.join(outdir, *p)).read()
    # the SUNK database is the one the reference run used (kmer.loc byte for byte; jellyfish.db is in hash order there)
    assert _sha(rd("mrsfast", "kmer.loc")) == case["loc_sha"]
    _check_final(case, rd)
    for hn in ("1", "2"):  # combine_ont_nofilt (tagONT.smk:39-55)
        det = rd("sunkpos", f"hap{hn}_detailed.sunkpos")
        assert det.count("\n") == case["detailed"][hn]["rows"] and _sha(det) == case["detailed"][hn]["sha"]
    if j1["name"] == "j1_amy_hg02723":  # README.md:36-37
        assert "AMY_h1\t284861\t324275\n" in rd("final_out", "hap1.gaps.bed")
        assert "AMY_h1\t84861\t524275\n" in rd("final_out", "hap1.gaps.slop.bed")
    # covprob rule on the fused outputs (float64, 1e-6 relative)
    for hn in ("1", "2"):
        want = case["final_out"][f"hap{hn}.gaps.covprob.tsv"]
        tsv = outdir / "final_out" / f"hap{hn}.gaps.covprob.tsv"
        rc = cli.main(["covprob", "--bed", str(outdir / "final_out" / f"hap{hn}.gaps.bed"), "--locs", str(outdir / "mrsfast" / "kmer.loc"),
                       "--rlen", str(outdir / "sunkpos" / f"hap{hn}.rlen"), "--fai", j1["fai"][int(hn) - 1], "--sunk-len", str(case["k"]),
                       "--tsv", str(tsv)])
        assert (rc == 0) == (case["final_out"][f"hap{hn}.covprob_rc"] == 0)
        if rc == 0:
            got, exp = tsv.read_text().splitlines(), want.splitlines()
            assert len(got) == len(exp) and got[0] == exp[0]
            for g, e in zip(got[1:], exp[1:]):
                g, e = g.split("\t"), e.split("\t")
                assert g[:6] == e[:6]
                assert float(g[6]) == pytest.approx(float(e[6]), rel=1e-6, abs=1e-15)


@pytest.mark.gpu
def test_rule_chain_equals_reference_outputs(j1):
    """the per-rule shims chained through files as workflow/rules/tagONT.smk chains the reference programs: SUNK_annot,
    read_lengths, diag_filter_step / _final per chunk, combine_ont, bad_sunks, split_sunkpos, process_by_contig,
    get_gaps, slop_gaps"""
    import io
    from contextlib import redirect_stdout
    case, tmp = j1["case"], j1["tmp"]
    work = tmp / "rules"
    for sub in ("db", "mrsfast", "sunkpos", "breaks", "inter_outs", "bed_files", "final_out"):
        os.makedirs(work / sub, exist_ok=True)
    src = tmp / "results_b0"  # the database files of the fused run (kmer.loc checked there against the reference run's)
    if not (src / "mrsfast" / "kmer.loc").exists():
        pytest.skip("needs test_fused_equals_reference_outputs[0] of the same sample")
    db_p, loc_p = str(src / "db" / "jellyfish.db"), str(src / "mrsfast" / "kmer.loc")
    for hi in range(2):
        parts, rl = [], []
        for ci, reads_p in enumerate(j1["chunks"][hi]):
            sp = work / "sunkpos" / f"hap{hi + 1}_{ci}.sunkpos"
            assert cli.main(["kmerpos_annot3", reads_p, db_p, loc_p, str(sp)]) == 0
            assert cli.main(["rlen", reads_p, str(work / "sunkpos" / f"hap{hi + 1}_{ci}.rlen")]) == 0
            buf = io.StringIO()
            with redirect_stdout(buf):
                assert cli.main(["diag_filter_v3", str(sp), j1["fai"][hi]]) == 0
            dp = work / "sunkpos" / f"hap{hi + 1}_{ci}_diag.sunkpos"
            dp.write_text(buf.getvalue())
            buf = io.StringIO()
            with redirect_stdout(buf):
                assert cli.main(["diag_filter_step2", str(sp), str(dp)]) == 0
            parts.append(buf.getvalue())
            rl.append((work / "sunkpos" / f"hap{hi + 1}_{ci}.rlen").read_text())
        (work / "sunkpos" / f"hap{hi + 1}.sunkpos").write_text("".join(parts))  # combine_ont: cat in scatter order
        (work / "sunkpos" / f"hap{hi + 1}.rlen").write_text("".join(rl))
        assert cli.main(["combine_ont_nofilt", *[str(work / "sunkpos" / f"hap{hi + 1}_{ci}.sunkpos") for ci in range(len(j1["chunks"][hi]))],
                         str(work / "sunkpos" / f"hap{hi + 1}_detailed.sunkpos")]) == 0
        det = (work / "sunkpos" / f"hap{hi + 1}_detailed.sunkpos").read_text()
        assert _sha(det) == case["detailed"][str(hi + 1)]["sha"]
    assert cli.main(["badsunks_AR", j1["fai"][0], j1["fai"][1], str(work / "sunkpos" / "hap1.sunkpos"), str(work / "sunkpos" / "hap2.sunkpos"),
                     str(work / "sunkpos" / "bad_sunks.txt")]) == 0
    for hn in (1, 2):
        flag = work / "breaks" / f"hap{hn}_splits_pos.done"
        assert cli.main(["split_locs", "--ont-pos", str(work / "sunkpos" / f"hap{hn}.sunkpos"), "--kmer-loc", loc_p, "--flag", str(flag),
                         "--hap", f"hap{hn}"]) == 0
        for fn in sorted(os.listdir(work / "breaks")):
            if not fn.endswith(f"_hap{hn}.sunkpos"):
                continue
            stem = fn[:-len(".sunkpos")]
            tsv, bed = work / "inter_outs" / f"{stem}.tsv", work / "bed_files" / f"{stem}.bed"
            assert cli.main(["process_by_contig", str(work / "breaks" / f"{stem}.loc"), str(work / "breaks" / fn),
                             str(work / "sunkpos" / f"hap{hn}.rlen"), str(work / "sunkpos" / "bad_sunks.txt"), str(tsv), str(bed)]) == 0
            if not bed.exists():
                bed.write_text("")  # `touch {output.bed}` (tagONT.smk:190)
    assert cli.main(["get_gaps", j1["fai"][0], j1["fai"][1], "sample", str(work / "bed_files") + "/", str(work / "final_out") + "/"]) == 0
    for hn in (1, 2):
        assert cli.main(["slop_gaps", str(work / "final_out" / f"hap{hn}.gaps.bed"), j1["fai"][hn - 1],
                         str(work / "final_out" / f"hap{hn}.gaps.slop.bed")]) == 0
        beds = "".join(open(work / "bed_files" / f).read() for f in sorted(os.listdir(work / "bed_files")) if f.endswith(f"_hap{hn}.bed"))
        (work / "final_out" / f"hap{hn}.valid.bed").write_text(beds)  # gather_process_by_contig: cat
    _check_final(case, lambda *p: open(os.path.join(work, *p)).read())


def test_oracle_python_stages_on_the_bundled_samples():
    """the oracle's restatement of badsunks / process-by-contig / get_gaps on the reference's own sunkpos rows of
    configs 1-2 equals the reference's Python scripts' outputs (no GPU), and the README's known answer is among them"""
    import gavisunk_oracle as O
    for name in SAMPLES:
        case = load_golden(name)
        rows = {h: gio.parse_sunkpos(case["hap"][h]["sunkpos"]) for h in ("1", "2")}
        fai = {h: [(l.split("\t")[0], int(l.split("\t")[1])) for l in case[f"fai{h}"].splitlines()] for h in ("1", "2")}
        bad = O.bad_sunks(rows["1"], {n for n, _ in fai["1"]}, rows["2"], {n for n, _ in fai["2"]})
        assert {f"{c}:{g}" for c, g in bad} == set(case["bad_sunks"])
        for h in ("1", "2"):
            rlen = {l.split("\t")[0]: int(l.split("\t")[1]) for l in case["hap"][h]["rlen"].splitlines()}
            byc, beds = {}, {}
            for r in rows[h]:
                byc.setdefault(r[2], []).append(r)
            for ctg, rr in byc.items():
                inter, bed = O.process_by_contig(rr, rlen, bad, ctg)
                stem = f"{ctg}_hap{h}"
                want = case["inter_outs"][stem]
                assert ("".join(f"{g}\t{n}\n" for g, n in inter) if inter else ctg + "\n") == want, stem
                assert "".join(f"{c}\t{s}\t{e}\n" for c, s, e in (bed or [])) == (case["bed_files"][stem] or ""), stem
                if bed is not None:
                    beds[ctg] = [(s, e) for _, s, e in bed]
            gaps, nodata = O.get_gaps(fai[h], beds)
            assert "".join(f"{c}\t{s}\t{e}\n" for c, s, e in gaps) == (case["final_out"][f"hap{h}.gaps.bed"] or "")
            assert "".join(f"{c}\t{s}\t{e}\n" for c, s, e in nodata) == (case["final_out"][f"hap{h}.nodata.bed"] or "")
    hg = load_golden("j1_amy_hg02723")["final_out"]
    assert "AMY_h1\t284861\t324275\n" in hg["hap1.gaps.bed"] and "AMY_h1\t84861\t524275\n" in hg["hap1.gaps.slop.bed"]


def test_simulated_reads_are_reproducible():
    case = load_golden("j1_amy_hg02723")
    haps = [[(n, s.encode()) for n, s in h] for h in case["asm"]]
    reads = S.simulate(haps[1], case["lengths"][1], case["seed"] + 1, "h2r", forbid=tuple(case["forbid"]), skip=case["skip"])
    assert S.digest(reads) == case["reads_sha"][1]
    # no simulated read of haplotype 1 may span the desert; spot-check the generator's own rule on a few lengths
    r1 = S.simulate(haps[0], case["lengths"][0][:40], case["seed"], "h1r", forbid=tuple(case["forbid"]), skip=case["skip"])
    assert len(r1) == 40 and all(len(s) > 0 for _, s in r1)


@pytest.mark.gpu
def test_fused_on_two_contexts_equals_reference_outputs(j1):
    """`--devices 0,0`: two contexts (one host thread each) share the chunk files of the sample and exchange the
    histogram and the forests inside the process (parallel.ThreadExchange) -- the multi-GPU path of the fused rule; the
    files are the reference's, byte for byte"""
    case, tmp = j1["case"], j1["tmp"]
    outdir = tmp / "results_2ctx"
    argv = ["fused", "--k", str(case["k"]), "--hap1-asm", j1["asm"][0], "--hap2-asm", j1["asm"][1], "--hap1-reads", *j1["chunks"][0],
            "--hap2-reads", *j1["chunks"][1], "--outdir", str(outdir), "--devices", "0,0", "--batch-files", "3"]
    assert cli.main(argv) == 0
    rd = lambda *p: open(os.path.join(outdir, *p)).read()
    assert _sha(rd("mrsfast", "kmer.loc")) == case["loc_sha"]
    _check_final(case, rd)


@pytest.mark.gpu
def test_split_ont_then_fused_equals_reference_outputs(j1):
    """split_ONT emulation (cli split_ont: FASTQ with '#' qualities, round-robin over 10 outputs, gzip) on the whole
    read set of each haplotype, then the fused rule: the chunk files hold the same records as the reference run's, so
    every output is the reference's (parity of the split itself is unpinned: seqtk / rustybam are absent)"""
    case, tmp = j1["case"], j1["tmp"]
    haps = [[(n, s.encode()) for n, s in h] for h in case["asm"]]
    forbid = tuple(case["forbid"]) if case["forbid"] else None
    chunks = [[], []]
    for hi in range(2):
        reads = S.simulate(haps[hi], case["lengths"][hi], case["seed"] + hi, f"h{hi + 1}r", forbid=forbid, skip=case["skip"])
        whole = tmp / f"hap{hi + 1}.ONT.fa.gz"
        whole.write_bytes(gzip.compress(b"".join(b">" + n.encode() + b" some comment\n" + s + b"\n" for n, s in reads), compresslevel=1))
        outs = [str(tmp / f"split_hap{hi + 1}_{i + 1}-of-{case['nchunks']}.fq.gz") for i in range(case["nchunks"])]
        assert cli.main(["split_ont", "--reads", str(whole), "--out", *outs]) == 0
        chunks[hi] = outs
        first = gio.read_fastx(outs[0])
        assert [n for n, _ in first] == [n for n, _ in reads[0::case["nchunks"]]]
        assert gzip.open(outs[1]).read().split(b"\n")[3] == b"#" * len(reads[1][1])
    outdir = tmp / "results_split"
    assert cli.main(["fused", "--k", str(case["k"]), "--hap1-asm", j1["asm"][0], "--hap2-asm", j1["asm"][1], "--hap1-reads", *chunks[0],
                     "--hap2-reads", *chunks[1], "--outdir", str(outdir)]) == 0
    _check_final(case, lambda *p: open(os.path.join(outdir, *p)).read())

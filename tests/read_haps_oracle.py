"""CPU restatement of the read haplotypes (test infrastructure; no reference counterpart, DESIGN.md section 5.5e).

From the definition in include/gavisunk_b200.h: the oracle's diag_filter_v3 is run over each chunk once with each
haplotype's contig set, and the two outputs give the votes, the assignment, the kept rows and the file haplotype.  No
logic is shared with the device code or with gavisunk_b200.cli."""
import gavisunk_oracle as G

ANY = 2  # GVS_HAP_ANY: a chunk of unbinned reads


def chunk_votes(rows, hap_contigs):
    """rows: (read, pos, contig, start, group) of ONE chunk in file order; hap_contigs: the two haplotypes' contig sets ->
    {read: [vote_0, vote_1]}, vote = (contig, n, dir) or None, for every read with rows"""
    out = {r[0]: [None, None] for r in rows}
    for h in range(2):
        for r, c, n, d, _ in G.diag_filter_v3(rows, hap_contigs[h]):
            out[r][h] = (c, n, d)
    return out


def n_of(v):
    return v[1] if v else 0


def assign(votes):
    """0 / 1, 'tie' (n_0 == n_1 >= 2) or None (no vote on either)"""
    n0, n1 = n_of(votes[0]), n_of(votes[1])
    if n0 > n1:
        return 0
    if n1 > n0:
        return 1
    return "tie" if n0 else None


def read_haps(chunks, hap_contigs):
    """chunks: [(chunk haplotype 0 / 1 / ANY, rows)] in run order, read names unique across the run.
    -> dict with
         records  [(read, vote_0, vote_1, assigned)] of the reads with a vote on either haplotype, in run order;
         kept     the rows the diag filter keeps, in run order (binned: the chunk haplotype's vote, unbinned: the
                  assigned haplotype's, tie / none: nothing);
         assigned {read: assign()} of every read with rows."""
    records, kept, assigned = [], [], {}
    for ch_hap, rows in chunks:
        votes = chunk_votes(rows, hap_contigs)
        best = []
        for r, v in votes.items():  # dict order = first-row order = read order
            a = assign(v)
            if v[0] or v[1]:
                records.append((r, v[0], v[1], a))
            k = ch_hap if ch_hap != ANY else (a if a in (0, 1) else None)
            assigned[r] = a
            if k is not None and v[k]:
                best.append((r, v[k][0]))
        kept += G.diag_filter_step2(rows, best)
    return dict(records=records, kept=kept, assigned=assigned)


def file_haps(read_names, read_bin, assigned):
    """read_names / read_bin: every read of the run in run-wide index order and its chunk haplotype; assigned: read ->
    assignment (read_haps()["assigned"]; reads without rows are absent) -> file haplotype per read: the chunk's when
    binned, the assigned one when unbinned, else the parity of the run-wide index (even: 0)"""
    out = []
    for i, (r, b) in enumerate(zip(read_names, read_bin)):
        a = assigned.get(r)
        out.append(b if b != ANY else (a if a in (0, 1) else i & 1))
    return out

"""CPU restatement of the support tracks (test infrastructure; no reference counterpart, DESIGN.md section 5.5a).

Placements come from the oracle's own process_by_contig (the validated IDs of every read, exactly as inter_outs holds
them); the strand is the orientation majority of the read's rows (process-by-contig_lowmem_AR.py:140-152); the depth is
a difference array over the coordinates -- no logic shared with the device algorithm, which works on group ranks."""
import os
import sys
from collections import OrderedDict, defaultdict

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
import gavisunk_oracle as O  # noqa: E402


def support_depth(placements, fai):
    """placements: (contig, start, end, ...) tuples; fai: [(contig, length)] in .fai order.  Depth at base x = number of
    placements of the contig with start <= x < end.  -> runs [(contig, start, end, depth)] tiling every contig, maximal
    (adjacent runs of a contig differ in depth)."""
    by_c = defaultdict(list)
    for p in placements:
        by_c[p[0]].append((int(p[1]), int(p[2])))
    runs = []
    for c, L in fai:
        d = np.zeros(L + 1, np.int64)
        for a, b in by_c.get(c, []):
            d[a] += 1
            d[b] -= 1
        depth = np.cumsum(d[:L])
        starts = np.concatenate([[0], np.flatnonzero(np.diff(depth)) + 1]).astype(np.int64)
        ends = np.append(starts[1:], L)
        runs.extend((c, int(a), int(b), int(depth[a])) for a, b in zip(starts, ends))
    return runs


def _orientation(rows):
    """majority sign of the pairs that pass the ratio test, rows = distinct (pos, start) of one read sorted by start;
    a tie is 0 (np.unique + argmax, :151-152)"""
    n = [0, 0]
    for i in range(len(rows)):
        pi, si = rows[i]
        for j in range(i + 1, len(rows)):
            pj, sj = rows[j]
            ds, dp = abs(si - sj), abs(pi - pj)
            if 9 * ds < 10 * dp < 11 * ds:  # 0.9 < dpos/dstart < 1.1 (:145-147, Q12)
                n[1 if pi > pj else 0] += 1
    return 1 if n[1] > n[0] else 0


def support_tracks(rows, rlen, bad, fai, minlen=10000):
    """rows: (read, pos, contig, start, ID) of one haplotype, rlen / bad / minlen as O.process_by_contig, fai: [(contig,
    length)].  A placement is a read with >= 2 distinct validated IDs on a contig: (contig, min ID, max ID, read,
    n distinct IDs, '+' when the orientation majority is 0 else '-').
    -> (placements sorted by (.fai order, start, end, read name), support_depth runs)"""
    order = {c: i for i, (c, _) in enumerate(fai)}
    by_c = OrderedDict()
    for r in rows:
        by_c.setdefault(r[2], []).append(r)
    pls = []
    for contig, rs in by_c.items():
        inter, _ = O.process_by_contig(rs, rlen, bad, contig, minlen)
        ids = OrderedDict()
        for i, rname in inter or []:
            ids.setdefault(rname, set()).add(int(i))
        for rname, v in ids.items():
            if len(v) < 2:
                continue
            own = sorted({(int(r[1]), int(r[3])) for r in rs if r[0] == rname and (r[2], int(r[4])) not in bad}, key=lambda t: t[1])
            pls.append((contig, min(v), max(v), rname, len(v), "-" if _orientation(own) else "+"))
    pls.sort(key=lambda p: (order[p[0]], p[1], p[2], p[3].encode()))
    return pls, support_depth(pls, fai)

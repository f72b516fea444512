"""The GPU SUNK database build (csrc/dbbuild.cu k_db_count / k_db_mark / k_db_rows, then table.cu k_tab_finalize)
against gavisunk_oracle.build_sunk_db at the shapes where it can go wrong: every SUNK_len from 1 to 32, contig
boundaries on the 4096-base tiles and 16-byte loads of the count kernel, bytes outside ACGT, group heads that reach
into the previous word of the SUNK bitmap, tandem repeats and palindromes, empty and SUNK-less assemblies, forced
hash-partitioned passes and rebuilds on one engine.  Then the match over databases this code built against
gavisunk_oracle.match_chunk at every k, and hit-dense batches that overflow the first hit buffer of a context."""
import numpy as np
import pytest

import gavisunk_oracle as O

pytestmark = pytest.mark.gpu

DTILE = 4096  # bases per tile of k_db_count
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = bytes.maketrans(b"ACGTacgtN", b"TGCAtgcaN")


def _rand(rng, n, alphabet=ACGT):
    return alphabet[rng.integers(0, len(alphabet), n)].tobytes()


def _rc(s):
    return s.translate(_COMP)[::-1]


def _snps(rng, s, rate):
    b = np.frombuffer(s, dtype=np.uint8).copy()
    m = rng.random(len(b)) < rate
    b[m] = ACGT[(np.searchsorted(ACGT, b[m]) + rng.integers(1, 4, int(m.sum()))) % 4]
    return b.tobytes()


def _split(rng, s, n, prefix):
    cuts = sorted(int(x) for x in rng.integers(0, len(s) + 1, n - 1))
    b = [0] + cuts + [len(s)]
    return [(f"{prefix}{i}", s[b[i]:b[i + 1]]) for i in range(n)]


def _windows(contigs, k):
    """canonical values of every valid window (only ACGT/acgt, inside one contig), as jellyfish counts them"""
    ws = [np.zeros(0, np.uint64)]
    for _, s in contigs:
        b = np.frombuffer(s, dtype=np.uint8)
        n = len(b) - k + 1
        if n <= 0:
            continue
        bad = np.concatenate([[0], np.cumsum(~O._ACGT_VALID[b])])
        ws.append(O.canonical_windows(O.BASE_LUT[b], k)[(bad[k:k + n] - bad[:n]) == 0])
    return np.concatenate(ws)


def _n_groups(db):
    return len(np.unique(db["contig"].astype(np.int64) << 32 | db["group"]))


def _has_repeat(contigs, k):
    _, c = np.unique(_windows(contigs, k), return_counts=True)
    return bool((c > 1).any())


# ---- assemblies ------------------------------------------------------------------------------------------------------
def _b1_contigs(k, seed):
    """two haplotypes sized to the k-mer space (a few times 4^k / 8 bases up to k = 7, 240 kb above), a duplication
    inside a hap-1 contig, hap 2 = hap 1 with SNPs and a reverse-complemented copy of a hap-1 segment; the first seed
    whose database has more than one group (k = 1: one) and at least one repeated k-mer"""
    for attempt in range(200):
        rng = np.random.default_rng(seed * 1000 + attempt)
        n1 = max(4 ** k // 4, 24) if k <= 7 else 120_000
        h1 = bytearray(_rand(rng, n1, np.frombuffer(b"AT", np.uint8) if k == 1 else ACGT))
        if k == 1:
            h1[int(rng.integers(0, n1))] = ord("C")
        d = max(k + 2, n1 // 16)
        a = int(rng.integers(0, n1 - 2 * d))
        b = int(rng.integers(a + d, n1 - d + 1))
        h1[b:b + d] = h1[a:a + d]
        h1 = bytes(h1)
        h2 = _snps(rng, h1, 0.02 if k > 7 else 0.25) if k > 1 else _rand(rng, n1, np.frombuffer(b"AT", np.uint8))
        if k > 7:
            c = int(rng.integers(0, n1 - 3000))
            h2 = h2[:n1 // 2] + _rc(h1[c:c + 3000]) + h2[n1 // 2:]
        contigs = _split(rng, h1, 3, "h1_") + _split(rng, h2, 2, "h2_")
        db = O.build_sunk_db(contigs, k)
        if _n_groups(db) >= (1 if k == 1 else 2) and _has_repeat(contigs, k):
            return contigs
    raise AssertionError(f"no non-vacuous assembly at k={k}")


def _tile_edges_contigs(k, seed):
    """contig boundaries at tile starts + {-k, -(k-1), -1, 0, +1, k-2, k-1, k}; more than 256 boundaries (contigs of
    length 0, 1, k-1, k, k+1) inside one tile; leading and trailing empty contigs; a final tile of 1..15 bytes"""
    rng = np.random.default_rng(seed)
    deltas = [-k, -(k - 1), -1, 0, 1, k - 2, k - 1, k]
    bounds = [DTILE * (m + 1) + d for m, d in enumerate(deltas)]
    t0 = DTILE * (len(deltas) + 1) + 5
    cyc = [0, 1, k - 1, k, k + 1, 0, 1, 0]
    pos, i = t0, 0
    while pos + k + 1 < t0 + DTILE - 8:
        pos += cyc[i % len(cyc)]
        bounds.append(pos)
        i += 1
    total = DTILE * (len(deltas) + 3) + 1 + (k + seed) % 15
    seq = bytearray(_rand(rng, total))
    seg = max(k + 2, 700)
    seq[total - seg - 3:total - 3] = seq[100:100 + seg]  # repeats that end in the last tile
    seq[DTILE * 3 - 300:DTILE * 3 + 300] = seq[DTILE * 7 - 300:DTILE * 7 + 300]  # and straddle tile starts
    seq = bytes(seq)
    b = [0, 0] + bounds + [total, total, total]
    contigs = [(f"c{j}", seq[b[j]:b[j + 1]]) for j in range(len(b) - 1)]
    per_tile = np.bincount(np.asarray(bounds) // DTILE)
    assert per_tile.max() > 256 and total % DTILE in range(1, 16)
    return contigs


def _bytes_contigs(k, seed):
    """N runs that start and end on tile and 16-byte boundaries, lower case, and every byte value: only ACGT/acgt
    are bases of the database (U/u and 0x01-0x03, which the probe reads as bases, break windows here)"""
    rng = np.random.default_rng(seed)
    n = 3 * DTILE + 77
    s = bytearray(_rand(rng, n))
    for a, b in ((DTILE, DTILE + 32), (2 * DTILE - 48, 2 * DTILE), (80, 96), (2 * DTILE + 16, 2 * DTILE + 17),
                 (3 * DTILE - 1, 3 * DTILE + 16)):
        s[a:b] = b"N" * (b - a)
    s[500:1300] = s[500:1300].lower()
    low = rng.random(n) < 0.1
    s = bytearray(bytes(c | 0x20 if l and c != ord("N") else c for c, l in zip(s, low)))
    vals = list(range(256))
    rng.shuffle(vals)
    for j, v in enumerate(vals):  # one byte of every value, at least k + 3 apart
        s[40 + j * (k + 3) % (n - 80)] = v
    h1 = bytes(s)
    h2 = _snps(rng, h1[:DTILE + 500].upper().replace(b"N", b"A"), 0.03) + b"uUuU" + h1[DTILE + 500:DTILE + 1500].lower()
    contigs = [("h1_0", h1[:2 * DTILE + 3]), ("h1_1", h1[2 * DTILE + 3:]), ("h2_0", h2)]
    assert set(h1) == set(range(256))
    return contigs


def _heads_contigs(k, seed):
    """SUNKs placed one by one in an N background: pairs exactly k apart (book-ended: one group) and k+1 apart (two
    groups) whose earlier SUNK lies at every offset of the previous 32-bit bitmap word that the pair can straddle,
    chains of book-ended SUNKs over many words, and pairs k apart across a contig boundary inside one word (two
    groups).  Every window between the planted SUNKs also occurs in a decoy, so it is not a SUNK.
    Returns (contigs, planted, same, split): planted SUNK positions per contig, pairs of (contig, position) that must
    share a group and pairs that must not."""
    rng = np.random.default_rng(seed)
    L = 64 * 32 * (k + 8)
    main = bytearray(b"N" * L)
    decoys = []
    planted, same, split = set(), [], []

    def put(p, units, gap):
        s = b""
        starts = []
        for j, u in enumerate(units):
            if j:
                s += gap
            starts.append(p + len(s))
            s += u
        main[p:p + len(s)] = s
        for j in range(len(units) - 1):
            a, b = starts[j] - p, starts[j + 1] - p + k
            decoys.append(s[a + 1:b - 1])  # every window that straddles the junction, and neither unit
        planted.update(starts)
        return starts

    w = 1
    for j in range(min(k, 32)):
        for g in (0, 1):  # earlier SUNK at bit 31 - j of word w, the later one k (+1) on
            p = 32 * w + 31 - j
            st = put(p, [_rand(rng, k), _rand(rng, k)], _rand(rng, g))
            (same if g == 0 else split).append(((0, st[0]), (0, st[1])))
            w += (2 * k + 40) // 32 + 1
    for n_units in (12, 40):
        st = put(32 * w + int(rng.integers(0, 32)), [_rand(rng, k) for _ in range(n_units)], b"")
        same += [((0, st[0]), (0, x)) for x in st[1:]]
        w += (n_units * k + 40) // 32 + 1
    assert 32 * w + 64 < L
    contigs = [("h1_0", bytes(main))]
    # across contig boundaries: contig A ends with a SUNK, contig B (after 0 or 1 empty contigs) starts with one
    for empties in (0, 1, 0):
        g0 = sum(len(c) for _, c in contigs)  # A's SUNK at bit 0 of a word, B's k bases on (same word below k = 32)
        a = b"N" * (32 * int(rng.integers(1, 4)) + (-g0) % 32) + _rand(rng, k)
        ci = len(contigs)
        planted_a = (ci, len(a) - k)
        contigs.append((f"x{ci}", a))
        contigs += [(f"e{ci}_{e}", b"") for e in range(empties)]
        cb = len(contigs)
        contigs.append((f"x{cb}", _rand(rng, k) + b"N" * int(rng.integers(0, 40))))
        split.append((planted_a, (cb, 0)))
    dec = b"N".join(decoys)
    contigs.append(("h2_0", b"N" + dec + b"N"))
    return contigs, planted, same, split


def _repeats_contigs(k, seed):
    """homopolymers and period-2/3 tandem runs (one thread's 16 windows insert the same k-mer several times), and at
    even k palindromic k-mers that occur once (a SUNK) and twice (not a SUNK).  Returns (contigs, once, twice):
    positions in contig 0 of the palindromes."""
    rng = np.random.default_rng(seed)
    parts = [_rand(rng, 3000)]
    for run in (b"A" * (3 * k + 17), b"C" * (2 * k + 5), b"g" * (k + 1), b"AC" * (2 * k + 9), b"GT" * (k + 3),
                b"ACG" * (2 * k + 11), b"tta" * (k + 2), b"T" * 40):
        parts += [run, _rand(rng, 200)]
    once, twice = [], []
    s = b"".join(parts)
    if k % 2 == 0:
        p1 = _rand(rng, k // 2)
        p1 += _rc(p1)
        p2 = _rand(rng, k // 2)
        p2 += _rc(p2)
        s += b"N"
        once.append(len(s))
        s += p1 + b"N" + _rand(rng, 300) + b"N"
        twice.append(len(s))
        s += p2 + b"N" + _rand(rng, 100) + b"N"
        twice.append(len(s))
        s += p2 + b"N"
    h2 = _snps(rng, s[:3000], 0.02) + b"A" * (2 * k) + b"CA" * (3 * k)
    return [("h1_0", s), ("h2_0", h2)], once, twice


# ---- build and compare ---------------------------------------------------------------------------------------------
def _build(eng, contigs, device):
    if not device:
        eng.build_db(contigs)
        return
    import torch
    seq = b"".join(s for _, s in contigs)
    buf = torch.zeros(len(seq) + 16, dtype=torch.uint8, device="cuda")  # the caching allocator aligns to 512 bytes
    if seq:
        buf[:len(seq)].copy_(torch.frombuffer(bytearray(seq), dtype=torch.uint8))
    off = np.zeros(len(contigs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(s) for _, s in contigs])
    doff = torch.from_numpy(off).cuda()
    assert buf.data_ptr() % 16 == 0
    torch.cuda.synchronize()
    eng.build_db_device(buf.data_ptr(), doff.data_ptr(), [n for n, _ in contigs])


def _check_db(eng, contigs, k, exp=None):
    """every column of the export against the oracle: kmer, contig, start, group and the dense group index in
    (contig, group) order"""
    exp = O.build_sunk_db(contigs, k) if exp is None else exp
    got = eng.db_export()
    assert len(got["kmer"]) == len(exp["kmer"])
    assert np.array_equal(got["contig"].astype(np.int64), exp["contig"].astype(np.int64))
    assert np.array_equal(got["start"].astype(np.int64), exp["start"])
    assert np.array_equal(got["kmer"], exp["kmer"])
    assert np.array_equal(got["group"].astype(np.int64), exp["group"])
    key = exp["contig"].astype(np.int64) << 32 | exp["group"]
    _, inv = np.unique(key, return_inverse=True)
    assert np.array_equal(got["gidx"].astype(np.int64), inv)
    assert eng.db_size() == (len(exp["kmer"]), _n_groups(exp))
    return got


def _check_both(k, contigs, passes=0, exp=None):
    """build on the host and from a 16-byte-aligned device buffer: both equal to the oracle"""
    from gavisunk_b200.engine import Engine
    exp = O.build_sunk_db(contigs, k) if exp is None else exp
    eng = Engine(k)
    if passes:
        eng.set_db_passes(passes)
    out = []
    for device in (False, True):
        _build(eng, contigs, device)
        out.append(_check_db(eng, contigs, k, exp))
    eng.close()
    return exp, out[0]


# ---- B1: every k ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", range(1, 33))
def test_db_every_k(k):
    contigs = _b1_contigs(k, 100 + k)
    exp, _ = _check_both(k, contigs)
    assert len(exp["kmer"]) >= 1  # k = 32 included: jellyfish counts 32-mers, and so does the build


# ---- B2: tiles and 16-byte loads -----------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 8, 11, 16, 20, 31, 32])
def test_db_tile_edges(k):
    contigs = _tile_edges_contigs(k, 7 * k)
    exp, _ = _check_both(k, contigs)
    if k >= 11:
        assert len(exp["kmer"]) > 10000


# ---- B3: bytes -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [8, 9, 11, 16, 20, 31, 32])
def test_db_bytes(k):
    contigs = _bytes_contigs(k, 11 * k)
    exp, _ = _check_both(k, contigs)
    assert len(exp["kmer"]) > 100


# ---- B4: group heads across bitmap words ---------------------------------------------------------------------------
@pytest.mark.parametrize("k", [11, 16, 20, 31, 32])
def test_db_group_heads(k):
    contigs, planted, same, split = _heads_contigs(k, 13 * k)
    exp, _ = _check_both(k, contigs)
    # the planted SUNKs are exactly the oracle's, so each pair below tests one head decision
    sunk0 = set(exp["start"][exp["contig"] == 0].tolist())
    assert sunk0 == planted
    grp = {(int(c), int(s)): int(g) for c, s, g in zip(exp["contig"], exp["start"], exp["group"])}
    assert all(grp[a] == grp[b] for a, b in same) and len(same) > 50
    assert all(a in grp and b in grp for a, b in split) and len(split) == min(k, 32) + 3
    assert all(grp[a] != grp[b] for a, b in split if a[0] == b[0])


# ---- B5: repeats ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 3, 4, 6, 11, 12, 20, 31, 32])
def test_db_repeats(k):
    contigs, once, twice = _repeats_contigs(k, 17 * k)
    exp, _ = _check_both(k, contigs)
    if k >= 12 and k % 2 == 0:
        s0 = set(exp["start"][exp["contig"] == 0].tolist())
        assert all(p in s0 for p in once) and not any(p in s0 for p in twice) and once


# ---- B6: empty and SUNK-less assemblies ----------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 20, 31, 32])
def test_db_empty_assemblies(k):
    """every contig empty, and a total shorter than k: an empty database, no error"""
    for contigs in ([("a", b"")], [("a", b""), ("b", b""), ("c", b"")], [("a", b"ACG"[:max(k - 1, 0)]), ("b", b"")],
                    [("a", (b"AC" * 32)[:k - 1])]):
        exp, _ = _check_both(k, contigs)
        assert len(exp["kmer"]) == 0


@pytest.mark.parametrize("k", [4, 20, 32])
def test_db_sunkless_assembly_runs(k):
    """hap 2 identical to hap 1: no SUNK, no group; a read batch matches to 0 rows and a batches run finishes with
    empty rows"""
    from gavisunk_b200.engine import Engine
    rng = np.random.default_rng(k)
    h = _split(rng, _rand(rng, 20000), 3, "")
    contigs = [("h1_" + n, s) for n, s in h] + [("h2_" + n, s) for n, s in h]
    exp, _ = _check_both(k, contigs)
    assert len(exp["kmer"]) == 0
    eng = Engine(k)
    eng.build_db(contigs)
    assert eng.db_size() == (0, 0)
    reads = [h[0][1][100:9000], _rc(h[1][1][:5000]), b"ACGTN" * 300]
    seq = np.frombuffer(b"".join(reads), dtype=np.uint8)
    off = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.uint64)
    eng.set_reads(seq, off)
    assert eng.match() == 0
    hap = [0, 0, 0, 1, 1, 1]
    seen = []

    def on_batch(e, b, base):
        seen.append((b, base, len(e.rows(0)["read"]), len(e.rows(1)["read"])))

    iv, bases = eng.run_batches([lambda e: e.set_reads(seq, off), lambda e: e.set_reads(seq, off)], hap, min_read_len=1000,
                                on_batch=on_batch)
    assert bases == [0, 3] and seen == [(0, 0, 0, 0), (1, 3, 0, 0)]
    assert (eng.n_rows, eng.n_kept, eng.n_reads) == (0, 0, 6)
    assert all(len(v) == 0 for v in iv.values())


# ---- B7: forced passes ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 11, 20, 31])
def test_db_forced_passes(k):
    """the hash-partitioned build (n passes, each inserting the k-mers whose hash is its part) exports bit for bit
    what the default build and the oracle do, on the assemblies of every other build test"""
    from gavisunk_b200.engine import Engine, GavisunkError
    cases = [_b1_contigs(k, 100 + k), _tile_edges_contigs(k, 7 * k), _bytes_contigs(k, 11 * k),
             _repeats_contigs(k, 17 * k)[0]]
    if k >= 11:
        cases.append(_heads_contigs(k, 13 * k)[0])
    for contigs in cases:
        exp = O.build_sunk_db(contigs, k)
        eng = Engine(k)
        eng.build_db(contigs)
        want = _check_db(eng, contigs, k, exp)
        for n in (1, 2, 3, 7, 64):
            eng.set_db_passes(n)
            for device in (False, True):
                _build(eng, contigs, device)
                got = eng.db_export()
                assert all(np.array_equal(got[c], want[c]) for c in want), (n, device)
        eng.close()
    with pytest.raises(GavisunkError):
        Engine(k).set_db_passes(65)


# ---- B8: rebuilds on one engine ------------------------------------------------------------------------------------
def test_db_rebuild_one_engine():
    """larger, smaller, larger again on one engine: the reused buffers (bitmap, count table, probe table, filters)
    carry nothing over, and the probe sees only the current database"""
    from gavisunk_b200.engine import Engine
    k = 20
    big1, small, big2 = _b1_contigs(k, 3), _heads_contigs(k, 5)[0], _b1_contigs(k, 4)
    eng = Engine(k)
    for contigs in (big1, small, big2, small):
        for device in (False, True):
            _build(eng, contigs, device)
            _check_db(eng, contigs, k)
        exp = O.build_sunk_db(contigs, k)
        names = [n for n, _ in contigs]
        rng = np.random.default_rng(len(contigs))
        reads = _reads_from(big1, k, rng, 40)
        seq, off = _concat(reads)
        eng.set_reads(seq, off)
        eng.match()
        assert _rows(eng, names) == _oracle_rows(reads, [0, len(reads)], exp, names, k)


# ---- C: the match over GPU-built databases -------------------------------------------------------------------------
def _reads_from(contigs, k, rng, n):
    """error-free forward and reverse-complement substrings, substrings with SNPs and N runs, and reads of length
    k-1, k and k+1 at SUNK-rich places"""
    src = [s for _, s in contigs if len(s) >= k + 2]
    out = []
    for i in range(n):
        s = src[int(rng.integers(0, len(src)))]
        kind = i % 6
        if kind < 3:
            ln = max([k - 1, k, k + 1][kind], 1)
        else:
            ln = int(rng.integers(k + 2, min(len(s), 3000) + 1))
        a = int(rng.integers(0, len(s) - ln + 1))
        r = s[a:a + ln].upper()
        if kind == 4:
            r = _snps(rng, r.replace(b"N", b"A"), 0.01)
        if kind == 5 and ln > 40:
            b = int(rng.integers(0, ln - 20))
            r = r[:b] + b"N" * int(rng.integers(1, 20)) + r[b + 20:]
        if rng.random() < 0.5:
            r = _rc(r)
        out.append(r)
    return out


def _concat(reads):
    seq = np.frombuffer(b"".join(reads), dtype=np.uint8)
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(r) for r in reads])
    return seq, off


def _oracle_rows(reads, chunk_first, db, names, k):
    loc = [(names[c], int(s), int(km), int(g)) for c, s, km, g in zip(db["contig"], db["start"], db["kmer"], db["group"])]
    out = []
    for c in range(len(chunk_first) - 1):
        chunk = [(r, reads[r]) for r in range(chunk_first[c], chunk_first[c + 1])]
        out += O.match_chunk(chunk, db["kmer"], loc, k)
    return out


def _rows(eng, names):
    r = eng.rows(0)
    return list(zip(r["read"].tolist(), r["pos"].tolist(), [names[c] for c in r["contig"]], r["start"].tolist(),
                    r["group"].tolist()))


@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("k", range(1, 33))
def test_match_on_built_db_every_k(k, variant):
    """k_tab_finalize's sub-mer insertions and the probe's extraction, on tables this code built: both probe
    variants, ASCII and 2-bit packed reads (k = 32: the reference's k = 32 windows, match_k32)"""
    from gavisunk_b200.engine import Engine, pack_2bit
    contigs = _b1_contigs(k, 100 + k)
    names = [n for n, _ in contigs]
    eng = Engine(k)
    eng.set_probe_variant(variant)
    eng.build_db(contigs)
    db = _check_db(eng, contigs, k)
    rng = np.random.default_rng(1000 * variant + k)
    reads = _reads_from(contigs, k, rng, 120)
    chunk_first = [0, 50, len(reads)]
    seq, off = _concat(reads)
    exp = _oracle_rows(reads, chunk_first, {c: db[c] for c in ("contig", "start", "kmer", "group")}, names, k)
    assert len(exp) > (0 if k <= 2 else 5 if k == 32 else 20)  # k = 32: in effect only window 0 of a read can hit
    eng.set_reads(seq, off, chunk_first, [0, 1])
    assert eng.match() == len(exp)
    assert _rows(eng, names) == exp
    eng.set_reads_packed(pack_2bit(seq), off, chunk_first, [0, 1])
    assert eng.match() == len(exp)
    assert _rows(eng, names) == exp


# ---- D: hit-dense batches ------------------------------------------------------------------------------------------
_DENSE = {}


def _dense_case(k, mbp, n_chunks=1):
    """a database of N-separated islands (about 4 SUNKs per group) and a batch of reads that are SUNK k-mers of
    different groups back to back (consecutive groups distinct, random strand): one hit record per k bases, far
    above the first hit buffer of a context (1/32 of the windows).  Cached with its oracle rows."""
    key = (k, mbp, n_chunks)
    if key in _DENSE:
        return _DENSE[key]
    rng = np.random.default_rng(k * 7 + n_chunks)
    isl = [_rand(rng, k + 3) for _ in range(12000)]
    contigs = [("h1_0", b"N".join(isl[:6000])), ("h2_0", b"N".join(isl[6000:]))]
    names = [n for n, _ in contigs]
    db = O.build_sunk_db(contigs, k)
    assert _n_groups(db) == 12000
    gi = np.unique(db["contig"].astype(np.int64) << 32 | db["group"], return_inverse=True)[1]
    first = np.nonzero(np.diff(np.concatenate([[-1], gi])))[0]  # first SUNK of every group
    mers = []
    for c, s in zip(db["contig"][first], db["start"][first]):
        mers.append(contigs[c][1][s:s + k])
    fw = np.frombuffer(b"".join(mers), dtype=np.uint8).reshape(-1, k)
    rv = np.frombuffer(b"".join(_rc(m) for m in mers), dtype=np.uint8).reshape(-1, k)
    per_read = 16000 // k
    n_reads = int(mbp * 1e6) // (per_read * k) + 1
    g = np.cumsum(rng.integers(1, len(mers), n_reads * per_read)) % len(mers)  # consecutive groups distinct
    strand = rng.random(len(g)) < 0.5
    bases = np.where(strand[:, None], rv[g], fw[g]).reshape(n_reads, per_read * k)
    reads = [bases[r].tobytes() for r in range(n_reads)]
    cf = np.linspace(0, n_reads, n_chunks + 1).astype(int).tolist()
    exp = _oracle_rows(reads, cf, db, names, k)
    assert len(exp) > n_reads * per_read * 0.95
    seq, off = _concat(reads)
    _DENSE[key] = (contigs, names, reads, seq, off, cf, exp)
    return _DENSE[key]


def _dense_engine(k, contigs):
    from gavisunk_b200.engine import Engine
    eng = Engine(k)
    eng.build_db(contigs)
    return eng


@pytest.mark.parametrize("k", [16, 20])
def test_match_dense_fresh_engine(k):
    """a fresh engine: the first attempt overflows (records ~ windows / k > windows / 32) and the retry, sized by the
    densest span, gives the oracle's rows; a second match of the batch needs no retry and launches fewer kernels"""
    contigs, names, reads, seq, off, cf, exp = _dense_case(k, 4.2)
    assert len(exp) > len(seq) / 32 + 4096
    eng = _dense_engine(k, contigs)
    eng.set_reads(seq, off)
    l0 = eng.launches
    assert eng.match() == len(exp)
    l1 = eng.launches
    assert _rows(eng, names) == exp
    l2 = eng.launches
    assert eng.match() == len(exp)
    l3 = eng.launches
    assert _rows(eng, names) == exp
    assert l3 - l2 < l1 - l0


def test_match_dense_after_small_batch():
    """one engine: a batch under 1 kb sets the hit buffer to ~4100 records; a 4 Mbp dense batch then gets ~4 records
    per 4096-base span, a 17.5 Mbp one gets 0, and a small batch after them; every one equals the oracle"""
    k = 16
    contigs, names, reads, seq, off, cf, exp = _dense_case(k, 4.2)
    _, _, reads_b, seq_b, off_b, _, exp_b = _dense_case(k, 17.5)
    small = reads[0][:600], reads[1][:300]
    sseq, soff = _concat(list(small))
    db = O.build_sunk_db(contigs, k)
    exp_s = _oracle_rows(list(small), [0, 2], db, names, k)
    assert len(exp_s) > 40
    for big_seq, big_off, big_exp in ((seq, off, exp), (seq_b, off_b, exp_b)):
        eng = _dense_engine(k, contigs)
        for s, o, e in ((sseq, soff, exp_s), (big_seq, big_off, big_exp), (sseq, soff, exp_s), (big_seq, big_off, big_exp)):
            eng.set_reads(s, o)
            assert eng.match() == len(e)
            assert _rows(eng, names) == e
        eng.close()


@pytest.mark.parametrize("mode", ["ascii0", "ascii2", "ascii3", "packed"])
def test_match_dense_copy_pipeline(mode):
    """the dense batch through the copy pipeline (7 segments), its segments sent as they are / all packed / every
    other one packed, or packed on the host: the retry runs after the copies and packers of the first attempt"""
    from gavisunk_b200.engine import pack_2bit
    k = 16
    contigs, names, reads, seq, off, cf, exp = _dense_case(k, 4.2)
    eng = _dense_engine(k, contigs)
    eng.set_copy_pipeline(0, 7)
    if mode == "packed":
        eng.set_reads_packed(pack_2bit(seq), off)
    else:
        eng.set_host_pack(int(mode[-1]), 3)
        eng.set_reads(seq, off)
    assert eng.match() == len(exp)
    assert _rows(eng, names) == exp
    assert eng.copy_stats()[1] == 7


def test_match_dense_many_chunks():
    """the dense batch in 37 chunks: the consecutive-group suppression restarts per chunk (Q4) across the retry"""
    k = 16
    contigs, names, reads, seq, off, cf, exp = _dense_case(k, 4.2, n_chunks=37)
    eng = _dense_engine(k, contigs)
    eng.set_reads(seq, off, cf, [0] * 37)
    assert eng.match() == len(exp)
    assert _rows(eng, names) == exp

"""The support-track oracle (tests/support_oracle.py) against brute-force per-base counting.  CPU only."""
import random

import support_oracle as O


def _brute(placements, fai):
    runs = []
    for c, L in fai:
        depth = [sum(1 for p in placements if p[0] == c and p[1] <= x < p[2]) for x in range(L)]
        s = 0
        for x in range(1, L + 1):
            if x == L or depth[x] != depth[s]:
                runs.append((c, s, x, depth[s]))
                s = x
    return runs


def test_depth_equals_per_base_count():
    rng = random.Random(7)
    for trial in range(40):
        fai = [(f"c{i}", rng.randint(1, 120)) for i in range(rng.randint(1, 4))]
        pls = []
        for c, L in fai:
            if rng.random() < 0.25:
                continue  # a contig without placements: one depth-0 run
            for _ in range(rng.randint(0, 8)):
                a = rng.randrange(0, L)
                b = rng.randint(a + 1, L)
                pls.append((c, a, b))
            if pls and pls[-1][0] == c and rng.random() < 0.5:
                a, b = pls[-1][1:3]
                pls.append((c, b, min(L, b + 3)) if b < L else (c, a, b))  # touching, or the same span twice
                pls.append((c, a, max(a + 1, (a + b) // 2)))            # nested
        assert O.support_depth(pls, fai) == _brute(pls, fai), trial


def test_support_tracks_placements():
    """one read of two rows in the same direction on contig a, one read with a single ID, one reversed read on b"""
    rows = [("r1", 100, "a", 1000, 1000), ("r1", 1100, "a", 2000, 2000), ("r1", 2100, "a", 3000, 3000),
            ("r2", 100, "a", 1000, 1000), ("r2", 150, "a", 1000, 1000),
            ("r3", 100, "b", 3000, 3000), ("r3", 1100, "b", 2000, 2000), ("r3", 2100, "b", 1000, 1000)]
    fai = [("b", 4000), ("a", 5000), ("e", 10)]
    rlen = {"r1": 20000, "r2": 20000, "r3": 20000}
    pls, runs = O.support_tracks(rows, rlen, set(), fai)
    assert pls == [("b", 1000, 3000, "r3", 3, "-"), ("a", 1000, 3000, "r1", 3, "+")]
    assert runs == [("b", 0, 1000, 0), ("b", 1000, 3000, 1), ("b", 3000, 4000, 0),
                    ("a", 0, 1000, 0), ("a", 1000, 3000, 1), ("a", 3000, 5000, 0), ("e", 0, 10, 0)]
    # a bad group removes the read's first ID
    pls, _ = O.support_tracks(rows, rlen, {("a", 1000)}, fai)
    assert ("a", 2000, 3000, "r1", 2, "+") in pls

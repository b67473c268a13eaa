"""CPU: the findpath reference (tests/findpath_ref.c, bf_findpath's breadth-limited search over direct paths in plain C, every
structure scored by orc_eval) against an exact subset DP over all direct paths, with the properties the engine's definition
guarantees: valid paths, saddle = max of the path's energies, a saddle that does not increase over the powers of two, and k = 0 for
equal structures."""
import numpy as np

from conftest import PAR1999
from findpath_ref import FindpathOracle, check_path, perturb, random_structure


def _instances(O, rng):
    out = []
    for x in range(220):
        n = int(rng.integers(20, 61))
        alpha, p = ("ACGU", None) if x % 4 else ("GC", None)   # low-complexity sequences make energy ties
        seq = "".join(rng.choice(list(alpha), n, p=p))
        s1 = O.mfe(seq)[1]
        if x % 5 == 4:
            s2 = random_structure(rng, n, int(rng.integers(0, 12)))
        else:
            s2 = perturb(rng, s1, int(rng.integers(0, 6)), int(rng.integers(0, 6)))
        out.append((seq, s1, s2))
    return out


def test_findpath_reference():
    O = FindpathOracle(PAR1999)
    rng = np.random.default_rng(5)
    n_dp = n_trunc = 0
    for seq, s1, s2 in _instances(O, rng):
        prev = None
        for W in (1, 2, 4, 8, 16):
            r = O.findpath(seq, s1, s2, W)
            structs = check_path(s1, s2, r["moves"])
            assert r["path_e"] == [O.eval(seq, s) for s in structs], (seq, s1, s2, W)
            assert r["saddle"] == max(r["path_e"]), (seq, s1, s2, W)
            assert prev is None or r["saddle"] <= prev, (seq, s1, s2, W, r["saddle"], prev)
            prev = r["saddle"]
            n_trunc += r["max_level"] > W
        k = len(r["moves"])
        if k <= 12:
            full = O.findpath(seq, s1, s2, 1 << k)   # wider than any level: nothing is cut
            assert full["max_level"] <= 1 << k
            assert full["saddle"] == O.findpath_dp(seq, s1, s2) <= prev, (seq, s1, s2)
            n_dp += 1
    assert n_dp >= 150 and n_trunc >= 50, (n_dp, n_trunc)


def test_findpath_equal_structures():
    O = FindpathOracle(PAR1999)
    rng = np.random.default_rng(6)
    for _ in range(20):
        n = int(rng.integers(20, 61))
        seq = "".join(rng.choice(list("ACGU"), n))
        s = O.mfe(seq)[1] if rng.random() < 0.5 else random_structure(rng, n)
        r = O.findpath(seq, s, s, 4)
        assert r["moves"] == [] and r["path_e"] == [O.eval(seq, s)] and r["saddle"] == O.eval(seq, s)

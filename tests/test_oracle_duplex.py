"""CPU: the duplex reference (tests/duplex_ref.c, the recurrence and tie rules of bf_duplex in plain C) against a brute force over
every duplex chain scored by the oracle's two-strand eval_structure on a&b."""
import numpy as np

from conftest import PAR1999
from duplex_ref import INF, DuplexOracle


def _cases(rng):
    """random pairs of 1-9 nt, GC-rich pairs, pairs whose only possible pairs are GU, pairs with no possible pair"""
    rnd = lambda alpha, p=None: "".join(rng.choice(list(alpha), int(rng.integers(1, 10)), p=p))  # noqa: E731
    cases = [(rnd("ACGU"), rnd("ACGU")) for _ in range(200)]
    cases += [(rnd("ACGU", [0.1, 0.4, 0.4, 0.1]), rnd("ACGU", [0.1, 0.4, 0.4, 0.1])) for _ in range(60)]
    cases += [(rnd("GA"), rnd("UA")) for _ in range(30)]   # GU and AU pairs only
    cases += [(rnd("G"), rnd("U")) for _ in range(15)]     # GU pairs only
    cases += [(rnd("AC"), rnd("AC")) for _ in range(15)]   # no possible pair
    cases += [("G", "C"), ("A", "U"), ("GGGGGGGGG", "CCCCCCCCC"), ("GCGCGCGCG", "CGCGCGCGC"), ("A", "A"), ("GUGUGUGUG", "UGUGUGUGU")]
    return cases


def test_duplex_reference_equals_brute_force():
    O = DuplexOracle(PAR1999)
    rng = np.random.default_rng(11)
    cases = _cases(rng)
    assert len(cases) >= 300
    n_none = 0
    for a, b in cases:
        e, ss = O.duplex(a, b)
        bf = O.duplex_brute(a, b)
        assert e == bf, (a, b, e, bf, ss)
        assert len(ss) == len(a) + len(b) + 1 and ss[len(a)] == "&"
        if e >= INF:
            n_none += 1
            assert ss == "." * len(a) + "&" + "." * len(b), (a, b, ss)
            continue
        pa, pb = ss[:len(a)], ss[len(a) + 1:]
        assert set(pa) <= set("(.") and set(pb) <= set(").") and pa.count("(") == pb.count(")") >= 1, (a, b, ss)
        assert O.eval_duplex(a, b, ss) == e, (a, b, ss, e)
    assert n_none >= 15

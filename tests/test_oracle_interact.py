"""CPU: the interaction reference (tests/interact_ref.c, the fixed-start recurrence, spans, score, tie and trace rules of
bf_interact in plain C) against a brute force over every chain scored by the oracle's two-strand eval on a&b, with opening energies
from exact masked partition functions Z(stretch unpaired) / Z (tests/unpaired_ref.c)."""
from fractions import Fraction

import numpy as np

from conftest import PAR1999
from interact_ref import INF, KT, InteractOracle
from unpaired_ref import UnpairedOracle


def _cases(rng):
    """random pairs of 1-8 nt, GC-rich pairs, pairs whose only possible pairs are GU, pairs with no possible pair"""
    rnd = lambda alpha, p=None: "".join(rng.choice(list(alpha), int(rng.integers(1, 9)), p=p))  # noqa: E731
    cases = [(rnd("ACGU"), rnd("ACGU")) for _ in range(150)]
    cases += [(rnd("ACGU", [0.1, 0.4, 0.4, 0.1]), rnd("ACGU", [0.1, 0.4, 0.4, 0.1])) for _ in range(60)]
    cases += [(rnd("GA"), rnd("UA")) for _ in range(20)]
    cases += [(rnd("AC"), rnd("AC")) for _ in range(10)]
    cases += [("G", "C"), ("GGGGGGGG", "CCCCCCCC"), ("GCGCGCGC", "GCGCGCGC"), ("GUGUGUGU", "UGUGUGUG")]
    return cases


def _exact_ed(uo, seq, span, cache):
    """[len, span] opening energies -(kT/1000) ln(Z(k .. k+u-1 unpaired) / Z), +inf past the strand's end"""
    if (seq, span) not in cache:
        n = len(seq)
        lnz = uo.masked_lnz(seq)
        ed = np.full((n, span), np.inf)
        for k in range(1, n + 1):
            for u in range(1, min(span, n - k + 1) + 1):
                mask = [1 if k <= p < k + u else 0 for p in range(1, n + 1)]
                ed[k - 1, u - 1] = -(KT / 1000.0) * (uo.masked_lnz(seq, mask) - lnz)
        cache[(seq, span)] = ed
    return cache[(seq, span)]


def _check_structure(O, a, b, r):
    ss = r["ss"]
    assert len(ss) == len(a) + len(b) + 1 and ss[len(a)] == "&"
    if r["h"] >= INF:
        assert ss == "." * len(a) + "&" + "." * len(b) and r["site"] == (0, 0, 0, 0)
        return
    pa, pb = ss[:len(a)], ss[len(a) + 1:]
    k1, km, lm, l1 = r["site"]
    assert pa.index("(") + 1 == k1 and pa.rindex("(") + 1 == km and pb.index(")") + 1 == lm and pb.rindex(")") + 1 == l1, (a, b, r)
    assert O.eval_duplex(a, b, ss) == r["h"], (a, b, r)


def test_interact_reference_equals_brute_force():
    O = InteractOracle(PAR1999)
    uo = UnpairedOracle(PAR1999)
    rng = np.random.default_rng(12)
    cases = _cases(rng)
    assert len(cases) >= 200
    cache = {}
    n_site = n_checks = 0
    for a, b in cases:
        for span in range(1, max(len(a), len(b)) + 1):
            modes = [(None, None), (_exact_ed(uo, a, span, cache), _exact_ed(uo, b, span, cache)), (None, _exact_ed(uo, b, span, cache))]
            for eda, edb in modes:
                r = O.interact(a, b, span, eda, edb)
                e, h, site = O.interact_brute(a, b, span, eda, edb)
                assert (r["e"], r["h"], r["site"]) == (e, h, site), (a, b, span, r, e, h, site)
                _check_structure(O, a, b, r)
                n_checks += 1
                if h < INF:
                    n_site += 1
                    ea = 0.0 if eda is None else eda[site[0] - 1, site[1] - site[0]]
                    eb = 0.0 if edb is None else edb[site[2] - 1, site[3] - site[2]]
                    assert r["e"] == h / 100.0 + ea + eb, (a, b, span, r, ea, eb)
                    assert r["gap"] >= 0.0
            if span >= max(len(a), len(b)):   # no accessibility and no span limit: bf_duplex's energy, E = H / 100 exactly
                r, ed = O.interact(a, b, span), O.duplex(a, b)[0]
                assert r["h"] == ed and (r["e"] == ed / 100.0 if ed < INF else r["e"] == np.inf), (a, b, r, ed)
    assert n_checks >= 1500 and n_site >= 1000


def test_division_by_100_without_a_divide():
    """bf_interact.cu forms H / 100.0 as q = H * 0.01 corrected by one fma step; that equals the correctly rounded quotient for
    every integer |H| <= 200000 (each fma rounds the exact value once: emulated here in exact rational arithmetic)"""
    c = Fraction(0.01)
    for v in range(-200000, 200001):
        q = float(v) * 0.01
        r = float(v - Fraction(q) * 100)
        assert float(Fraction(q) + Fraction(r) * c) == v / 100.0, v

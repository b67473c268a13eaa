"""The masked-partition-function reference for unpaired stretches (tests/unpaired_ref.c) against exact enumeration: the oracle's
per-structure Boltzmann weights (pf_smooth included) summed over every structure of short sequences."""
import os
import random

import pytest

from struct_weight import WeightOracle
from unpaired_ref import UnpairedOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAR = os.path.join(ROOT, "desirna_b200", "params", "turner1999_37C.par")


@pytest.fixture(scope="module")
def oracles():
    from oracle.pyoracle import build
    build()
    return UnpairedOracle(PAR), WeightOracle(PAR)


def _seqs():
    rng = random.Random(11)
    out = ["GGGGAAAACCCC", "GGGAAACCCAAAGGG", "GCGCUUCGGCGCAA"]
    while len(out) < 20:
        out.append("".join(rng.choice("ACGU") for _ in range(rng.randint(12, 16))))
    return out


@pytest.mark.parametrize("seq", _seqs())
def test_masked_reference_matches_enumeration(oracles, seq):
    U, Wo = oracles
    structs = [db for _, db in Wo.enumerate_band(seq, 10 ** 6, cap=200000)]
    w = [Wo.weight(seq, db) for db in structs]
    Z = sum(w)
    n = len(seq)
    st = [(i, u) for i in range(1, n + 1) for u in range(1, n - i + 2)]
    ref = U.unpaired(seq, st, nthreads=1)
    for (i, u), r in zip(st, ref):
        e = sum(wk for wk, db in zip(w, structs) if db[i - 1:i - 1 + u] == "." * u) / Z
        assert abs(r - e) <= 1e-12, (seq, i, u, r, e)

"""CPU: the per-structure partition-function weight the sampling tests compare against.  Summed over every structure it is the
oracle's Z; where no smoothed dangle or mismatch factor applies it is plain exp(-E / kT)."""
import math
import os
import random

import pytest

from struct_weight import WeightOracle

PAR1999 = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "desirna_b200", "params", "turner1999_37C.par")


@pytest.fixture(scope="module")
def wo():
    from oracle.pyoracle import build
    build()
    return WeightOracle(PAR1999)


@pytest.mark.parametrize("seed", range(6))
def test_weights_sum_to_z(wo, seed):
    rng = random.Random(seed)
    s = "".join(rng.choice("ACGU") for _ in range(rng.randint(10, 16)))
    band = wo.enumerate_band(s, 10 ** 6, cap=500000)
    Z = math.fsum(wo.weight(s, db) for _, db in band)
    assert abs(Z / wo.Z(s) - 1.0) < 1e-12, (s, Z, wo.Z(s))


@pytest.mark.parametrize("seq,db", [
    ("GGGGAAAACCCC", "............"),
    ("GGGGAAAACCCC", "((((....))))"),
    ("GCGCGGGGACGCGC", "(((((....)))))"),
    ("GCAUCGAAAGAUGC", "(((((....)))))"),
    ("GGCAGGGGACUGCC", "(((((....)))))"),
])
def test_weight_without_smoothed_terms_is_boltzmann(wo, seq, db):
    """the empty structure, and a helix from nucleotide 1 to n closed by a hairpin: no dangle, no mismatch outside the hairpin"""
    w = wo.weight(seq, db)
    e = wo.eval(seq, db)
    assert abs(w / math.exp(-e * 10.0 / wo.kT) - 1.0) < 1e-12, (seq, db, w, e)

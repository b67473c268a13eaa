"""CPU: avoid mode (-o on, oligo_state "avoid") of the lock-step host path.  score_sequences folds the self-dimers seq&seq of a
whole batch in one engine call and must score every mutant exactly as score_sequence does, one dimer compound at a time
(utils/energy_scores.py:118-119, 412-419).  The CPU oracle stands in for the GPU engine."""
import math
import types

import pytest

import oracle_backend

from conftest import PAR1999, load_golden


@pytest.fixture(scope="module")
def rna_on_oracle(oracle):
    from oracle_backend import OracleBackend
    old = oracle_backend.current()
    be = OracleBackend(PAR1999)
    oracle_backend.install(be)
    yield be
    oracle_backend.install(old)


def options(**kw):
    o = types.SimpleNamespace(oligo_state="avoid", pks="off", scoring_f=[("Ed-Epf", 1.0)], subopt="off", motifs={})
    o.__dict__.update(kw)
    return o


def input_file(target):
    return types.SimpleNamespace(sec_struct=target, alt_sec_struct=None, alt_sec_structs=None)


def same(a, b):
    """field equality that lets NaN equal NaN"""
    return a == b or (isinstance(a, float) and isinstance(b, float) and math.isnan(a) and math.isnan(b))


def batch():
    rows = load_golden("G1")[:5]
    target = rows[0]["target"]
    # poly-A has no pair between its two copies: FcAB is the 999 sentinel (QAB <= 1e-17) and the reference's arithmetic gives
    # rhs = 0, a 0/0 fraction and a NaN score
    return [r["sequence"] for r in rows] + ["A" * len(target)], input_file(target)


@pytest.mark.filterwarnings("ignore:invalid value:RuntimeWarning")
@pytest.mark.parametrize("scoring", [[("Ed-Epf", 1.0)], [("Edef", 5.0), ("Ed-Epf", 0.3)]])
def test_batched_avoid_equals_one_by_one(rna_on_oracle, scoring):
    from desirna_b200.utils import energy_scores as es
    seqs, inp = batch()
    opt = options(scoring_f=scoring)
    got = es.score_sequences(seqs, inp, opt)
    want = [es.score_sequence(s, inp, opt) for s in seqs]
    for a, b in zip(got, want):
        va, vb = vars(a), vars(b)
        assert va.keys() == vb.keys() and "monomer_bonus" in va and "oligo_fraction" in va
        for k in va:
            assert same(va[k], vb[k]), (a.sequence, k, va[k], vb[k])
    assert all(0.0 <= s.oligo_fraction < 1.0 and s.monomer_bonus >= 0.0 for s in got[:-1])
    assert math.isnan(got[-1].oligo_fraction) and math.isnan(got[-1].scoring_function)


@pytest.mark.filterwarnings("ignore:invalid value:RuntimeWarning")
def test_one_engine_call_for_the_self_dimers_of_a_batch(rna_on_oracle):
    """-sf Ed-Epf: a sub-step of R mutants costs two engine calls in avoid mode (folds + evals, then the R self-dimers), one without"""
    from desirna_b200.utils import energy_scores as es
    seqs, inp = batch()
    c0 = rna_on_oracle.calls
    es.score_sequences(seqs, inp, options(oligo_state="none"))
    c1 = rna_on_oracle.calls
    es.score_sequences(seqs, inp, options())
    c2 = rna_on_oracle.calls
    assert (c1 - c0, c2 - c1) == (1, 2)
    # one sequence at a time, the self-dimer is one more engine call per sequence
    es.score_sequence(seqs[0], inp, options(oligo_state="none"))
    c3 = rna_on_oracle.calls
    es.score_sequence(seqs[0], inp, options())
    c4 = rna_on_oracle.calls
    assert (c4 - c3) - (c3 - c2) == 1

"""CPU: the brute-force two-strand enumeration (tests/twostrand_enum.py) that the GPU second-best tests compare with, checked
against the oracle's two-strand MFE and single-strand band enumeration, and `-nd on` scoring of a heterodimer on the host mirror."""
import random
import struct
import types

import pytest

import oracle_backend
import twostrand_enum as te

from conftest import PAR1999


def f32(x):
    return struct.unpack("f", struct.pack("f", x))[0]


def random_dimers(count, seed):
    rng = random.Random(seed)
    out = []
    for k in range(count):
        la = rng.randint(1, 9) if k % 5 else rng.randint(1, 2)   # every fifth: a strand of 1-2 nt
        lb = rng.randint(1, 9)
        a = "".join(rng.choice("ACGU") for _ in range(la))
        b = a if k % 7 == 0 else "".join(rng.choice("ACGU") for _ in range(lb))   # every seventh: a homodimer
        out.append(a + "&" + b)
    return out + ["A&A", "AAAA&AAAA", "AAAAAAA&AAAAA", "GC&GC", "G&C", "GGGAAACCC&GGGUUUCCC"]


def pair_table(db):
    st, pt = [], {}
    for i, ch in enumerate(db):
        if ch == "(":
            st.append(i)
        elif ch == ")":
            j = st.pop()
            pt[i], pt[j] = j, i
    assert not st
    return pt


def test_minimum_is_the_two_strand_mfe(oracle):
    seqs = random_dimers(120, 11)
    connected = 0
    for seq in seqs:
        band = te.enumerate_band(oracle, seq)
        assert band[0][0] == oracle.mfe(seq)[0], (seq, band[:2], oracle.mfe(seq))
        a = len(seq.split("&")[0])
        connected += any(i < a <= j for i, j in pair_table(band[0][1]).items())
    assert connected >= 10   # the minimum is often a duplex, so the nick-loop and DuplexInit terms are exercised
    for seq in ("AAAA&AAAA", "AAAAAAA&AAAAA", "A&A"):   # no canonical pair: the open structure only
        assert te.enumerate_band(oracle, seq) == [(0, "." * len(seq.replace("&", "")))]
        assert te.second_best(oracle, seq) == (0, te.INF_DCAL)


def test_listed_structures_are_distinct_and_scored_by_eval(oracle):
    for seq in random_dimers(40, 12):
        s = seq.replace("&", "")
        cp = len(seq.split("&")[0])   # 0-based first index of strand B
        band = te.enumerate_band(oracle, seq)
        assert len({db for _, db in band}) == len(band), seq
        for e, db in band:
            assert len(db) == len(s) and e == oracle.eval(seq, db)
            for i, j in pair_table(db).items():
                if i < j:
                    assert (s[i], s[j]) in te._PAIRS and ((i < cp) != (j < cp) or j - i > te.TURN), (seq, db)


def test_single_strand_equals_the_oracle_band():
    from oracle.pyoracle import Oracle
    O = Oracle(PAR1999)
    rng = random.Random(13)
    for n in (4, 8, 12, 15):
        for _ in range(6):
            s = "".join(rng.choice("ACGU") for _ in range(n))
            assert te.enumerate_band(O, s) == O.enumerate_band(s, te.INF_DCAL), s
            assert te.enumerate_band(O, s, 0) == O.enumerate_band(s, 0), s


@pytest.fixture
def rna_on_dimer_oracle(oracle):
    old = oracle_backend.current()
    be = te.DimerOracleBackend(PAR1999)
    oracle_backend.install(be)
    yield be
    oracle_backend.install(old)


def options(**kw):
    o = types.SimpleNamespace(oligo_state="heterodimer", pks="off", scoring_f=[("Ed-Epf", 1.0)], subopt="off", motifs={})
    o.__dict__.update(kw)
    return o


def test_subopt_term_of_a_heterodimer_score(rna_on_dimer_oracle, oracle):
    """`-nd on` for a two-strand target whose MFE structure the sequence already folds into: subopt_e is the float32 of the
    enumeration's second energy and enters the score before the oligomer term (energy_scores.py:104-116)."""
    from desirna_b200.utils import energy_scores as es
    seq = "CGCAUGCA&UGCAUGCGA"
    mfe, ss = oracle.mfe(seq)
    a = len(seq.split("&")[0])
    target = ss[:a] + "&" + ss[a:]
    assert "(" in ss[:a] and ")" in ss[a:] and "." in ss   # a duplex with unpaired bases: the mcc term can reach 0
    inp = types.SimpleNamespace(sec_struct=target, alt_sec_struct=None, alt_sec_structs=None)
    plain = es.score_sequence(seq, inp, options())
    nd = es.score_sequence(seq, inp, options(subopt="on"))
    assert plain.mcc == 0
    band = te.enumerate_band(oracle, seq)
    assert band[0][0] == mfe and band[1][0] - mfe <= 4900
    assert nd.subopt_e == f32(band[1][0] / 100.0)
    assert abs(nd.scoring_function - ((plain.scoring_function - plain.oligomer_bonus) - (nd.subopt_e - plain.Epf) + nd.oligomer_bonus)) < 1e-9
    # one structure only: the term is 0
    from desirna_b200 import RNA
    assert es.get_first_suboptimal_energy("AAAA&AAAA", RNA.fold_compound("AAAA&AAAA")) == 0

"""GPU: the second-best energy of two-strand ('A&B') sequences -- bf_second_best's nick-aware 2-best DP (csrc/bf_twobest.cu) against
brute-force enumeration under the engine's two-strand loop model (tests/twostrand_enum.py), against the engine's own two-strand MFE,
through the RNA shim, and inside the device design loop with `-nd on`."""
import random
import struct

import pytest

import twostrand_enum as te

pytestmark = pytest.mark.gpu


def f32(x):
    return struct.unpack("f", struct.pack("f", x))[0]


def rand_seq(rng, n):
    return "".join(rng.choice("ACGU") for _ in range(n))


def pair_table(db):
    st, pt = [], {}
    for i, ch in enumerate(db):
        if ch == "(":
            st.append(i)
        elif ch == ")":
            j = st.pop()
            pt[i], pt[j] = j, i
    return pt


def test_short_dimers_against_brute_force(engine, oracle):
    seqs = []
    for seed in range(4):
        rng = random.Random(100 + seed)
        for n in range(6, 21):
            s = rand_seq(rng, n)
            cut = rng.randint(1, n - 1)
            seqs.append(s[:cut] + "&" + s[cut:])
            if n % 2 == 0 and seed < 2:
                h = rand_seq(rng, n // 2)
                seqs.append(h + "&" + h)   # homodimer
    seqs += ["AAAA&AAAA", "A&AAAAAA", "G&C", "GC&GC", "GGGAAACCC&GGGUUUCCC"]
    e1, e2 = engine.second_best(seqs)
    finite = 0
    for k, seq in enumerate(seqs):
        b1, b2 = te.second_best(oracle, seq)
        assert int(e1[k]) == b1 == oracle.mfe(seq)[0], (seq, int(e1[k]), b1)
        if b2 >= te.INF_DCAL:
            assert int(e2[k]) >= 10000000, (seq, int(e2[k]))
        else:
            assert int(e2[k]) == b2, (seq, int(e2[k]), b2)
            finite += 1
    assert finite > 30


def test_mixed_batch_equals_separate_calls(engine):
    rng = random.Random(7)
    singles = [rand_seq(rng, n) for n in (12, 25, 40, 61)]
    twos = [rand_seq(rng, a) + "&" + rand_seq(rng, b) for a, b in ((5, 9), (17, 18), (30, 20), (1, 40))]
    mixed = [x for pair in zip(singles, twos) for x in pair]
    m1, m2 = engine.second_best(mixed)
    s1, s2 = engine.second_best(singles)
    t1, t2 = engine.second_best(twos)
    assert (m1[0::2] == s1).all() and (m2[0::2] == s2).all()
    assert (m1[1::2] == t1).all() and (m2[1::2] == t2).all()


def opened_hairpin(db, cut0):
    """the structure with the closing pair of a hairpin opened, the hairpin stacked on its outer pair and on one strand (so the
    opened structure is one the folding grammar generates); None if there is no such hairpin"""
    pt = pair_table(db)
    for i, j in sorted(pt.items()):
        if i < j and (i < cut0) == (j < cut0) and all(db[k] == "." for k in range(i + 1, j)) and pt.get(i - 1) == j + 1:
            return db[:i] + "." + db[i + 1:j] + "." + db[j + 1:]
    return None


def test_long_dimers_bound_the_second_best(engine, oracle):
    rng = random.Random(23)
    h = rand_seq(rng, 60)
    seqs = ["AACUGAGGGGAAACCAA&GUCUAGUGACCACUCGUU"]   # 17&18, the shape of the reference's RNA-RNA complex example
    seqs += [rand_seq(rng, a) + "&" + rand_seq(rng, a) for a in (30, 50, 100)]
    seqs += [h + "&" + h]
    homo = {len(seqs) - 1}
    e1, e2 = engine.second_best(seqs)
    out = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)
    hairpins = connected = 0
    for k, seq in enumerate(seqs):
        a, b = seq.split("&")
        ss = out["mfe_ss"][k]
        assert int(e1[k]) == int(out["mfe_dcal"][k]), (k, int(e1[k]), int(out["mfe_dcal"][k]))
        assert int(e1[k]) <= int(e2[k]) < 10000000
        opened = opened_hairpin(ss, len(a))
        if opened is not None:
            assert int(e2[k]) <= oracle.eval(seq, opened), (k, int(e2[k]), oracle.eval(seq, opened))
            hairpins += 1
        if any(i < len(a) <= j for i, j in pair_table(ss).items()):
            assert int(e2[k]) <= oracle.mfe(a)[0] + oracle.mfe(b)[0]
            connected += 1
        if k in homo:
            L = len(a)
            mirror = ["."] * len(ss)
            for i, j in pair_table(ss).items():
                x, y = sorted(((i + L) % len(ss), (j + L) % len(ss)))
                mirror[x], mirror[y] = "(", ")"
            if "".join(mirror) != ss:   # the strand-swapped structure has the same energy: a tie
                assert int(e2[k]) == int(e1[k])
    assert hairpins >= 3 and connected >= 3


def test_shim_and_first_suboptimal_energy(engine, oracle):
    from desirna_b200 import RNA
    from desirna_b200.utils import energy_scores as es
    for seq in ("CGCAUGCA&UGCAUGCGA", "GGGAAUCCA&UGGGCAAGCC", "GCAUG&CAUGC"):
        b1, b2 = te.second_best(oracle, seq)
        fc = RNA.fold_compound(seq)
        assert fc.second_best_energy() == (f32(b1 / 100.0), f32(b2 / 100.0))
        assert es.get_first_suboptimal_energy(seq, fc) == (f32(b2 / 100.0) if b2 - b1 <= 4900 else 0)
    fc = RNA.fold_compound("AAAA&AAAA")
    assert fc.second_best_energy() == (0.0, None)
    assert es.get_first_suboptimal_energy("AAAA&AAAA", fc) == 0
    with pytest.raises(NotImplementedError):
        fc.subopt_cb(100, lambda *a: None)


HETERO_SHORT = ("((((((....&))))))", "NNNNNNNNNN&NNNNNN")
HOMO_SHORT = ("((((....))))..&((((....))))..", "NNNNNNNNNNNNNN&NNNNNNNNNNNNNN")
HOMO_DUPLEX = ("((((((......&......))))))", "NNNNNNNNNNNN&NNNNNNNNNNNN")
FULL_DUPLEX = ("((((((&))))))", "NNNNNN&NNNNNN")   # every position paired: folding into it leaves mcc at 0, so the term stays off


def test_negative_design_of_dimers_on_the_device(engine):
    """-nd on for two-strand jobs: the device loop's subopt_e and score of every replica equal the host mirror's (the term comes
    before the oligomer term, utils/energy_scores.py:104-116); a heterodimer and a homodimer replica reach their target"""
    from desirna_b200 import design
    from desirna_b200.utils import energy_scores as es
    from desirna_b200.utils import stats_inputs_outputs as sio
    hits = {"heterodimer": 0, "homodimer": 0}
    for case, state in ((HETERO_SHORT, "heterodimer"), (HOMO_SHORT, "homodimer"), (HOMO_DUPLEX, "homodimer"), (FULL_DUPLEX, "heterodimer")):
        inp = sio.make_input("dimer", *case)
        o = design.DesignOptions(replicas=8, RE_attempt=25, oligo_state=state, scoring_f=[("Ed-Epf", 1.0)], subopt="on")
        random.seed(17)
        loop = design.DesignLoop([inp], o, seed=29)
        loop.run(10)
        rep = loop.replicas()
        loop.close()
        ref = es.score_sequences(rep["sequence"], inp, o)
        for g, (s, h) in enumerate(zip(rep["sequence"], ref)):
            rec = dict(zip(design.REC_FIELDS, rep["rec"][g]))
            assert rep["mfe_ss"][g] == h.mfe_ss
            assert rec["subopt_e"] == h.subopt_e, (case[0], s, rec["subopt_e"], h.subopt_e)
            assert (rec["subopt_e"] != 0) <= (h.mcc == 0)
            hits[state] += h.mcc == 0
            assert rec["oligomer_bonus"] == pytest.approx(h.oligomer_bonus, abs=1e-9)
            assert rec["scoring_function"] == pytest.approx(h.scoring_function, abs=1e-5), (case[0], s)
    assert hits["heterodimer"] > 0 and hits["homodimer"] > 0, hits   # replicas folded into their target: the term was exercised

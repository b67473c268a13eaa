"""GPU: avoid designs (-o on, oligo_state "avoid", bf_design_t.oligo = 3) in the device-resident design loop.  Every mutant's
self-dimer seq&seq is folded by the two-strand partition function beside the single-strand fills, and the accept kernel adds
-kT ln(1 - dimer fraction) (utils/energy_scores.py:118-119, 412-419).  Records against the host mirror of score_sequence, the
fraction against the CPU oracle, the combinations with the other device terms, the trajectory output and the refusal of
two-strand jobs."""
import ctypes as C
import math
import random
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

KT = 0.001987204259 * (273.15 + 37)


def f32(x):
    import struct
    return struct.unpack("f", struct.pack("f", x))[0]


def small_inputs(max_len=48, limit=6):
    from desirna_b200.utils import stats_inputs_outputs as sio
    rows = [r for r in load_golden("E1") if len(r["target"]) <= max_len and not set(r["target"]) - set(".()")]
    return [sio.make_input(r["file"], r["target"]) for r in rows[:limit]]


def check_against_host(loop, inputs, o, exact_epf=False):
    """every replica's record against es.score_sequences of the same sequences; returns the replicas and the host records"""
    from desirna_b200 import design
    from desirna_b200.utils import energy_scores as es
    rep = loop.replicas()
    recs = loop.records(o, 0)
    R = loop.R
    refs = []
    for j, inp in enumerate(inputs):
        seqs = rep["sequence"][j * R:(j + 1) * R]
        ref = es.score_sequences(seqs, inp, o)
        refs += ref
        for r, (s, h) in enumerate(zip(seqs, ref)):
            g = j * R + r
            rec = dict(zip(design.REC_FIELDS, rep["rec"][g]))
            row = recs[j][r]
            assert rep["mfe_ss"][g] == h.mfe_ss, (inp.name, s)
            assert rec["edesired"] == h.edesired
            assert rec["Epf"] == h.Epf if exact_epf else abs(rec["Epf"] - h.Epf) <= 4e-6
            assert row["oligo_fraction"] == pytest.approx(h.oligo_fraction, rel=1e-6), (inp.name, s)
            assert row["monomer_bonus"] == pytest.approx(h.monomer_bonus, abs=1e-6), (inp.name, s)
            assert "oligomer_bonus" not in row
            assert row["scoring_function"] == pytest.approx(h.scoring_function, abs=1e-5), (inp.name, s)
    return rep, refs


@pytest.mark.parametrize("overlap", ["0", "1"])
@pytest.mark.parametrize("scoring", [[("Ed-Epf", 1.0)], [("Edef", 5.0), ("Ed-Epf", 0.3)]])
def test_avoid_records_match_host_scoring(engine, monkeypatch, scoring, overlap):
    monkeypatch.setenv("BF_DESIGN_OVERLAP", overlap)
    from desirna_b200 import design
    inputs = small_inputs()
    o = design.DesignOptions(replicas=6, RE_attempt=15, scoring_f=scoring, oligo_state="avoid")
    random.seed(5)
    loop = design.DesignLoop(inputs, o, seed=7)
    loop.run(3)
    rep, _ = check_against_host(loop, inputs, o, exact_epf=overlap == "0")
    assert (rep["counts"][:, 0] + rep["counts"][:, 2] == 3 * 15).all()
    loop.close()


def test_avoid_fraction_against_the_oracle(engine, oracle):
    """the self-dimer fraction from the CPU oracle's pf(s&s) columns FA, FB, FcAB, independent of the CUDA two-strand kernel"""
    from desirna_b200 import design
    inputs = small_inputs(limit=4)
    o = design.DesignOptions(replicas=5, RE_attempt=10, oligo_state="avoid")
    random.seed(11)
    loop = design.DesignLoop(inputs, o, seed=3)
    loop.run(2)
    rep = loop.replicas()
    loop.close()
    for g, s in enumerate(rep["sequence"]):
        rec = dict(zip(design.REC_FIELDS, rep["rec"][g]))
        cols = [f32(x) for x in oracle.pf(s + "&" + s)[:3]]
        dF = cols[2] - cols[0] - cols[1]
        rhs = 1e-3 / 55.14 * math.exp(-dF / KT)
        frac = 1 - (math.sqrt(1 + 4 * rhs) - 1) / (2 * rhs)
        # the columns agree to 1e-5 relative (test_device_records_against_the_oracle's Epf bound); the fraction moves by at most
        # |d dF| / kT
        tol = sum(1e-5 * max(1.0, abs(c)) for c in cols) / KT + 1e-9
        assert abs(rec["oligo_fraction"] - frac) <= tol, (s, rec["oligo_fraction"], frac)
        assert rec["oligomer_bonus"] == pytest.approx(-KT * math.log(1 - rec["oligo_fraction"]), abs=1e-12)


ALT = ("Alt_Struct_Example", "((((((.((((((((....))))).)).).))))))", ["(((((((((((((....)))..)).)).).))))).", "(((((((((((((....)))))...)).).)))))."])


@pytest.mark.parametrize("combo", ["alt_motifs", "subopt", "pks"])
def test_avoid_combines_with_the_other_device_terms(engine, combo):
    """avoid with alternative structures plus motifs, with -nd on, and with the pseudoknot overlay (the reference's avoid branch of
    get_mfe_e_ss runs it): records against the host mirror, whose term order is that of score_sequence"""
    from desirna_b200 import design
    from desirna_b200.utils import stats_inputs_outputs as sio
    if combo == "alt_motifs":
        alt = sio.make_input(ALT[0], ALT[1])
        alt.add_alt_sec_struct(ALT[2])
        inputs = [alt, sio.make_input("plain", "((((....))))....((((...)))).")]
        o = design.DesignOptions(replicas=6, RE_attempt=12, scoring_f=[("Ed-Epf", 0.7), ("1-MCC", 0.3)], motifs={"GNRA": -3.5, "UUCG": 2.0},
                                 oligo_state="avoid")
    elif combo == "subopt":
        inputs = [sio.make_input("hp", "((((....))))"), sio.make_input("two", "((((....))))..(((....)))"), sio.make_input("std", ALT[1])]
        o = design.DesignOptions(replicas=8, RE_attempt=25, subopt="on", oligo_state="avoid")
    else:
        inputs = [sio.make_input("Pseudoknot_Example", "((((((....[[[[..))))))......]]]]...."), sio.make_input("plain", "((((....))))....((((...)))).")]
        o = design.DesignOptions(replicas=6, RE_attempt=12, scoring_f=[("Ed-Epf", 0.5), ("1-MCC", 0.5)], pks="on", oligo_state="avoid")
    random.seed(21)
    loop = design.DesignLoop(inputs, o, seed=9)
    loop.run(4)
    rep, refs = check_against_host(loop, inputs, o)
    from desirna_b200.utils import energy_scores as es
    exercised = 0
    for g, h in enumerate(refs):
        rec = dict(zip(design.REC_FIELDS, rep["rec"][g]))
        if combo == "alt_motifs":
            assert rec["edesired2"] == pytest.approx(h.edesired2, abs=1e-12) and rec["motif_bonus"] == es.score_motifs(h.sequence, o)
            exercised += rec["motif_bonus"] != 0
        elif combo == "subopt":
            assert rec["subopt_e"] == h.subopt_e
            exercised += h.mfe_ss == inputs[g // loop.R].sec_struct
        else:
            exercised += "[" in h.mfe_ss
    assert exercised > 0
    loop.close()


def test_avoid_self_dimer_without_pairs(engine):
    """poly-A: no pair between the two copies, FcAB is the 999 sentinel; the fraction, the bonus and the score are what the host
    arithmetic makes of it (0/0: NaN), and a NaN mutant is never accepted"""
    from desirna_b200 import design
    from desirna_b200.utils import energy_scores as es
    from desirna_b200.utils import stats_inputs_outputs as sio
    inp = sio.make_input("polyA", "." * 12, "A" * 12)
    o = design.DesignOptions(replicas=2, RE_attempt=5, oligo_state="avoid")
    loop = design.DesignLoop([inp], o, seed=1)
    loop.run(2)
    rep = loop.replicas()
    loop.close()
    with np.errstate(invalid="ignore"):
        h = es.score_sequences(rep["sequence"], inp, o)
    for g in range(2):
        rec = dict(zip(design.REC_FIELDS, rep["rec"][g]))
        assert rep["sequence"][g] == "A" * 12
        for f_dev, f_host in (("oligo_fraction", "oligo_fraction"), ("oligomer_bonus", "monomer_bonus"), ("scoring_function", "scoring_function")):
            assert math.isnan(rec[f_dev]) and math.isnan(getattr(h[g], f_host)), (f_dev, rec[f_dev], getattr(h[g], f_host))
    assert (rep["counts"][:, 0] == 0).all() and (rep["counts"][:, 2] == 10).all()


def test_avoid_trajectory_and_result_files(engine, tmp_path):
    from desirna_b200 import design
    from desirna_b200.utils import stats_inputs_outputs as sio
    inputs = small_inputs(max_len=30, limit=2)
    o = design.DesignOptions(replicas=4, RE_attempt=20, oligo_state="avoid")
    results, info = design.design_batch(inputs, o, global_steps=3, seed=2, stop_when_solved=False, trajectory=True)
    for k, inp in enumerate(inputs):
        assert results[k]["monomer_bonus"] == results[k]["oligomer_bonus"] and math.isfinite(results[k]["oligo_fraction"])
        data = info["simulation_data"][k]
        assert len(data) == 4 * (3 + 1)
        for d in data:
            assert d["monomer_bonus"] == pytest.approx(-KT * math.log(1 - d["oligo_fraction"]), abs=1e-12)
        so = SimpleNamespace(infile=inp.name, outname=str(tmp_path / ("run%d" % k)), num_results=10, oligo="on", dimer="off", subopt="off", timlim=60)
        best, solved = sio.parse_and_output_results(data, inp, info["stats"][k], info["seconds"], so, "now")
        assert best[0]["mcc"] == min(d["mcc"] for d in data)
        traj = (tmp_path / ("run%d_traj.csv" % k)).read_text()
        assert traj.count("\n") == len(data) + 1 and "monomer_bonus" in traj.split("\n")[0]
        best_str = (tmp_path / ("run%d_best_str" % k)).read_text()
        assert ("oligo fraction" in best_str) == solved


def test_avoid_refused_for_two_strand_jobs(engine):
    """bf_design_create: oligo = 3 with a two-strand job is BF_ERR_ARG; the same job as a heterodimer, and oligo = 3 on one strand,
    are accepted"""
    from desirna_b200 import design
    L = design._bind()
    S = 8

    def create(oligo, len_a):
        keep = [design._chars(["(((())))"], S), np.array([8], np.int32), np.array([len_a], np.int32), np.full((1, S), 15, np.uint8),
                design._chars(["GGGGCCCC"], S), np.array([1.0]), np.array([0.5])]
        cfg = design.bf_design_t()
        cfg.n_jobs, cfg.replicas, cfg.stride = 1, 1, S
        cfg.target, cfg.len, cfg.len_a, cfg.allowed, cfg.init_seq, cfg.temps, cfg.tm_prob = (a.ctypes.data for a in keep)
        cfg.n_terms, cfg.re_attempt, cfg.metropolis_L, cfg.oligo = 1, 1, 504.12, oligo
        cfg.term[0], cfg.weight[0] = 0, 1.0
        h = C.c_void_p()
        rc = L.bf_design_create(C.byref(cfg), C.byref(h))
        if rc == 0:
            L.bf_design_destroy(h)
        return rc

    assert create(3, 4) == 5   # BF_ERR_ARG
    assert "single-strand" in L.bf_last_error().decode()
    assert create(1, 4) == 0
    assert create(3, 0) == 0

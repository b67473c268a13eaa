"""GPU: bf_interact (accessibility-aware RNA-RNA interaction, engine.interact) against the plain-C fixed-start recurrence of
tests/interact_ref.c fed the engine's own P_u (engine.unpaired / engine.plfold), against bf_duplex, and against the engine's
two-strand eval."""
import ctypes as C
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import PAR1999, ROOT
from interact_ref import INF, KT, InteractOracle, ed_rows

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def iref(oracle):
    return InteractOracle(PAR1999)


def rseq(rng, lo, hi):
    return "".join("ACGU"[x] for x in rng.integers(0, 4, int(rng.integers(lo, hi + 1))))


def pu_rows(engine, seqs, acc, span):
    """P_u rows [len, span] of every strand for accessibility mode acc, as bf_interact computes them (None for acc = -1)"""
    if acc < 0:
        return [None] * len(seqs)
    if acc == 0:
        S = max(map(len, seqs))
        pu = engine.unpaired(seqs, min(span, S))
        out = [pu[k, :len(s)] for k, s in enumerate(seqs)]
    else:
        out = [p for _, p in engine.plfold(seqs, acc, max_u=span, pairs=False)]
    return [np.pad(p, ((0, 0), (0, span - p.shape[1]))) for p in out]


def check_against_ref(engine, iref, A, B, pairs, span, acc_a, acc_b, exact=False):
    r = engine.interact(A, B, pairs=pairs, max_span=span, acc_a=acc_a, acc_b=acc_b)
    pa, pb = pu_rows(engine, A, acc_a, span), pu_rows(engine, B, acc_b, span)
    eda = [None if p is None else ed_rows(p, span) for p in pa]
    edb = [None if p is None else ed_rows(p, span) for p in pb]
    with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        refs = list(ex.map(lambda ab: iref.interact(A[ab[0]], B[ab[1]], span, eda[ab[0]], edb[ab[1]]), pairs))
    n_site = 0
    for p, ((ia, ib), x) in enumerate(zip(pairs, refs)):
        site, ss = tuple(int(v) for v in r["site"][p]), r["structures"][p]
        what = (p, A[ia], B[ib], span, acc_a, acc_b, float(r["e"][p]), int(r["h"][p]), site, x)
        if exact:   # no accessibility: everything bit for bit, ties included
            assert (float(r["e"][p]), int(r["h"][p]), site, ss) == (x["e"], x["h"], x["site"], x["ss"]), what
            assert r["ed_a"][p] == 0.0 and r["ed_b"][p] == 0.0
        else:
            assert (r["e"][p] == x["e"]) if x["e"] == np.inf else abs(r["e"][p] - x["e"]) <= 1e-9, what
            if x["gap"] > 1e-9:
                assert (int(r["h"][p]), site, ss) == (x["h"], x["site"], x["ss"]), what
        if int(r["h"][p]) < INF:
            n_site += 1
            k1, km, lm, l1 = site
            for ed, rows, k, u in ((r["ed_a"][p], pa[ia], k1, km - k1 + 1), (r["ed_b"][p], pb[ib], lm, l1 - lm + 1)):
                want = 0.0 if rows is None else -(KT / 1000.0) * np.log(rows[k - 1, u - 1])
                assert abs(ed - want) <= 1e-12 * max(1.0, abs(want)), what
            assert abs(r["e"][p] - (int(r["h"][p]) / 100.0 + r["ed_a"][p] + r["ed_b"][p])) == 0.0, what
        else:
            assert r["e"][p] == np.inf and site == (0, 0, 0, 0) and ss == "." * len(A[ia]) + "&" + "." * len(B[ib]), what
    return r, n_site


def test_ragged_short_pairs(engine, iref):
    rng = np.random.default_rng(1)
    A = [rseq(rng, 1, 40) for _ in range(300)]
    B = [rseq(rng, 1, 40) for _ in range(300)]   # accessibility below: strands of 1 .. 40 nt through the PF fill and outside pass
    pairs = [(k, k) for k in range(300)]
    _, n = check_against_ref(engine, iref, A, B, pairs, 25, -1, -1, exact=True)
    assert n >= 250
    check_against_ref(engine, iref, A, B, pairs, 25, 0, 0)
    check_against_ref(engine, iref, A, B, pairs, 25, -1, 40)


def test_span_1_and_64(engine, iref):
    rng = np.random.default_rng(2)
    A = [rseq(rng, 5, 80) for _ in range(60)]
    B = [rseq(rng, 5, 80) for _ in range(60)]
    pairs = [(k, k) for k in range(60)]
    for span in (1, 64):
        check_against_ref(engine, iref, A, B, pairs, span, -1, -1, exact=True)
        check_against_ref(engine, iref, A, B, pairs, span, 0, 0)


def test_guides_against_plfold_targets(engine, iref):
    """21-nt guides, global accessibility, against 500-2000 nt targets with RNAplfold window averages (W = 150)"""
    rng = np.random.default_rng(3)
    A = [rseq(rng, 21, 21) for _ in range(8)]
    B = [rseq(rng, 500, 2000) for _ in range(8)]
    check_against_ref(engine, iref, A, B, [(k, k) for k in range(8)], 25, 0, 150)


def test_200x200_global(engine, iref):
    rng = np.random.default_rng(4)
    A = [rseq(rng, 200, 200) for _ in range(4)]
    B = [rseq(rng, 200, 200) for _ in range(4)]
    check_against_ref(engine, iref, A, B, [(k, k) for k in range(4)], 25, 0, 0)


def test_length_cap(engine, iref):
    """2000 nt on both sides, with windowed accessibility on both as for long transcripts"""
    rng = np.random.default_rng(5)
    A = [rseq(rng, 2000, 2000), rseq(rng, 21, 21)]
    B = [rseq(rng, 2000, 2000)]
    check_against_ref(engine, iref, A, B, [(0, 0), (1, 0)], 4, -1, -1, exact=True)
    check_against_ref(engine, iref, A, B, [(0, 0), (1, 0)], 4, 80, 80)


def test_several_launches(engine, iref):
    """a 2000-nt a strand sets 2000 (pair, k1) slots per pair, so 5000 pairs exceed one launch's slot budget: two launches of
    bf_k_interact + bf_k_interact_reduce, results written at each launch's offset"""
    rng = np.random.default_rng(6)
    A = [rseq(rng, 2000, 2000)] + [rseq(rng, 8, 30) for _ in range(4999)]
    B = [rseq(rng, 8, 30) for _ in range(5000)]
    pairs = [(k, k) for k in range(5000)]
    n0 = engine.kernel_launches()
    r2 = engine.interact(A, B, pairs=pairs, max_span=16, acc_a=-1, acc_b=-1, structures=False)
    assert engine.kernel_launches() - n0 == 4
    r = engine.interact(A, B, pairs=pairs, max_span=16, acc_a=-1, acc_b=-1)
    for k in ("e", "h", "ed_a", "ed_b", "site"):
        assert (r2[k] == r[k]).all(), k
    for p in list(range(0, 5000, 41)) + [4194, 4195, 4999]:
        x = iref.interact(A[p], B[p], 16)
        assert (float(r["e"][p]), int(r["h"][p]), tuple(int(v) for v in r["site"][p]), r["structures"][p]) == \
            (x["e"], x["h"], x["site"], x["ss"]), (p, x)
    check_against_ref(engine, iref, A[4000:4400], B[4000:4400], [(k, k) for k in range(400)], 16, 0, 0)


def test_duplex_grid_and_modes(engine):
    """no accessibility and max_span >= both lengths: 100 E is bf_duplex's energy on every pair of a 64 x 64 grid; grid equals
    pair list; energies-only equals structure mode"""
    rng = np.random.default_rng(7)
    A = [rseq(rng, 5, 64) for _ in range(64)]
    B = [rseq(rng, 5, 64) for _ in range(64)]
    g = engine.interact(A, B, max_span=64, acc_a=-1, acc_b=-1)
    d = engine.duplex(A, B, structures=False)
    assert g["e"].shape == (64, 64) and g["site"].shape == (64, 64, 4) and len(g["structures"]) == 64
    assert (g["h"] == d).all()
    assert (g["e"] == np.where(d < INF, d / 100.0, np.inf)).all()
    pairs = [(a, b) for a in range(64) for b in range(64)]
    for acc in ((-1, -1), (0, 0)):
        gg = engine.interact(A, B, max_span=20, acc_a=acc[0], acc_b=acc[1])
        pl = engine.interact(A, B, pairs=pairs, max_span=20, acc_a=acc[0], acc_b=acc[1])
        en = engine.interact(A, B, max_span=20, acc_a=acc[0], acc_b=acc[1], structures=False)
        for k in ("e", "h", "ed_a", "ed_b"):
            assert (pl[k] == gg[k].reshape(-1)).all() and (en[k] == gg[k]).all(), (acc, k)
        assert (pl["site"] == gg["site"].reshape(-1, 4)).all() and (en["site"] == gg["site"]).all()
        assert pl["structures"] == [s for row in gg["structures"] for s in row] and "structures" not in en


def test_engine_eval_of_sites(engine):
    """H equals the engine's two-strand eval of the returned structure on a&b"""
    rng = np.random.default_rng(8)
    A = [rseq(rng, 10, 60) for _ in range(200)]
    B = [rseq(rng, 10, 60) for _ in range(200)]
    r = engine.interact(A, B, pairs=[(k, k) for k in range(200)], max_span=25, acc_a=0, acc_b=0)
    keep = [k for k in range(200) if r["h"][k] < INF]
    assert len(keep) >= 180
    out = engine.score_batch([A[k] + "&" + B[k] for k in keep], [[r["structures"][k].replace("&", "")] for k in keep],
                             want=engine.WANT_EVAL)
    assert (out["eval_dcal"][:, 0] == r["h"][keep]).all()


def test_same_strand_set_on_both_sides(engine):
    rng = np.random.default_rng(9)
    A = [rseq(rng, 20, 50) for _ in range(12)]
    g = engine.interact(A, A, max_span=25, acc_a=0, acc_b=0)
    h = engine.interact(A, list(A), max_span=25, acc_a=0, acc_b=0)
    for k in ("e", "h", "ed_a", "ed_b", "site"):
        assert (g[k] == h[k]).all(), k


def test_errors(engine):
    from desirna_b200 import engine as E
    L = E.lib()

    def call(a_seqs, a_lens, b_seqs, b_lens, pairs=None, n_pairs=0, stride_a=None, span=8, acc_a=-1, acc_b=-1, e_buf=True):
        q = E.bf_interact_t()
        keep = []
        for st, seqs, lens, stride in ((q.a, a_seqs, a_lens, stride_a), (q.b, b_seqs, b_lens, None)):
            buf, _, _ = E.pack(seqs, stride)
            ln = np.asarray(lens, np.int32)
            st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, ln.ctypes.data
            keep += [buf, ln]
        if pairs is not None:
            pr = np.asarray(pairs, np.int32).reshape(-1, 2)
            q.pairs, q.n_pairs = pr.ctypes.data, n_pairs
            keep.append(pr)
        q.max_span, q.acc_a, q.acc_b = span, acc_a, acc_b
        e = np.zeros(max(1, len(a_seqs) * len(b_seqs), n_pairs), np.float64)
        return L.bf_interact(C.byref(q), e.ctypes.data if e_buf else None, None, None, None, None)

    ARG, UNAV = 5, 4
    assert call(["GGGG"], [4], ["CCCC"], [4]) == 0
    assert L.bf_interact(None, None, None, None, None, None) == ARG                      # null query
    assert call(["GGGG"], [4], ["CCCC"], [4], e_buf=False) == ARG                        # null e
    assert call(["GGGG"], [5], ["CCCC"], [4]) == ARG                                     # bad strand set
    assert call(["GGGG"], [4], ["CCCC"], [4], span=0) == ARG                             # max_span outside 1 .. 64
    assert call(["GGGG"], [4], ["CCCC"], [4], span=65) == ARG
    assert call(["GGGG"], [4], ["CCCC"], [4], acc_a=-2) == ARG                           # acc < -1
    assert call(["GGGG"], [4], ["CCCC"], [4], acc_b=7) == ARG                            # window below max_span
    assert call(["GGGG"], [4], ["CCCC"], [4], pairs=[(0, 0)], n_pairs=-1) == ARG         # n_pairs < 0
    assert call(["GGGG"], [4], ["CCCC"], [4], pairs=[(0, 1)], n_pairs=1) == ARG          # pair index out of range
    assert call(["GGGG"], [4], ["C" * 2001], [2001], acc_b=-1) == ARG                    # over the 2000-nt cap
    assert call(["GGGG"], [4], ["CCCC"], [4], acc_b=2001) == UNAV                        # window longer than the fill path
    with pytest.raises(ValueError):
        engine.interact(["GG&CC"], ["GGCC"])
    # strands longer than the PF fill path covers, and BF_FORCE_GENERIC with accessibility on: a fresh process each
    code = ("import ctypes as C, sys, numpy as np; sys.path.insert(0, %r); from desirna_b200 import engine as E; L = E.lib(); "
            "q = E.bf_interact_t(); e = (C.c_double * 1)(); r0 = L.bf_interact(C.byref(q), e, None, None, None, None); "
            "L.bf_init(0); r1 = L.bf_interact(C.byref(q), e, None, None, None, None); print(r0, r1)") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=ROOT)
    assert out.stdout.split() == ["2", "2"], out                                        # BF_ERR_NOT_INIT before init / parameters
    code = ("import sys; sys.path.insert(0, %r); from desirna_b200 import engine as E\n"
            "try:\n    E.interact(['GGGGAAAACCCC'], ['GGGGAAAACCCC'], acc_a=0, acc_b=-1)\nexcept E.EngineError as x:\n    print(x.code)\n"
            "print(int(E.interact(['GGGG'], ['CCCC'], acc_a=-1, acc_b=-1)['h'][0, 0]))") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=ROOT,
                         env=dict(os.environ, BF_FORCE_GENERIC="1"))
    assert out.stdout.split()[0] == str(UNAV) and int(out.stdout.split()[1]) < 0, out   # BF_FORCE_GENERIC: no accessibility

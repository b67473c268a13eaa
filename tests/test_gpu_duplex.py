"""GPU: bf_duplex (RNA-RNA hybridization, engine.duplex, RNA.duplexfold) against a brute force over every duplex chain, against the
plain-C recurrence of tests/duplex_ref.c (energies and structures bit for bit), and against the engine's own two-strand eval and
cofold MFE."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import PAR1999, ROOT
from duplex_ref import INF, DuplexOracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dref(oracle):
    return DuplexOracle(PAR1999)


def rseq(rng, lo, hi):
    return "".join("ACGU"[x] for x in rng.integers(0, 4, int(rng.integers(lo, hi + 1))))


def check_against_ref(engine, dref, A, B, pairs):
    e, ss = engine.duplex(A, B, pairs=pairs)
    for p, (ia, ib) in enumerate(pairs):
        er, sr = dref.duplex(A[ia], B[ib])
        assert int(e[p]) == er, (p, A[ia], B[ib], int(e[p]), er)
        assert ss[p] == sr, (p, A[ia], B[ib], ss[p], sr)
    return e, ss


def test_brute_force(engine, dref):
    rng = np.random.default_rng(1)
    A = [rseq(rng, 1, 9) for _ in range(220)]
    B = [rseq(rng, 1, 9) for _ in range(220)]
    pairs = [(k, k) for k in range(len(A))]
    e, ss = engine.duplex(A, B, pairs=pairs)
    n_pair = 0
    for k in range(len(A)):
        assert int(e[k]) == dref.duplex_brute(A[k], B[k]), (A[k], B[k], int(e[k]))
        if e[k] < INF:
            n_pair += 1
            assert dref.eval_duplex(A[k], B[k], ss[k]) == int(e[k]), (A[k], B[k], ss[k])
        else:
            assert ss[k] == "." * len(A[k]) + "&" + "." * len(B[k])
    assert n_pair >= 150


def test_against_reference_ragged(engine, dref):
    rng = np.random.default_rng(2)
    A = [rseq(rng, 1, 60) for _ in range(500)]
    B = [rseq(rng, 1, 60) for _ in range(500)]
    check_against_ref(engine, dref, A, B, [(k, k) for k in range(500)])


def test_against_reference_guide_vs_long_targets(engine, dref):
    rng = np.random.default_rng(3)
    A = [rseq(rng, 21, 21) for _ in range(64)]
    B = [rseq(rng, 500, 2000) for _ in range(64)]
    check_against_ref(engine, dref, A, B, [(k, k) for k in range(64)])


def test_against_reference_200x200(engine, dref):
    rng = np.random.default_rng(4)
    A = [rseq(rng, 200, 200) for _ in range(16)]
    B = [rseq(rng, 200, 200) for _ in range(16)]
    check_against_ref(engine, dref, A, B, [(k, k) for k in range(16)])


def test_against_reference_length_caps(engine, dref):
    """1 and 2000 nt on either side; 2000 x 2000 keeps its c ring in HBM (it does not fit shared memory)"""
    rng = np.random.default_rng(5)
    A = [rseq(rng, 1, 1), rseq(rng, 2000, 2000), "G"]
    B = [rseq(rng, 1, 1), rseq(rng, 2000, 2000), "C"]
    e, _ = check_against_ref(engine, dref, A, B, [(0, 0), (0, 1), (1, 0), (1, 1), (2, 2)])
    assert int(e[4]) < INF and int(e[3]) < 0
    e2 = engine.duplex(A, B, pairs=[(0, 0), (0, 1), (1, 0), (1, 1), (2, 2)], structures=False)
    assert (e2 == e).all()


def test_chunked_launches_with_hbm_ring(engine, dref):
    """one 2000 x 2000 pair moves every ring of the call to HBM; with 2000 more pairs of 21 x 200 nt, rings and c tables exceed one
    launch's workspace, so the call runs in several launches (c tables placed after the rings, results written at each chunk's offset)"""
    rng = np.random.default_rng(9)
    A = [rseq(rng, 21, 21) for _ in range(2000)] + [rseq(rng, 2000, 2000)]
    B = [rseq(rng, 200, 200) for _ in range(2000)] + [rseq(rng, 2000, 2000)]
    pairs = [(k, k) for k in range(1000)] + [(2000, 2000)] + [(k, k) for k in range(1000, 2000)]
    n0 = engine.kernel_launches()
    e, _ = check_against_ref(engine, dref, A, B, pairs)
    assert engine.kernel_launches() - n0 >= 3
    assert (engine.duplex(A, B, pairs=pairs, structures=False) == e).all()


def test_engine_eval_and_cofold(engine):
    """the engine's two-strand eval of every returned structure equals its energy; the cofold MFE is no higher"""
    rng = np.random.default_rng(6)
    A = [rseq(rng, 5, 40) for _ in range(300)]
    B = [rseq(rng, 5, 40) for _ in range(300)]
    e, ss = engine.duplex(A, B, pairs=[(k, k) for k in range(300)])
    keep = [k for k in range(300) if e[k] < INF]
    assert len(keep) >= 250
    seqs = [A[k] + "&" + B[k] for k in keep]
    out = engine.score_batch(seqs, [[ss[k].replace("&", "")] for k in keep], want=engine.WANT_MFE | engine.WANT_EVAL)
    assert (out["eval_dcal"][:, 0] == e[keep]).all()
    assert (out["mfe_dcal"] <= e[keep]).all()


def test_grid_and_modes(engine, dref):
    rng = np.random.default_rng(7)
    A = [rseq(rng, 8, 45) for _ in range(23)]
    B = [rseq(rng, 3, 50) for _ in range(17)]
    eg, sg = engine.duplex(A, B)
    assert eg.shape == (23, 17) and len(sg) == 23 and len(sg[0]) == 17
    pairs = [(a, b) for a in range(23) for b in range(17)]
    el, sl = engine.duplex(A, B, pairs=pairs)
    assert (el == eg.reshape(-1)).all()
    assert sl == [s for row in sg for s in row]
    assert (engine.duplex(A, B, structures=False) == eg).all()
    assert (engine.duplex(A, B, pairs=pairs, structures=False) == el).all()
    # a pair list in any order, with repeats
    perm = [pairs[k] for k in rng.permutation(len(pairs))[:200]] + [pairs[0]] * 3
    ep, sp = engine.duplex(A, B, pairs=perm)
    for p, (a, b) in enumerate(perm):
        assert ep[p] == eg[a, b] and sp[p] == sg[a][b]


def test_full_gpu_grid(engine, dref):
    """512 x 512 strands of 30-60 nt (every SM busy), energies only, sampled entries against the reference"""
    rng = np.random.default_rng(8)
    A = [rseq(rng, 30, 60) for _ in range(512)]
    B = [rseq(rng, 30, 60) for _ in range(512)]
    e = engine.duplex(A, B, structures=False)
    assert e.shape == (512, 512)
    for a, b in zip(rng.integers(0, 512, 2000), rng.integers(0, 512, 2000)):
        assert int(e[a, b]) == dref.duplex(A[a], B[b])[0], (a, b)


def test_errors(engine):
    from desirna_b200 import engine as E
    L = E.lib()

    def call(a_seqs, a_lens, b_seqs, b_lens, pairs=None, n_pairs=0, stride_a=None, stride_b=None, e_buf=True):
        q = E.bf_duplex_t()
        keep = []
        for st, seqs, lens, stride in ((q.a, a_seqs, a_lens, stride_a), (q.b, b_seqs, b_lens, stride_b)):
            buf, _, _ = E.pack(seqs, stride)
            ln = np.asarray(lens, np.int32)
            st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, ln.ctypes.data
            keep += [buf, ln]
        if pairs is not None:
            pr = np.asarray(pairs, np.int32).reshape(-1, 2)
            q.pairs, q.n_pairs = pr.ctypes.data, n_pairs
            keep.append(pr)
        e = np.zeros(max(1, len(a_seqs) * len(b_seqs), n_pairs), np.int32)
        return L.bf_duplex(C.byref(q), e.ctypes.data if e_buf else None, None)

    ARG = 5
    assert call(["GGGG"], [4], ["CCCC"], [4]) == 0
    assert call(["GGGG"], [4], ["CCCC"], [4], e_buf=False) == ARG                   # null output
    assert L.bf_duplex(None, None, None) == ARG                                     # null query
    assert call(["GGGG"], [5], ["CCCC"], [4]) == ARG                                # len > stride
    assert call(["GGGG"], [-1], ["CCCC"], [4]) == ARG
    assert call(["G" * 2001], [2001], ["CCCC"], [4]) == ARG                         # over the 2000-nt cap
    assert call(["GGGG"], [4], ["C" * 2001], [2001]) == ARG
    assert call(["GGGG"], [4], ["CCCC"], [4], pairs=[(1, 0)], n_pairs=1) == ARG     # pair index out of range
    assert call(["GGGG"], [4], ["CCCC"], [4], pairs=[(0, 1)], n_pairs=1) == ARG
    assert call(["GGGG"], [4], ["CCCC"], [4], pairs=[(0, -1)], n_pairs=1) == ARG
    assert call(["GGGG"], [4], ["CCCC"], [4], pairs=[(0, 0)], n_pairs=-1) == ARG
    assert call(["GGGG"], [4], ["CCCC"], [4], stride_a=(1 << 16) + 1) == ARG          # stride over the bound
    with pytest.raises(ValueError):
        engine.duplex(["GG&CC"], ["GGCC"])                                          # one strand per entry
    with pytest.raises(E.EngineError) as ei:
        engine.duplex(["G" * 2001], ["C"])
    assert ei.value.code == ARG
    # before bf_init and before parameters are loaded: BF_ERR_NOT_INIT (a fresh process)
    code = ("import ctypes as C, sys; sys.path.insert(0, %r); from desirna_b200 import engine as E; L = E.lib(); q = E.bf_duplex_t();"
            "e = (C.c_int32 * 1)(); r0 = L.bf_duplex(C.byref(q), e, None); L.bf_init(0); r1 = L.bf_duplex(C.byref(q), e, None);"
            "print(r0, r1)") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=ROOT)
    assert out.stdout.split() == ["2", "2"], out


def test_rna_duplexfold(engine):
    from desirna_b200 import RNA
    cases = [
        ("GGGG", "CCCC", "((((&))))", -5.8, 4, 1),                                  # pairs at every strand end
        ("AAAAGGGGAAAA", "CCCC", ".((((.&))))", -7.1, 9, 1),
        ("GGGG", "AAACCCCAAA", "((((&.)))).", -8.0, 4, 3),
        ("UGCAUCGAUCGAU", "AUCGAUCGAUGCA", ".((((((((((((&)))))))))))).", -20.3, 13, 1),
        ("ACGUAGGCAUCUA", "GAUGCCUACG", ".((((((((((.&))))))))))", -17.9, 12, 1),
        ("ACGTAGGCATCTA", "GATGCCTACG", ".((((((((((.&))))))))))", -17.9, 12, 1),   # T read as U
    ]
    for s1, s2, st, en, i, j in cases:
        d = RNA.duplexfold(s1, s2)
        assert (d.structure, d.i, d.j) == (st, i, j), (s1, s2, d)
        assert isinstance(d.energy, float) and abs(d.energy - en) < 1e-9, (s1, s2, d)
    d = RNA.duplexfold("AAAA", "CCCC")
    assert (d.structure, d.energy, d.i, d.j) == ("....&....", 100000.0, 4, 1)

"""GPU: bf_findpath (direct refolding paths, engine.findpath, fc.path_findpath_saddle / fc.path_findpath) against the plain-C beam
of tests/findpath_ref.c bit for bit, against the exact subset DP, and against the engine's own eval."""
import ctypes as C
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import PAR1999, ROOT
from findpath_ref import INF, FindpathOracle, check_path, perturb, random_structure

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fref(oracle):
    return FindpathOracle(PAR1999)


def rseq(rng, n, alpha="ACGU"):
    return "".join(rng.choice(list(alpha), n))


def instances(engine, rng, count, lo, hi, max_moves=None):
    """(seq, s1, s2): s1 the MFE; s2 a Boltzmann sample, a perturbed MFE (non-canonical pairs included) or a random structure.  Every
    third sequence is low-complexity (GC or AU only), so that energy ties occur."""
    seqs = []
    for x in range(count):
        n = int(rng.integers(lo, hi + 1))
        seqs.append(rseq(rng, n, ("ACGU", "GC", "AU")[x % 3]))
    mfe = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]
    samp = engine.sample(seqs, 1, seed=int(rng.integers(1 << 30)))
    out = []
    for x, (s, s1) in enumerate(zip(seqs, mfe)):
        kind = x % 4 if max_moves is None else 1
        if kind == 0:
            s2 = samp[x][0]
        elif kind in (1, 2):
            m = max_moves or 12
            s2 = perturb(rng, s1, int(rng.integers(0, m // 2 + 1)), int(rng.integers(0, m // 2 + 1)))
        else:
            s2 = random_structure(rng, len(s))
        out.append((s, s1, s2))
    return out


def run_ref(fref, cases, W):
    with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda c: fref.findpath(c[0], c[1], c[2], W), cases))


def check_exact(engine, fref, cases, W):
    sad, paths = engine.findpath([c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], W)
    refs = run_ref(fref, cases, W)
    n_moves = 0
    for r, (c, x) in enumerate(zip(cases, refs)):
        mv, pe = paths[r]
        got = (int(sad[r]), [tuple(int(v) for v in m) for m in mv], [int(v) for v in pe])
        assert got == (x["saddle"], x["moves"], x["path_e"]), (W, c, got, x)
        assert int(sad[r]) == max(got[2])
        check_path(c[1], c[2], got[1])
        n_moves += len(got[1])
    return n_moves


@pytest.mark.parametrize("W,count,lo,hi", [(1, 24, 20, 300), (2, 24, 20, 300), (3, 24, 20, 300), (10, 16, 20, 150), (64, 12, 20, 80),
                                           (1024, 8, 20, 60)])
def test_exact_against_reference(engine, fref, W, count, lo, hi):
    rng = np.random.default_rng(100 + W)
    cases = instances(engine, rng, count, lo, hi, max_moves=14 if W == 1024 else None)
    assert check_exact(engine, fref, cases, W) > 0


def test_against_dp(engine, fref):
    """k <= 12: no level holds more than C(12, 6) = 924 states, so W = 1024 keeps them all and finds the optimum"""
    rng = np.random.default_rng(7)
    cases = [c for c in instances(engine, rng, 40, 20, 80, max_moves=12)]
    sad, paths = engine.findpath([c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], 1024)
    with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        dp = list(ex.map(lambda c: fref.findpath_dp(c[0], c[1], c[2]), cases))
    for r, c in enumerate(cases):
        assert len(paths[r][0]) <= 12 and dp[r] < INF
        assert int(sad[r]) == dp[r], (c, int(sad[r]), dp[r])


@pytest.mark.parametrize("n,W", [(400, 8), (2000, 2)])
def test_energies_against_eval(engine, n, W):
    rng = np.random.default_rng(n)
    seqs = [rseq(rng, n) for _ in range(2)]
    s1 = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]
    s2 = [perturb(rng, s1[0], 60, 60), perturb(rng, s1[1], 5, 5)]   # non-canonical pairs on the way
    sad, paths = engine.findpath(seqs, s1, s2, W)
    for r in range(2):
        structs = check_path(s1[r], s2[r], [tuple(int(v) for v in m) for m in paths[r][0]])
        ev = engine.score_batch([seqs[r]], [structs], want=engine.WANT_EVAL)["eval_dcal"][0]
        assert [int(v) for v in paths[r][1]] == [int(v) for v in ev], r
        assert int(sad[r]) == max(int(v) for v in ev)
        assert r == 1 or len(structs) > 50


def test_ragged_batch(engine):
    rng = np.random.default_rng(11)
    cases = instances(engine, rng, 60, 10, 200)
    cases.append(("GGGGAAAACCCC", "((((....))))", "((((....))))"))   # equal structures: k = 0
    cases.append(("GGGGAAAACCCC", "............", "............"))
    seqs, s1, s2 = [c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases]
    sad, paths = engine.findpath(seqs, s1, s2, 64)
    assert engine.findpath(seqs, s1, s2, 64, path=False).tolist() == sad.tolist()
    for r in (0, 17, 59, 60, 61):   # each alone, with its own stride
        s1r, p1r = engine.findpath([seqs[r]], [s1[r]], [s2[r]], 64)
        assert int(s1r[0]) == int(sad[r]) and (p1r[0][0] == paths[r][0]).all() and (p1r[0][1] == paths[r][1]).all(), r
    assert len(paths[60][0]) == 0 and int(sad[60]) == int(paths[60][1][0]) == int(engine.score_batch(
        [seqs[60]], [[s1[60]]], want=engine.WANT_EVAL)["eval_dcal"][0, 0])
    assert int(sad[61]) == 0 and len(paths[61][0]) == 0


def test_launch_split(engine):
    """a 1 MB budget splits the call into several launches (back-pointers) on a smaller grid (workspaces): the same results"""
    rng = np.random.default_rng(12)
    seqs = [rseq(rng, int(rng.integers(300, 401))) for _ in range(16)]
    s1 = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]
    s2 = [random_structure(rng, len(s)) for s in seqs]
    sad, paths = engine.findpath(seqs, s1, s2, 64)
    engine.set_option("findpath_mb", 1)
    try:
        n0 = engine.kernel_launches()
        sad2, paths2 = engine.findpath(seqs, s1, s2, 64)
        assert engine.kernel_launches() - n0 > 4
    finally:
        engine.set_option("findpath_mb", -1)
    assert sad2.tolist() == sad.tolist()
    for r in range(len(seqs)):
        assert (paths2[r][0] == paths[r][0]).all() and (paths2[r][1] == paths[r][1]).all(), r


def test_shim(engine, fref):
    from desirna_b200 import RNA
    rng = np.random.default_rng(21)
    for seq, s1, s2 in instances(engine, rng, 6, 30, 120):
        fc = RNA.fold_compound(seq)
        x = fref.findpath(seq, s1, s2, 4)
        assert fc.path_findpath_saddle(s1, s2, 4) == x["saddle"]
        assert fc.path_findpath_saddle(s1, s2) == fref.findpath(seq, s1, s2, 1)["saddle"]
        p = fc.path_findpath(s1, s2, 4)
        structs = check_path(s1, s2, x["moves"])
        assert [q.s for q in p] == structs
        assert [q.en for q in p] == [RNA.f32(e / 100.0) for e in x["path_e"]]
    with pytest.raises(NotImplementedError):
        RNA.fold_compound("GGGGAAAA&CCCCAAAA").path_findpath_saddle("((((....&))))....", "........&........")
    with pytest.raises(NotImplementedError):
        RNA.fold_compound("GGGGAAAA&CCCCAAAA").path_findpath("((((....&))))....", "........&........")


def test_errors(engine):
    from desirna_b200 import engine as E
    L = E.lib()

    def call(seqs, lens, s1, s2, width=2, stride=None, sad_buf=True, n=None):
        buf, _, _ = E.pack(seqs, stride)
        S = buf.shape[1]
        t1 = np.frombuffer("".join(x.ljust(S, ".")[:S] for x in s1).encode(), np.uint8).copy()
        t2 = np.frombuffer("".join(x.ljust(S, ".")[:S] for x in s2).encode(), np.uint8).copy()
        ln = np.asarray(lens, np.int32)
        q = E.bf_findpath_t()
        q.n, q.stride, q.seq, q.len, q.s1, q.s2, q.width = len(seqs) if n is None else n, S, buf.ctypes.data, ln.ctypes.data, \
            t1.ctypes.data, t2.ctypes.data, width
        sad = np.zeros(max(1, len(seqs)), np.int32)
        return L.bf_findpath(C.byref(q), sad.ctypes.data if sad_buf else None, None, None, None)

    ARG = 5
    ok = ("GGGGAAAACCCC", "((((....))))", "............")
    assert call([ok[0]], [12], [ok[1]], [ok[2]]) == 0
    assert call([ok[0]], [12], [ok[1]], [ok[2]], width=1) == 0 and call([ok[0]], [12], [ok[1]], [ok[2]], width=1024) == 0
    assert L.bf_findpath(None, None, None, None, None) == ARG                                # null query
    assert call([ok[0]], [12], [ok[1]], [ok[2]], sad_buf=False) == ARG                       # null saddle buffer
    assert call([ok[0]], [12], [ok[1]], [ok[2]], n=-1) == ARG                                # n < 0
    assert call([ok[0]], [13], [ok[1]], [ok[2]]) == ARG                                      # len > stride
    assert call(["G" * 2001], [2001], ["." * 2001], ["." * 2001]) == ARG                     # stride > 2000
    assert call([ok[0]], [12], [ok[1]], [ok[2]], width=0) == ARG                             # width outside 1 .. 1024
    assert call([ok[0]], [12], [ok[1]], [ok[2]], width=1025) == ARG
    assert call([ok[0]], [12], ["(((.....))))"], [ok[2]]) == ARG                             # unbalanced
    assert call([ok[0]], [12], [ok[1]], ["((((....)))("]) == ARG
    assert call([ok[0]], [12], ["((((....))))"], ["((((.x..))))"]) == ARG                    # another character
    assert call([ok[0]], [12], [ok[1]], ["((((.))))..."]) == ARG                             # a pair with j - i < 4
    assert call(["GGGGAANACCCC"], [12], [ok[1]], [ok[2]]) == ARG                             # a sequence character other than ACGUT
    assert call(["G" * 2000], [2000], ["." * 2000], ["." * 2000], width=1) == 0              # the 2000-nt cap
    with pytest.raises(ValueError):
        engine.findpath(["GG&CC"], ["(...)"], ["....."])
    code = ("import ctypes as C, sys, numpy as np; sys.path.insert(0, %r); from desirna_b200 import engine as E; L = E.lib(); "
            "q = E.bf_findpath_t(); q.width = 1; q.stride = 1; s = (C.c_int32 * 1)(); r0 = L.bf_findpath(C.byref(q), s, None, None, None); "
            "L.bf_init(0); r1 = L.bf_findpath(C.byref(q), s, None, None, None); print(r0, r1)") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=ROOT)
    assert out.stdout.split() == ["2", "2"], out                                            # BF_ERR_NOT_INIT before init / parameters

"""GPU: accessibility -- probabilities of unpaired stretches (bf_unpaired, engine.unpaired) and RNAplfold window averages
(bf_plfold, engine.plfold, RNA.pfl_fold_up / RNA.pfl_fold).

References computed without the new kernels: exact enumeration of every structure of short sequences (the oracle's per-structure
weights), Z(stretch masked) / Z from tests/unpaired_ref.c, the identity P_u(i, 1) = 1 - sum_j p_ij against the outside pass's
WANT_BPP for every fill family, and window averages taken on the host from bf_unpaired / WANT_BPP of the window substrings."""
import ctypes as C
import os

import numpy as np
import pytest

from struct_weight import WeightOracle
from unpaired_ref import UnpairedOracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAR1999 = os.path.join(ROOT, "desirna_b200", "params", "turner1999_37C.par")
SHORT = ["GGGGAAAACCCC", "GGCAGGGGACUGCC", "GAGCACGGGAGAC", "GCCUGGAUUAACAGGC", "GGGAGCAAAGCACCC", "GCGCUUCGGCGC", "AAAAAAAAAA"]


@pytest.fixture(scope="module")
def oracles():
    from oracle.pyoracle import build
    build()
    return UnpairedOracle(PAR1999), WeightOracle(PAR1999)


def rand_seqs(rng, lo, hi, B):
    return ["".join("ACGU"[x] for x in rng.integers(0, 4, int(rng.integers(lo, hi + 1)))) for _ in range(B)]


def unpaired_from_bpp(engine, seqs):
    """1 - sum_j p_ij per position from the outside pass (WANT_BPP), [B, stride]"""
    P = engine.score_batch(seqs, want=engine.WANT_BPP)["bpp"]
    return 1.0 - P.sum(axis=1) - P.sum(axis=2)


def check_invariants(pu, lens, tol=1e-12):
    for b, n in enumerate(lens):
        x = pu[b, :n]
        assert (x >= 0.0).all() and (x <= 1.0).all()
        U = x.shape[1]
        for u in range(1, min(U, n)):
            # P(i, u+1) <= min(P(i, u), P(i+1, u)) where i+u <= n
            a, left, right = x[:n - u, u], x[:n - u, u - 1], x[1:n - u + 1, u - 1]
            assert (a <= left + tol).all() and (a <= right + tol).all(), (b, u)
        for i in range(n):
            assert (x[i, n - i:] == 0.0).all()
        assert (pu[b, n:] == 0.0).all()


def test_short_sequences_against_enumeration(engine, oracles):
    _, wo = oracles
    rng = np.random.default_rng(3)
    seqs = SHORT + rand_seqs(rng, 12, 16, 13)
    stride = max(map(len, seqs))
    pu = engine.unpaired(seqs, stride)
    for b, s in enumerate(seqs):
        structs = [db for _, db in wo.enumerate_band(s, 10 ** 6, cap=200000)]
        w = np.array([wo.weight(s, db) for db in structs])
        Z = w.sum()
        n = len(s)
        for i in range(1, n + 1):
            for u in range(1, n - i + 2):
                e = w[[db[i - 1:i - 1 + u] == "." * u for db in structs]].sum() / Z
                assert abs(pu[b, i - 1, u - 1] - e) <= 1e-10, (s, i, u, pu[b, i - 1, u - 1], e)
    check_invariants(pu, [len(s) for s in seqs])


@pytest.mark.parametrize("L", [60, 100, 200])
def test_every_short_stretch_against_masked_reference(engine, oracles, L):
    uo, _ = oracles
    seqs = rand_seqs(np.random.default_rng(L), L, L, 2)
    pu = engine.unpaired(seqs, 8)
    for b, s in enumerate(seqs):
        st = [(i, u) for i in range(1, L + 1) for u in range(1, 9) if i + u - 1 <= L]
        ref = uo.unpaired(s, st)
        got = np.array([pu[b, i - 1, u - 1] for i, u in st])
        big = ref > 1e-12
        rel = np.abs(got[big] - ref[big]) / ref[big]
        assert rel.max() <= 1e-8, (L, b, st[int(np.flatnonzero(big)[rel.argmax()])], rel.max())
        assert np.abs(got[~big] - ref[~big]).max(initial=0.0) <= 1e-12
    check_invariants(pu, [L] * 2)


def test_sampled_stretches_400(engine, oracles):
    uo, _ = oracles
    rng = np.random.default_rng(400)
    s = rand_seqs(rng, 400, 400, 1)[0]
    pu = engine.unpaired([s], 31)
    st = [(int(i), int(u)) for i, u in zip(rng.integers(1, 370, 40), rng.integers(1, 32, 40))]
    ref = uo.unpaired(s, st)
    for (i, u), r in zip(st, ref):
        g = pu[0, i - 1, u - 1]
        assert (abs(g - r) <= 1e-8 * r) if r > 1e-12 else abs(g - r) <= 1e-12, (i, u, g, r)


# (family, batch, switches) as in the outside-pass tests: each fill family leaves the qb / qm / qm1 tables the passes read
def family_batch(name):
    rng = np.random.default_rng({"tap": 1, "round1": 2, "cluster": 3, "wide16": 4}[name])
    if name == "tap":
        return rand_seqs(rng, 60, 140, 40), {}
    if name == "round1":
        return rand_seqs(rng, 150, 260, 60), {"BF_FILL3": "0"}
    if name == "cluster":
        return rand_seqs(rng, 150, 400, 6), {"BF_CL": "1"}
    return rand_seqs(rng, 180, 260, 12), {"BF_FILL3_SMALL": "0", "BF_CL": "0"}


@pytest.mark.parametrize("name", ["tap", "round1", "cluster", "wide16"])
def test_single_positions_against_bpp(engine, monkeypatch, name):
    seqs, env = family_batch(name)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    pu = engine.unpaired(seqs, 4)
    ref = unpaired_from_bpp(engine, seqs)
    for b, s in enumerate(seqs):
        n = len(s)
        assert np.abs(pu[b, :n, 0] - ref[b, :n]).max() <= 1e-10, (name, b)
    check_invariants(pu, [len(s) for s in seqs])


def test_identity_and_bounds_longest(engine):
    # 668 nt: the longest stride the PF fill path covers (WANT_BPP and bf_unpaired are unavailable beyond it)
    seqs = rand_seqs(np.random.default_rng(668), 668, 668, 2)
    pu = engine.unpaired(seqs, 31)
    ref = unpaired_from_bpp(engine, seqs)
    assert np.abs(pu[:, :, 0] - ref).max() <= 1e-10
    check_invariants(pu, [668, 668])


def test_unpaired_errors(engine):
    L = engine.lib()

    def call(seqs, max_u, nopair=None, out=True, stride=None):
        buf, lens, cuts = engine.pack(seqs)
        b = engine.bf_batch_t()
        b.B, b.stride, b.seq, b.len = len(seqs), stride or buf.shape[1], buf.ctypes.data, lens.ctypes.data
        b.cut = cuts.ctypes.data if cuts.any() else None
        if nopair is not None:
            b.nopair = nopair.ctypes.data
        o = np.zeros((len(seqs), buf.shape[1], max(max_u, 1)), np.float64)
        return L.bf_unpaired(C.byref(b), max_u, o.ctypes.data if out else None)

    assert call(["GGGGAAAACCCC"], 4) == 0
    assert call(["GGGGAAAACCCC&GGGGAAAACCCC"], 4) == 4      # BF_ERR_UNAVAILABLE
    assert call(["GGGGAAAACCCC"], 4, nopair=np.zeros((1, 12), np.uint8)) == 4
    assert call(["A" * 669], 4) == 4
    assert call(["A" * 2001], 4) == 4
    assert call(["GGGGAAAACCCC"], 0) == 5                    # BF_ERR_ARG
    assert call(["GGGGAAAACCCC"], 13) == 5
    assert call(["GGGGAAAACCCC"], 4, out=False) == 5
    assert call(["GGGGAAAACCCC"], 4, stride=8) == 5
    with pytest.raises(engine.EngineError) as ei:
        engine.unpaired(["GGGGAAAACCCC"], 0)
    assert ei.value.code == 5


# ---------------------------------------------------------------------------------------------------------------- bf_plfold
def host_plfold(engine, s, W, max_u):
    """window averages from bf_unpaired / WANT_BPP of the window substrings: band [n, W], pu [n, max_u]"""
    n = len(s)
    Wp = min(W, n)
    wins = [s[k:k + Wp] for k in range(n - Wp + 1)]
    pu_w = engine.unpaired(wins, max_u)
    bpp_w = engine.score_batch(wins, want=engine.WANT_BPP)["bpp"]
    band, pu = np.zeros((n, W)), np.zeros((n, max_u))
    cb, cu = np.zeros((n, W)), np.zeros((n, max_u))
    for k in range(len(wins)):
        for a in range(Wp):
            i = k + a
            for d in range(4, Wp - a):
                band[i, d] += bpp_w[k, a, a + d]
                cb[i, d] += 1
            for u in range(1, min(max_u, Wp - a) + 1):
                pu[i, u - 1] += pu_w[k, a, u - 1]
                cu[i, u - 1] += 1
    return np.where(cb > 0, band / np.maximum(cb, 1), 0.0), np.where(cu > 0, pu / np.maximum(cu, 1), 0.0)


@pytest.mark.parametrize("W", [20, 70, "n", "n+"])
def test_plfold_against_window_averages(engine, W):
    rng = np.random.default_rng(77)
    seqs = [rand_seqs(rng, L, L, 1)[0] for L in (30, 95, 180, 300)]
    for s in seqs:
        n = len(s)
        w = n if W == "n" else n + 9 if W == "n+" else W
        mu = min(8, w)
        (band, pu), = engine.plfold([s], w, mu)
        rb, ru = host_plfold(engine, s, w, mu)
        assert band.shape == (n, w) and pu.shape == (n, mu)
        assert np.abs(band - rb).max() <= 1e-12, (n, w)
        assert np.abs(pu - ru).max() <= 1e-12, (n, w)
        if w >= n:   # one window: the global result
            g = engine.unpaired([s], mu)[0]
            P = engine.score_batch([s], want=engine.WANT_BPP)["bpp"][0]
            assert np.abs(pu - g).max() <= 1e-12
            for d in range(4, n):
                assert np.abs(band[:n - d, d] - np.diagonal(P, d)).max() <= 1e-12


def test_plfold_chunking_is_invisible(engine):
    rng = np.random.default_rng(5)
    seqs = rand_seqs(rng, 300, 450, 3) + ["GGGGAAAACCCC"]
    one = engine.plfold(seqs, 70, 31)
    engine.set_option("plfold_mb", 1)   # a few windows per chunk
    try:
        many = engine.plfold(seqs, 70, 31)
    finally:
        engine.set_option("plfold_mb", -1)
    for (b1, p1), (b2, p2) in zip(one, many):
        assert np.array_equal(b1, b2) and np.array_equal(p1, p2)


def test_plfold_long_transcript_in_chunks(engine):
    s = rand_seqs(np.random.default_rng(10000), 10000, 10000, 1)[0]
    (b1, p1), = engine.plfold([s], 70, 31)     # ~9900 windows: more than one chunk of the default budget
    engine.set_option("plfold_mb", 8192)
    try:
        (b2, p2), = engine.plfold([s], 70, 31)
    finally:
        engine.set_option("plfold_mb", -1)
    assert np.array_equal(b1, b2) and np.array_equal(p1, p2)
    assert (p1 >= 0).all() and (p1 <= 1).all() and (b1 >= 0).all() and (b1 <= 1).all()


def test_plfold_strands_together_equal_alone(engine):
    rng = np.random.default_rng(6)
    seqs = rand_seqs(rng, 40, 260, 5) + ["GGGGAAAACCCC", "ACGU"]
    together = engine.plfold(seqs, 50, 12)
    for s, (b, p) in zip(seqs, together):
        (b1, p1), = engine.plfold([s], 50, 12)
        assert np.abs(b - b1).max() <= 1e-12 and np.abs(p - p1).max() <= 1e-12


def test_plfold_errors(engine):
    L = engine.lib()
    buf, lens, _ = engine.pack(["GGGGAAAACCCCAAAGGG"])
    st = engine.bf_strands_t()
    st.n, st.stride, st.seq, st.len = 1, buf.shape[1], buf.ctypes.data, lens.ctypes.data
    o = np.zeros(buf.shape[1] * 3000, np.float64)
    p = np.zeros(buf.shape[1] * 3000, np.float64)
    assert L.bf_plfold(C.byref(st), 10, 4, o.ctypes.data, p.ctypes.data) == 0
    assert L.bf_plfold(C.byref(st), 10, 4, None, None) == 5
    assert L.bf_plfold(C.byref(st), 0, 1, o.ctypes.data, None) == 5
    assert L.bf_plfold(C.byref(st), 10, 0, None, p.ctypes.data) == 5
    assert L.bf_plfold(C.byref(st), 10, 11, None, p.ctypes.data) == 5
    assert L.bf_plfold(C.byref(st), 2001, 4, o.ctypes.data, None) == 4
    assert L.bf_plfold(C.byref(st), 1000, 4, o.ctypes.data, None) == 0   # W' = min(W, n)
    buf2, lens2, _ = engine.pack(["A" * 700])
    st2 = engine.bf_strands_t()
    st2.n, st2.stride, st2.seq, st2.len = 1, 700, buf2.ctypes.data, lens2.ctypes.data
    o2 = np.zeros(700 * 700, np.float64)
    assert L.bf_plfold(C.byref(st2), 700, 4, o2.ctypes.data, None) == 4   # a 700-nt window: beyond the PF fill path
    st.stride = 8
    assert L.bf_plfold(C.byref(st), 10, 4, o.ctypes.data, None) == 5
    with pytest.raises(ValueError):
        engine.plfold(["GGGG&CCCC"], 10)


def test_rna_shim_plfold(engine):
    from desirna_b200 import RNA
    s = rand_seqs(np.random.default_rng(8), 120, 120, 1)[0]
    n = len(s)
    up = RNA.pfl_fold_up(s, 10, 60, 60)
    (band, pu), = engine.plfold([s], 60, 10)
    assert len(up) == n + 1 and all(len(r) == 11 for r in up)
    assert all(x == 0.0 for x in up[0]) and all(r[0] == 0.0 for r in up)
    for i in range(1, n + 1):
        for u in range(1, 11):
            assert up[i][u] == (pu[i - u, u - 1] if u <= i else 0.0), (i, u)
    with pytest.raises(NotImplementedError):
        RNA.pfl_fold_up(s, 10, 60, 40)
    assert len(RNA.pfl_fold_up(s, 4, 500, 200)) == n + 1   # both spans clamp to n
    eps = RNA.pfl_fold(s, 60, 60, 0.01)
    got = {(e.i, e.j): e.p for e in eps}
    want = {(i + 1, i + 1 + d): band[i, d] for i in range(n) for d in range(60) if band[i, d] >= 0.01}
    assert got.keys() == want.keys() and all(got[k] == want[k] for k in got)
    assert all(e.i < e.j and e.p >= 0.01 and e.type == 0 for e in eps)
    with pytest.raises(NotImplementedError):
        RNA.pfl_fold(s, 60, 30, 0.01)

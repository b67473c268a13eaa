"""GPU: stochastic backtracking (bf_sample, engine.sample, RNA fold_compound.pbacktrack).

The samples are checked against quantities computed without the sampler: the exact distribution weight / Z over every structure
of short sequences (the oracle's per-structure weight, brute-force enumeration), the base-pair probabilities of the outside pass
(WANT_BPP) for every fill-kernel family, and the MFE structure's weight / Z of long Eterna100 solutions."""
import collections
import ctypes as C
import json
import math
import os

import numpy as np
import pytest

from struct_weight import WeightOracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAR1999 = os.path.join(ROOT, "desirna_b200", "params", "turner1999_37C.par")

# 12-16 nt; GGCAGGGGACUGCC closes a GGGGAC tetraloop with G-C; in GAGCACGGGAGAC the smoothed dangles change the distribution most
# (chosen by brute force over random sequences), so it carries the power check
EXACT = ["GGCAGGGGACUGCC", "GAGCACGGGAGAC", "GCCUGGAUUAACAGGC", "GGAUCACAGUCUACAC", "GGGUGGGGGUGCUGGC", "AGUAUGUAUACCAC"]
POWER = "GAGCACGGGAGAC"


@pytest.fixture(scope="module")
def wo():
    from oracle.pyoracle import build
    build()
    return WeightOracle(PAR1999)


def rand_seqs(rng, L, B):
    return ["".join("ACGU"[x] for x in rng.integers(0, 4, L)) for _ in range(B)]


def pair_counts(samples, n):
    """counts[i, j] (0-based, i < j) of pairs over the samples, and per-position unpaired counts"""
    a = np.frombuffer("".join(samples).encode(), np.uint8).reshape(len(samples), n)
    S = len(samples)
    stack = np.zeros((S, n + 1), np.int64)
    sp = np.zeros(S, np.int64)
    cnt = np.zeros((n, n), np.int64)
    rows = np.arange(S)
    for j in range(n):
        op = a[:, j] == ord("(")
        stack[rows[op], sp[op]] = j
        sp[op] += 1
        cl = a[:, j] == ord(")")
        sp[cl] -= 1
        i = stack[rows[cl], sp[cl]]
        np.add.at(cnt, (i, np.full(i.shape, j)), 1)
    unp = (a == ord(".")).sum(axis=0)
    return cnt, unp


def chi2_test(counts, probs, N):
    """Pearson chi-square of observed counts against N * probs, bins of expected count < 5 pooled; returns (p-value, TVD)"""
    from scipy.stats import chi2
    exp = N * probs
    big = exp >= 5
    obs_b, exp_b = list(counts[big]), list(exp[big])
    if (~big).any():
        obs_b.append(counts[~big].sum())
        exp_b.append(exp[~big].sum())
    obs_b, exp_b = np.array(obs_b, float), np.array(exp_b, float)
    stat = ((obs_b - exp_b) ** 2 / exp_b).sum()
    return chi2.sf(stat, len(obs_b) - 1), 0.5 * np.abs(counts / N - probs).sum()


def test_exact_distribution(engine, wo):
    """histogram of sampled structures against weight / Z over every structure; the unsmoothed weights are rejected"""
    N = 200000
    rows = EXACT + [POWER] * 4      # the smoothing shifts few structures by small factors: 10^6 samples for the power check
    out = engine.sample(rows, N, seed=11)
    for k, s in enumerate(EXACT):
        band = wo.enumerate_band(s, 10 ** 6, cap=500000)
        index = {db: x for x, (_, db) in enumerate(band)}
        w = np.array([wo.weight(s, db) for _, db in band])
        samples = out[k] if s != POWER else sum((out[r] for r in range(len(rows)) if rows[r] == POWER), [])
        hist = collections.Counter(samples)
        assert set(hist) <= set(index), [db for db in hist if db not in index][:5]
        counts = np.zeros(len(band))
        for db, c in hist.items():
            counts[index[db]] = c
        p, tvd = chi2_test(counts, w / w.sum(), len(samples))
        assert p > 1e-6 and tvd <= 0.01, (s, p, tvd)
        if s == "GGCAGGGGACUGCC":
            assert hist["(((((....)))))"] > 0
        if s == POWER:
            u = np.array([math.exp(-e * 10.0 / wo.kT) for e, _ in band])
            p_u, _ = chi2_test(counts, u / u.sum(), len(samples))
            assert p_u < 1e-6, (s, p_u)


def off_bound(counts, p, ns):
    """entries whose frequency is outside 6 sigma + 1/n of p.  That bound is the normal approximation; where the expected count
    n p is below 5 it does not hold (a rare pair drawn twice in 10^4 samples, n p = 0.02, is a 2e-4 event, and a 400-nt sequence has
    thousands of such pairs), so there an entry only counts when its exact binomial tail is below 1e-9 too."""
    from scipy.stats import binom
    p = np.clip(p, 0.0, 1.0)
    f = counts / ns
    bad = np.abs(f - p) > 6.0 * np.sqrt(p * (1.0 - p) / ns) + 1.0 / ns
    rare = bad & (ns * np.minimum(p, 1.0 - p) < 5)
    if rare.any():
        x, q = counts[rare], p[rare]
        tail = np.where(x > ns * q, binom.sf(x - 1, ns, q), binom.cdf(x, ns, q))
        keep = bad[rare]
        keep[tail >= 1e-9] = False
        bad[rare] = keep
    return bad


def check_bpp(engine, seqs, ns, seed=3):
    out = engine.score_batch(seqs, want=engine.WANT_BPP)
    samples = engine.sample(seqs, ns, seed=seed)
    for k, s in enumerate(seqs):
        n = len(s)
        P = np.triu(out["bpp"][k, :n, :n], 1)
        cnt, unp = pair_counts(samples[k], n)
        bad = np.argwhere(off_bound(cnt, P, ns))
        assert len(bad) == 0, (n, k, [(int(i) + 1, int(j) + 1, cnt[i, j] / ns, P[i, j]) for i, j in bad[:5]])
        pu = 1.0 - P.sum(axis=0) - P.sum(axis=1)
        badu = np.flatnonzero(off_bound(unp, pu, ns))
        assert len(badu) == 0, (n, k, [(int(i) + 1, unp[i] / ns, pu[i]) for i in badu[:5]])


@pytest.mark.parametrize("L", [50, 100, 200, 300, 400])
def test_pair_frequencies_default(engine, L):
    check_bpp(engine, rand_seqs(np.random.default_rng(L), L, 2), 10000)


@pytest.mark.parametrize("L", [50, 100, 200, 300, 400])
def test_pair_frequencies_round1(engine, L):
    engine.set_option("fill3", 0)
    try:
        check_bpp(engine, rand_seqs(np.random.default_rng(L + 1), L, 2), 10000)
    finally:
        engine.set_option("fill3", -1)


@pytest.mark.parametrize("L", [300, 400])
def test_pair_frequencies_cluster(engine, L):
    engine.set_option("cl", 1)
    try:
        check_bpp(engine, rand_seqs(np.random.default_rng(L + 2), L, 2), 10000)
    finally:
        engine.set_option("cl", -1)


def test_pair_frequencies_big_batch(engine):
    check_bpp(engine, rand_seqs(np.random.default_rng(512), 100, 512), 64)


def test_pair_frequencies_ragged(engine):
    rng = np.random.default_rng(20)
    seqs = ["".join("ACGU"[x] for x in rng.integers(0, 4, int(L))) for L in np.linspace(20, 180, 9).astype(int)]
    check_bpp(engine, seqs, 10000)


@pytest.mark.parametrize("target_len", [100, 400])
def test_mfe_structure_frequency(engine, wo, target_len):
    """Eterna100 solutions: frequency of the MFE structure against its weight / Z (per structure, no outside recursion)"""
    rows = [json.loads(l) for l in open(os.path.join(ROOT, "tests", "golden", "E1.jsonl"))]
    # eteV1_22 (400 nt) folds into its MFE structure with probability ~1 and would test nothing; eteV1_63 (400 nt) does so with ~0.62
    pick = {100: "eteV1_05.txt", 400: "eteV1_63.txt"}[target_len]
    s = next(r["sequence"] for r in rows if r["file"] == pick)
    e, mfe_ss = wo.mfe(s)
    p = wo.weight(s, mfe_ss) / wo.Z(s)
    ns = 10000
    f = engine.sample([s], ns, seed=5)[0].count(mfe_ss) / ns
    assert abs(f - p) <= 6.0 * math.sqrt(p * (1.0 - p) / ns) + 1.0 / ns, (pick, f, p)


def test_samples_are_valid_structures(engine):
    rng = np.random.default_rng(4)
    seqs = rand_seqs(rng, 60, 4) + rand_seqs(rng, 150, 2) + ["GGGGAAAACCCC" * 3]
    out = engine.sample(seqs, 200, seed=9)
    canon = {("A", "U"), ("U", "A"), ("G", "C"), ("C", "G"), ("G", "U"), ("U", "G")}
    for s, row in zip(seqs, out):
        n = len(s)
        for db in row:
            assert len(db) == n and set(db) <= set(".()"), db
            pt, st = [0] * (n + 1), []
            for i, ch in enumerate(db, 1):
                if ch == "(":
                    st.append(i)
                elif ch == ")":
                    assert st, db
                    o = st.pop()
                    pt[o], pt[i] = i, o
            assert not st, db
            for i in range(1, n + 1):
                j = pt[i]
                if j <= i:
                    continue
                assert (s[i - 1], s[j - 1]) in canon, (db, i, j)
                inner = [k for k in range(i + 1, j) if pt[k] > k]
                stems = []
                k = i + 1
                while k < j:
                    if pt[k] > k:
                        stems.append((k, pt[k]))
                        k = pt[k] + 1
                    else:
                        k += 1
                if not inner:
                    assert j - i - 1 >= 3, (db, i, j)
                if len(stems) == 1:
                    p, q = stems[0]
                    assert (p - i - 1) + (j - q - 1) <= 30, (db, i, j)
        ev = engine.score_batch([s] * len(row), [[db] for db in row], want=engine.WANT_EVAL)["eval_dcal"][:, 0]
        assert (ev < engine.INF_DCAL).all(), s
    short = engine.sample(["G", "GC", "GGC", "GGCC", "A" * 30], 50, seed=1)
    for s, row in zip(["G", "GC", "GGC", "GGCC", "A" * 30], short):
        assert row == ["." * len(s)] * 50


def test_determinism(engine):
    seqs = rand_seqs(np.random.default_rng(6), 120, 3)
    a = engine.sample(seqs, 300, seed=42)
    assert engine.sample(seqs, 300, seed=42) == a
    b = engine.sample(seqs, 37, seed=42)
    assert [r[:37] for r in a] == b
    c = engine.sample(seqs, 300, seed=43)
    assert c != a and sum(x != y for r, q in zip(a, c) for x, y in zip(r, q)) > 100


def test_errors(engine):
    L = engine.lib()

    def call(seqs, ns, nopair=None):
        buf, lens, cuts = engine.pack(seqs)
        b = engine.bf_batch_t()
        b.B, b.stride, b.seq, b.len = len(seqs), buf.shape[1], buf.ctypes.data, lens.ctypes.data
        b.cut = cuts.ctypes.data if cuts.any() else None
        if nopair is not None:
            b.nopair = nopair.ctypes.data
        out = np.zeros((len(seqs), max(ns, 1), buf.shape[1] + 1), np.uint8)
        return L.bf_sample(C.byref(b), ns, 0, out.ctypes.data)

    assert call(["GGGGAAAACCCC&GGGGAAAACCCC"], 4) == 4       # BF_ERR_UNAVAILABLE
    assert call(["GGGGAAAACCCC"], 4, nopair=np.zeros((1, 12), np.uint8)) == 4
    assert call(["A" * 2001], 4) == 4
    assert call(["GGGGAAAACCCC"], 0) == 5                     # BF_ERR_ARG
    buf, lens, _ = engine.pack(["GGGGAAAACCCC"])
    b = engine.bf_batch_t()
    b.B, b.stride, b.seq, b.len = 1, 12, buf.ctypes.data, lens.ctypes.data
    assert L.bf_sample(C.byref(b), 4, 0, None) == 5
    with pytest.raises(engine.EngineError) as ei:
        engine.sample(["GGGGAAAACCCC"], 0)
    assert ei.value.code == 5


def test_rna_shim_pbacktrack(engine):
    from desirna_b200 import RNA
    fc = RNA.fold_compound("AUGCUAGCUAGGCUAUCGAUCGAUGCAUCGAUGCUAGCUAGCUAGCAUCGAUCG")
    one = fc.pbacktrack()
    assert isinstance(one, str) and len(one) == fc.length
    many = fc.pbacktrack(50)
    assert isinstance(many, list) and len(many) == 50 and all(isinstance(x, str) and len(x) == fc.length for x in many)
    RNA.init_rand(123)
    r1 = [fc.pbacktrack(20), fc.pbacktrack(20)]
    RNA.init_rand(123)
    r2 = [fc.pbacktrack(20), fc.pbacktrack(20)]
    assert r1 == r2 and r1[0] != r1[1]
    with pytest.raises(RuntimeError):
        RNA.fold_compound("GGGGAAAACCCC&GGGGAAAACCCC").pbacktrack()
    fc.hc_add_from_db("x" + "." * (fc.length - 1))
    with pytest.raises(RuntimeError):
        fc.pbacktrack()

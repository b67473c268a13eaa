"""GPU parity: the CUDA path through the C-ABI against the CPU oracle and the golden fixtures."""
import struct

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu


def f32(x):
    return struct.unpack("f", struct.pack("f", x))[0]


def rand_seqs(seed, B, L):
    rng = np.random.default_rng(seed)
    return ["".join("ACGU"[x] for x in row) for row in rng.integers(0, 4, (B, L))]


@pytest.mark.parametrize("tag", ["G1", "G2", "G3", "G4"])
def test_golden_single_strand(engine, tag):
    rows = load_golden(tag)
    seqs = [r["sequence"] for r in rows]
    targets = [[r["target"]] + r["alts"] for r in rows]
    out = engine.score_batch(seqs, targets, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF | engine.WANT_EVAL)
    bad_ss = 0
    for k, r in enumerate(rows):
        assert f32(out["eval_dcal"][k, 0] / 100.0) == r["Ed"]
        assert abs(out["pf"][k, 4] - r["Epf"]) <= 2e-6 * max(1.0, abs(r["Epf"]))
        if r["alts"]:
            ed2 = sum(f32(e / 100.0) for e in out["eval_dcal"][k, 1:]) / len(r["alts"])
            assert abs(ed2 - r["Ed2"]) < 1e-9
        g = r["mfe_ss"]
        for ch in "[]<>{}":
            g = g.replace(ch, ".")
        if out["mfe_ss"][k] != g:
            bad_ss += 1
    # the single known tie anomaly of the 2023 reference run lives in G2 (SURVEY A.5)
    assert bad_ss <= (1 if tag == "G2" else 0)


@pytest.mark.parametrize("tag", ["G5", "G6"])
def test_golden_two_strands(engine, tag):
    rows = load_golden(tag)
    seqs = [r["sequence"] for r in rows]
    targets = [[r["target"]] for r in rows]
    out = engine.score_batch(seqs, targets, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF | engine.WANT_EVAL)
    for k, r in enumerate(rows):
        assert f32(out["eval_dcal"][k, 0] / 100.0) == r["Ed"]
        assert abs(out["pf"][k, 3] - r["Epf"]) <= 2e-6 * max(1.0, abs(r["Epf"]))  # FAB
        a = len(r["sequence"].split("&")[0])
        ss = out["mfe_ss"][k]
        assert ss[:a] + "&" + ss[a:] == r["mfe_ss"]


def test_eterna_v1_kats(engine):
    rows = load_golden("E1")
    seqs = [r["sequence"] for r in rows]
    targets = [[r["target"]] for r in rows]
    out = engine.score_batch(seqs, targets, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF | engine.WANT_EVAL)
    for k, r in enumerate(rows):
        assert out["mfe_ss"][k] == r["target"], r["file"]
        assert out["eval_dcal"][k, 0] == out["mfe_dcal"][k]
        assert out["pf"][k, 4] <= out["mfe_dcal"][k] / 100.0 + 1e-9


@pytest.mark.parametrize("wide", ["1", "0"])
@pytest.mark.parametrize("L,B", [(50, 256), (100, 128), (150, 64), (200, 48), (300, 16), (400, 12)])
def test_random_vs_oracle(engine, oracle, monkeypatch, L, B, wide):
    """wide = 0 forces the 8-warp kernels big batches use (batches of <= 148 sequences otherwise take the 16-warp variants)"""
    monkeypatch.setenv("BF_WIDE", wide)
    seqs = rand_seqs(20240000 + L, B, L)
    out = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF)
    mfe, ss, epf, ed = oracle.fold_batch(seqs, nthreads=8)
    # Ed of the MFE structure == MFE (free invariant), second target = neighbour's structure (NS pairs)
    targets = [[ss[k], ss[(k + 1) % B]] for k in range(B)]
    out2 = engine.score_batch(seqs, targets, want=engine.WANT_EVAL)
    for k in range(B):
        assert out["mfe_dcal"][k] == mfe[k]
        assert out["mfe_ss"][k] == ss[k]
        assert abs(out["pf"][k, 4] - epf[k]) <= 1e-6 * max(1.0, abs(epf[k]))
        assert out2["eval_dcal"][k, 0] == mfe[k]
        assert out2["eval_dcal"][k, 1] == oracle.eval(seqs[k], targets[k][1])


def test_ragged_and_edge_cases(engine, oracle):
    seqs = ["A", "GC", "GGGAAACCC", "ACGU" * 3, "G" * 20 + "AAAA" + "C" * 20, "GGGGAAAACCCC&GGGGAAAACCCC", "GCGC&GCGC",
            "A&U", "GGGG&CCCC", "ACGUACGUAGCUAGCUAGCUAGCAUCGAUCGAUGCAUCGUAGCUAGCUAGCUAGCUAGCAUGCAUCGAUGC"]
    out = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF)
    for k, s in enumerate(seqs):
        e, ss = oracle.mfe(s)
        pf = oracle.pf(s)
        assert out["mfe_dcal"][k] == e, s
        assert out["mfe_ss"][k] == ss, s
        for c in ((0, 1, 2, 3, 4) if "&" in s else (4,)):
            assert abs(out["pf"][k, c] - pf[c]) <= 1e-6 * max(1.0, abs(pf[c])), (s, c)


def test_hard_constraints(engine, oracle):
    seqs = rand_seqs(77, 32, 60)
    rng = np.random.default_rng(5)
    mask = (rng.random((32, 60)) < 0.3).astype(np.uint8)
    out = engine.score_batch(seqs, nopair=mask, want=engine.WANT_MFE | engine.WANT_SS)
    for k, s in enumerate(seqs):
        e, ss = oracle.mfe(s, nopair=mask[k])
        assert out["mfe_dcal"][k] == e
        assert out["mfe_ss"][k] == ss
        assert all(ss[i] == "." for i in range(60) if mask[k, i])


def test_empty_batch(engine):
    out = engine.score_batch([], want=engine.WANT_MFE)
    assert len(out["len"]) == 0


@pytest.mark.parametrize("L,B", [(30, 24), (100, 24), (150, 8)])
def test_bpp_and_defect_vs_oracle(engine, oracle, L, B):
    """Outside pass: not pinned by any ViennaRNA value in the reference tree; the oracle's outside recursion is
    checked against exhaustive enumeration on CPU (tests/test_oracle_golden.py).  Tolerance of north_star: 1e-5 absolute."""
    seqs = rand_seqs(4242 + L, B, L)
    mfe, ss, epf, ed = oracle.fold_batch(seqs, nthreads=8)
    out = engine.score_batch(seqs, [[s] for s in ss], want=engine.WANT_MFE | engine.WANT_PF | engine.WANT_BPP | engine.WANT_DEFECT)
    for k, s in enumerate(seqs):
        pf, bpp = oracle.pf(s, bpp=True)
        assert abs(out["pf"][k, 4] - pf[4]) <= 1e-6 * max(1.0, abs(pf[4]))
        got = out["bpp"][k][:L, :L]
        assert np.abs(got - bpp).max() < 1e-9, (L, k, np.abs(got - bpp).max())
        assert abs(out["defect"][k] - oracle.ensemble_defect(bpp, ss[k])) < 1e-9
    # row sums are probabilities
    full = out["bpp"] + out["bpp"].transpose(0, 2, 1)
    assert full.sum(axis=2).max() <= 1.0 + 1e-9


def test_bpp_ragged_and_unavailable_cases(engine, oracle):
    seqs = ["GGGGAAAACCCC", "ACGUACGUAGCUAGCUAGCUAGCAUCGAUCGAUGCAUCG", "AAAAAA", "GCGCAAAAGCGCAAAAGCGCUUUUGCGC"]
    tg = [["((((....))))"], ["." * len(seqs[1])], ["......"], ["((((....))))....((((....))))"]]
    out = engine.score_batch(seqs, tg, want=engine.WANT_DEFECT | engine.WANT_BPP)
    for k, s in enumerate(seqs):
        pf, bpp = oracle.pf(s, bpp=True)
        n = len(s)
        assert np.abs(out["bpp"][k][:n, :n] - bpp).max() < 1e-9
        assert abs(out["defect"][k] - oracle.ensemble_defect(bpp, tg[k][0])) < 1e-9
    with pytest.raises(engine.EngineError) as ei:
        engine.score_batch(["GGGG&CCCC"], [["((((&))))"]], want=engine.WANT_DEFECT)
    assert ei.value.code == 4


def test_blocked_split_matches_oracle(engine, oracle, monkeypatch):
    """The blocked split (tile-major mirrors + 4x4 block products, long sequences by default) forced on for every length:
    MFE energies and structures bit-exact, ensemble free energy within 1e-6 relative of the oracle."""
    monkeypatch.setenv("BF_BLK_MIN", "1")
    monkeypatch.setenv("BF_BLK_MIN_PF", "1")
    rng = np.random.default_rng(77)
    seqs = ["".join("ACGU"[x] for x in rng.integers(0, 4, int(L))) for L in rng.integers(20, 180, 96)]
    seqs += rand_seqs(5, 4, 300) + rand_seqs(6, 2, 401)
    out = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF)
    for k, s in enumerate(seqs):
        e, ss = oracle.mfe(s)
        assert out["mfe_dcal"][k] == e and out["mfe_ss"][k] == ss, (len(s), k)
        f = oracle.pf(s)[4]
        assert abs(out["pf"][k, 4] - f) <= 1e-6 * max(1.0, abs(f)), (len(s), k)


@pytest.mark.parametrize("thr, L, B", [(300, 253, 1), (400, 365, 1), (400, 317, 149)])
def test_raised_blocked_split_threshold(engine, oracle, monkeypatch, thr, L, B):
    """BF_BLK_MIN_PF raised above a length: the round-1 PF fill runs that length without the blocked split (16 warps with the
    full or the shared partial buffers, 8 warps with shared ones).  Same ensemble energies as the default rule and the oracle."""
    monkeypatch.setenv("BF_CL", "0")
    seqs = rand_seqs(900 + L, B, L)
    want = engine.WANT_MFE | engine.WANT_PF
    ref = engine.score_batch(seqs, want=want)
    monkeypatch.setenv("BF_BLK_MIN_PF", str(thr))
    out = engine.score_batch(seqs, want=want)
    assert (out["mfe_dcal"] == ref["mfe_dcal"]).all()
    assert np.allclose(out["pf"][:, 4], ref["pf"][:, 4], rtol=1e-10, atol=0)
    for k in range(0, B, 50):
        f = oracle.pf(seqs[k])[4]
        assert abs(out["pf"][k, 4] - f) <= 1e-6 * max(1.0, abs(f))


@pytest.mark.parametrize("L", [30, 100, 260, 400])
def test_small_batch_16_warp_variant_matches_8_warp(engine, oracle, monkeypatch, L):
    """Batches of at most one sequence per SM run the fill kernels with 16 warps per CTA (latency of a replica-exchange
    sub-step); same tables, same results as the 8-warp configuration, and as the oracle."""
    seqs = rand_seqs(77 + L, 24, L) + rand_seqs(78 + L, 6, max(5, L // 2))
    want = engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF
    monkeypatch.setenv("BF_WIDE", "1")
    wide = engine.score_batch(seqs, want=want)
    monkeypatch.setenv("BF_WIDE", "0")
    narrow = engine.score_batch(seqs, want=want)
    assert (wide["mfe_dcal"] == narrow["mfe_dcal"]).all()
    assert wide["mfe_ss"] == narrow["mfe_ss"]
    assert np.allclose(wide["pf"][:, 4], narrow["pf"][:, 4], rtol=1e-12, atol=0)
    for k in range(0, len(seqs), 5 if L > 100 else 1):
        e, ss = oracle.mfe(seqs[k])
        assert wide["mfe_dcal"][k] == e and wide["mfe_ss"][k] == ss
        f = oracle.pf(seqs[k])[4]
        assert abs(wide["pf"][k, 4] - f) <= 1e-6 * max(1.0, abs(f))


@pytest.mark.parametrize("L", [100, 400])
def test_full_size_batch_invariants(engine, L):
    """BASELINE.json's sweep size (4096 sequences per launch): properties that need no CPU reference -- the energy of the
    backtracked structure equals the MFE (bit-exact), the structure is a valid pairing of pairable bases with loops >= 3,
    the ensemble free energy lies below the MFE, results do not depend on the batch a sequence travels in."""
    B = 4096 if L == 100 else 1024
    seqs = rand_seqs(20240000 + L, B, L)
    want = engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF
    out = engine.score_batch(seqs, want=want)
    ev = engine.score_batch(seqs, [[s] for s in out["mfe_ss"]], want=engine.WANT_EVAL)["eval_dcal"][:, 0]
    assert (ev == out["mfe_dcal"]).all()
    assert (out["pf"][:, 4] * 100.0 <= out["mfe_dcal"] + 1e-6).all()
    ok = {("A", "U"), ("U", "A"), ("G", "C"), ("C", "G"), ("G", "U"), ("U", "G")}
    for k in range(0, B, 37):
        stack = []
        for i, ch in enumerate(out["mfe_ss"][k]):
            if ch == "(":
                stack.append(i)
            elif ch == ")":
                j = stack.pop()
                assert i - j > 3 and (seqs[k][j], seqs[k][i]) in ok
        assert not stack
    sub = list(range(0, B, 41))
    again = engine.score_batch([seqs[k] for k in sub], want=want)     # a small batch: other kernel variants, same answers
    assert (again["mfe_dcal"] == out["mfe_dcal"][sub]).all()
    assert again["mfe_ss"] == [out["mfe_ss"][k] for k in sub]
    assert np.allclose(again["pf"][:, 4], out["pf"][sub, 4], rtol=1e-12, atol=0)

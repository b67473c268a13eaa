"""The c table the third-generation MFE fill writes (one coalesced row per diagonal from its combine step, every cell) and the
exterior recursions on both sides of the batch-size rule (one CTA per sequence for small batches, one warp per sequence with
the column look-ups in flight for big ones).

The c and fML tables are compared cell by cell, INF included, with the round-1 fill kernels (BF_FILL3=0), which write every
cell of both tables themselves; energies and structures are compared with the CPU oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def rand_seqs(seed, lens):
    rng = np.random.default_rng(seed)
    return ["".join("ACGU"[x] for x in rng.integers(0, 4, n)) for n in lens]


def tables_both_fills(engine, monkeypatch, seqs, nopair=None):
    want = engine.WANT_MFE | engine.WANT_SS
    monkeypatch.setenv("BF_FILL3", "1")
    new = engine.score_batch(seqs, nopair=nopair, want=want)
    tc, tf = engine.debug_table(0, len(seqs)).copy(), engine.debug_table(1, len(seqs)).copy()
    monkeypatch.setenv("BF_FILL3", "0")
    old = engine.score_batch(seqs, nopair=nopair, want=want)
    monkeypatch.delenv("BF_FILL3")
    return new, old, tc, tf


# strides 100 / 101 / 102 / 103: the ring row stride steps 102 -> 103 -> 106 there; 150: the longest the 8-warp fill takes.
# B = 400 takes the 8-warp instance, B = 64 the 16-warp one.
@pytest.mark.parametrize("B", [400, 64])
@pytest.mark.parametrize("stride", [100, 101, 102, 103, 150])
def test_c_table_ragged_batch(engine, oracle, monkeypatch, stride, B):
    lens = [5 + (k * 37) % (stride - 4) for k in range(B)]
    lens[0] = stride
    seqs = rand_seqs(4000 + stride + B, lens)
    new, old, tc, tf = tables_both_fills(engine, monkeypatch, seqs)
    assert (tc == engine.debug_table(0, len(seqs))).all()
    assert (tf == engine.debug_table(1, len(seqs))).all()
    assert (new["mfe_dcal"] == old["mfe_dcal"]).all() and new["mfe_ss"] == old["mfe_ss"]
    for k in range(0, B, 7):
        e, ss = oracle.mfe(seqs[k])
        assert new["mfe_dcal"][k] == e and new["mfe_ss"][k] == ss, (k, lens[k])


@pytest.mark.parametrize("B", [400, 64])
def test_c_table_with_nopair_mask(engine, oracle, monkeypatch, B):
    lens = [5 + (k * 29) % 96 for k in range(B)]
    lens[0] = 100
    seqs = rand_seqs(5000 + B, lens)
    rng = np.random.default_rng(B)
    mask = np.zeros((B, 100), np.uint8)
    for k in range(B):
        mask[k, :lens[k]] = rng.random(lens[k]) < 0.3
    new, old, tc, tf = tables_both_fills(engine, monkeypatch, seqs, nopair=mask)
    assert (tc == engine.debug_table(0, len(seqs))).all()
    assert (tf == engine.debug_table(1, len(seqs))).all()
    for k in range(0, B, 5):
        e, ss = oracle.mfe(seqs[k], nopair=mask[k, :lens[k]])
        assert new["mfe_dcal"][k] == e and new["mfe_ss"][k] == ss, (k, lens[k])


@pytest.mark.parametrize("B", [400, 64])
def test_no_pairable_cell(engine, monkeypatch, B):
    """all-A sequences: no cell can pair, every c entry is INF and the structure is open"""
    seqs = ["A" * (5 + k % 96) for k in range(B - 1)] + ["A" * 100]
    new, old, tc, tf = tables_both_fills(engine, monkeypatch, seqs)
    assert (tc == engine.debug_table(0, len(seqs))).all()
    assert (new["mfe_dcal"] == 0).all()
    assert new["mfe_ss"] == ["." * len(s) for s in seqs]
    inf = tc[-1, :(96 * 100 - (100 * 99 // 2 - 6))]   # the whole triangle of the 100-nt sequence
    assert (inf == inf.max()).all() and inf.max() > 10 ** 6


@pytest.mark.parametrize("B", [4096, 16])
def test_exterior_recursions_both_batch_sides(engine, oracle, B):
    seqs = rand_seqs(6000 + B, [100] * B)
    out = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF)
    rows = range(B) if B <= 64 else range(0, B, 8)
    sub = [seqs[k] for k in rows]
    mfe, ss, epf, ed = oracle.fold_batch(sub, nthreads=8)
    for r, k in enumerate(rows):
        assert out["mfe_dcal"][k] == mfe[r] and out["mfe_ss"][k] == ss[r], k
        assert abs(out["pf"][k, 4] - epf[r]) <= 1e-6 * max(1.0, abs(epf[r])), k

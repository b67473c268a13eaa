"""GPU: minimum-free-energy outside pass (bf_pair_mfe, engine.pair_mfe) and Zuker suboptimals (bf_subopt_zuker,
engine.subopt_zuker, RNA fold_compound.subopt_zuker).

E_pair(i,j), the lowest energy of any structure containing the pair (i,j), is checked bit for bit against brute force over every
structure of short sequences, and against a plain C outside recursion on the CPU oracle's energy functions
(tests/pair_mfe_ref.c) for every fill-kernel family; the Zuker list against E_pair, the MFE and both structure evaluators."""
import ctypes as C
import os

import numpy as np
import pytest

from pair_mfe_ref import PairMfeOracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAR1999 = os.path.join(ROOT, "desirna_b200", "params", "turner1999_37C.par")
INF = 10000000

# hairpins and stems among the short cases: a tetraloop stem, a long stem with a bulge, two stems side by side
SHORT_FIXED = ["GGGGAAACCCC", "GGCAGGGGACUGCC", "GGGAGCAAAGCACCC", "GGGAAACCCGGGAAACCC", "GCGCUUCGGCGC", "AAAAAAAAAA"]


@pytest.fixture(scope="module")
def po():
    from oracle.pyoracle import build
    build()
    return PairMfeOracle(PAR1999)


def rand_seqs(rng, lo, hi, B):
    return ["".join("ACGU"[x] for x in rng.integers(0, 4, int(rng.integers(lo, hi + 1)))) for _ in range(B)]


def pairs_of(db):
    st, out = [], []
    for k, ch in enumerate(db):
        if ch == "(":
            st.append(k)
        elif ch == ")":
            out.append((st.pop(), k))
    assert not st
    return out


def masks_for(rng, seqs, stride, every=3):
    m = np.zeros((len(seqs), stride), np.uint8)
    for b, s in enumerate(seqs):
        if b % every == 1:
            m[b, rng.integers(0, len(s), max(1, len(s) // 8))] = 1
    return m


def short_cases():
    rng = np.random.default_rng(11)
    seqs = SHORT_FIXED + rand_seqs(rng, 8, 18, 34)
    return seqs, masks_for(rng, seqs, max(map(len, seqs)))


def brute_force(po, seq, mask):
    """per-pair minimum over every structure that pairs no masked position, and the structures themselves"""
    n = len(seq)
    ref = np.full((n, n), INF, np.int64)
    kept = []
    for e, db in po.enumerate_band(seq, 10 ** 6, cap=400000):
        prs = pairs_of(db)
        if any(mask[i] or mask[j] for i, j in prs):
            continue
        kept.append((e, db))
        for i, j in prs:
            ref[i, j] = min(ref[i, j], e)
    return ref, kept


def check_rows(E, seqs, refs):
    stride = E.shape[1]
    for b, (s, ref) in enumerate(zip(seqs, refs)):
        n = len(s)
        assert np.array_equal(E[b, :n, :n], ref), (b, s, np.argwhere(E[b, :n, :n] != ref)[:5])
        assert (E[b, n:, :] == INF).all() and (E[b, :, n:] == INF).all()
        assert stride >= n


def test_pair_mfe_equals_brute_force(engine, po):
    seqs, mask = short_cases()
    E = engine.pair_mfe(seqs, nopair=mask)
    refs = [brute_force(po, s, mask[b, :len(s)])[0] for b, s in enumerate(seqs)]
    check_rows(E, seqs, refs)
    assert sum((r < INF).sum() for r in refs) > 200


# (family, batch, switches): each fill family leaves the c / fML triangles the pass reads
def family_batch(name):
    rng = np.random.default_rng({"tap": 1, "round1": 2, "cluster": 3, "wide16": 4, "mask": 5}[name])
    if name == "tap":
        seqs = rand_seqs(rng, 1, 150, 300) + ["GGGGAAACCCC" * 13]
        return seqs, {}
    if name == "round1":
        return rand_seqs(rng, 200, 300, 200), {"BF_FILL3": "0"}
    if name == "cluster":
        return rand_seqs(rng, 150, 400, 6), {"BF_CL": "1"}
    if name == "wide16":
        return rand_seqs(rng, 180, 260, 12), {"BF_FILL3_SMALL": "0", "BF_CL": "0"}
    return rand_seqs(rng, 20, 220, 120), {}


@pytest.mark.parametrize("name", ["tap", "round1", "cluster", "wide16", "mask"])
def test_pair_mfe_equals_cpu_restatement(engine, po, monkeypatch, name):
    seqs, env = family_batch(name)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    stride = max(map(len, seqs))
    mask = masks_for(np.random.default_rng(7), seqs, stride, every=2) if name == "mask" else None
    E = engine.pair_mfe(seqs, nopair=mask)
    refs, mfes = [], []
    for b, s in enumerate(seqs):
        mfe, ref = po.pair_mfe(s, mask[b, :len(s)] if mask is not None else None)
        refs.append(ref)
        mfes.append(mfe)
    check_rows(E, seqs, refs)
    # the CPU restatement's own fill agrees with the engine's MFE
    out = engine.score_batch(seqs, nopair=mask, want=engine.WANT_MFE)
    assert [int(x) for x in out["mfe_dcal"]] == mfes


def eval_both(engine, po, seq, dbs):
    out = engine.score_batch([seq], targets=[list(dbs)], want=engine.WANT_EVAL)
    eng = [int(x) for x in out["eval_dcal"][0]]
    orc = [po.eval(seq, db) for db in dbs]
    return eng, orc


@pytest.mark.parametrize("n", [400, 1000])
def test_invariants_and_zuker_structures_at_length(engine, po, n):
    rng = np.random.default_rng(n)
    seq = rand_seqs(rng, n, n, 1)[0]
    E = engine.pair_mfe([seq])[0]
    out = engine.score_batch([seq], want=engine.WANT_MFE | engine.WANT_SS)
    mfe, ss = int(out["mfe_dcal"][0]), out["mfe_ss"][0]
    fin = E < INF
    assert fin.any() and (E[fin] >= mfe).all()
    for i, j in pairs_of(ss):
        assert E[i, j] == mfe
    zl = engine.subopt_zuker(seq)
    assert zl[0][1] == mfe and all(e >= mfe for _, e in zl)
    # a structure containing (i,j) has energy >= E_pair(i,j), and the one listed for (i,j) has exactly E_pair(i,j): look among those
    by_e = {}
    for k, (_, e) in enumerate(zl):
        by_e.setdefault(e, []).append(k)
    idx = np.argwhere(fin)
    pick = idx[rng.choice(len(idx), min(200, len(idx)), replace=False)]
    chosen = []
    for i, j in pick:
        hit = [k for k in by_e.get(int(E[i, j]), []) if zl[k][0][i] == "(" and (int(i), int(j)) in pairs_of(zl[k][0])]
        assert hit, (i, j)
        chosen.append(hit[0])
    chosen = sorted(set(chosen))
    eng, orc = eval_both(engine, po, seq, [zl[k][0] for k in chosen])
    assert eng == orc == [zl[k][1] for k in chosen]


def check_zuker_list(engine, po, seq, zl, E, mfe):
    dbs = [db for db, _ in zl]
    assert len(set(dbs)) == len(dbs)
    assert zl == sorted(zl, key=lambda x: (x[1], x[0]))
    assert zl[0][1] == mfe
    union = set()
    for db, e in zl:
        assert len(db) == len(seq)
        for i, j in pairs_of(db):
            assert j - i > 3 and (seq[i] + seq[j]) in ("AU", "UA", "GC", "CG", "GU", "UG")
            assert E[i, j] <= e
            union.add((i, j))
    assert union == {(int(i), int(j)) for i, j in np.argwhere(E < INF)}
    eng, orc = eval_both(engine, po, seq, dbs)
    assert eng == orc == [e for _, e in zl]


@pytest.mark.parametrize("n", [60, 150, 400])
def test_zuker_list(engine, po, n):
    seq = rand_seqs(np.random.default_rng(100 + n), n, n, 1)[0]
    E = engine.pair_mfe([seq])[0]
    mfe = int(engine.score_batch([seq], want=engine.WANT_MFE)["mfe_dcal"][0])
    check_zuker_list(engine, po, seq, engine.subopt_zuker(seq), E, mfe)


def test_zuker_list_short_against_brute_force(engine, po):
    seqs, mask = short_cases()
    for b, s in enumerate(seqs):
        m = mask[b, :len(s)]
        ref, kept = brute_force(po, s, m)
        if not (ref < INF).any():
            assert engine.subopt_zuker(s, nopair=m if m.any() else None) == []
            continue
        zl = engine.subopt_zuker(s, nopair=m if m.any() else None)
        mfe = min(e for e, _ in kept)
        if any(db.count("(") for e, db in kept if e == mfe):   # the MFE structure has a pair: it is the first entry
            assert zl[0][1] == mfe
        union = set()
        for db, e in zl:
            prs = pairs_of(db)
            assert not any(m[i] or m[j] for i, j in prs)
            assert (e, db) in kept
            # listed for one of its pairs: a minimum-energy structure containing that pair (its other pairs may have lower E_pair)
            assert any(ref[i, j] == e for i, j in prs)
            union.update(prs)
        assert union == {(int(i), int(j)) for i, j in np.argwhere(ref < INF)}


def test_errors_and_shim(engine):
    from desirna_b200 import RNA
    with pytest.raises(engine.EngineError) as ei:
        engine.pair_mfe(["GGGAAACCC&GGGAAACCC"])
    assert ei.value.code == 4
    with pytest.raises(NotImplementedError):
        RNA.fold_compound("GGGAAACCC&GGGAAACCC").subopt_zuker()
    for call in (lambda: engine.pair_mfe(["A" * 2001]), lambda: engine.subopt_zuker("A" * 2001)):
        with pytest.raises(engine.EngineError) as ei:
            call()
        assert ei.value.code == 4
    buf, lens, _ = engine.pack(["GGGGAAACCCC"])
    b = engine.bf_batch_t()
    b.B, b.stride, b.seq, b.len = 1, buf.shape[1], buf.ctypes.data, lens.ctypes.data
    assert engine.lib().bf_pair_mfe(C.byref(b), None) == 5
    out = np.zeros((1, 11, 11), np.int32)
    lens2 = np.array([12], np.int32)
    b.len = lens2.ctypes.data
    assert engine.lib().bf_pair_mfe(C.byref(b), out.ctypes.data) == 5


def test_shim_subopt_zuker_honours_constraints(engine):
    from desirna_b200 import RNA
    seq = "GGGAGCAAAGCACCCAUGGGAAACCCAU"
    cons = "..x.........x......x........"[:len(seq)]
    fc = RNA.fold_compound(seq)
    fc.hc_add_from_db(cons)
    sols = fc.subopt_zuker()
    mask = np.array([ch == "x" for ch in cons], np.uint8)
    E = engine.pair_mfe([seq], nopair=mask[None, :])[0]
    union = set()
    for s in sols:
        prs = pairs_of(s.structure)
        assert not any(mask[i] or mask[j] for i, j in prs)
        assert s.energy == RNA.f32(fc.eval_structure(s.structure))
        union.update(prs)
    assert union == {(int(i), int(j)) for i, j in np.argwhere(E < INF)}
    assert sols[0].energy == RNA.f32(fc.mfe()[1])
    plain = RNA.fold_compound(seq).subopt_zuker()
    assert any(mask[i] or mask[j] for s in plain for i, j in pairs_of(s.structure))

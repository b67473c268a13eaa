"""CPU: the folding-kinetics reference (tests/kinfold_ref.c, bf_kinfold's model in plain C, every neighbour scored by orc_eval)
against the definition: its move lists against a brute force over all pairs, its dE against eval differences, and its trajectories
against the exact master equation of two short sequences."""
from concurrent.futures import ThreadPoolExecutor
import os

import numpy as np
import scipy.linalg
import scipy.stats

from conftest import PAR1999
from kinfold_ref import KinfoldOracle, boltzmann, brute_moves, master_equation, pairs_of, to_db


def random_canonical(rng, seq, tries):
    """a random structure of canonical pairs, built by inserting random valid moves"""
    db = "." * len(seq)
    for _ in range(tries):
        mv = [m for m in brute_moves(seq, db) if db[m[0] - 1] == "."]
        if not mv:
            break
        i, j = mv[int(rng.integers(len(mv)))]
        db = to_db(len(seq), sorted(set(pairs_of(db)) | {(i, j)}))
    return db


def test_moves_against_brute_force():
    O = KinfoldOracle(PAR1999)
    rng = np.random.default_rng(31)
    n_moves = 0
    for x in range(60):
        n = int(rng.integers(8, 41))
        seq = "".join(rng.choice(list(("ACGU", "GC", "AU")[x % 3]), n))
        for db in ("." * n, O.mfe(seq)[1], random_canonical(rng, seq, int(rng.integers(1, 8)))):
            got = O.moves(seq, db)
            assert [(i, j) for i, j, _ in got] == brute_moves(seq, db), (seq, db)
            e0 = O.eval(seq, db)
            pairs = set(pairs_of(db))
            for i, j, de in got:
                assert de == O.eval(seq, to_db(n, sorted(pairs ^ {(i, j)}))) - e0, (seq, db, i, j)
            n_moves += len(got)
    assert n_moves > 3000


def chi2_tvd(ss, states, p, N):
    """(chi-square p-value over the cells with expectation >= 5, the rest pooled; total variation distance; its bound)"""
    idx = {s: x for x, s in enumerate(states)}
    cnt = np.zeros(len(states))
    for s in ss:
        cnt[idx[s]] += 1
    exp = p * N
    big = exp >= 5
    obs_c = np.append(cnt[big], cnt[~big].sum())
    exp_c = np.append(exp[big], exp[~big].sum())
    keep = exp_c > 0
    chi2 = float(((obs_c[keep] - exp_c[keep]) ** 2 / exp_c[keep]).sum())
    pv = float(scipy.stats.chi2.sf(chi2, keep.sum() - 1))
    tvd = 0.5 * float(np.abs(cnt / N - p).sum())
    return pv, tvd, float(np.sqrt(p * (1 - p) / N).sum())


def test_trajectories_against_master_equation():
    """the reference's snapshot distributions from the open chain against p0 expm(Q t); the latest time against Boltzmann"""
    O = KinfoldOracle(PAR1999)
    N = 4000
    for seq in ("AUGGGGACAUGG", "AUCAAACCGUAAGG"):
        states, E, Q = master_equation(O, seq, "kawasaki")
        gap = -np.sort(np.linalg.eigvals(Q).real)[-2]
        ts = [0.1 / gap, 0.5 / gap, 1.5 / gap, 12 / gap]
        p0 = np.zeros(len(states))
        p0[states.index("." * len(seq))] = 1
        with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
            runs = list(ex.map(lambda k: O.traj(seq, rule="kawasaki", t_max=ts[-1], seed=9, k=k, t_snap=ts), range(N)))
        assert all(r["status"] == 0 and r["t_end"] == ts[-1] for r in runs)
        for s, t in enumerate(ts):
            p = p0 @ scipy.linalg.expm(Q * t)
            pv, tvd, bound = chi2_tvd([r["ss_snap"][s] for r in runs], states, p, N)
            assert pv > 1e-4 and tvd < bound, (seq, t, pv, tvd, bound)
        pb = boltzmann(O, E)
        pv, tvd, bound = chi2_tvd([r["ss_snap"][-1] for r in runs], states, pb, N)
        assert pv > 1e-4 and tvd < bound, (seq, pv, tvd, bound)

"""GPU: bf_kinfold (folding kinetics, engine.kinfold) against the plain-C reference of tests/kinfold_ref.c bit for bit, against the
exact master equation and mean first-passage times of short sequences, and against the engine's own eval at scale."""
import ctypes as C
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import scipy.linalg

from conftest import PAR1999, ROOT
from kinfold_ref import INF, KinfoldOracle, boltzmann, master_equation, mfpt, pairs_of, to_db
from test_oracle_kinfold import chi2_tvd

pytestmark = pytest.mark.gpu

ME_SEQS = ("AUGGGGACAUGG", "GAUCGGAUAACCGA", "AGGCCGAUACGGUAGA")


@pytest.fixture(scope="module")
def kref(oracle):
    return KinfoldOracle(PAR1999)


def rseq(rng, n, alpha="ACGU"):
    return "".join(rng.choice(list(alpha), n))


def close(a, b):
    return abs(a - b) <= 1e-9 * max(abs(a), abs(b), 1e-300)


def test_exact_against_reference(engine, kref):
    """ragged batches of 20-150 nt, a third GC- or AU-only (ties); open chain, MFE or sampled starts; stop at none or the MFE;
    all three rules.  max_steps shrinks with the length, so that the reference (a full eval per neighbour) stays affordable."""
    rng = np.random.default_rng(41)
    seqs = [rseq(rng, int(rng.integers(20, 151)), ("ACGU", "GC", "AU")[x % 3]) for x in range(150)]
    mfe = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]
    samp = [s[0] for s in engine.sample(seqs, 1, seed=5)]
    jobs = []
    for lo, hi, max_steps in ((20, 60, 400), (61, 110, 80), (111, 150, 15)):
        rows = [r for r, s in enumerate(seqs) if lo <= len(s) <= hi]
        for rule in ("kawasaki", "metropolis", "descent"):
            for kind in range(3):
                sel = [r for r in rows if r % 3 == kind]
                start = None if kind == 0 else [(samp if kind == 1 else mfe)[r] for r in sel]
                stop = [mfe[r] for r in sel] if kind != 1 else None
                t_max = float(rng.uniform(0.05, 3.0))
                ts = sorted(float(x) for x in rng.uniform(0, t_max, 3))
                seed = int(rng.integers(1 << 63))
                got = engine.kinfold([seqs[r] for r in sel], start, stop, n_traj=2, rule=rule, t_max=t_max, seed=seed, t_snap=ts,
                                     max_steps=max_steps)
                for x, r in enumerate(sel):
                    for k in range(2):
                        jobs.append((got, x, k, seqs[r], start[x] if start else None, stop[x] if stop else None, rule, t_max, seed,
                                     max_steps, ts))

    def ref(j):
        _, x, k, s, st, sp, rule, t_max, seed, ms, ts = j
        return kref.traj(s, st, sp, rule, t_max, seed, x, k, ms, ts)

    with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        refs = list(ex.map(ref, jobs))
    excluded = 0
    status = np.zeros(3, int)
    for j, w in zip(jobs, refs):
        got, x, k = j[:3]
        if w["margin"] < 1e-9:
            excluded += 1
            continue
        g = {key: got[key][x, k] for key in ("status", "t_end", "steps", "e_end", "ss_end", "e_snap", "ss_snap")}
        ctx = (j[3:], g, w)
        assert (int(g["status"]), int(g["steps"]), int(g["e_end"]), str(g["ss_end"])) == \
            (w["status"], w["steps"], w["e_end"], w["ss_end"]), ctx
        assert close(float(g["t_end"]), w["t_end"]), ctx
        assert [int(v) for v in g["e_snap"]] == w["e_snap"] and [str(v) for v in g["ss_snap"]] == w["ss_snap"], ctx
        assert int(g["e_end"]) == kref.eval(j[3], str(g["ss_end"])), ctx
        status[w["status"]] += 1
    print(f"kinfold exact: {len(jobs)} trajectories, {excluded} excluded at a time boundary, status counts {status.tolist()}")
    assert excluded <= len(jobs) // 100
    assert status[0] >= 20 and status[2] >= 20, status


def snap_dist(engine, seq, rule, ts, N, seed):
    got = engine.kinfold([seq], n_traj=N, rule=rule, t_max=ts[-1], seed=seed, t_snap=ts)
    assert (got["status"] == 0).all() and (got["t_end"] == ts[-1]).all()
    return got["ss_snap"][0]


@pytest.mark.parametrize("rule", ["kawasaki", "metropolis"])
def test_master_equation(engine, kref, rule):
    """2e5 trajectories per sequence from the open chain: snapshot distributions against p0 expm(Q t), the latest against
    Boltzmann"""
    N = 200000
    for q, seq in enumerate(ME_SEQS):
        states, E, Q = master_equation(kref, seq, rule)
        gap = -np.sort(np.linalg.eigvals(Q).real)[-2]
        ts = [0.1 / gap, 0.5 / gap, 1.5 / gap, 12 / gap]
        ss = snap_dist(engine, seq, rule, ts, N, seed=100 + q)
        p0 = np.zeros(len(states))
        p0[states.index("." * len(seq))] = 1
        for s, t in enumerate(ts):
            p = p0 @ scipy.linalg.expm(Q * t)
            pv, tvd, bound = chi2_tvd(list(ss[:, s]), states, p, N)
            assert pv > 1e-4 and tvd < bound, (seq, rule, t, pv, tvd, bound)
        pv, tvd, bound = chi2_tvd(list(ss[:, -1]), states, boltzmann(kref, E), N)
        assert pv > 1e-4 and tvd < bound, (seq, rule, pv, tvd, bound)


@pytest.mark.parametrize("rule", ["kawasaki", "metropolis"])
def test_first_passage(engine, kref, rule):
    """mean first-passage time open chain -> MFE against the linear solve of the absorbing chain, within 5 standard errors"""
    N = 100000
    for q, seq in enumerate(ME_SEQS):
        states, E, Q = master_equation(kref, seq, rule)
        target = states[int(np.argmin(E))]
        m = mfpt(Q, states.index("." * len(seq)), int(np.argmin(E)))
        got = engine.kinfold([seq], stop=[target], n_traj=N, rule=rule, t_max=1e9, seed=7 + q, structures=False)
        assert (got["status"] == 1).all()
        t = got["t_end"][0]
        se = t.std() / np.sqrt(N)
        assert abs(t.mean() - m) < 5 * se, (seq, rule, t.mean(), m, se)


def neighbours(seq, db):
    """every valid move's structure (a pair deleted or a canonical pair inserted into its loop)"""
    n = len(seq)
    pt = [0] * (n + 2)
    for i, j in pairs_of(db):
        pt[i], pt[j] = j, i
    lid, cur = [0] * (n + 2), 0
    for x in range(1, n + 1):
        if pt[x] == 0:
            lid[x] = cur
        elif pt[x] > x:
            lid[x] = lid[pt[x]] = cur
            cur = x
        else:
            cur = lid[x]
    canon = {("A", "U"), ("U", "A"), ("C", "G"), ("G", "C"), ("G", "U"), ("U", "G")}
    out = []
    for i in range(1, n + 1):
        if pt[i] > i:
            out.append(db[:i - 1] + "." + db[i:pt[i] - 1] + "." + db[pt[i]:])
        elif pt[i] == 0:
            hi = pt[lid[i]] - 1 if lid[i] else n
            for j in range(i + 4, hi + 1):
                if pt[j] == 0 and lid[j] == lid[i] and (seq[i - 1], seq[j - 1]) in canon:
                    out.append(db[:i - 1] + "(" + db[i:j - 1] + ")" + db[j:])
    return out


@pytest.mark.parametrize("n,count", [(100, 16), (400, 8), (2000, 2)])
def test_descent_at_scale(engine, n, count):
    """from Boltzmann samples (bf_sample covers up to 400 nt) or, at 2000 nt, the MFE structure less a third of its pairs"""
    rng = np.random.default_rng(n)
    seqs = [rseq(rng, n) for _ in range(count)]
    if n <= 400:
        start = [s[0] for s in engine.sample(seqs, 1, seed=3)]
    else:
        start = []
        for s in engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]:
            pairs = pairs_of(s)
            start.append(to_db(n, [p for x, p in enumerate(pairs) if x % 3]))
    got = engine.kinfold(seqs, start, n_traj=1, rule="descent")
    ss = [str(got["ss_end"][r, 0]) for r in range(count)]
    ev = engine.score_batch(seqs, [[s] for s in ss], want=engine.WANT_EVAL)["eval_dcal"][:, 0]
    assert [int(v) for v in got["e_end"][:, 0]] == [int(v) for v in ev]
    assert (got["status"] == 0).all() and (got["t_end"] == 0).all() and (got["steps"] > 0).sum() >= count // 2
    st = engine.score_batch(seqs, [[s] for s in start], want=engine.WANT_EVAL)["eval_dcal"][:, 0]
    assert (got["e_end"][:, 0] <= st).all()
    if n <= 400:
        for r in range(count):
            nb = neighbours(seqs[r], ss[r])
            e = engine.score_batch([seqs[r]], [nb], want=engine.WANT_EVAL)["eval_dcal"][0]
            assert int(e.min()) >= int(got["e_end"][r, 0]), r


def test_determinism_and_chunking(engine):
    rng = np.random.default_rng(13)
    seqs = [rseq(rng, int(rng.integers(30, 121))) for _ in range(12)]
    mfe = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]
    kw = dict(stop=mfe, rule="kawasaki", t_max=20.0, seed=77, t_snap=[0.5, 1.0, 5.0, 20.0], max_steps=400)
    a = engine.kinfold(seqs, n_traj=200, **kw)
    b = engine.kinfold(seqs, n_traj=200, **kw)
    c = engine.kinfold(seqs, n_traj=7, **kw)
    engine.set_option("kinfold_mb", 1)
    try:
        n0 = engine.kernel_launches()
        d = engine.kinfold(seqs, n_traj=200, **kw)   # about 800 trajectories per launch
        assert engine.kernel_launches() - n0 > 1
    finally:
        engine.set_option("kinfold_mb", -1)
    for key in a:
        assert (a[key] == b[key]).all(), key
        assert (a[key][:, :7] == c[key]).all(), key
        assert (a[key] == d[key]).all(), key
    assert len(set(a["status"].ravel().tolist())) >= 2
    assert (a["steps"] > 0).any()
    e = engine.kinfold(seqs, n_traj=200, **dict(kw, seed=78))
    assert not (e["t_end"] == a["t_end"]).all()
    # start = stop: a hit at time 0; a sequence without a possible pair: absorbing until t_max
    h = engine.kinfold(["GGGGAAAACCCC", "AAAAAAAA"], ["((((....))))", "........"], ["((((....))))", "........"],
                       n_traj=2, t_snap=[0.0, 1.0], t_max=2.0)
    assert h["status"].tolist() == [[1, 1], [1, 1]] and (h["t_end"] == 0).all() and (h["steps"] == 0).all()
    z = engine.kinfold(["AAAAAAAA"], n_traj=3, t_snap=[0.0, 2.0], t_max=2.0)
    assert (z["status"] == 0).all() and (z["t_end"] == 2.0).all() and (z["ss_snap"] == "........").all() and (z["e_snap"] == 0).all()
    # a cap: the snapshots after the last move are blank
    cap = engine.kinfold(["GGGGAAAACCCCAGGGAAACCCA"], n_traj=4, t_snap=[1e3], t_max=1e3, max_steps=3)
    assert (cap["status"] == 2).all() and (cap["steps"] == 3).all() and (cap["e_snap"] == INF).all() and (cap["ss_snap"] == "").all()


def test_errors(engine):
    from desirna_b200 import engine as E
    L = E.lib()

    def call(seqs, lens, start=None, stop=None, n_traj=1, rule=0, t_max=10.0, max_steps=100, ts=(), n=None, status=True, stride=None):
        buf, _, _ = E.pack(seqs, stride)
        S = buf.shape[1]
        keep = []
        q = E.bf_kinfold_t()
        q.n, q.stride, q.seq = len(seqs) if n is None else n, S, buf.ctypes.data
        ln = np.asarray(lens, np.int32)
        q.len = ln.ctypes.data
        for name, dbs in (("start", start), ("stop", stop)):
            if dbs is not None:
                t = np.frombuffer("".join(x.ljust(S, ".")[:S] for x in dbs).encode(), np.uint8).copy()
                keep.append(t)
                setattr(q, name, t.ctypes.data)
        tsa = np.asarray(ts, np.float64)
        q.n_traj, q.rule, q.t_max, q.max_steps, q.n_snap = n_traj, rule, t_max, max_steps, tsa.size
        q.t_snap = tsa.ctypes.data if tsa.size else None
        st = np.zeros(max(1, len(seqs) * max(n_traj, 1)), np.int32)
        return L.bf_kinfold(C.byref(q), st.ctypes.data if status else None, None, None, None, None, None, None)

    ARG = 5
    ok = ("GGGGAAAACCCC", "((((....))))")
    assert call([ok[0]], [12]) == 0
    assert call([ok[0]], [12], [ok[1]], [ok[1]], rule=1, ts=(0.0, 10.0)) == 0
    assert call([ok[0]], [12], rule=2, t_max=float("nan"), ts=(5.0, 1.0)) == 0                # descent reads neither
    assert L.bf_kinfold(None, None, None, None, None, None, None, None) == ARG                   # null query
    assert call([ok[0]], [12], status=False) == ARG                                             # null status buffer
    assert call([ok[0]], [12], n=-1) == ARG                                                     # n < 0
    assert call([ok[0]], [12], n_traj=0) == ARG                                                 # T < 1
    assert call(["G" * 2001], [2001]) == ARG                                                    # stride above 2000
    assert call([ok[0]], [13]) == ARG                                                           # len > stride
    assert call(["GGGGAANACCCC"], [12]) == ARG                                                  # a character other than ACGUT
    assert call([ok[0]], [12], ["(((.....))))"]) == ARG                                        # unbalanced start
    assert call([ok[0]], [12], None, ["((((....)))("]) == ARG                                  # unbalanced stop
    assert call([ok[0]], [12], ["((((.x..))))"]) == ARG                                        # another character
    assert call(["GGGGAAAACCCA"], [12], ["((((....))))"]) == ARG                               # a non-canonical pair (G-A)
    assert call([ok[0]], [12], None, ["((.))......."]) == ARG   # stop pair with j - i < 4
    assert call([ok[0]], [12], rule=3) == ARG and call([ok[0]], [12], rule=-1) == ARG          # rule outside 0 .. 2
    assert call([ok[0]], [12], t_max=0.0) == ARG and call([ok[0]], [12], t_max=float("inf")) == ARG   # t_max
    assert call([ok[0]], [12], rule=1, t_max=float("nan")) == ARG
    assert call([ok[0]], [12], ts=(2.0, 1.0)) == ARG                                            # unsorted snapshots
    assert call([ok[0]], [12], ts=(-1.0,)) == ARG and call([ok[0]], [12], ts=(11.0,)) == ARG    # outside [0, t_max]
    assert call([ok[0]], [12], max_steps=0) == ARG                                              # max_steps < 1
    assert call(["G" * 1000 + "C" * 1000], [2000], rule=2, max_steps=1) == 0                    # the 2000-nt cap
    with pytest.raises(ValueError):
        engine.kinfold(["GG&CC"])
    with pytest.raises(ValueError):
        engine.kinfold(["GGGGAAAACCCC"], rule="glauber")
    code = ("import ctypes as C, sys; sys.path.insert(0, %r); from desirna_b200 import engine as E; L = E.lib(); "
            "q = E.bf_kinfold_t(); q.stride = 1; q.n_traj = 1; q.t_max = 1.0; q.max_steps = 1; s = (C.c_int32 * 1)(); "
            "r0 = L.bf_kinfold(C.byref(q), s, None, None, None, None, None, None); "
            "L.bf_init(0); r1 = L.bf_kinfold(C.byref(q), s, None, None, None, None, None, None); print(r0, r1)") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=ROOT)
    assert out.stdout.split() == ["2", "2"], out                                               # BF_ERR_NOT_INIT

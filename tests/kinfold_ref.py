"""Folding kinetics (bf_kinfold's trajectories and descent walks) on the CPU, restated on the oracle's eval (test infrastructure):
tests/kinfold_ref.c, compiled with oracle/orc_fold.c into a temporary directory so that nothing is written into the tree.  Also the
exact master equation of short sequences: the state space, the rate matrix Q and its solutions."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from oracle.pyoracle import Oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_lib = None
_lock = threading.Lock()   # the tests call the reference from a thread pool: build and load it once
INF = 10000000
RULES = {"kawasaki": 0, "metropolis": 1, "descent": 2}
CANON = {("A", "U"), ("U", "A"), ("C", "G"), ("G", "C"), ("G", "U"), ("U", "G")}


def lib():
    global _lib
    with _lock:
        return _lib or _load()


def _load():
    global _lib
    srcs = [os.path.join(_HERE, "kinfold_ref.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"), os.path.join(_ROOT, "oracle", "orc_fold.h")]
    h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"kinfold_ref_{os.getuid()}_{h}.so")
    if not os.path.exists(out):
        tmp = out + f".{os.getpid()}"
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                               "-o", tmp, srcs[0], "-lm"])
        os.replace(tmp, out)
    L = C.CDLL(out)
    L.kf_moves.restype = C.c_int
    L.kf_moves.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_void_p, C.c_void_p]
    L.kf_kT.restype = C.c_double
    L.kf_kT.argtypes = [C.c_void_p]
    L.kf_rate_table.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.kf_traj.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int, C.c_double, C.c_uint64, C.c_int, C.c_int,
                          C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_double),
                          C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.c_char_p, C.c_void_p, C.c_char_p, C.POINTER(C.c_double)]
    _lib = L
    return _lib


class KinfoldOracle(Oracle):
    def __init__(self, par_path):
        super().__init__(par_path)
        self._rates = {}

    @property
    def kT(self):
        return lib().kf_kT(self.P)

    def rate_table(self, rule):
        if rule not in self._rates:
            t = np.zeros(65536, np.float64)
            lib().kf_rate_table(self.P, RULES[rule], t.ctypes.data)
            self._rates[rule] = t
        return self._rates[rule]

    def moves(self, seq, db):
        """[(i, j, dE)] of the valid moves of db in canonical order, dE from orc_eval"""
        n = len(seq)
        cap = n * n // 2 + 32
        mv = np.zeros(cap, np.int32)
        de = np.zeros(cap, np.int32)
        c = lib().kf_moves(self.P, seq.encode(), n, db.encode(), mv.ctypes.data, de.ctypes.data)
        return [(int(m) >> 16, int(m) & 0xFFFF, int(d)) for m, d in zip(mv[:c], de[:c])]

    def traj(self, seq, start=None, stop=None, rule="kawasaki", t_max=500.0, seed=0, r=0, k=0, max_steps=10**6, t_snap=()):
        """one trajectory (instance r, trajectory k) by the rules of bf_kinfold: dict(status, t_end, steps, e_end, ss_end, e_snap,
        ss_snap, margin); margin is the least relative distance of a time comparison that decided the outcome"""
        n = len(seq)
        ts = np.ascontiguousarray(t_snap, np.float64)
        ns = ts.size
        st, te, sp, ee, mg = C.c_int(), C.c_double(), C.c_longlong(), C.c_int(), C.c_double()
        sse = C.create_string_buffer(n + 1)
        es = np.zeros(max(ns, 1), np.int32)
        sss = C.create_string_buffer(max(ns, 1) * (n + 1))
        rate = self.rate_table(rule if rule != "descent" else "kawasaki")
        lib().kf_traj(self.P, seq.encode(), n, start.encode() if start else None, stop.encode() if stop else None, RULES[rule],
                      float(t_max), int(seed) & ((1 << 64) - 1), int(r), int(k), int(max_steps), ns, ts.ctypes.data if ns else None,
                      rate.ctypes.data, C.byref(st), C.byref(te), C.byref(sp), C.byref(ee), sse, es.ctypes.data, sss, C.byref(mg))
        raw = sss.raw
        snaps = [raw[s * (n + 1):(s + 1) * (n + 1)].split(b"\0")[0].decode() for s in range(ns)]
        return dict(status=st.value, t_end=te.value, steps=sp.value, e_end=ee.value, ss_end=sse.value.decode(),
                    e_snap=[int(x) for x in es[:ns]], ss_snap=snaps, margin=mg.value)


def brute_moves(seq, db):
    """every valid move of db by the definition alone: [(i, j)] in canonical order"""
    n = len(seq)
    pairs = set(pairs_of(db))
    out = []
    for i in range(1, n + 1):
        for j in range(i + 4, n + 1):
            if (i, j) in pairs:
                out.append((i, j))
            elif (seq[i - 1], seq[j - 1]) in CANON and all(
                    p not in (i, j) and q not in (i, j) and not (p < i < q < j) and not (i < p < j < q) for p, q in pairs):
                out.append((i, j))
    return out


def pairs_of(db):
    st, out = [], []
    for i, c in enumerate(db, 1):
        if c == "(":
            st.append(i)
        elif c == ")":
            out.append((st.pop(), i))
    return sorted(out)


def to_db(n, pairs):
    ss = ["."] * n
    for i, j in pairs:
        ss[i - 1], ss[j - 1] = "(", ")"
    return "".join(ss)


def master_equation(O, seq, rule):
    """(states, energies, Q) of the kinetic chain of seq: every structure (oracle.enumerate_band), energies by orc_eval, Q[x, y] the
    rate x -> y (rows sum to 0)"""
    states = [s for _, s in O.enumerate_band(seq, 10**6)]
    idx = {s: x for x, s in enumerate(states)}
    E = np.array([O.eval(seq, s) for s in states], np.int64)
    rate = O.rate_table(rule)
    Q = np.zeros((len(states), len(states)))
    n = len(seq)
    for x, s in enumerate(states):
        pairs = set(pairs_of(s))
        for i, j in brute_moves(seq, s):
            y = idx[to_db(n, sorted(pairs ^ {(i, j)}))]
            Q[x, y] = rate[E[y] - E[x] + 32768]
        Q[x, x] = -Q[x].sum()
    return states, E, Q


def boltzmann(O, E):
    w = np.exp(-(E - E.min()) * 10.0 / O.kT)
    return w / w.sum()


def mfpt(Q, x0, target):
    """mean first-passage time from state x0 to state target"""
    keep = [x for x in range(Q.shape[0]) if x != target]
    m = np.linalg.solve(-Q[np.ix_(keep, keep)], np.ones(len(keep)))
    return float(m[keep.index(x0)])

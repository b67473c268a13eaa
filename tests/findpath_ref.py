"""Direct refolding paths (bf_findpath's breadth-limited findpath search) on the CPU, restated on the oracle's eval (test
infrastructure): tests/findpath_ref.c, compiled with oracle/orc_fold.c into a temporary directory so that nothing is written into the
tree."""
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


def lib():
    global _lib
    with _lock:
        return _lib or _load()


def _load():
    global _lib
    srcs = [os.path.join(_HERE, "findpath_ref.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"), os.path.join(_ROOT, "oracle", "orc_fold.h")]
    h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"findpath_ref_{os.getuid()}_{h}.so")
    if not os.path.exists(out):
        tmp = out + f".{os.getpid()}"
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                               "-o", tmp, srcs[0], "-lm"])
        os.replace(tmp, out)
    L = C.CDLL(out)
    IP = C.POINTER(C.c_int)
    L.orc_findpath.restype = C.c_int
    L.orc_findpath.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int, IP, C.c_void_p, C.c_void_p, IP]
    L.orc_findpath_dp.restype = C.c_int
    L.orc_findpath_dp.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p]
    _lib = L
    return _lib


def apply_moves(s1, moves):
    """the structures of the path from s1: one per prefix of moves ((i, j) > 0 insert, < 0 delete; 1-based)"""
    ss = list(s1)
    out = [s1]
    for i, j in moves:
        if i > 0:
            ss[i - 1], ss[j - 1] = "(", ")"
        else:
            ss[-i - 1], ss[-j - 1] = ".", "."
        out.append("".join(ss))
    return out


class FindpathOracle(Oracle):
    def findpath(self, seq, s1, s2, width):
        """dict(saddle, moves [(i, j)], path_e [k + 1], max_level) by the rules of bf_findpath; the reference takes any width"""
        n = len(seq)
        moves = np.zeros(2 * n + 2, np.int32)
        pe = np.zeros(n + 2, np.int32)
        k, ml = C.c_int(), C.c_int()
        sad = lib().orc_findpath(self.P, seq.encode(), n, s1.encode(), s2.encode(), int(width), C.byref(k), moves.ctypes.data,
                                 pe.ctypes.data, C.byref(ml))
        k = k.value
        return dict(saddle=sad, moves=[(int(moves[2 * s]), int(moves[2 * s + 1])) for s in range(k)], path_e=[int(x) for x in pe[:k + 1]],
                    max_level=ml.value)

    def findpath_dp(self, seq, s1, s2):
        """the least saddle over all direct paths (exact subset DP; INF when more than 20 moves)"""
        return lib().orc_findpath_dp(self.P, seq.encode(), len(seq), s1.encode(), s2.encode())


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


def compatible(pairs, i, j):
    """pair (i, j) can join the valid pair set `pairs`: no shared position, no crossing, j - i >= 4"""
    if j - i < 4:
        return False
    for p, q in pairs:
        if p in (i, j) or q in (i, j) or (p < i < q < j) or (i < p < j < q):
            return False
    return True


def random_structure(rng, n, tries=None):
    """a random valid structure (pairs need not be canonical)"""
    pairs = []
    for _ in range(tries if tries is not None else int(rng.integers(0, n))):
        i = int(rng.integers(1, n + 1))
        j = int(rng.integers(1, n + 1))
        i, j = min(i, j), max(i, j)
        if compatible(pairs, i, j):
            pairs.append((i, j))
    return to_db(n, pairs)


def perturb(rng, s1, n_del, n_add):
    """s1 without n_del of its pairs plus up to n_add random compatible pairs: at most n_del + n_add moves away"""
    pairs = pairs_of(s1)
    drop = set(rng.choice(len(pairs), min(n_del, len(pairs)), replace=False).tolist()) if pairs else set()
    keep = [p for x, p in enumerate(pairs) if x not in drop]
    n = len(s1)
    added = 0
    for _ in range(200 * max(n_add, 1)):
        if added >= n_add:
            break
        i, j = sorted(int(x) for x in rng.integers(1, n + 1, 2))
        if compatible(keep, i, j):
            keep.append((i, j))
            added += 1
    return to_db(n, keep)


def check_path(s1, s2, moves):
    """every structure of the path from s1 is valid and the path ends at s2; returns the structures"""
    cur = set(pairs_of(s1))
    out = [s1]
    for i, j in moves:
        if i > 0:
            assert (i, j) not in cur and compatible(list(cur), i, j), (s1, s2, moves, (i, j))
            cur.add((i, j))
        else:
            assert (-i, -j) in cur, (s1, s2, moves, (i, j))
            cur.remove((-i, -j))
        out.append(to_db(len(s1), sorted(cur)))
    assert out[-1] == s2, (s1, s2, moves)
    return out

"""Accessibility-aware RNA-RNA interaction (bf_interact's site model) on the CPU, restated on the oracle's energy functions (test
infrastructure): tests/interact_ref.c, compiled with tests/duplex_ref.c and oracle/orc_fold.c into a temporary directory so that
nothing is written into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from duplex_ref import DuplexOracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_lib = None
_lock = threading.Lock()   # the tests call the reference from a thread pool: build and load it once
INF = 10000000
KT = (37.0 + 273.15) * 1.98717   # cal/mol: the kT of the oracle's and the engine's parameter sets at 37 C


def lib():
    global _lib
    with _lock:
        return _lib or _load()


def _load():
    global _lib
    srcs = [os.path.join(_HERE, "interact_ref.c"), os.path.join(_HERE, "duplex_ref.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"),
            os.path.join(_ROOT, "oracle", "orc_fold.h")]
    h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"interact_ref_{os.getuid()}_{h}.so")
    if not os.path.exists(out):
        tmp = out + f".{os.getpid()}"
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                               "-o", tmp, srcs[0], "-lm"])
        os.replace(tmp, out)
    L = C.CDLL(out)
    D = C.POINTER(C.c_double)
    L.orc_interact.restype = None
    L.orc_interact.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, D,
                               C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, D]
    L.orc_interact_brute.restype = None
    L.orc_interact_brute.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, D,
                                     C.POINTER(C.c_int), C.POINTER(C.c_int)]
    _lib = L
    return _lib


def ed_rows(pu, span):
    """opening energies (kcal/mol) from P_u rows [n, >= span], entry [k-1, u-1]: -(kT/1000) ln P_u, +inf where P_u <= 0"""
    p = np.ascontiguousarray(np.asarray(pu, np.float64)[:, :span])
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.ascontiguousarray(np.where(p > 0.0, -(KT / 1000.0) * np.log(np.where(p > 0.0, p, 1.0)), np.inf))


def _ptr(x):
    return None if x is None else np.ascontiguousarray(x, np.float64).ctypes.data


class InteractOracle(DuplexOracle):
    def interact(self, a, b, span, ed_a=None, ed_b=None):
        """dict(e, h, site (k1, km, lm, l1), ss, gap) by the fixed-start recurrence and the rules of bf_interact.  ed_a / ed_b:
        None (no accessibility) or opening energies [len, span], entry [k-1, u-1] for the stretch k .. k+u-1."""
        ea = None if ed_a is None else np.ascontiguousarray(ed_a, np.float64)
        eb = None if ed_b is None else np.ascontiguousarray(ed_b, np.float64)
        e, gap, h, site = C.c_double(), C.c_double(), C.c_int(), (C.c_int * 4)()
        ss = C.create_string_buffer(len(a) + len(b) + 2)
        lib().orc_interact(self.P, a.encode(), len(a), b.encode(), len(b), span, _ptr(ea), _ptr(eb), C.byref(e), C.byref(h), site, ss,
                           C.byref(gap))
        return dict(e=e.value, h=h.value, site=tuple(site), ss=ss.value.decode("ascii"), gap=gap.value)

    def interact_brute(self, a, b, span, ed_a=None, ed_b=None):
        """(e, h, site) of the least-E site over every chain, scored by orc_eval on a&b"""
        ea = None if ed_a is None else np.ascontiguousarray(ed_a, np.float64)
        eb = None if ed_b is None else np.ascontiguousarray(ed_b, np.float64)
        e, h, site = C.c_double(), C.c_int(), (C.c_int * 4)()
        lib().orc_interact_brute(self.P, a.encode(), len(a), b.encode(), len(b), span, _ptr(ea), _ptr(eb), C.byref(e), C.byref(h), site)
        return e.value, h.value, tuple(site)

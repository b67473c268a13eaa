"""Probabilities of unpaired stretches on the CPU as ratios of masked partition functions (test infrastructure):
tests/unpaired_ref.c, compiled with oracle/orc_fold.c into a temporary directory so that nothing is written into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.pyoracle import Oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_HERE, "unpaired_ref.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"), os.path.join(_ROOT, "oracle", "orc_fold.h")]
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), f"unpaired_ref_{os.getuid()}_{h}.so")
        if not os.path.exists(out):
            tmp = out + f".{os.getpid()}"
            subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                                   "-o", tmp, srcs[0], "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.orc_masked_lnz.restype = C.c_double
        L.orc_masked_lnz.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p]
        L.orc_unpaired.restype = None
        L.orc_unpaired.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


class UnpairedOracle(Oracle):
    def unpaired(self, seq, stretches, nthreads=None):
        """float64 [len(stretches)]: P(positions i .. i+u-1 unpaired) = Z(masked) / Z for each 1-based (i, u)"""
        st = np.ascontiguousarray(np.asarray(stretches, np.int32).reshape(-1, 2))
        i, u = np.ascontiguousarray(st[:, 0]), np.ascontiguousarray(st[:, 1])
        out = np.zeros(len(st), np.float64)
        nt = nthreads or min(32, os.cpu_count() or 1)
        lib().orc_unpaired(self.P, seq.encode(), len(seq), len(st), i.ctypes.data, u.ctypes.data, out.ctypes.data, nt)
        return out

    def masked_lnz(self, seq, nopair=None):
        mask = bytes(np.asarray(nopair, np.uint8)) if nopair is not None else None
        return lib().orc_masked_lnz(self.P, seq.encode(), len(seq), mask)

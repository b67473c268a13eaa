"""E_pair (lowest energy of a structure containing each pair) on the CPU, restated on the oracle's energy functions (test
infrastructure): tests/pair_mfe_ref.c, compiled with oracle/orc_fold.c into a temporary directory so that nothing is written into
the tree."""
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
        srcs = [os.path.join(_HERE, "pair_mfe_ref.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"), os.path.join(_ROOT, "oracle", "orc_fold.h")]
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), f"pair_mfe_ref_{os.getuid()}_{h}.so")
        if not os.path.exists(out):
            tmp = out + f".{os.getpid()}"
            subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                                   "-o", tmp, srcs[0], "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.orc_pair_mfe.restype = C.c_int
        L.orc_pair_mfe.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_void_p]
        _lib = L
    return _lib


class PairMfeOracle(Oracle):
    def pair_mfe(self, seq, nopair=None):
        """(MFE, int32 [n, n] E_pair) of single-strand seq; nopair: optional n-byte mask"""
        n = len(seq)
        out = np.zeros((n, n), np.int32)
        mask = bytes(np.asarray(nopair, np.uint8)) if nopair is not None else None
        mfe = lib().orc_pair_mfe(self.P, seq.encode(), n, mask, out.ctypes.data)
        return mfe, out

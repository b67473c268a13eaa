"""Per-structure Boltzmann weights under the CPU oracle's partition-function model (test infrastructure).

Because of pf_smooth, a structure's probability is weight / Z with the smoothed dangle and mismatch factors, not
exp(-eval / kT) / Z.  `WeightOracle.weight(seq, db)` exposes the oracle's own per-structure weight (the function its brute-force
enumeration sums), compiled from oracle/orc_fold.c by tests/struct_weight.c into a temporary directory, so that nothing is
written into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

from oracle.pyoracle import Oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_HERE, "struct_weight.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"), os.path.join(_ROOT, "oracle", "orc_fold.h")]
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), f"struct_weight_{os.getuid()}_{h}.so")
        if not os.path.exists(out):
            tmp = out + f".{os.getpid()}"
            subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                                   "-o", tmp, srcs[0], "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.orc_struct_weight.restype = C.c_double
        L.orc_struct_weight.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.POINTER(C.c_int)]
        L.orc_kT.restype = C.c_double
        L.orc_kT.argtypes = [C.c_void_p]
        _lib = L
    return _lib


class WeightOracle(Oracle):
    @property
    def kT(self):
        """cal/mol"""
        return lib().orc_kT(self.P)

    def weight(self, seq, db):
        """Boltzmann weight of structure db of single-strand seq under the partition function's model"""
        assert len(db) == len(seq) and "&" not in seq
        e = C.c_int()
        w = lib().orc_struct_weight(self.P, seq.encode(), len(seq), db.encode(), C.byref(e))
        assert w >= 0.0, ("unbalanced structure", db)
        return w

    def Z(self, seq):
        """partition function from orc_pf's ensemble free energy"""
        import math
        return math.exp(-self.pf(seq)[4] * 1000.0 / self.kT)

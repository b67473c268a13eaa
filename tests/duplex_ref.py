"""Duplex MFE (RNA-RNA hybridization, ViennaRNA duplexfold's recurrence) on the CPU, restated on the oracle's energy functions
(test infrastructure): tests/duplex_ref.c, compiled with oracle/orc_fold.c into a temporary directory so that nothing is written
into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

from oracle.pyoracle import Oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_lib = None
INF = 10000000


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(_HERE, "duplex_ref.c"), os.path.join(_ROOT, "oracle", "orc_fold.c"), os.path.join(_ROOT, "oracle", "orc_fold.h")]
        h = hashlib.sha1(b"".join(open(p, "rb").read() for p in srcs)).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), f"duplex_ref_{os.getuid()}_{h}.so")
        if not os.path.exists(out):
            tmp = out + f".{os.getpid()}"
            subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-pthread", "-fPIC", "-Wall", "-Wno-unused-function", "-shared",
                                   "-o", tmp, srcs[0], "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.orc_duplex.restype = C.c_int
        L.orc_duplex.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p]
        L.orc_duplex_brute.restype = C.c_int
        L.orc_duplex_brute.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_int]
        _lib = L
    return _lib


class DuplexOracle(Oracle):
    def duplex(self, a, b):
        """(energy in dcal/mol, 'a-part&b-part' full length) by the recurrence and the tie rules of bf_duplex"""
        ss = C.create_string_buffer(len(a) + len(b) + 2)
        e = lib().orc_duplex(self.P, a.encode(), len(a), b.encode(), len(b), ss)
        return e, ss.value.decode("ascii")

    def duplex_brute(self, a, b):
        """least orc_eval energy on a&b over every duplex chain (INF: no chain)"""
        return lib().orc_duplex_brute(self.P, a.encode(), len(a), b.encode(), len(b))

    def eval_duplex(self, a, b, ss):
        """orc_eval of 'a-part&b-part' on the two-strand compound a&b"""
        return self.eval(a + "&" + b, ss.replace("&", ""))

"""TEST INFRASTRUCTURE: brute-force ground truth for the second-best energy of short two-strand ('A&B') sequences.

Every secondary structure the folding recursions allow is listed -- canonical pairs, non-crossing, TURN unpaired bases at least
in a hairpin on one strand, a pair across the nick at any span -- and scored with the CPU oracle's eval_structure, whose
two-strand loop model (nick loops, strand-aware dangles, DuplexInit once for a connected structure) the G5/G6 goldens pin.
Unconnected structures are listed too.  Short sequences only (the count grows exponentially).  Never imported by the product.
"""
import functools

import numpy as np

from oracle.pyoracle import split
from oracle_backend import OracleBackend

TURN = 3
INF_DCAL = 10000000
_PAIRS = {("A", "U"), ("U", "A"), ("G", "C"), ("C", "G"), ("G", "U"), ("U", "G")}


def structures(seq):
    """every structure of `seq` ('A&B' or one strand) as a dot-bracket without '&', each exactly once"""
    s, cut = split(seq.upper().replace("T", "U"))
    n = len(s)
    cp = cut if cut else n + 1   # 1-based first base of strand B

    def can_pair(i, j):
        if (s[i - 1], s[j - 1]) not in _PAIRS:
            return False
        return (i >= cp) != (j >= cp) or j - i > TURN

    @functools.lru_cache(maxsize=None)
    def frag(i, j):   # structures of positions i..j: i unpaired, or i paired with k
        if i > j:
            return ("",)
        out = ["." + r for r in frag(i + 1, j)]
        for k in range(i + 1, j + 1):
            if can_pair(i, k):
                inner, outer = frag(i + 1, k - 1), frag(k + 1, j)
                out += ["(" + a + ")" + b for a in inner for b in outer]
        return tuple(out)

    return list(frag(1, n))


def enumerate_band(oracle, seq, bound=INF_DCAL):
    """sorted [(energy_dcal, structure)] of every structure of `seq` with energy <= bound"""
    return sorted(x for x in ((oracle.eval(seq, db), db) for db in structures(seq)) if x[0] <= bound)


def second_best(oracle, seq):
    """(e1, e2) in dcal/mol; e2 = 10000000 when the sequence has a single structure"""
    band = enumerate_band(oracle, seq)
    return band[0][0], (band[1][0] if len(band) > 1 else INF_DCAL)


class DimerOracleBackend(OracleBackend):
    """OracleBackend whose second_best also takes 'A&B' sequences (brute force, up to ~20 nt)"""

    def second_best(self, seqs, nopair=None):
        assert nopair is None
        e1, e2 = np.zeros(len(seqs), np.int32), np.zeros(len(seqs), np.int32)
        for k, seq in enumerate(seqs):
            assert len(seq.replace("&", "")) <= 20
            e1[k], e2[k] = second_best(self.O, seq)
        return e1, e2

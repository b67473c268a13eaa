"""ViennaRNA-shaped front end of the B200 engine: the subset of the SWIG module `RNA` that DesiRNA calls.

DesiRNA has no FFI of its own; its hot path enters native code through `import RNA`
(utils/energy_scores.py:20, utils/dimer_multichain_energy.py:27, utils/sequence_utils.py:46,
DesiRNA.py:35).  A maintainer switches engines with `from desirna_b200 import RNA`.  Call sites covered:

    RNA.params_load(path)                         DesiRNA.py:456
    RNA.md(), md.compute_bpp                      energy_scores.py:27-28, 369
    RNA.fold_compound(seq[, md])                  energy_scores.py:147, 370, 416; dimer_multichain_energy.py:89, 104
    fc.pf() / fc.mfe() / fc.eval_structure(db)    energy_scores.py:75, 99, 150-151, 371-373
    fc.mfe_dimer() / fc.pf_dimer()                energy_scores.py:156-157; dimer_multichain_energy.py:47, 90, 105
    fc.hc_add_from_db(db)                         sequence_utils.py:1181, 1198, 1214
    fc.exp_params_rescale(mfe)                    energy_scores.py:372   (numerical no-op here: the kernels rescale per sequence)
    fc.ensemble_defect(db)                        energy_scores.py:374
    fc.pbacktrack([num_samples]), RNA.init_rand(seed)   stochastic backtracking (not called by DesiRNA; ViennaRNA's API)
    fc.subopt_zuker()                             Zuker suboptimals (not called by DesiRNA; ViennaRNA's API)
    fc.path_findpath_saddle(s1, s2, width)        findpath saddle (not called by DesiRNA; ViennaRNA's API; conventions recalled)
    fc.path_findpath(s1, s2, width)               findpath refolding path (not called by DesiRNA; ViennaRNA's API; conventions recalled)
    RNA.duplexfold(s1, s2)                        RNA-RNA hybridization, RNAduplex (not called by DesiRNA; ViennaRNA's API)
    RNA.pfl_fold_up(seq, ulength, W, L)           accessibility, RNAplfold -u (not called by DesiRNA; ViennaRNA's API; conventions recalled)
    RNA.pfl_fold(seq, W, L, cutoff)               RNAplfold pair probabilities (not called by DesiRNA; ViennaRNA's API; conventions recalled)
    RNA.fold(seq) / RNA.co_pf_fold(seq)           energy_scores.py:354; dimer_multichain_energy.py:109, 113-114

Conventions kept: energies come back as Python floats holding float32-rounded kcal/mol (ViennaRNA returns C
float), structures from mfe_dimer() carry no '&', pf() returns (string, energy) and DesiRNA ignores element 0.
Results of one fold compound are cached, and a whole batch of compounds can be evaluated by ONE engine call
through `prefetch()` -- that is how the lock-step replica loop keeps the GPU busy while callers still see
the per-object API.  There is no CPU fallback: every number comes from libb200fold.so.
"""
import random
import struct

import numpy as np

from . import engine as _eng


def f32(x):
    """round to C float, widen back to double (what SWIG hands to Python)"""
    return struct.unpack("f", struct.pack("f", float(x)))[0]


class _Cvar:
    uniq_ML = 0


cvar = _Cvar()

# seeds of fc.pbacktrack(): each call draws the next one, so successive calls give new samples and init_rand(seed) repeats a run
_rand = random.Random()


def init_rand(seed=None):
    """Seed the generator behind fc.pbacktrack() (ViennaRNA RNA.init_rand); no seed: from the system's entropy source."""
    _rand.seed(seed)


def params_load(path):
    _eng.params_load(path)
    return 1


class md:
    """model details: only the fields DesiRNA touches; the rest are ViennaRNA's defaults baked into the kernels
    (T=37C, dangles=2, noLP=0, noGU=0, special hairpins, TURN=3, MAXLOOP=30, pf_smooth=1)."""

    def __init__(self):
        self.compute_bpp = 1
        self.temperature = 37.0
        self.dangles = 2
        self.uniq_ML = 0


class fold_compound:
    def __init__(self, sequence, model_details=None, *_):
        self.sequence = sequence
        self.md = model_details if model_details is not None else md()
        self.length = len(sequence.replace("&", ""))
        self._nopair = None          # accumulated hard constraints ('x' positions)
        self._cache = {}

    # ---- batching hook -------------------------------------------------------------------------
    @staticmethod
    def prefetch(compounds, targets=None, want=None):
        """Evaluate many fold compounds with one engine call and fill their caches.
        targets: optional list (per compound) of lists of dot-bracket strings for eval_structure."""
        if not compounds:
            return
        E = _eng
        w = want if want is not None else (E.WANT_MFE | E.WANT_SS | E.WANT_PF)
        seqs = [c.sequence for c in compounds]
        tg = None
        if targets is not None:
            T = max(len(t) for t in targets)
            if T:
                tg = [list(t) + [t[-1] if t else "." * c.length] * (T - len(t)) for t, c in zip(targets, compounds)]
                w |= E.WANT_EVAL
        out = E.score_batch(seqs, tg, want=w)
        for k, c in enumerate(compounds):
            if "mfe_dcal" in out:
                c._cache["mfe"] = (out["mfe_ss"][k], int(out["mfe_dcal"][k])) if "mfe_ss" in out else (None, int(out["mfe_dcal"][k]))
            if "pf" in out:
                c._cache["pf"] = [float(x) for x in out["pf"][k]]
            if tg is not None:
                for t, db in enumerate(targets[k]):
                    c._cache[("eval", db.replace("&", ""))] = int(out["eval_dcal"][k, t])

    @staticmethod
    def prefetch_constrained(compounds):
        """One engine call for the constrained MFE folds (hc_add_from_db 'x' masks) of many compounds: the refolds of one
        round of the pseudoknot overlay (sequence_utils.py:1181-1216) across all mutants of a Monte-Carlo sub-step."""
        todo = [c for c in compounds if c._nopair is not None and ("mfe", bytes(c._nopair)) not in c._cache]
        if not todo:
            return
        E = _eng
        stride = max(c.length for c in todo)
        mask = np.zeros((len(todo), stride), np.uint8)
        for k, c in enumerate(todo):
            mask[k, :c.length] = c._nopair
        out = E.score_batch([c.sequence for c in todo], None, nopair=mask, want=E.WANT_MFE | E.WANT_SS)
        for k, c in enumerate(todo):
            c._cache[("mfe", bytes(c._nopair))] = (out["mfe_ss"][k], int(out["mfe_dcal"][k]))

    # ---- single-object API ---------------------------------------------------------------------
    def _run(self, want, targets=None):
        mask = None
        if self._nopair is not None:
            mask = np.asarray(self._nopair, np.uint8)[None, :]
        return _eng.score_batch([self.sequence], targets, nopair=mask, want=want)

    def _mfe(self):
        key = "mfe" if self._nopair is None else ("mfe", bytes(self._nopair))
        if key not in self._cache:
            E = _eng
            out = self._run(E.WANT_MFE | E.WANT_SS)
            self._cache[key] = (out["mfe_ss"][0], int(out["mfe_dcal"][0]))
        return self._cache[key]

    def _pf(self):
        if "pf" not in self._cache:
            if self._nopair is not None and any(self._nopair):
                # the partition-function kernels ignore hard constraints; DesiRNA always calls pf() before hc_add_from_db
                raise RuntimeError("fold_compound.pf() after hc_add_from_db(): constrained partition functions are not supported")
            out = self._run(_eng.WANT_PF)
            self._cache["pf"] = [float(x) for x in out["pf"][0]]
        return self._cache["pf"]

    def mfe(self):
        ss, e = self._mfe()
        return ss, f32(e / 100.0)

    def mfe_dimer(self):
        return self.mfe()

    def pf(self):
        p = self._pf()
        col = 3 if "&" in self.sequence else 4
        return "", f32(p[col])

    def pf_dimer(self):
        p = self._pf()
        if "&" not in self.sequence:
            return "", f32(p[4]), 0.0, 0.0, f32(p[4])
        return "", f32(p[0]), f32(p[1]), f32(p[2]), f32(p[3])

    def eval_structure(self, structure):
        db = structure.replace("&", "")
        key = ("eval", db)
        if key not in self._cache:
            out = self._run(_eng.WANT_EVAL, targets=[[db]])
            self._cache[key] = int(out["eval_dcal"][0, 0])
        return f32(self._cache[key] / 100.0)

    def hc_add_from_db(self, constraint, *_):
        """only 'x' (position may not pair) is used by DesiRNA; constraints accumulate on the compound"""
        db = constraint.replace("&", "")
        if self._nopair is None:
            self._nopair = [0] * self.length
        for i, ch in enumerate(db[:self.length]):
            if ch == "x":
                self._nopair[i] = 1
        return 1

    def exp_params_rescale(self, mfe=None):
        return None

    def bpp(self):
        if "bpp" not in self._cache:
            E = _eng
            out = self._run(E.WANT_MFE | E.WANT_PF | E.WANT_BPP)
            self._cache["bpp"] = out["bpp"][0]
            self._cache["pf"] = [float(x) for x in out["pf"][0]]
        return self._cache["bpp"]

    def ensemble_defect(self, structure):
        """vrna_ensemble_defect: (1/n) sum_i (1 - p_i,pt(i)) for paired i, sum_j p_ij for unpaired i"""
        db = structure.replace("&", "")
        key = ("defect", db)
        if key not in self._cache:
            E = _eng
            out = self._run(E.WANT_MFE | E.WANT_PF | E.WANT_DEFECT, targets=[[db]])
            self._cache[key] = float(out["defect"][0])
        return self._cache[key]

    def pbacktrack(self, num_samples=None, *_):
        """vrna_pbacktrack: a secondary structure drawn from the Boltzmann ensemble, or a list of num_samples independent ones"""
        if "&" in self.sequence:
            raise NotImplementedError("pbacktrack on two-strand compounds is not part of the accelerated path")
        if self._nopair is not None and any(self._nopair):
            raise RuntimeError("fold_compound.pbacktrack() after hc_add_from_db(): sampling under hard constraints is not supported")
        n = 1 if num_samples is None else int(num_samples)
        out = _eng.sample([self.sequence], n, seed=_rand.getrandbits(64))[0]
        return out[0] if num_samples is None else out

    def second_best_energy(self):
        """(MFE, energy of the second-best structure) in kcal/mol as C floats, or (MFE, None) when the sequence has a single
        structure: bf_second_best, a 2-best DP on the unambiguous grammar -- the number DesiRNA reads off subopt_cb's enumeration
        (energy_scores.py:453-488) without the enumeration.  'A&B' compounds: structures of the two-strand loop model of mfe_dimer()
        and eval_structure(), connected or not.  Extension of the shim; ViennaRNA has no such call."""
        nopair = np.asarray(self._nopair, np.uint8)[None, :] if self._nopair is not None and any(self._nopair) else None
        e1, e2 = _eng.second_best([self.sequence], nopair)
        return f32(int(e1[0]) / 100.0), (f32(int(e2[0]) / 100.0) if int(e2[0]) < 10000000 else None)

    def subopt_cb(self, delta, cb, data=None):
        """vrna_subopt_cb as DesiRNA calls it (energy_scores.py:465-474, uniq_ML = 1): cb(structure, energy, data) for every
        structure within `delta` dcal/mol of the MFE, then once more with structure None."""
        if "&" in self.sequence:
            raise NotImplementedError("subopt_cb on two-strand compounds is not part of the accelerated path")
        nopair = np.asarray(self._nopair, np.uint8) if self._nopair is not None and any(self._nopair) else None
        # the walk stops at max_out structures in search order, not energy order: a truncated band is not a band.  Grow the
        # buffer until the whole band fits (ViennaRNA enumerates it completely, whatever its size).
        cap = 4096
        while True:
            found, truncated = _eng.subopt(self.sequence, int(delta), nopair, max_out=cap)
            if not truncated:
                break
            if cap >= (1 << 22):
                raise RuntimeError("subopt_cb: more than %d structures within %d dcal/mol of the MFE" % (cap, int(delta)))
            cap *= 8
        for structure, e in found:
            cb(structure, f32(e / 100.0), data)
        cb(None, 0.0, data)

    def subopt_zuker(self):
        """vrna_subopt_zuker: for every base pair that some structure contains, a minimum-free-energy structure containing it
        (each structure listed once), sorted by energy; hard constraints of hc_add_from_db() apply"""
        if "&" in self.sequence:
            raise NotImplementedError("subopt_zuker on two-strand compounds is not part of the accelerated path")
        nopair = np.asarray(self._nopair, np.uint8) if self._nopair is not None and any(self._nopair) else None
        return [subopt_solution(s, f32(e / 100.0)) for s, e in _eng.subopt_zuker(self.sequence, nopair)]

    def path_findpath_saddle(self, s1, s2, width=1):
        """vrna_path_findpath_saddle: the saddle energy (int, dcal/mol) of the best direct refolding path from s1 to s2 found by the
        breadth-limited search of width `width` (engine.findpath).  The width schedule, direction alternation and tie order are
        ViennaRNA's as recalled; no ViennaRNA output pins them here."""
        if "&" in self.sequence:
            raise NotImplementedError("path_findpath_saddle on two-strand compounds is not part of the accelerated path")
        return int(_eng.findpath([self.sequence], [s1], [s2], width, path=False)[0])

    def path_findpath(self, s1, s2, width=1):
        """vrna_path_findpath: the best direct refolding path from s1 to s2, a list of path objects (.s structure, .en kcal/mol) from
        s1 to s2, with the structures expanded from the moves.  Conventions recalled as for path_findpath_saddle."""
        if "&" in self.sequence:
            raise NotImplementedError("path_findpath on two-strand compounds is not part of the accelerated path")
        _, res = _eng.findpath([self.sequence], [s1], [s2], width)
        moves, pe = res[0]
        ss = list(s1)
        out = [path(s1, f32(int(pe[0]) / 100.0))]
        for (i, j), e in zip(moves.tolist(), pe[1:].tolist()):
            if i > 0:
                ss[i - 1], ss[j - 1] = "(", ")"
            else:
                ss[-i - 1], ss[-j - 1] = ".", "."
            out.append(path("".join(ss), f32(int(e) / 100.0)))
        return out


class path:
    """one step of fc.path_findpath(): .s (structure) and .en (kcal/mol, C float) as ViennaRNA's path object"""

    def __init__(self, s, en):
        self.s = s
        self.en = en

    def __repr__(self):
        return "path(%r, %r)" % (self.s, self.en)


class subopt_solution:
    """one entry of fc.subopt_zuker(): .structure and .energy (kcal/mol, C float) as ViennaRNA's subopt_solution"""

    def __init__(self, structure, energy):
        self.structure = structure
        self.energy = energy

    def __repr__(self):
        return "subopt_solution(%r, %r)" % (self.structure, self.energy)


class duplexT:
    """result of RNA.duplexfold(), in ViennaRNA's duplexT convention as recalled (no ViennaRNA output pins it here):
    .structure  'a-part&b-part', trimmed to the paired region plus one flanking nucleotide on each side where one exists;
    .i          last position of the a-part, 1-based;
    .j          first position of the b-part, 1-based;
    .energy     kcal/mol (double)"""

    def __init__(self, structure, energy, i, j):
        self.structure = structure
        self.energy = energy
        self.i = i
        self.j = j

    def __repr__(self):
        return "duplexT(%r, %r, i=%d, j=%d)" % (self.structure, self.energy, self.i, self.j)


def duplexfold(s1, s2):
    """vrna_duplexfold: the lowest-energy structure of strands s1 and s2 made of intermolecular pairs only (bf_duplex).  With no
    possible intermolecular pair: the untrimmed all-dot structure, i = len(s1), j = 1 and energy 100000.0."""
    e, ss = _eng.duplex([s1], [s2], pairs=[(0, 0)])
    e, ss = int(e[0]), ss[0]
    n1, n2 = len(s1), len(s2)
    if e >= _eng.INF_DCAL:
        return duplexT(ss, e / 100.0, n1, 1)
    pa, pb = ss[:n1], ss[n1 + 1:]
    # 1-based bounds: the paired region and one flanking nucleotide on each side where one exists
    a0, a1 = max(pa.index("("), 1), min(pa.rindex("(") + 2, n1)
    b0, b1 = max(pb.index(")"), 1), min(pb.rindex(")") + 2, n2)
    return duplexT(pa[a0 - 1:a1] + "&" + pb[b0 - 1:b1], e / 100.0, a1, b0)


def _plfold_span(sequence, window_size, max_bp_span):
    n = len(sequence)
    W, L = min(int(window_size), n), min(int(max_bp_span), n)
    if W != L:
        raise NotImplementedError("RNAplfold with a maximum base-pair span below the window size is not supported (L must equal W)")
    return W


def pfl_fold_up(sequence, ulength, window_size, max_bp_span):
    """RNAplfold -u (ViennaRNA RNA.pfl_fold_up), span = window: n+1 lists of ulength+1 floats, [i][u] the window-averaged probability
    that the u nucleotides ending at i (i-u+1 .. i, 1-based) are unpaired.  Row 0, column 0 and entries with u > i are 0.0.  This
    pU layout is ViennaRNA's as recalled; no ViennaRNA output pins it here."""
    n, U = len(sequence), int(ulength)
    out = [[0.0] * (U + 1) for _ in range(n + 1)]
    if n == 0 or U < 1:
        return out
    W = _plfold_span(sequence, window_size, max_bp_span)
    mu = min(U, W, n)
    _, pu = _eng.plfold([sequence], W, mu, pairs=False)[0]
    for i in range(1, n + 1):
        row = out[i]
        for u in range(1, min(mu, i) + 1):
            row[u] = float(pu[i - u, u - 1])
    return out


class ep:
    """one pair probability of RNA.pfl_fold: .i < .j (1-based), .p, .type (0: a base pair)"""

    def __init__(self, i, j, p, type=0):
        self.i, self.j, self.p, self.type = i, j, p, type

    def __repr__(self):
        return f"ep({self.i}, {self.j}, {self.p:.6g})"


def pfl_fold(sequence, w, L, cutoff):
    """RNAplfold pair probabilities (ViennaRNA RNA.pfl_fold), span = window: the pairs whose window-averaged probability is at least
    cutoff, as ep objects in (i, j) order.  Conventions recalled; no ViennaRNA output pins them here."""
    n = len(sequence)
    if n == 0:
        return []
    W = _plfold_span(sequence, w, L)
    band, _ = _eng.plfold([sequence], W, 1, pairs=True)[0]
    return [ep(i + 1, i + 1 + d, float(band[i, d])) for i in range(n) for d in range(band.shape[1]) if band[i, d] > 0.0 and band[i, d] >= cutoff]


def fold(sequence):
    return fold_compound(sequence).mfe()


def co_pf_fold(sequence):
    return fold_compound(sequence).pf_dimer()

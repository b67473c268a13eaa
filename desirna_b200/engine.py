"""ctypes binding of libb200fold.so (C-ABI: include/b200fold.h).

The library is the product: there is no CPU fallback.  Importing this module without the
built shared object raises; calling into it without a B200 returns BF_ERR_CUDA, surfaced
as EngineError.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libb200fold.so")
PARAMS_DIR = os.path.join(_PKG, "params")

WANT_MFE, WANT_SS, WANT_PF, WANT_EVAL, WANT_BPP, WANT_DEFECT = 1, 2, 4, 8, 16, 32
INF_DCAL = 10000000


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200fold error {code}: {msg}")
        self.code = code


class bf_batch_t(C.Structure):
    _fields_ = [("B", C.c_int32), ("stride", C.c_int32), ("seq", C.c_void_p), ("len", C.c_void_p),
                ("cut", C.c_void_p), ("nopair", C.c_void_p), ("targets", C.c_void_p),
                ("n_targets", C.c_int32), ("want", C.c_uint32)]


class bf_result_t(C.Structure):
    _fields_ = [("mfe_dcal", C.c_void_p), ("mfe_ss", C.c_void_p), ("pf", C.c_void_p),
                ("eval_dcal", C.c_void_p), ("defect", C.c_void_p), ("bpp", C.c_void_p)]


class bf_strands_t(C.Structure):
    _fields_ = [("n", C.c_int32), ("stride", C.c_int32), ("seq", C.c_void_p), ("len", C.c_void_p)]


class bf_duplex_t(C.Structure):
    _fields_ = [("a", bf_strands_t), ("b", bf_strands_t), ("n_pairs", C.c_int32), ("pairs", C.c_void_p)]


class bf_interact_t(C.Structure):
    _fields_ = [("a", bf_strands_t), ("b", bf_strands_t), ("n_pairs", C.c_int32), ("pairs", C.c_void_p), ("max_span", C.c_int32),
                ("acc_a", C.c_int32), ("acc_b", C.c_int32)]


class bf_findpath_t(C.Structure):
    _fields_ = [("n", C.c_int32), ("stride", C.c_int32), ("seq", C.c_void_p), ("len", C.c_void_p), ("s1", C.c_void_p), ("s2", C.c_void_p),
                ("width", C.c_int32)]


class bf_kinfold_t(C.Structure):
    _fields_ = [("n", C.c_int32), ("stride", C.c_int32), ("seq", C.c_void_p), ("len", C.c_void_p), ("start", C.c_void_p),
                ("stop", C.c_void_p), ("n_traj", C.c_int32), ("rule", C.c_int32), ("t_max", C.c_double), ("seed", C.c_uint64),
                ("max_steps", C.c_int64), ("n_snap", C.c_int32), ("t_snap", C.c_void_p)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(the engine has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.bf_last_error.restype = C.c_char_p
        L.bf_init.argtypes = [C.c_int]
        L.bf_params_load.argtypes = [C.c_char_p]
        L.bf_params_builtin.argtypes = [C.c_int, C.c_char_p]
        L.bf_params_get.argtypes = [C.c_char_p] + [C.c_int] * 6 + [C.POINTER(C.c_int32)]
        L.bf_score_batch.argtypes = [C.POINTER(bf_batch_t), C.POINTER(bf_result_t)]
        L.bf_score_batch_device.argtypes = [C.POINTER(bf_batch_t), C.POINTER(bf_result_t), C.c_void_p]
        L.bf_kernel_launches.restype = C.c_int64
        L.bf_last_kernel_ms.argtypes = [C.POINTER(C.c_double)]
        L.bf_microbench.argtypes = [C.POINTER(C.c_double)]
        L.bf_second_best.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.bf_subopt.argtypes = [C.c_char_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.bf_sample.argtypes = [C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p]
        L.bf_pair_mfe.argtypes = [C.c_void_p, C.c_void_p]
        L.bf_subopt_zuker.argtypes = [C.c_char_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int32)]
        L.bf_duplex.argtypes = [C.POINTER(bf_duplex_t), C.c_void_p, C.c_void_p]
        L.bf_interact.argtypes = [C.POINTER(bf_interact_t), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.bf_findpath.argtypes = [C.POINTER(bf_findpath_t), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.bf_kinfold.argtypes = [C.POINTER(bf_kinfold_t)] + [C.c_void_p] * 7
        L.bf_unpaired.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.bf_plfold.argtypes = [C.POINTER(bf_strands_t), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
        L.bf_set_option.argtypes = [C.c_char_p, C.c_int]
        L.bf_debug_copy_table.argtypes = [C.c_int, C.c_int32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise EngineError(rc, lib().bf_last_error().decode())


_state = {"inited": False, "params": None}


def init(device=None):
    """Select the GPU (default: LOCAL_RANK or 0) and create the engine."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    _check(lib().bf_init(int(device)))
    _state["inited"] = True


def shutdown():
    lib().bf_shutdown()
    _state["inited"] = False


def params_load(path):
    """RNA.params_load(path) (DesiRNA.py:456)."""
    _check(lib().bf_params_load(os.fsencode(path)))
    _state["params"] = path


def params_builtin(year=1999):
    """`-p 1999|2004` selection of DesiRNA.py:455; 2004 raises EngineError(BF_ERR_UNAVAILABLE)."""
    _check(lib().bf_params_builtin(int(year), os.fsencode(PARAMS_DIR)))
    _state["params"] = f"builtin:{year}"


def params_get(name, *idx):
    idx = list(idx) + [0] * (6 - len(idx))
    out = C.c_int32()
    _check(lib().bf_params_get(name.encode(), *idx, C.byref(out)))
    return out.value


def ensure_ready(device=None):
    if not _state["inited"]:
        init(device)
    if _state["params"] is None:
        params_builtin(1999)


def kernel_launches():
    return int(lib().bf_kernel_launches())


def last_kernel_ms():
    """(mfe_ms, pf_ms, eval_ms) of the most recent call, CUDA-event timed on the launch stream."""
    out = (C.c_double * 3)()
    _check(lib().bf_last_kernel_ms(out))
    return list(out)


def subopt(seq, delta_dcal, nopair=None, max_out=4096):
    """bf_subopt: every structure of one single-strand sequence within delta_dcal of the MFE, sorted by energy.
    Returns (list of (structure, energy_dcal), truncated)."""
    ensure_ready()
    s = seq.upper().replace("T", "U").encode("ascii")
    n = len(s)
    ss = np.zeros((max_out, n + 1), np.uint8)
    en = np.zeros(max_out, np.int32)
    cnt, trunc = C.c_int32(0), C.c_int32(0)
    mask = None
    if nopair is not None:
        mask = np.ascontiguousarray(nopair, np.uint8)
        assert mask.shape == (n,)
    _check(lib().bf_subopt(s, n, mask.ctypes.data if mask is not None else None, int(delta_dcal), max_out, ss.ctypes.data, en.ctypes.data,
                           C.byref(cnt), C.byref(trunc)))
    return [(bytes(ss[k, :n]).decode("ascii"), int(en[k])) for k in range(cnt.value)], bool(trunc.value)


def second_best(seqs, nopair=None):
    """bf_second_best: (e1, e2) int32 arrays, dcal/mol -- energies of the best and the second-best structure of every sequence
    ('A&B' for two strands); e2 >= 10000000 where a sequence has no second structure."""
    ensure_ready()
    buf, lens, cuts = pack([s.upper().replace("T", "U") for s in seqs])
    b = bf_batch_t()
    b.B, b.stride = len(seqs), buf.shape[1]
    b.seq, b.len = buf.ctypes.data, lens.ctypes.data
    b.cut = cuts.ctypes.data if cuts.any() else None
    keep = [buf, lens, cuts]
    if nopair is not None:
        nopair = np.ascontiguousarray(nopair, np.uint8)
        assert nopair.shape == buf.shape
        b.nopair = nopair.ctypes.data
        keep.append(nopair)
    e1, e2 = np.zeros(len(seqs), np.int32), np.zeros(len(seqs), np.int32)
    _check(lib().bf_second_best(C.byref(b), e1.ctypes.data, e2.ctypes.data))
    return e1, e2


def sample(seqs, n_samples, seed=0):
    """bf_sample: stochastic backtracking (ViennaRNA fc.pbacktrack()).  n_samples secondary structures of every single-strand
    sequence, drawn independently from its Boltzmann ensemble; returns a list (per sequence) of lists of dot-bracket strings.
    The samples are a function of (seed, sequence index, sample index) only: the same call repeats, and the first k samples of a
    call with more are those of a call with k."""
    ensure_ready()
    buf, lens, cuts = pack([s.upper().replace("T", "U") for s in seqs])
    b = bf_batch_t()
    b.B, b.stride = len(seqs), buf.shape[1]
    b.seq, b.len = buf.ctypes.data, lens.ctypes.data
    b.cut = cuts.ctypes.data if cuts.any() else None
    n_samples = int(n_samples)
    out = np.zeros((len(seqs), max(n_samples, 1), b.stride + 1), np.uint8)
    _check(lib().bf_sample(C.byref(b), n_samples, int(seed) & ((1 << 64) - 1), out.ctypes.data))
    res = []
    for r in range(len(seqs)):
        n = int(lens[r])
        raw = out[r, :, :n].tobytes().decode("ascii")
        res.append([raw[k * n:(k + 1) * n] for k in range(n_samples)])
    return res


def pair_mfe(seqs, nopair=None):
    """bf_pair_mfe: int32 [B, stride, stride], entry [i-1, j-1] (i < j) the lowest energy in dcal/mol of any structure of single-strand
    sequence b that contains the pair (i,j) -- the matrix of Zuker suboptimals (RNAsubopt -z); 10000000 where no structure contains it
    and on and below the diagonal.  nopair: optional uint8 [B, stride] mask ('x' hard constraint), honoured as by the MFE."""
    ensure_ready()
    buf, lens, cuts = pack([s.upper().replace("T", "U") for s in seqs])
    b = bf_batch_t()
    b.B, b.stride = len(seqs), buf.shape[1]
    b.seq, b.len = buf.ctypes.data, lens.ctypes.data
    b.cut = cuts.ctypes.data if cuts.any() else None
    if nopair is not None:
        nopair = np.ascontiguousarray(nopair, np.uint8)
        assert nopair.shape == buf.shape
        b.nopair = nopair.ctypes.data
    out = np.zeros((len(seqs), b.stride, b.stride), np.int32)
    _check(lib().bf_pair_mfe(C.byref(b), out.ctypes.data))
    return out


def subopt_zuker(seq, nopair=None):
    """bf_subopt_zuker: Zuker suboptimals of one single-strand sequence, [(structure, energy_dcal)] sorted by (energy, structure):
    for every pair (i,j) that some structure contains, a structure of energy E_pair(i,j) that contains it."""
    ensure_ready()
    s = seq.upper().replace("T", "U").encode("ascii")
    n = len(s)
    mask = None
    if nopair is not None:
        mask = np.ascontiguousarray(nopair, np.uint8)
        assert mask.shape == (n,)
    # one structure per uncovered pair: grow the buffer until every pair is covered
    cap = 1024
    while True:
        ss = np.zeros((cap, n + 1), np.uint8)
        en = np.zeros(cap, np.int32)
        cnt, trunc = C.c_int32(0), C.c_int32(0)
        _check(lib().bf_subopt_zuker(s, n, mask.ctypes.data if mask is not None else None, cap, ss.ctypes.data, en.ctypes.data,
                                     C.byref(cnt), C.byref(trunc)))
        if not trunc.value:
            return [(bytes(ss[k, :n]).decode("ascii"), int(en[k])) for k in range(cnt.value)]
        cap *= 8


def duplex(seqs_a, seqs_b, pairs=None, structures=True):
    """bf_duplex: RNA-RNA hybridization (ViennaRNA's duplexfold recurrence, RNAduplex), intermolecular pairs only.  The duplex MFE
    in dcal/mol of every requested pair of strands (10000000: no intermolecular pair is possible).  pairs: [(index into seqs_a,
    index into seqs_b)], or None for the full grid.  Returns int32 energies, shape [P] or [len(seqs_a), len(seqs_b)] for the grid;
    with structures, (energies, structures): 'a-part&b-part' strings, full length, '(' in a and ')' in b, in the same layout (a
    list, or a list of rows for the grid).  Each strand holds at most 2000 nt; T is read as U."""
    if any("&" in s for s in seqs_a) or any("&" in s for s in seqs_b):
        raise ValueError("engine.duplex: a strand may not contain '&' (pass the two strands separately)")
    ensure_ready()
    q = bf_duplex_t()
    keep = []
    for st, seqs in ((q.a, seqs_a), (q.b, seqs_b)):
        buf, lens, _ = pack([s.upper().replace("T", "U") for s in seqs])
        st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, lens.ctypes.data
        keep += [buf, lens]
    la, lb = keep[1], keep[3]
    if pairs is None:
        P, shape = len(seqs_a) * len(seqs_b), (len(seqs_a), len(seqs_b))
        ia, ib = np.repeat(np.arange(len(seqs_a)), len(seqs_b)), np.tile(np.arange(len(seqs_b)), len(seqs_a))
    else:
        pr = np.ascontiguousarray(np.asarray(pairs, np.int32).reshape(-1, 2))
        P, shape = pr.shape[0], (pr.shape[0],)
        q.n_pairs, q.pairs = P, pr.ctypes.data
        keep.append(pr)
        ia, ib = pr[:, 0], pr[:, 1]
    e = np.zeros(P, np.int32)
    ss = np.zeros((P, q.a.stride + q.b.stride + 2), np.uint8) if structures else None
    _check(lib().bf_duplex(C.byref(q), e.ctypes.data, ss.ctypes.data if structures else None))
    e = e.reshape(shape)
    if not structures:
        return e
    out = [bytes(ss[p, :int(la[ia[p]]) + int(lb[ib[p]]) + 1]).decode("ascii") for p in range(P)]
    if pairs is None:
        out = [out[r * len(seqs_b):(r + 1) * len(seqs_b)] for r in range(len(seqs_a))]
    return e, out


def interact(seqs_a, seqs_b, pairs=None, max_span=25, acc_a=0, acc_b=0, structures=True):
    """bf_interact: accessibility-aware RNA-RNA interaction, the best site of every requested pair of strands.  A site is a duplex
    chain as in engine.duplex whose span on each strand is at most max_span (1 .. 64; the default is RNAup's -w 25); its score is
    E = H / 100 + ED_a + ED_b in kcal/mol, H the chain's hybridization energy in dcal/mol and ED = -kT ln P_u the free energy
    that opens the site on each strand.  acc_a / acc_b choose P_u: -1 none (ED = 0), 0 the global ensemble of the whole strand
    (engine.unpaired), W > 0 RNAplfold window averages with span W >= max_span (engine.plfold).  pairs: [(index into seqs_a,
    index into seqs_b)], or None for the full grid.

    Returns a dict of numpy arrays, each of shape [P] or [len(seqs_a), len(seqs_b)] plus a trailing axis where noted: 'e'
    (float64, +inf where no site exists), 'h' (int32, 10000000 where none), 'ed_a', 'ed_b' (float64), 'site' (int32, [..., 4]:
    1-based k1, km in a and lm, l1 in b, 0 where none) and, with structures, 'structures': full-length 'a-part&b-part' strings
    as engine.duplex returns them.  Each strand holds at most 2000 nt; T is read as U.

    ViennaRNA's Python API has no call with this model: RNAup's pf_interact is a partition-function model over all sites, while
    this returns the single site of least E, as RNAplex -a and IntaRNA's MFE mode do, so there is no RNA.py counterpart."""
    if any("&" in s for s in seqs_a) or any("&" in s for s in seqs_b):
        raise ValueError("engine.interact: a strand may not contain '&' (pass the two strands separately)")
    ensure_ready()
    q = bf_interact_t()
    keep = []
    for st, seqs in ((q.a, seqs_a), (q.b, seqs_b)):
        buf, lens, _ = pack([s.upper().replace("T", "U") for s in seqs])
        st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, lens.ctypes.data
        keep += [buf, lens]
    la, lb = keep[1], keep[3]
    q.max_span, q.acc_a, q.acc_b = int(max_span), int(acc_a), int(acc_b)
    if pairs is None:
        P, shape = len(seqs_a) * len(seqs_b), (len(seqs_a), len(seqs_b))
        ia, ib = np.repeat(np.arange(len(seqs_a)), len(seqs_b)), np.tile(np.arange(len(seqs_b)), len(seqs_a))
    else:
        pr = np.ascontiguousarray(np.asarray(pairs, np.int32).reshape(-1, 2))
        P, shape = pr.shape[0], (pr.shape[0],)
        q.n_pairs, q.pairs = P, pr.ctypes.data
        keep.append(pr)
        ia, ib = pr[:, 0], pr[:, 1]
    e = np.zeros(P, np.float64)
    h = np.zeros(P, np.int32)
    ed = np.zeros((P, 2), np.float64)
    site = np.zeros((P, 4), np.int32)
    ss = np.zeros((P, q.a.stride + q.b.stride + 2), np.uint8) if structures else None
    _check(lib().bf_interact(C.byref(q), e.ctypes.data, h.ctypes.data, ed.ctypes.data, site.ctypes.data,
                             ss.ctypes.data if structures else None))
    out = {"e": e.reshape(shape), "h": h.reshape(shape), "ed_a": ed[:, 0].reshape(shape).copy(), "ed_b": ed[:, 1].reshape(shape).copy(),
           "site": site.reshape(shape + (4,))}
    if structures:
        st = [bytes(ss[p, :int(la[ia[p]]) + int(lb[ib[p]]) + 1]).decode("ascii") for p in range(P)]
        if pairs is None:
            st = [st[r * len(seqs_b):(r + 1) * len(seqs_b)] for r in range(len(seqs_a))]
        out["structures"] = st
    return out


def findpath(seqs, s1, s2, width=1, path=True):
    """bf_findpath: direct refolding paths (ViennaRNA's findpath), a breadth-limited search over the paths from s1[r] to s2[r] that
    remove the pairs of s1 that s2 lacks and add the pairs of s2 that s1 lacks, one pair per step.  width: W, 1 .. 1024; the call
    runs widths 1, 2, 4, ... below W, then W, each in both directions, and keeps the path of least saddle (definition in
    include/b200fold.h).  Energies are the engine's eval (dcal/mol); sequences are single strands of at most 2000 nt, T read as U.

    Returns saddles (int32 [n], dcal/mol) and, with path=True, also a list (per instance) of (moves, path_e): moves an int32 [k, 2]
    array of 1-based (i, j), positive for an insertion and negative for a deletion, path_e an int32 [k + 1] array of the energies of
    the structures along the path, E(s1) first."""
    if any("&" in s for s in seqs):
        raise ValueError("engine.findpath: single strands only")
    ensure_ready()
    n = len(seqs)
    buf, lens, _ = pack([s.upper().replace("T", "U") for s in seqs])
    S = buf.shape[1]
    if len(s1) != n or len(s2) != n or any(len(s1[r]) != lens[r] or len(s2[r]) != lens[r] for r in range(n)):
        raise ValueError("engine.findpath: one s1 and one s2 of the sequence's length per sequence")
    t1 = pack_targets([[x] for x in s1], S).reshape(n, S) if n else np.zeros((0, S), np.uint8)
    t2 = pack_targets([[x] for x in s2], S).reshape(n, S) if n else np.zeros((0, S), np.uint8)
    q = bf_findpath_t()
    q.n, q.stride, q.seq, q.len, q.s1, q.s2, q.width = n, S, buf.ctypes.data, lens.ctypes.data, t1.ctypes.data, t2.ctypes.data, int(width)
    sad = np.zeros(n, np.int32)
    k = np.zeros(n, np.int32)
    mv = np.zeros((n, S, 2), np.int32) if path else None
    pe = np.zeros((n, S + 1), np.int32) if path else None
    _check(lib().bf_findpath(C.byref(q), sad.ctypes.data, k.ctypes.data, mv.ctypes.data if path else None, pe.ctypes.data if path else None))
    if not path:
        return sad
    return sad, [(mv[r, :k[r]].copy(), pe[r, :k[r] + 1].copy()) for r in range(n)]


KINFOLD_RULES = {"kawasaki": 0, "metropolis": 1, "descent": 2}


def kinfold(seqs, start=None, stop=None, n_traj=1, rule="kawasaki", t_max=500.0, seed=0, t_snap=None, max_steps=10**6,
            structures=True):
    """bf_kinfold: folding kinetics over single-pair moves (insert or delete one canonical pair; no shift moves), n_traj
    trajectories per sequence.  rule: "kawasaki" (k = exp(-dE / 2kT)) or "metropolis" (k = min(1, exp(-dE / kT))), simulated
    with Gillespie's method up to time t_max, or "descent", the deterministic steepest-descent walk to a local minimum.  start:
    one structure per sequence or None (open chain); stop: one structure per sequence or None, absorbing (a "hit").  t_snap:
    ascending times in [0, t_max] at which the occupied state is recorded.  The trajectories are a function of (seed, sequence
    index, trajectory index) alone.  Definition in include/b200fold.h; single strands of at most 2000 nt, T read as U.

    Returns a dict of numpy arrays shaped [len(seqs), n_traj, ...]: 'status' (int32: 0 t_max reached or, for descent, a local
    minimum; 1 stop structure reached; 2 max_steps moves), 't_end' (float64), 'steps' (int64), 'e_end' (int32, dcal/mol) and,
    with t_snap, 'e_snap' (int32 [..., n_snap]; 10000000 after a cap and for descent); with structures also 'ss_end' and
    'ss_snap' (str, '' where e_snap is 10000000).

    ViennaRNA's Python module has no Kinfold, so there is no RNA.py counterpart."""
    if any("&" in s for s in seqs):
        raise ValueError("engine.kinfold: single strands only")
    if rule not in KINFOLD_RULES:
        raise ValueError("engine.kinfold: rule must be one of " + ", ".join(KINFOLD_RULES))
    ensure_ready()
    n, T = len(seqs), int(n_traj)
    buf, lens, _ = pack([s.upper().replace("T", "U") for s in seqs])
    S = buf.shape[1]
    q = bf_kinfold_t()
    q.n, q.stride, q.seq, q.len, q.n_traj, q.rule = n, S, buf.ctypes.data, lens.ctypes.data, T, KINFOLD_RULES[rule]
    q.t_max, q.seed, q.max_steps = float(t_max), int(seed) & ((1 << 64) - 1), int(max_steps)
    keep = []
    for name, dbs in (("start", start), ("stop", stop)):
        if dbs is None:
            continue
        if len(dbs) != n or any(len(dbs[r]) != lens[r] for r in range(n)):
            raise ValueError(f"engine.kinfold: one {name} structure of the sequence's length per sequence")
        tb = pack_targets([[x] for x in dbs], S).reshape(n, S) if n else np.zeros((0, S), np.uint8)
        keep.append(tb)
        setattr(q, name, tb.ctypes.data)
    ts = np.ascontiguousarray(t_snap if t_snap is not None else [], np.float64).reshape(-1)
    q.n_snap, q.t_snap = ts.size, ts.ctypes.data if ts.size else None
    ns, U = ts.size, n * max(T, 1)
    status = np.zeros(U, np.int32)
    t_end = np.zeros(U, np.float64)
    steps = np.zeros(U, np.int64)
    e_end = np.zeros(U, np.int32)
    e_snap = np.zeros((U, ns), np.int32)
    ss_end = np.zeros((U, S + 1), np.uint8) if structures else None
    ss_snap = np.zeros((U, ns, S + 1), np.uint8) if structures and ns else None
    _check(lib().bf_kinfold(C.byref(q), status.ctypes.data, t_end.ctypes.data, steps.ctypes.data, e_end.ctypes.data,
                            ss_end.ctypes.data if ss_end is not None else None, e_snap.ctypes.data if ns else None,
                            ss_snap.ctypes.data if ss_snap is not None else None))
    shape = (n, T)
    out = {"status": status.reshape(shape), "t_end": t_end.reshape(shape), "steps": steps.reshape(shape), "e_end": e_end.reshape(shape)}
    if ns:
        out["e_snap"] = e_snap.reshape(shape + (ns,))
    if structures:
        out["ss_end"] = ss_end.view(f"S{S + 1}").reshape(shape).astype(str)
        if ns:
            out["ss_snap"] = ss_snap.view(f"S{S + 1}").reshape(shape + (ns,)).astype(str)
    return out


def unpaired(seqs, max_u):
    """bf_unpaired: float64 [B, stride, max_u], entry [b, i-1, u-1] the probability that positions i .. i+u-1 (1-based) of
    single-strand sequence b are all unpaired, in the ensemble of WANT_BPP (RNAplfold -u over the whole sequence); 0 where
    i+u-1 > len.  T is read as U."""
    ensure_ready()
    buf, lens, cuts = pack([s.upper().replace("T", "U") for s in seqs])
    b = bf_batch_t()
    b.B, b.stride = len(seqs), buf.shape[1]
    b.seq, b.len = buf.ctypes.data, lens.ctypes.data
    b.cut = cuts.ctypes.data if cuts.any() else None
    out = np.zeros((len(seqs), b.stride, max(int(max_u), 1)), np.float64)
    _check(lib().bf_unpaired(C.byref(b), int(max_u), out.ctypes.data))
    return out


def plfold(seqs, winsize, max_u=31, pairs=True):
    """bf_plfold: RNAplfold with span = window size over single strands.  Returns one (band, pu) per sequence of length n:
    band float64 [n, winsize], band[i-1, d] the mean pair probability of (i, i+d) over the windows that hold both (None unless
    pairs), and pu float64 [n, max_u], pu[i-1, u-1] the mean probability that i .. i+u-1 is unpaired over the windows that hold
    it.  T is read as U."""
    if any("&" in s for s in seqs):
        raise ValueError("engine.plfold: single strands only (a sequence contains '&')")
    ensure_ready()
    buf, lens, _ = pack([s.upper().replace("T", "U") for s in seqs])
    st = bf_strands_t()
    st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, lens.ctypes.data
    W, U = int(winsize), int(max_u)
    band = np.zeros((len(seqs), st.stride, max(W, 1)), np.float64) if pairs else None
    pu = np.zeros((len(seqs), st.stride, max(U, 1)), np.float64)
    _check(lib().bf_plfold(C.byref(st), W, U, band.ctypes.data if pairs else None, pu.ctypes.data))
    return [(band[r, :int(lens[r])] if pairs else None, pu[r, :int(lens[r])]) for r in range(len(seqs))]


def set_option(key, value):
    """Test / measurement hook (bf_set_option): sets the engine's BF_<KEY> variable, e.g. set_option("cl", 0) switches the
    cluster-per-sequence fill kernels off, set_option("cl", -1) restores the default rule.  The keys are listed in
    include/b200fold.h; any other key raises."""
    ensure_ready()
    _check(lib().bf_set_option(key.encode(), int(value)))


def debug_table(which, n_seq):
    """Test hook: the packed diagonal-major DP table (0 = c, 1 = fML, 2 = qb) of the most recent call, [n_seq, slot]."""
    slot = C.c_size_t(0)
    _check(lib().bf_debug_copy_table(which, n_seq, None, 0, C.byref(slot)))
    out = np.zeros((n_seq, slot.value), np.float64 if which == 2 else np.int32)
    _check(lib().bf_debug_copy_table(which, n_seq, out.ctypes.data, out.nbytes, C.byref(slot)))
    return out


def microbench():
    """{'int32_ops', 'fp64_flops', 'smem_bytes'} per second, measured on the current GPU."""
    ensure_ready()
    out = (C.c_double * 3)()
    _check(lib().bf_microbench(out))
    return {"int32_ops_per_s": out[0], "fp64_flops_per_s": out[1], "smem_bytes_per_s": out[2]}


def score_batch_device(seq, lens, want, cut=None, nopair=None, targets=None, mfe=None, ss=None, pf=None, ev=None, stream=0, defect=None,
                       bpp=None):
    """Device-resident entry point (bf_score_batch_device).  Arguments are torch CUDA tensors:
    seq uint8[B,stride], lens int32[B], cut int32[B], nopair uint8[B,stride], targets uint8[B,T,stride];
    outputs mfe int32[B], ss uint8[B,stride+1], pf float64[B,5], ev int32[B,T].  Enqueues on `stream`
    (a raw cudaStream_t handle, e.g. torch.cuda.current_stream().cuda_stream) without synchronising."""
    ensure_ready()
    b, r = bf_batch_t(), bf_result_t()
    b.B, b.stride = int(seq.shape[0]), int(seq.shape[1])
    b.seq, b.len = seq.data_ptr(), lens.data_ptr()
    b.cut = cut.data_ptr() if cut is not None else None
    b.nopair = nopair.data_ptr() if nopair is not None else None
    if targets is not None:
        b.targets, b.n_targets = targets.data_ptr(), int(targets.shape[1])
    b.want = want
    r.mfe_dcal = mfe.data_ptr() if mfe is not None else None
    r.mfe_ss = ss.data_ptr() if ss is not None else None
    r.pf = pf.data_ptr() if pf is not None else None
    r.eval_dcal = ev.data_ptr() if ev is not None else None
    r.defect = defect.data_ptr() if defect is not None else None   # float64[B]
    r.bpp = bpp.data_ptr() if bpp is not None else None            # float64[B,stride,stride]
    _check(lib().bf_score_batch_device(C.byref(b), C.byref(r), C.c_void_p(stream)))


def sm_count():
    return int(lib().bf_sm_count())


def pack(seqs, stride=None):
    """list of str (optionally 'A&B') -> (chars[B,stride] uint8, len[B] int32, cut[B] int32)."""
    B = len(seqs)
    clean, cuts = [], np.zeros(B, np.int32)
    for k, s in enumerate(seqs):
        if "&" in s:
            a, b = s.split("&")[:2]
            cuts[k] = len(a) + 1
            s = a + b
        clean.append(s)
    lens = np.array([len(s) for s in clean], np.int32)
    if stride is None:
        stride = max(1, int(lens.max()) if B else 1)
    # one join + one frombuffer instead of a numpy assignment per row (rows padded with NUL to the stride)
    flat = "".join(s if len(s) == stride else s.ljust(stride, "\0") for s in clean).encode("ascii")
    buf = np.frombuffer(flat, np.uint8).reshape(B, stride).copy() if B else np.zeros((0, stride), np.uint8)
    return buf, lens, cuts


def pack_targets(targets, stride):
    """targets: list (per sequence) of list of dot-bracket strings ('&' dropped) -> uint8[B,T,stride]"""
    B = len(targets)
    T = len(targets[0]) if B else 0
    rows = []
    for row in targets:
        assert len(row) == T, "every sequence needs the same number of targets"
        for db in row:
            if "&" in db:
                db = db.replace("&", "")
            rows.append(db if len(db) == stride else db.ljust(stride, "."))
    if not rows:
        return np.full((B, T, stride), ord("."), np.uint8)
    return np.frombuffer("".join(rows).encode("ascii"), np.uint8).reshape(B, T, stride).copy()


def score_batch(seqs, targets=None, nopair=None, want=WANT_MFE | WANT_SS | WANT_PF):
    """Host-buffer entry point (bf_score_batch).  seqs: list of str; targets: list of lists of
    dot-bracket strings; nopair: optional uint8[B, stride] mask.  Returns a dict of numpy arrays."""
    ensure_ready()
    B = len(seqs)
    if B == 0:
        return {"len": np.zeros(0, np.int32), "cut": np.zeros(0, np.int32), "mfe_dcal": np.zeros(0, np.int32),
                "mfe_ss": [], "pf": np.zeros((0, 5)), "eval_dcal": np.zeros((0, 0), np.int32)}
    buf, lens, cuts = pack(seqs)
    stride = buf.shape[1]
    b, r = bf_batch_t(), bf_result_t()
    b.B, b.stride = B, stride
    b.seq, b.len = buf.ctypes.data, lens.ctypes.data
    b.cut = cuts.ctypes.data if cuts.any() else None
    keep = [buf, lens, cuts]
    if nopair is not None:
        nopair = np.ascontiguousarray(nopair, np.uint8)
        assert nopair.shape == (B, stride)
        b.nopair = nopair.ctypes.data
        keep.append(nopair)
    out = {}
    if targets is not None and (want & (WANT_EVAL | WANT_DEFECT)):
        tb = pack_targets(targets, stride)
        b.targets, b.n_targets = tb.ctypes.data, tb.shape[1]
        keep.append(tb)
        if want & WANT_EVAL:
            out["eval_dcal"] = np.zeros((B, tb.shape[1]), np.int32)
            r.eval_dcal = out["eval_dcal"].ctypes.data
    else:
        want &= ~(WANT_EVAL | WANT_DEFECT)
    if want & (WANT_BPP | WANT_DEFECT):
        want |= WANT_MFE | WANT_PF   # the MFE sets the partition function's scale (energy_scores.py:371-372)
    if want & WANT_DEFECT:
        out["defect"] = np.zeros(B, np.float64)
        r.defect = out["defect"].ctypes.data
    if want & WANT_BPP:
        out["bpp"] = np.zeros((B, stride, stride), np.float64)
        r.bpp = out["bpp"].ctypes.data
    if want & (WANT_MFE | WANT_SS):
        want |= WANT_MFE
        out["mfe_dcal"] = np.zeros(B, np.int32)
        r.mfe_dcal = out["mfe_dcal"].ctypes.data
    if want & WANT_SS:
        ss = np.zeros((B, stride + 1), np.uint8)
        r.mfe_ss = ss.ctypes.data
    if want & WANT_PF:
        out["pf"] = np.zeros((B, 5), np.float64)
        r.pf = out["pf"].ctypes.data
    b.want = want
    _check(lib().bf_score_batch(C.byref(b), C.byref(r)))
    if want & WANT_SS:
        raw, w = ss.tobytes().decode("ascii"), stride + 1
        out["mfe_ss"] = [raw[k * w:k * w + int(lens[k])] for k in range(B)]
    out["len"], out["cut"] = lens, cuts
    return out

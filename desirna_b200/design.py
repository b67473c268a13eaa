"""Many design problems x replicas in ONE device-resident Replica-Exchange Monte-Carlo loop (C-ABI bf_design_*).

The reference designs one target per process: `DesiRNA.py:331-383` runs, per global step, `remc.mutate_sequence_re`
(R worker processes x RE_attempt Metropolis sub-steps, utils/replica_exchange_monte_carlo.py:233-271) and
`remc.replica_exchange` (:113-173).  With R = 10..64 mutants per sub-step a B200 idles (SURVEY.md section 0, finding 6), so
this driver advances ALL targets of a benchmark (e.g. the 100 Eterna puzzles) together: jobs are bucketed by length,
each bucket is one `bf_design_*` loop on its own CUDA stream, and a sub-step of a bucket is
propose -> MFE fill + backtrack -> PF fill -> eval -> accept for (jobs x replicas) sequences without leaving the GPU.

Host work per poll: read the per-job best records, retire solved jobs (`-sws on`), check the clock.
"""
import ctypes as C
import random
import re
import time

import numpy as np

from . import engine
from .utils import sequence_utils as seq_utils

TERM_ID = {"Ed-Epf": 0, "1-MCC": 1, "sln_Epf": 2, "Ed-MFE": 3, "1-precision": 4, "1-recall": 5, "Edef": 6}
REC_FIELDS = ("scoring_function", "edesired", "Epf", "mcc", "precision", "recall", "MFE", "ensemble_defect", "distance", "global_step",
              "oligo_fraction", "oligomer_bonus", "edesired2", "motif_bonus", "subopt_e")
REC = len(REC_FIELDS)


class DesignOptions:
    """The fields of DesiRNA.py's DesignOptions (:520-633) the loop reads, with the CLI defaults (:92-139)."""

    def __init__(self, replicas=10, RE_attempt=100, T_min=10.0, T_max=150.0, scoring_f=(("Ed-Epf", 1.0),), point_mutations="on",
                 tm_max=0.7, tm_min=0.0, acgu_percentages="off", nt_percentages=None, diff_start_replicas="one", oligo_state="none",
                 motifs=None, pks="off", subopt="off"):
        self.replicas = replicas
        self.RE_attempt = RE_attempt
        self.T_min, self.T_max = T_min, T_max
        self.scoring_f = list(scoring_f)
        self.point_mutations = point_mutations
        self.tm_max, self.tm_min = tm_max, tm_min
        self.acgu_percentages = acgu_percentages
        self.nt_percentages = nt_percentages or {"A": 15, "C": 30, "G": 30, "U": 15}
        self.diff_start_replicas = diff_start_replicas
        self.L = 504.12
        self.oligo_state, self.pks, self.subopt = oligo_state, pks, subopt   # "none" | "heterodimer" | "homodimer" | "avoid" (-o on)
        # -motifs "KEY,bonus,KEY,bonus": IUPAC motif -> (compiled regex, bonus) as DesiRNA.py:212-224 builds it
        self.motifs = {k: (re.compile("".join("[%s]" % seq_utils.IUPAC.get(ch, ch) for ch in k)), float(v)) for k, v in (motifs or {}).items()} or None
        self.rep_temps_shelfs = seq_utils.get_rep_temps(self)


class bf_design_t(C.Structure):
    _fields_ = [("n_jobs", C.c_int32), ("replicas", C.c_int32), ("stride", C.c_int32), ("target", C.c_void_p), ("len", C.c_void_p),
                ("len_a", C.c_void_p), ("allowed", C.c_void_p), ("init_seq", C.c_void_p), ("temps", C.c_void_p), ("tm_prob", C.c_void_p),
                ("n_terms", C.c_int32), ("term", C.c_int32 * 8), ("weight", C.c_double * 8), ("metropolis_L", C.c_double),
                ("point_mutations", C.c_int32), ("re_attempt", C.c_int32), ("acgu", C.c_int32), ("nt_weight", C.c_double * 4),
                ("oligo", C.c_int32), ("seed", C.c_uint64), ("alt_targets", C.c_void_p), ("n_alt", C.c_void_p), ("max_alt", C.c_int32),
                ("n_motifs", C.c_int32), ("motif_mask", C.c_void_p), ("motif_len", C.c_void_p), ("motif_bonus", C.c_void_p), ("pks", C.c_int32), ("move_partner", C.c_void_p), ("snake_id", C.c_void_p),
                ("snake_letter", C.c_void_p), ("subopt", C.c_int32)]


def _bind():
    L = engine.lib()
    if not getattr(L, "_design_bound", False):
        L.bf_design_create.argtypes = [C.POINTER(bf_design_t), C.POINTER(C.c_void_p)]
        L.bf_design_run.argtypes = [C.c_void_p, C.c_int32]
        L.bf_design_sync.argtypes = [C.c_void_p]
        L.bf_design_busy.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
        L.bf_design_set_active.argtypes = [C.c_void_p, C.c_void_p]
        L.bf_design_read_jobs.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        L.bf_design_read_replicas.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        L.bf_design_read_swaps.argtypes = [C.c_void_p, C.c_void_p]
        L.bf_design_propose_only.argtypes = [C.c_void_p, C.c_void_p]
        L.bf_design_destroy.argtypes = [C.c_void_p]
        L._design_bound = True
    return L


def _chars(rows, stride):
    out = np.zeros((len(rows), stride), np.uint8)
    for k, s in enumerate(rows):
        out[k, :len(s)] = np.frombuffer(s.encode("ascii"), np.uint8)
    return out


def _strings(buf, lens, len_a=None):
    """rows of a char buffer -> str; two-strand rows get their '&' back after strand A"""
    out = [bytes(buf[k, :lens[k]]).decode("ascii") for k in range(buf.shape[0])]
    if len_a is not None:
        out = [s[:a] + "&" + s[a:] if a > 0 else s for s, a in zip(out, len_a)]
    return out


class DesignLoop:
    """One bf_design_* loop: the jobs of one length bucket."""

    def __init__(self, inputs, sim_options, seed=0, init_seqs=None):
        engine.ensure_ready()
        self.lib = _bind()
        self.inputs = list(inputs)
        self.J, self.R = len(self.inputs), sim_options.replicas
        for inp in self.inputs:
            pk_ok = sim_options.pks == "on" and "&" not in inp.sec_struct
            if set(inp.sec_struct) - set(".()&" + ("[]<>{}" if pk_ok else "")) or inp.sec_struct.count("&") > 1:
                raise ValueError("the device design loop takes targets made of . ( ), one strand or 'A&B' (with pks='on': also [ ] < > { }): %r" % (inp.name,))
            if "&" in inp.sec_struct and sim_options.oligo_state not in ("heterodimer", "homodimer"):
                raise ValueError("two-strand targets need oligo_state='heterodimer' or 'homodimer'")
            if sim_options.oligo_state == "homodimer" and len(set(map(len, inp.sec_struct.split("&")))) != 1:
                raise ValueError("homodimer targets need two strands of equal length: %r" % (inp.name,))
        # the reference's strings carry the '&'; the engine's do not: len_a remembers where it sat
        self.len_a = np.array([i.sec_struct.index("&") if "&" in i.sec_struct else 0 for i in self.inputs], np.int32)
        self.lens = np.array([len(i.sec_struct.replace("&", "")) for i in self.inputs], np.int32)
        self.stride = int(self.lens.max())
        for inp in self.inputs:   # alternative structures: conflict graphs before the per-position restraints (DesiRNA.py:277-284)
            if inp.alt_sec_struct is not None and "&" not in inp.sec_struct and inp.graphs is None and inp.excluded_alt_pairs is None:
                seq_utils.attach_alternatives(inp)
        nt_lists = [seq_utils.get_nt_list(i) for i in self.inputs]
        allowed = np.full((self.J, self.stride), 15, np.uint8)
        for j, nts in enumerate(nt_lists):
            allowed[j, :self.lens[j]] = seq_utils.allowed_masks([nt for nt in nts if nt.letters != ["&"]])
        if init_seqs is None:
            init_seqs = []
            for inp, nts in zip(self.inputs, nt_lists):
                first = seq_utils.initial_sequence_generator(nts, inp, sim_options)
                for _ in range(self.R):
                    init_seqs.append(seq_utils.initial_sequence_generator(nts, inp, sim_options)
                                     if sim_options.diff_start_replicas == "different" else first)
        init_seqs = [x.replace("&", "") for x in init_seqs]
        assert len(init_seqs) == self.J * self.R
        terms = [(TERM_ID[f], float(w)) for f, w in sim_options.scoring_f]
        cfg = bf_design_t()
        self._keep = [_chars([i.sec_struct.replace("&", "") for i in self.inputs], self.stride), self.lens, self.len_a, allowed, _chars(init_seqs, self.stride),
                      np.array(sim_options.rep_temps_shelfs, np.float64), np.array(seq_utils.targeted_move_probabilities(sim_options), np.float64)]
        cfg.n_jobs, cfg.replicas, cfg.stride = self.J, self.R, self.stride
        cfg.target, cfg.len, cfg.len_a, cfg.allowed, cfg.init_seq, cfg.temps, cfg.tm_prob = (a.ctypes.data for a in self._keep)
        cfg.oligo = {"heterodimer": 1, "homodimer": 2, "avoid": 3}.get(sim_options.oligo_state, 0)
        cfg.n_terms = len(terms)
        for k, (t, w) in enumerate(terms):
            cfg.term[k], cfg.weight[k] = t, w
        cfg.metropolis_L = sim_options.L
        cfg.point_mutations = int(sim_options.point_mutations == "on")
        cfg.re_attempt = sim_options.RE_attempt
        cfg.acgu = int(sim_options.acgu_percentages == "on")
        for k, l in enumerate("ACGU"):
            cfg.nt_weight[k] = float(sim_options.nt_percentages[l])
        cfg.seed = seed
        cfg.pks = int(sim_options.pks == "on")
        cfg.subopt = int(sim_options.subopt == "on")
        # alternative structures (scored as mean(eval) - Epf, energy_scores.py:98-102; the move generator keeps to the main target)
        alts = [list(i.alt_sec_structs) if i.alt_sec_struct is not None else [] for i in self.inputs]
        if any(alts):
            # the move generator's partners (the clash-free pairs of the alternatives are restraints too) and the conflict graphs
            mp = np.full((self.J, self.stride), -1, np.int16)
            sid = np.full((self.J, self.stride), -1, np.int8)
            sl = np.zeros((self.J, self.stride, 4), np.uint8)
            for j, nts in enumerate(nt_lists):
                for nt in nts:
                    if nt.pairs_with is not None:
                        mp[j, nt.number] = nt.pairs_with
                    if nt.snake:
                        sid[j, nt.number] = nt.snake_number
                        at = nt.snake_nts.index(nt.number)
                        for k, st in enumerate(nt.snake_states):
                            sl[j, nt.number, k] = ord(st[at])
            self._keep += [mp, sid, sl]
            cfg.move_partner, cfg.snake_id, cfg.snake_letter = mp.ctypes.data, sid.ctypes.data, sl.ctypes.data
            for inp, al in zip(self.inputs, alts):
                if any(set(a) - set(".()") or len(a) != len(inp.sec_struct) for a in al):
                    raise ValueError("alternative structures must be made of . ( ) and as long as the target: %r" % (inp.name,))
            max_alt = max(len(a) for a in alts)
            buf = np.full((self.J, max_alt, self.stride), ord("."), np.uint8)
            for j, al in enumerate(alts):
                for k, a in enumerate(al):
                    buf[j, k, :len(a)] = np.frombuffer(a.encode("ascii"), np.uint8)
            n_alt = np.array([len(a) for a in alts], np.int32)
            self._keep += [buf, n_alt]
            cfg.alt_targets, cfg.n_alt, cfg.max_alt = buf.ctypes.data, n_alt.ctypes.data, max_alt
        if sim_options.motifs:
            keys = list(sim_options.motifs)
            if len(keys) > 8 or any(len(k) > 32 or set(k) - set(seq_utils.IUPAC) - set("ACGU") for k in keys):
                raise ValueError("the device loop takes up to 8 IUPAC motifs of up to 32 letters")
            mm = np.zeros((len(keys), 32), np.uint8)
            for m, k in enumerate(keys):
                for p, ch in enumerate(k):
                    mm[m, p] = sum(1 << "ACGU".index(x) for x in seq_utils.IUPAC.get(ch, ch))
            ml = np.array([len(k) for k in keys], np.int32)
            mb = np.array([sim_options.motifs[k][1] for k in keys], np.float64)
            self._keep += [mm, ml, mb]
            cfg.n_motifs, cfg.motif_mask, cfg.motif_len, cfg.motif_bonus = len(keys), mm.ctypes.data, ml.ctypes.data, mb.ctypes.data
        self.h = C.c_void_p()
        engine._check(self.lib.bf_design_create(C.byref(cfg), C.byref(self.h)))
        self.active = np.ones(self.J, np.uint8)

    # -- stepping
    def run(self, global_steps=1):
        engine._check(self.lib.bf_design_run(self.h, int(global_steps)))

    def sync(self):
        engine._check(self.lib.bf_design_sync(self.h))

    def busy(self):
        flag = C.c_int32(0)
        engine._check(self.lib.bf_design_busy(self.h, C.byref(flag)))
        return bool(flag.value)

    def set_active(self, mask):
        self.active = np.ascontiguousarray(mask, np.uint8)
        engine._check(self.lib.bf_design_set_active(self.h, self.active.ctypes.data))

    # -- reading
    def jobs(self):
        seq = np.zeros((self.J, self.stride), np.uint8)
        ss = np.zeros((self.J, self.stride + 1), np.uint8)
        rec = np.zeros((self.J, REC))
        step = np.zeros(self.J, np.int32)
        nsol = np.zeros(self.J, np.uint32)
        engine._check(self.lib.bf_design_read_jobs(self.h, seq.ctypes.data, ss.ctypes.data, rec.ctypes.data, step.ctypes.data, nsol.ctypes.data))
        return {"sequence": _strings(seq, self.lens, self.len_a), "mfe_ss": _strings(ss, self.lens, self.len_a), "rec": rec,
                "solved_step": step, "n_solved": nsol}

    def replicas(self):
        G = self.J * self.R
        seq = np.zeros((G, self.stride), np.uint8)
        ss = np.zeros((G, self.stride + 1), np.uint8)
        rec = np.zeros((G, REC))
        shelf = np.zeros(G, np.int32)
        counts = np.zeros((G, 3), np.uint32)
        engine._check(self.lib.bf_design_read_replicas(self.h, seq.ctypes.data, ss.ctypes.data, rec.ctypes.data, shelf.ctypes.data, counts.ctypes.data))
        lens, la = np.repeat(self.lens, self.R), np.repeat(self.len_a, self.R)
        return {"sequence": _strings(seq, lens, la), "mfe_ss": _strings(ss, lens, la), "rec": rec, "shelf": shelf.reshape(self.J, self.R),
                "counts": counts}

    def swaps(self):
        """neighbour-swap counters per job: accepted, accepted because not worse, rejected"""
        out = np.zeros((self.J, 3), np.uint32)
        engine._check(self.lib.bf_design_read_swaps(self.h, out.ctypes.data))
        return out

    def records(self, sim_options, sim_step):
        """the current replica states as the dicts DesiRNA.py appends to `simulation_data` (vars(ScoreSeq), DesiRNA.py:373-375),
        one list per job"""
        rep = self.replicas()
        out = []
        for j in range(self.J):
            rows = []
            for r in range(self.R):
                g = j * self.R + r
                v = dict(zip(REC_FIELDS, rep["rec"][g]))
                n = len(rep["sequence"][g])
                row = {"sequence": rep["sequence"][g], "scoring_function": v["scoring_function"], "replica_num": r + 1,
                       "temp_shelf": sim_options.rep_temps_shelfs[rep["shelf"][j, r]], "sim_step": sim_step,
                       "edesired_minus_Epf": v["edesired"] - v["Epf"], "Epf": v["Epf"], "edesired": v["edesired"], "mcc": v["mcc"], "mcc_alt": 0,
                       "mfe_ss": rep["mfe_ss"][g], "subopt_e": v["subopt_e"], "esubopt_minus_Epf": (v["subopt_e"] - v["Epf"]) if sim_options.subopt == "on" and v["mcc"] == 0 else 0,
                       "sln_Epf": (v["Epf"] + 0.3759 * n + 5.7534) / 10 if any(f == "sln_Epf" for f, _ in sim_options.scoring_f) else 0,
                       "MFE": v["MFE"] if any(f == "Ed-MFE" for f, _ in sim_options.scoring_f) else 0,
                       "edesired_minus_MFE": v["edesired"] - v["MFE"] if any(f == "Ed-MFE" for f, _ in sim_options.scoring_f) else 0,
                       "recall": v["recall"], "precision": v["precision"]}
                has_alt = self.inputs[j].alt_sec_struct is not None
                row["edesired2"] = v["edesired2"] if has_alt else 0
                row["edesired2_minus_Epf"] = v["edesired2"] - v["Epf"] if has_alt else 0
                if any(f == "Edef" for f, _ in sim_options.scoring_f):
                    row["ensemble_defect"] = v["ensemble_defect"]
                if self.len_a[j] > 0:
                    row["oligo_fraction"], row["oligomer_bonus"] = v["oligo_fraction"], v["oligomer_bonus"]
                elif sim_options.oligo_state == "avoid":   # ScoreSeq.get_scoring_function_monomer's fields; the record slot is shared
                    row["oligo_fraction"], row["monomer_bonus"] = v["oligo_fraction"], v["oligomer_bonus"]
                rows.append(row)
            out.append(rows)
        return out

    def propose_only(self):
        """test hook: one draw of the move generator for every replica of every active job, not scored, not accepted"""
        rows = int(self.active.sum()) * self.R
        out = np.zeros((rows, self.stride), np.uint8)
        engine._check(self.lib.bf_design_propose_only(self.h, out.ctypes.data))
        act = self.active.astype(bool)
        return _strings(out, np.repeat(self.lens[act], self.R), np.repeat(self.len_a[act], self.R))

    def close(self):
        if self.h:
            self.lib.bf_design_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


BUCKET_EDGES = (40, 72, 104, 136, 200, 304, 400, 600, 1000, 2000)


def bucket_jobs(lengths, edges=BUCKET_EDGES):
    """indices of the jobs per length bucket (jobs of one loop share a table stride, so similar lengths go together)"""
    out = {}
    for k, n in enumerate(lengths):
        for e in edges:
            if n <= e:
                out.setdefault(e, []).append(k)
                break
        else:
            raise ValueError("target longer than %d nt" % edges[-1])
    return [out[e] for e in sorted(out)]


def shard_jobs(lengths, world):
    """Job indices per rank: longest first, each to the least loaded rank, load ~ L^3 (the fold's cost).  Every rank computes
    the same assignment; nothing is exchanged until the results are gathered (SURVEY.md section 8e: independent units)."""
    load = [0.0] * world
    out = [[] for _ in range(world)]
    for k in sorted(range(len(lengths)), key=lambda k: (-lengths[k], k)):
        r = min(range(world), key=lambda r: (load[r], r))
        out[r].append(k)
        load[r] += float(lengths[k]) ** 3
    return [sorted(x) for x in out]


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist
    except Exception:
        pass
    return None


def design_batch_sharded(inputs, sim_options, **kw):
    """design_batch with the jobs sharded over the ranks of torch.distributed (one process per GPU): each rank designs its
    own targets; the per-job results are all-gathered at the end.  Returns (results in input order, info of this rank with
    the job-weighted totals of all ranks) on every rank."""
    dist = _dist()
    inputs = list(inputs)
    if dist is None:
        return design_batch(inputs, sim_options, **kw)
    rank, world = dist.get_rank(), dist.get_world_size()
    mine = shard_jobs([len(i.sec_struct) for i in inputs], world)[rank]
    kw = dict(kw)
    kw["seed"] = kw.get("seed", 0) * 131 + rank
    res, info = design_batch([inputs[k] for k in mine], sim_options, **kw) if mine else ([], {"folds": 0, "seconds": 0.0, "solved": 0, "jobs": 0, "global_steps": 0, "buckets": []})
    gathered = [None] * world
    dist.all_gather_object(gathered, (mine, res, info))
    results = [None] * len(inputs)
    for idx, rr, _ in gathered:
        for k, r in zip(idx, rr):
            results[k] = r
    infos = [g[2] for g in gathered]
    total = dict(info)
    total.update(folds=sum(i["folds"] for i in infos), solved=sum(i["solved"] for i in infos), jobs=len(inputs),
                 seconds=max(i["seconds"] for i in infos), per_rank=[{"jobs": i["jobs"], "solved": i["solved"], "folds": i["folds"], "seconds": i["seconds"]} for i in infos])
    total["folds_per_s"] = total["folds"] / max(total["seconds"], 1e-9)
    return results, total


def design_batch(inputs, sim_options, time_limit=None, global_steps=None, stop_when_solved=True, seed=0, poll_steps=1,
                 edges=BUCKET_EDGES, verbose=False, trajectory=False):
    """Design every target of `inputs` (InputFile objects, utils/stats_inputs_outputs.py) concurrently.

    Stops when every job is solved (stop_when_solved, the reference's `-sws on` with `-r 1`), after `global_steps` global
    steps (`-s`), or after `time_limit` seconds (`-t`), whichever comes first.  Returns (results, info): one dict per input
    (REC_FIELDS + name, sequence, mfe_ss, solved, solved_step, solved_after_s; + monomer_bonus with oligo_state="avoid") and run
    statistics.

    trajectory=True (use poll_steps=1) also records, per job, what DesiRNA.py keeps as `simulation_data` -- the state of every
    replica after each global step -- and a Stats object, as info["simulation_data"][k] / info["stats"][k]: the inputs of
    utils.stats_inputs_outputs.parse_and_output_results, which writes the reference's result files."""
    if time_limit is None and global_steps is None:
        raise ValueError("give time_limit and/or global_steps")
    random.seed(seed)
    inputs = list(inputs)
    # two-strand jobs fold with the two-strand kernels: they get loops of their own
    one = [k for k, i in enumerate(inputs) if "&" not in i.sec_struct]
    two = [k for k, i in enumerate(inputs) if "&" in i.sec_struct]
    groups = [[sub[k] for k in grp] for sub in (one, two) if sub for grp in bucket_jobs([len(inputs[k].sec_struct) for k in sub], edges)]
    t_start = time.time()
    loops = [DesignLoop([inputs[k] for k in grp], sim_options, seed=seed * 1000003 + b) for b, grp in enumerate(groups)]
    results = [None] * len(inputs)
    solved_at = [None] * len(inputs)
    done = [0] * len(loops)          # global steps finished, per loop
    folds = sum(l.J * l.R for l in loops)   # start sequences
    sim_data = [[] for _ in inputs] if trajectory else None

    def harvest(b, now):
        """read loop b (waits for its stream), record results, retire solved jobs; returns its number of unsolved jobs"""
        grp, loop = groups[b], loops[b]
        jb = loop.jobs()
        mask = loop.active.copy()
        if trajectory:
            recs = loop.records(sim_options, done[b] * sim_options.RE_attempt)
            for pos, k in enumerate(grp):
                if loop.active[pos]:
                    sim_data[k].extend(recs[pos])
        for pos, k in enumerate(grp):
            solved = jb["solved_step"][pos] >= 0
            if solved and solved_at[k] is None:
                solved_at[k] = now
            res = {"name": inputs[k].name, "sequence": jb["sequence"][pos], "mfe_ss": jb["mfe_ss"][pos], "solved": bool(solved),
                   "solved_step": int(jb["solved_step"][pos]), "solved_after_s": solved_at[k]}
            res.update({f: float(jb["rec"][pos, c]) for c, f in enumerate(REC_FIELDS)})
            if sim_options.oligo_state == "avoid":
                res["monomer_bonus"] = res["oligomer_bonus"]
            results[k] = res
            if solved and stop_when_solved:
                mask[pos] = 0
        if (mask != loop.active).any():
            loop.set_active(mask)
        return int(loop.active.sum())

    # Every loop advances at its own pace: a bucket of short targets makes hundreds of global steps while the 400-nt bucket makes
    # one.  A loop gets `batch[b]` global steps at a time, sized from its measured pace to ~poll_seconds of GPU time (the host
    # reads results and retires solved jobs in between); with trajectory=True every poll_steps-th state must be seen instead.
    poll_seconds = 0.5
    batch = [poll_steps] * len(loops)
    pending = [None] * len(loops)     # (steps enqueued, enqueue time) of a running batch
    left = [harvest(b, time.time() - t_start) for b in range(len(loops))]
    while True:
        now = time.time() - t_start
        out_of_time = time_limit is not None and now >= time_limit
        progressed = False
        for b, loop in enumerate(loops):
            if pending[b] is not None:
                if loop.busy():
                    continue
                n, t0 = pending[b]
                pending[b] = None
                done[b] += n
                left[b] = harvest(b, time.time() - t_start)
                if not trajectory:
                    pace = max((time.time() - t_start - t0) / n, 1e-4)     # seconds per global step, as last observed
                    batch[b] = int(min(64, max(1, poll_seconds / pace)))
                progressed = True
                if verbose:
                    print("loop %d (stride %d): %d global steps, %d jobs unsolved, %.1f s" % (b, loop.stride, done[b], left[b], time.time() - t_start), flush=True)
            if left[b] > 0 and not out_of_time and (global_steps is None or done[b] < global_steps):
                n = batch[b] if global_steps is None else min(batch[b], global_steps - done[b])
                loop.run(n)
                pending[b] = (n, time.time() - t_start)
                folds += left[b] * loop.R * sim_options.RE_attempt * n
                progressed = True
        if all(p is None for p in pending):
            break     # nothing running and nothing could be started: solved, out of steps or out of time
        if not progressed:
            time.sleep(0.001)
    steps = max(done) if done else 0
    elapsed = time.time() - t_start
    info = {"global_steps": steps, "global_steps_per_loop": list(done), "seconds": elapsed, "folds": folds, "folds_per_s": folds / max(elapsed, 1e-9),
            "solved": sum(1 for r in results if r["solved"]), "jobs": len(inputs), "buckets": [(l.stride, l.J) for l in loops]}
    if trajectory:
        from .utils.stats_inputs_outputs import Stats
        stats = [None] * len(inputs)
        for grp, loop in zip(groups, loops):
            counts, swaps = loop.replicas()["counts"].reshape(loop.J, loop.R, 3).sum(axis=1), loop.swaps()
            for pos, k in enumerate(grp):
                st = Stats()
                st.acc_mc_step, st.acc_mc_better_e, st.rej_mc_step = (int(x) for x in counts[pos])
                st.acc_re_step, st.acc_re_better_e, st.rej_re_step = (int(x) for x in swaps[pos])
                st.step = (st.acc_mc_step + st.rej_mc_step) // loop.R
                st.global_step = st.step // sim_options.RE_attempt
                stats[k] = st
        info["simulation_data"], info["stats"] = sim_data, stats
    for loop in loops:
        loop.close()
    return results, info

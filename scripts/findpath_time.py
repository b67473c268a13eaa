"""wall time of bf_findpath (direct refolding paths) per call:  python scripts/findpath_time.py [--rounds 7] [--out FILE]

Workloads (random sequences, seed 1; s1 the MFE structure):
  - 4096 x 100 nt, s2 one Boltzmann sample (engine.sample, seed 1), W = 16;
  - 64 x 400 nt, s2 one Boltzmann sample, W = 64;
  - 1 x 1000 nt, W = 128, s2 the MFE structure less 60 of its pairs plus up to 30 random compatible pairs (bf_sample does not cover
    1000 nt).
Each call is timed at the C-ABI into preallocated host buffers (parsing, copies in and out included, moves and energies returned) and
ends in a device synchronise; every workload is warmed up once and the median over rounds is reported.  Move evaluations are given as
an upper bound counted from the shapes, sum over instances and runs of w k (k + 1) / 2 (every level full and every move of every
kept state valid), per second of call time.  In a separate profiled run (torch.profiler, CUDA activities) the device time of
bf_k_findpath in one call.  For context only, the single-thread time of the plain-C beam of tests/findpath_ref.c (the CPU reference of
the tests, a full orc_eval per candidate structure) on the first instances of the first workload, scaled to that workload; the
reference is not run on the longer workloads.  One JSON line per workload, the card's name and power limit first."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from desirna_b200 import engine


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, limit = (x.strip() for x in q.stdout.strip().split(","))
    return {"card": name, "power_limit": limit}


def widths(W):
    out, w = [], 1
    while w < W:
        out.append(w)
        w *= 2
    return out + [W]


def device_ms(run):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    tot = 0.0
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and ("bf_k_findpath(" in ev.name or "bf_k_findpathE" in ev.name):
            tot += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return tot / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    from conftest import PAR1999
    from findpath_ref import FindpathOracle, pairs_of, perturb
    ref = FindpathOracle(PAR1999)
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    for n_inst, L, W, n_ref in ((4096, 100, 16, 8), (64, 400, 64, 0), (1, 1000, 128, 0)):
        seqs = ["".join("ACGU"[x] for x in rng.integers(0, 4, L)) for _ in range(n_inst)]
        s1 = engine.score_batch(seqs, want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"]
        s2 = [x[0] for x in engine.sample(seqs, 1, seed=1)] if L <= 400 else [perturb(rng, x, 60, 30) for x in s1]
        buf, lens, _ = engine.pack(seqs)
        S = buf.shape[1]
        t1 = engine.pack_targets([[x] for x in s1], S).reshape(n_inst, S)
        t2 = engine.pack_targets([[x] for x in s2], S).reshape(n_inst, S)
        q = engine.bf_findpath_t()
        q.n, q.stride, q.seq, q.len, q.s1, q.s2, q.width = n_inst, S, buf.ctypes.data, lens.ctypes.data, t1.ctypes.data, t2.ctypes.data, W
        sad, k = np.zeros(n_inst, np.int32), np.zeros(n_inst, np.int32)
        mv, pe = np.zeros((n_inst, S, 2), np.int32), np.zeros((n_inst, S + 1), np.int32)
        run = lambda: engine._check(engine.lib().bf_findpath(ctypes.byref(q), sad.ctypes.data, k.ctypes.data, mv.ctypes.data,  # noqa: E731
                                                             pe.ctypes.data))
        run()
        ts = []
        for _ in range(a.rounds):
            t0 = time.perf_counter()
            run()
            ts.append((time.perf_counter() - t0) * 1e3)
        ms = statistics.median(ts)
        ks = [len(set(pairs_of(x)) ^ set(pairs_of(y))) for x, y in zip(s1, s2)]
        assert ks == k.tolist()
        bound = sum(2 * w * kk * (kk + 1) // 2 for kk in ks for w in widths(W))
        kern_ms = device_ms(run)
        rec = {"workload": "%d x %d nt, MFE -> %s, W = %d" % (n_inst, L, "one sample" if L <= 400 else "perturbed MFE", W), "instances": n_inst, "width": W, "rounds": a.rounds,
               "call_ms": round(ms, 3), "moves_k_mean": round(float(np.mean(ks)), 1), "moves_k_max": int(max(ks)),
               "move_evaluations_upper_bound": bound, "move_evaluations_upper_bound_per_s": float("%.4g" % (bound / ms * 1e3)),
               "bf_k_findpath_device_ms": round(kern_ms, 3), "saddle_mean_dcal": round(float(np.mean(sad)), 1)}
        if n_ref:
            t0 = time.perf_counter()
            for r in range(n_ref):
                x = ref.findpath(seqs[r], s1[r], s2[r], W)
                assert x["saddle"] == int(sad[r])
            rec["c_reference_host_1thread_ms_scaled"] = round((time.perf_counter() - t0) * 1e3 * n_inst / n_ref, 1)
            rec["c_reference_timed_instances"] = n_ref
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

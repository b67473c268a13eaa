"""wall time of bf_kinfold (folding kinetics) per call:  python scripts/kinfold_time.py [--rounds 5] [--t-max 10] [--out FILE]

Workloads (random sequences, seed 1):
  - 1 x 100 nt x 10^4 trajectories, open chain -> MFE structure (stop), Kawasaki;
  - 64 x 150 nt x 1000 trajectories from the open chain, Metropolis, 8 snapshots evenly spaced up to t_max;
  - steepest descent from 10^4 Boltzmann samples (engine.sample, seed 1) of one 400-nt sequence.
t_max (the two stochastic workloads) is a flag: the trajectories of 100-150 nt take thousands of moves per time unit.  Each call is
timed at the C-ABI into preallocated host buffers (parsing, copies in and out included, all outputs returned) and ends in a device
synchronise; every workload is warmed up once and the median over rounds is reported, with the moves made per second of call time.
In a separate profiled run (torch.profiler, CUDA activities) the device time of bf_k_kinfold in one call.  For context only, the
single-thread time per move of the plain-C reference of tests/kinfold_ref.c (the CPU reference of the tests, a full orc_eval per
neighbour), measured on the first moves of a few trajectories of the workload and scaled to the workload's moves; it is a test
reference, not a tuned Kinfold.  One JSON line per workload, the card's name and power limit first."""
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


def device_ms(run):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    tot = 0.0
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and ("bf_k_kinfold(" in ev.name or "bf_k_kinfoldE" in ev.name):
            tot += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return tot / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--t-max", type=float, default=10.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    from conftest import PAR1999
    from kinfold_ref import KinfoldOracle
    ref = KinfoldOracle(PAR1999)
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    s100 = "".join("ACGU"[x] for x in rng.integers(0, 4, 100))
    s150 = ["".join("ACGU"[x] for x in rng.integers(0, 4, 150)) for _ in range(64)]
    s400 = "".join("ACGU"[x] for x in rng.integers(0, 4, 400))
    mfe100 = engine.score_batch([s100], want=engine.WANT_MFE | engine.WANT_SS)["mfe_ss"][0]
    samples = engine.sample([s400], 10000, seed=1)[0]
    ts8 = [a.t_max * (s + 1) / 8 for s in range(8)]
    work = [
        ("1 x 100 nt x 10^4 trajectories, open chain -> MFE, Kawasaki, t_max %g" % a.t_max, [s100], None, [mfe100], 10000, 0, a.t_max, []),
        ("64 x 150 nt x 1000 trajectories, open chain, Metropolis, t_max %g, 8 snapshots" % a.t_max, s150, None, None, 1000, 1, a.t_max, ts8),
        ("descent from 10^4 Boltzmann samples of one 400-nt sequence", [s400] * 10000, samples, None, 1, 2, 1.0, []),
    ]
    for name, seqs, start, stop, T, rule, t_max, ts in work:
        n = len(seqs)
        buf, lens, _ = engine.pack(seqs)
        S = buf.shape[1]
        q = engine.bf_kinfold_t()
        q.n, q.stride, q.seq, q.len, q.n_traj, q.rule, q.t_max, q.seed, q.max_steps = n, S, buf.ctypes.data, lens.ctypes.data, T, rule, \
            t_max, 1, 10**6
        keep = []
        for field, dbs in (("start", start), ("stop", stop)):
            if dbs is not None:
                tb = engine.pack_targets([[x] for x in (dbs if len(dbs) == n else dbs * n)], S).reshape(n, S)
                keep.append(tb)
                setattr(q, field, tb.ctypes.data)
        tsa = np.asarray(ts, np.float64)
        q.n_snap, q.t_snap = tsa.size, tsa.ctypes.data if tsa.size else None
        U = n * T
        status, t_end, steps, e_end = np.zeros(U, np.int32), np.zeros(U), np.zeros(U, np.int64), np.zeros(U, np.int32)
        ss_end = np.zeros((U, S + 1), np.uint8)
        e_snap, ss_snap = np.zeros((U, max(1, tsa.size)), np.int32), np.zeros((U, max(1, tsa.size), S + 1), np.uint8)
        run = lambda: engine._check(engine.lib().bf_kinfold(ctypes.byref(q), status.ctypes.data, t_end.ctypes.data, steps.ctypes.data,  # noqa: E731
                                                             e_end.ctypes.data, ss_end.ctypes.data, e_snap.ctypes.data, ss_snap.ctypes.data))
        run()
        tm = []
        for _ in range(a.rounds):
            t0 = time.perf_counter()
            run()
            tm.append((time.perf_counter() - t0) * 1e3)
        ms = statistics.median(tm)
        moves = int(steps.sum())
        kern_ms = device_ms(run)
        rec = {"workload": name, "trajectories": U, "rounds": a.rounds, "call_ms": round(ms, 2), "bf_k_kinfold_device_ms": round(kern_ms, 2),
               "moves": moves, "moves_per_s": float("%.4g" % (moves / ms * 1e3)), "moves_per_trajectory_mean": round(moves / U, 1),
               "status_counts": np.bincount(status, minlength=3).tolist()}
        # the reference: the first moves of a few trajectories, per move
        r_moves = 0
        t0 = time.perf_counter()
        for x in range(3):
            r, k = x // T, x % T
            w = ref.traj(seqs[r], start[r] if start else None, stop[r] if stop else None, ("kawasaki", "metropolis", "descent")[rule], t_max,
                         1, r, k, 20 if rule != 2 else 3, ts)
            r_moves += w["steps"]
        ref_ms = (time.perf_counter() - t0) * 1e3
        if r_moves:
            rec["c_reference_host_1thread_ms_per_move"] = round(ref_ms / r_moves, 3)
            rec["c_reference_host_1thread_s_scaled"] = round(ref_ms / r_moves * moves / 1e3, 1)
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

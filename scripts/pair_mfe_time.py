"""wall time of bf_pair_mfe (MFE fill + minimum-free-energy outside pass + copy of E_pair) against the MFE fill and backtrack alone
(bf_score_batch, WANT_MFE | WANT_SS) on the same batch:  python scripts/pair_mfe_time.py [--rounds 7] [--out FILE]

Shapes: 4096 x 100 nt, 64 x 100 nt, 16 x 400 nt, 1 x 1000 nt (random sequences, seed 1).  Both calls are timed at the C-ABI into
preallocated host buffers and end in a device synchronise; they alternate, each shape warmed up once.  bf_pair_mfe copies B x
stride x stride int32 back to pageable host memory (e_pair_MB), which is part of its time.  After the timed rounds, one call per
shape runs under torch.profiler (CUDA activities) for the device time of bf_k_mfe_out alone.  Reported: medians over rounds, one
JSON line per shape, the card's name and power limit first."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desirna_b200 import engine

SHAPES = ((4096, 100), (64, 100), (16, 400), (1, 1000))


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, limit = (x.strip() for x in q.stdout.strip().split(","))
    return {"card": name, "power_limit": limit}


def timed(f):
    t0 = time.perf_counter()
    f()
    return (time.perf_counter() - t0) * 1e3


def kernel_ms(f, name):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if name in e.key) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    calls = []
    for B, L in SHAPES:
        seqs = ["".join("ACGU"[x] for x in rng.integers(0, 4, L)) for _ in range(B)]
        buf, lens, _ = engine.pack(seqs)
        b = engine.bf_batch_t()
        b.B, b.stride, b.seq, b.len = B, L, buf.ctypes.data, lens.ctypes.data
        ep = np.zeros((B, L, L), np.int32)
        r = engine.bf_result_t()
        mfe, ss = np.zeros(B, np.int32), np.zeros((B, L + 1), np.uint8)
        r.mfe_dcal, r.mfe_ss = mfe.ctypes.data, ss.ctypes.data
        bm = engine.bf_batch_t()
        bm.B, bm.stride, bm.seq, bm.len, bm.want = B, L, buf.ctypes.data, lens.ctypes.data, engine.WANT_MFE | engine.WANT_SS
        run_p = lambda b=b, ep=ep: engine._check(engine.lib().bf_pair_mfe(ctypes.byref(b), ep.ctypes.data))  # noqa: E731
        run_m = lambda bm=bm, r=r: engine._check(engine.lib().bf_score_batch(ctypes.byref(bm), ctypes.byref(r)))  # noqa: E731
        run_p(); run_m()
        tp, tm = [], []
        for _ in range(a.rounds):
            tp.append(timed(run_p))
            tm.append(timed(run_m))
        ms_p, ms_m = statistics.median(tp), statistics.median(tm)
        calls.append((B, L, run_p, ms_p, ms_m, ep.nbytes, (buf, lens)))   # the batch's arrays stay alive for the profiled call
    for B, L, run_p, ms_p, ms_m, nbytes, _ in calls:
        rec = {"B": B, "L": L, "rounds": a.rounds, "pair_mfe_call_ms": round(ms_p, 3), "mfe_bt_call_ms": round(ms_m, 3),
               "e_pair_MB": round(nbytes / 1e6, 1), "mfe_out_kernel_ms": round(kernel_ms(run_p, "bf_k_mfe_out"), 3)}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

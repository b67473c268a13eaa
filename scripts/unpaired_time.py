"""wall time of bf_unpaired and bf_plfold (accessibility) per call:  python scripts/unpaired_time.py [--rounds 7] [--out FILE]

Workloads (random sequences, seed 1): bf_unpaired at 4096 x 100 nt, 16 x 400 nt and 1 x 668 nt (the longest stride the PF fill
path covers; 1000 nt is unavailable, as for WANT_BPP) with max_u = 31, each beside a
WANT_BPP call alone on the same batch (MFE fill, PF fill and outside pass: what bf_unpaired runs before its own kernel); bf_plfold
on one 10 kb transcript at W = 70 and W = 200 and on 100 transcripts of 2 kb at W = 70, u = 31.  Each call is timed at the host
(engine entry points into host buffers, copies included, ending in a device synchronise), warmed up once, median over rounds.  One
extra run of every bf_unpaired shape under torch.profiler (CUDA activities) gives the device time of bf_k_unpaired and of the
outside pass alone.  One JSON line per workload, the card's name and power limit first."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from desirna_b200 import engine


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, limit = (x.strip() for x in q.stdout.strip().split(","))
    return {"card": name, "power_limit": limit}


def rseqs(rng, n, L):
    return ["".join("ACGU"[x] for x in rng.integers(0, 4, L)) for _ in range(n)]


def median_ms(f, rounds):
    f()
    ts = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def kernel_ms(f, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    ev = prof.key_averages()
    return {n: round(sum(e.device_time_total for e in ev if n in e.key) / 1e3, 3) for n in names}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    for B, L in ((4096, 100), (16, 400), (1, 668)):
        seqs = rseqs(rng, B, L)
        up = lambda: engine.unpaired(seqs, 31)  # noqa: E731
        bpp = lambda: engine.score_batch(seqs, want=engine.WANT_BPP)  # noqa: E731
        rec = {"workload": f"bf_unpaired {B} x {L} nt, max_u 31", "rounds": a.rounds, "call_ms": round(median_ms(up, a.rounds), 3),
               "want_bpp_call_ms": round(median_ms(bpp, a.rounds), 3)}
        k = kernel_ms(up, ["bf_k_unpaired", "bf_k_pf_out"])
        rec["unpaired_kernel_ms"], rec["outside_kernel_ms"] = k["bf_k_unpaired"], k["bf_k_pf_out"]
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    for name, seqs, W in (("bf_plfold 1 x 10 kb, W 70, u 31", rseqs(rng, 1, 10000), 70),
                          ("bf_plfold 1 x 10 kb, W 200, u 31", rseqs(rng, 1, 10000), 200),
                          ("bf_plfold 100 x 2 kb, W 70, u 31", rseqs(rng, 100, 2000), 70)):
        windows = sum(len(s) - W + 1 for s in seqs)
        ms = median_ms(lambda: engine.plfold(seqs, W, 31), a.rounds)
        rec = {"workload": name, "windows": windows, "rounds": a.rounds, "call_ms": round(ms, 3), "windows_per_s": round(windows / ms * 1e3, 1)}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

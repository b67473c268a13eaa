"""wall time of stochastic backtracking (bf_sample) against the partition function alone (bf_score_batch, WANT_PF) on the same batch:
python scripts/sample_time.py [--rounds 5] [--out FILE]

Shapes: 1 x 100 nt x 10^4 samples, 64 x 100 nt x 1000 samples, 16 x 400 nt x 1000 samples (random sequences, seed 1).  A bf_sample
call runs the MFE fill (for the scale), the PF fill with its qm / qm1 tables kept, the exterior prefix and the walk, and copies the
structures back (timed at the C-ABI, without Python's string decoding); the two calls alternate, each shape warmed up once, and every call ends in a device synchronise.  Reported: the
median over rounds, ms per call and us per sample of the sampling call beyond the PF call, and samples per second.  One JSON line per
shape, the card's name and power limit first."""
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

SHAPES = ((1, 100, 10000), (64, 100, 1000), (16, 400, 1000))


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, limit = (x.strip() for x in q.stdout.strip().split(","))
    return {"card": name, "power_limit": limit}


def timed(f):
    t0 = time.perf_counter()
    f()
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    for B, L, ns in SHAPES:
        seqs = ["".join("ACGU"[x] for x in rng.integers(0, 4, L)) for _ in range(B)]
        buf, lens, _ = engine.pack(seqs)
        b = engine.bf_batch_t()
        b.B, b.stride, b.seq, b.len = B, L, buf.ctypes.data, lens.ctypes.data
        out = np.zeros((B, ns, L + 1), np.uint8)
        run_s = lambda: engine._check(engine.lib().bf_sample(ctypes.byref(b), ns, 7, out.ctypes.data))  # noqa: E731
        run_pf = lambda: engine.score_batch(seqs, want=engine.WANT_PF)  # noqa: E731
        run_s(); run_pf()
        ts, tp = [], []
        for _ in range(a.rounds):
            ts.append(timed(run_s))
            tp.append(timed(run_pf))
        ms_s, ms_pf = statistics.median(ts), statistics.median(tp)
        rec = {"B": B, "L": L, "samples_per_seq": ns, "rounds": a.rounds, "sample_call_ms": round(ms_s, 3), "pf_call_ms": round(ms_pf, 3),
               "beyond_pf_us_per_sample": round((ms_s - ms_pf) * 1e3 / (B * ns), 4), "samples_per_s": round(B * ns / (ms_s / 1e3))}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

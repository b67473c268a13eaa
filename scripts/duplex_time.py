"""wall time of bf_duplex (RNA-RNA hybridization) per call:  python scripts/duplex_time.py [--rounds 7] [--out FILE]

Workloads (random strands, seed 1): 4096 pairs of 21 x 21 nt with structures; the 256 x 256 grid of 50-nt strands, energies only;
64 pairs of 21 x 2000 nt with structures; 1 pair of 100 x 100 nt with structures.  Each call is timed at the C-ABI into
preallocated host buffers (copies in and out included) and ends in a device synchronise; every workload is warmed up once, the
median over rounds is reported with pairs/s.  For context, the single-thread time of the plain-C recurrence of tests/duplex_ref.c
(the CPU reference of the tests, not ViennaRNA) on the same inputs, measured on the host of the same run; for the grid it is
timed on its first 4096 entries and scaled to the whole grid.  One JSON line per workload, the card's name and power limit first."""
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


def rseqs(rng, n, L):
    return ["".join("ACGU"[x] for x in rng.integers(0, 4, L)) for _ in range(n)]


def query(A, B, pairs):
    """a bf_duplex_t over packed strands; the arrays it points to are returned with it and must stay alive"""
    q = engine.bf_duplex_t()
    keep = []
    for st, seqs in ((q.a, A), (q.b, B)):
        buf, lens, _ = engine.pack(seqs)
        st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, lens.ctypes.data
        keep += [buf, lens]
    if pairs is not None:
        pr = np.ascontiguousarray(np.asarray(pairs, np.int32))
        q.pairs, q.n_pairs = pr.ctypes.data, len(pr)
        keep.append(pr)
    return q, keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    from conftest import PAR1999
    from duplex_ref import DuplexOracle
    ref = DuplexOracle(PAR1999)
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    work = []
    A, B = rseqs(rng, 4096, 21), rseqs(rng, 4096, 21)
    work.append(("4096 pairs 21 x 21", A, B, [(k, k) for k in range(4096)], True))
    A, B = rseqs(rng, 256, 50), rseqs(rng, 256, 50)
    work.append(("grid 256 x 256 at 50 nt", A, B, None, False))
    A, B = rseqs(rng, 64, 21), rseqs(rng, 64, 2000)
    work.append(("64 pairs 21 x 2000", A, B, [(k, k) for k in range(64)], True))
    A, B = rseqs(rng, 1, 100), rseqs(rng, 1, 100)
    work.append(("1 pair 100 x 100", A, B, [(0, 0)], True))
    for name, A, B, pairs, want_ss in work:
        q, keep = query(A, B, pairs)
        P = len(pairs) if pairs is not None else len(A) * len(B)
        e = np.zeros(P, np.int32)
        ss = np.zeros((P, q.a.stride + q.b.stride + 2), np.uint8) if want_ss else None
        run = lambda: engine._check(engine.lib().bf_duplex(ctypes.byref(q), e.ctypes.data, ss.ctypes.data if want_ss else None))  # noqa: E731
        run()
        ts = []
        for _ in range(a.rounds):
            t0 = time.perf_counter()
            run()
            ts.append((time.perf_counter() - t0) * 1e3)
        ms = statistics.median(ts)
        todo = pairs if pairs is not None else [(x // len(B), x % len(B)) for x in range(P)]
        sub = todo[:4096]
        t0 = time.perf_counter()
        for ia, ib in sub:
            ref.duplex(A[ia], B[ib])
        ref_ms = (time.perf_counter() - t0) * 1e3 * P / len(sub)
        rec = {"workload": name, "pairs": P, "structures": want_ss, "rounds": a.rounds, "call_ms": round(ms, 3),
               "pairs_per_s": round(P / ms * 1e3, 1), "c_reference_host_1thread_ms": round(ref_ms, 1),
               "c_reference_timed_pairs": len(sub)}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

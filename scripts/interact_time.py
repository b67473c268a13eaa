"""wall time of bf_interact (accessibility-aware RNA-RNA interaction) per call:  python scripts/interact_time.py [--rounds 7] [--out FILE]

Workloads (random strands, seed 1):
  - 1000 guides of 21 nt against one 2000-nt target, global accessibility on the guides, RNAplfold window W = 150 on the target,
    max_span 25, energies only (the siRNA / miRNA target-site scan);
  - the 256 x 256 grid of 50-nt strands, global accessibility on both sides, max_span 25, energies only (a crosstalk matrix);
  - 64 pairs of 100 x 100 nt, global accessibility on both sides, max_span 25, with structures.
Each call is timed at the C-ABI into preallocated host buffers (accessibility, copies in and out included) and ends in a device
synchronise; every workload is warmed up once and the median over rounds is reported.  Candidate evaluations are counted from the
shapes alone, as if every start and every window cell paired: for each start (k1, l1) and each cell (di, dj) of its window, the
(u1, u2) with u1 < di, u2 < dj, u1 + u2 <= 30; per second of call time.  In a separate profiled run (torch.profiler, CUDA
activities) the device time of bf_k_interact in one call.  For context only, the single-thread time of the plain-C recurrence of
tests/interact_ref.c (the CPU reference of the tests) on a stated subset of pairs, fed the same opening energies, scaled to the
workload.  One JSON line per workload, the card's name and power limit first."""
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


def query(A, B, pairs, span, acc_a, acc_b):
    """a bf_interact_t over packed strands; the arrays it points to are returned with it and must stay alive"""
    q = engine.bf_interact_t()
    keep = []
    for st, seqs in ((q.a, A), (q.b, B)):
        buf, lens, _ = engine.pack(seqs)
        st.n, st.stride, st.seq, st.len = len(seqs), buf.shape[1], buf.ctypes.data, lens.ctypes.data
        keep += [buf, lens]
    if pairs is not None:
        pr = np.ascontiguousarray(np.asarray(pairs, np.int32))
        q.pairs, q.n_pairs = pr.ctypes.data, len(pr)
        keep.append(pr)
    q.max_span, q.acc_a, q.acc_b = span, acc_a, acc_b
    return q, keep


def candidates(n1, n2, span):
    """candidate (u1, u2) evaluations of one pair of strands if every start and cell paired"""
    u = np.arange(span)
    # cnt[a, b]: (u1, u2) with u1 < a, u2 < b, u1 + u2 <= 30, for a cell at (di, dj) = (a, b)
    ok = ((u[:, None] + u[None, :]) <= 30).astype(np.int64)
    cnt = np.zeros((span + 1, span + 1), np.int64)
    cnt[1:, 1:] = ok.cumsum(0).cumsum(1)
    win = cnt[:span, :span].cumsum(0).cumsum(1)   # win[wa-1, wb-1]: sum over a window of wa x wb cells
    wa = np.minimum(span, n1 - np.arange(1, n1 + 1) + 1)
    wb = np.minimum(span, np.arange(1, n2 + 1))
    return int(win[wa[:, None] - 1, wb[None, :] - 1].sum())


def device_ms(run):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    tot = 0.0
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and ("bf_k_interact(" in ev.name or "bf_k_interactE" in ev.name):
            tot += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return tot / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    from conftest import PAR1999
    from interact_ref import InteractOracle, ed_rows
    ref = InteractOracle(PAR1999)
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(1)
    work = []
    A, B = rseqs(rng, 1000, 21), rseqs(rng, 1, 2000)
    work.append(("1000 guides 21 nt x 2000-nt target, global / W=150", A, B, [(k, 0) for k in range(1000)], 0, 150, False, 8))
    A, B = rseqs(rng, 256, 50), rseqs(rng, 256, 50)
    work.append(("grid 256 x 256 at 50 nt, global / global", A, B, None, 0, 0, False, 256))
    A, B = rseqs(rng, 64, 100), rseqs(rng, 64, 100)
    work.append(("64 pairs 100 x 100 nt, global / global, structures", A, B, [(k, k) for k in range(64)], 0, 0, True, 8))
    span = 25
    for name, A, B, pairs, acc_a, acc_b, want_ss, n_ref in work:
        q, keep = query(A, B, pairs, span, acc_a, acc_b)
        P = len(pairs) if pairs is not None else len(A) * len(B)
        e = np.zeros(P, np.float64)
        ss = np.zeros((P, q.a.stride + q.b.stride + 2), np.uint8) if want_ss else None
        run = lambda: engine._check(engine.lib().bf_interact(ctypes.byref(q), e.ctypes.data, None, None, None,  # noqa: E731
                                                             ss.ctypes.data if want_ss else None))
        run()
        ts = []
        for _ in range(a.rounds):
            t0 = time.perf_counter()
            run()
            ts.append((time.perf_counter() - t0) * 1e3)
        ms = statistics.median(ts)
        todo = pairs if pairs is not None else [(x // len(B), x % len(B)) for x in range(P)]
        cand = sum(candidates(len(A[ia]), len(B[ib]), span) for ia, ib in todo)
        kern_ms = device_ms(run)
        # the reference on the first n_ref pairs, fed the opening energies from engine.unpaired / engine.plfold
        sub = todo[:n_ref]
        ia_set, ib_set = sorted({x for x, _ in sub}), sorted({y for _, y in sub})

        def eds(seqs, idx, acc):
            S = [seqs[k] for k in idx]
            if acc == 0:
                pu = engine.unpaired(S, min(span, max(map(len, S))))
                rows = [pu[k, :len(s)] for k, s in enumerate(S)]
            else:
                rows = [p for _, p in engine.plfold(S, acc, max_u=span, pairs=False)]
            return {k: ed_rows(np.pad(r, ((0, 0), (0, span - r.shape[1]))), span) for k, r in zip(idx, rows)}
        EA, EB = eds(A, ia_set, acc_a), eds(B, ib_set, acc_b)
        t0 = time.perf_counter()
        for ia, ib in sub:
            ref.interact(A[ia], B[ib], span, EA[ia], EB[ib])
        ref_ms = (time.perf_counter() - t0) * 1e3 * P / len(sub)
        rec = {"workload": name, "pairs": P, "max_span": span, "structures": want_ss, "rounds": a.rounds, "call_ms": round(ms, 3),
               "candidates": cand, "candidates_per_s": float("%.4g" % (cand / ms * 1e3)), "bf_k_interact_device_ms": round(kern_ms, 3),
               "c_reference_host_1thread_ms_scaled": round(ref_ms, 1), "c_reference_timed_pairs": len(sub)}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

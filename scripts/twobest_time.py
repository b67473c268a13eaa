"""ms per bf_second_best call (the 2-best DP of negative design, csrc/bf_twobest.cu): host clock around the synchronising call,
after warm-up, for single strands and two-strand ('A&B') batches: python scripts/twobest_time.py"""
import os, sys, time, random
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desirna_b200 import engine

engine.ensure_ready()
rng = random.Random(5)


def seq(n):
    return "".join(rng.choice("ACGU") for _ in range(n))


shapes = (("36nt", lambda: seq(36)), ("100nt", lambda: seq(100)), ("17&18", lambda: seq(17) + "&" + seq(18)), ("50&50", lambda: seq(50) + "&" + seq(50)))
for B in (1, 64):
    for name, make in shapes:
        batch = [make() for _ in range(B)]
        for _ in range(3):
            engine.second_best(batch)   # warm-up: module load, workspace allocation
        reps = 20
        t0 = time.perf_counter()
        for _ in range(reps):
            engine.second_best(batch)   # returns after cudaStreamSynchronize
        dt = (time.perf_counter() - t0) / reps
        print(f"B={B:3d} {name:6s}: {dt * 1e3:.4f} ms per bf_second_best call", flush=True)

"""kernel times of two-strand batches (generic kernels): python scripts/two_time.py"""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desirna_b200 import engine
engine.init(); engine.params_builtin(1999)
want = engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF | engine.WANT_EVAL
for (a, b_), B in (((17, 18), 64), ((17, 18), 10), ((50, 50), 64), ((100, 100), 64), ((50, 50), 4096)):
    rng = np.random.default_rng(a + B)
    seqs = ["".join("ACGU"[x] for x in rng.integers(0, 4, a)) + "&" + "".join("ACGU"[x] for x in rng.integers(0, 4, b_)) for _ in range(B)]
    tg = [["." * (a + b_)]] * B
    for _ in range(2): engine.score_batch(seqs, tg, want=want)
    km = np.zeros(3); t0 = time.perf_counter()
    for _ in range(3):
        engine.score_batch(seqs, tg, want=want); km += np.array(engine.last_kernel_ms())
    print(f"{a}&{b_} B={B}: call {1e3 * (time.perf_counter() - t0) / 3:.3f} ms mfe {km[0] / 3:.3f} pf {km[1] / 3:.3f} eval {km[2] / 3:.3f}", flush=True)

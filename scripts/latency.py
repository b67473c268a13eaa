#!/usr/bin/env python
"""Small-batch latency of the fold pipeline (what one Monte-Carlo sub-step of a replica-exchange run costs):
ms per bf_score_batch call (MFE + backtrack + PF + eval) for B sequences of length L, kernel times from CUDA events."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from desirna_b200 import engine  # noqa: E402


def main():
    engine.init()
    engine.params_builtin(1999)
    want = engine.WANT_MFE | engine.WANT_SS | engine.WANT_PF | engine.WANT_EVAL
    out = {}
    for L in (36, 100, 200, 400):
        for B in (10, 64, 128, 296):
            rng = np.random.default_rng(L * 1000 + B)
            seqs = ["".join("ACGU"[x] for x in row) for row in rng.integers(0, 4, (B, L))]
            tg = [["." * L]] * B
            for _ in range(3):
                engine.score_batch(seqs, tg, want=want)
            t0 = time.perf_counter()
            n = 5
            km = np.zeros(3)
            for _ in range(n):
                engine.score_batch(seqs, tg, want=want)
                km += np.array(engine.last_kernel_ms())
            ms = (time.perf_counter() - t0) / n * 1e3
            out[f"L{L}_B{B}"] = {"call_ms": round(ms, 3), "mfe_ms": round(km[0] / n, 3), "pf_ms": round(km[1] / n, 3), "eval_ms": round(km[2] / n, 3)}
    print(json.dumps({"latency": out}))


if __name__ == "__main__":
    main()

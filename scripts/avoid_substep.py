"""sub-step time of avoid designs (oligo_state "avoid", -o on) against the same loops without the self-dimer term:
python scripts/avoid_substep.py [--rounds 3] [--out FILE]

Loops with oligo_state "none" and "avoid" run alternately (rounds x both modes) at 36 nt x 10 replicas and 104 nt x 64 replicas.
Each loop is warmed up by one global step, then timed over two global steps of 100 sub-steps ending in a device synchronise.
The device time of the self-dimer partition function alone (the R sequences seq&seq of the loop's final replicas, one
bf_score_batch call) is read from the kernel's CUDA events.  One JSON line per measurement, the card's name and power limit first."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desirna_b200 import design, engine
from desirna_b200.utils import stats_inputs_outputs as sio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, limit = (x.strip() for x in q.stdout.strip().split(","))
    return {"card": name, "power_limit": limit}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.ensure_ready()
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    rows = [json.loads(l) for l in open(os.path.join(ROOT, "tests", "golden", "E1.jsonl"))]
    one = min(rows, key=lambda r: (abs(len(r["target"]) - 104), r["file"]))
    sizes = (("36nt", sio.make_input("Standard_design", "((((((.((((((((....))))).)).).))))))"), 10), ("104nt", sio.make_input(one["file"], one["target"]), 64))
    for rnd in range(a.rounds):
        for name, inp, R in sizes:
            for mode in ("none", "avoid"):
                random.seed(0)
                loop = design.DesignLoop([inp], design.DesignOptions(replicas=R, RE_attempt=100, oligo_state=mode), seed=1)
                loop.run(1); loop.sync()
                t0 = time.perf_counter()
                loop.run(2); loop.sync()
                dt = time.perf_counter() - t0
                rec = {"round": rnd, "size": name, "n": len(inp.sec_struct), "replicas": R, "oligo_state": mode, "ms_per_substep": round(dt / 200 * 1e3, 4)}
                if mode == "avoid":
                    dimers = [s + "&" + s for s in loop.replicas()["sequence"]]
                    ms = []
                    for _ in range(5):
                        engine.score_batch(dimers, want=engine.WANT_PF)
                        ms.append(engine.last_kernel_ms()[1])
                    rec["self_dimer_pf_ms"] = round(min(ms[1:]), 4)
                loop.close()
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

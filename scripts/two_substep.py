"""sub-step time of the reference's two-strand example in the device design loop, without and with negative design (-nd on):
python scripts/two_substep.py"""
import os, sys, time, random
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desirna_b200 import design
from desirna_b200.utils import stats_inputs_outputs as sio
for subopt in ("off", "on"):
    for R in (64, 10):
        random.seed(0)
        o = design.DesignOptions(replicas=R, RE_attempt=100, oligo_state="heterodimer", subopt=subopt)
        loop = design.DesignLoop([sio.make_input("RNA_RNA_complex", "(((.(((((....))..&(((....)))..))))))", "NNNNNNNNNNNNNNNNN&NNNNNNNNNNNNNNNNNN")], o, seed=3)
        loop.run(1); loop.sync()
        t0 = time.perf_counter()
        loop.run(2); loop.sync()
        dt = time.perf_counter() - t0
        loop.close()
        print(f"heterodimer 17&18 R={R} subopt={subopt} env={ {k: v for k, v in os.environ.items() if k.startswith('BF_')} }: {dt / 200 * 1e3:.4f} ms per sub-step", flush=True)

#!/usr/bin/env python3
"""bench.py -- MFE+PF folds/sec on the synthetic batched fold sweep (BASELINE.json configs[1]).

One "step" = one pass of the hot path (MFE fill + backtrack, partition function, eval of the
target) over a batch of B=4096 random sequences of length L (default L=100; the other lengths
of the sweep are timed in the same run and reported under "by_length").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--L 100] [--B 4096] [--dump-outputs DIR]
  python bench.py --impl reference ...      # CPU arm: the oracle port on all host threads

--dump-outputs DIR writes what the last timed step returned to its caller (mfe_dcal, mfe_ss, pf, eval_dcal of
score_batch_device) as DIR/<name>.npy, so that two builds can be compared output for output on identical inputs.

Our arm prints ONE JSON line with the driver's contract keys plus `roofline`, `cpu_baseline`,
`e2e`, `by_length`, `clocks`, `gpu_launches`.  Timing: CUDA events on the launch stream, >= 3
warm-up steps, L2 flushed between timed steps, max over ranks.  ViennaRNA itself is not
installable here (no wheel, no network), so the CPU arm is the repo's C oracle
(cpu_baseline.kind = "port"), threaded over the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: no __pycache__ next to the sources

SWEEP = (50, 100, 200, 400)
P_PAIR = 6.0 / 16.0
DUMP_BYTES = (64 << 20) - (1 << 16)   # --dump-outputs: at most 64 MiB in all, .npy headers included


# ---------------------------------------------------------------- algorithmic work (SURVEY.md 8d / DESIGN.md)
def relaxations(N):
    """Closed-form DP relaxation counts per fold of a uniform random sequence of length N
    (TURN=3, MAXLOOP=30, pair probability 6/16).  Returns (R_MFE, R_PFin)."""
    T = lambda m: (m + 1) * (m + 2) // 2 if m >= 0 else 0
    r_int = P_PAIR * sum((N - d) * T(min(30, d - 6)) for d in range(4, N))
    r_mlc = P_PAIR * sum((N - d) * max(0, d - 9) for d in range(4, N))
    r_fml = sum((N - d) * max(0, d - 7) for d in range(4, N))
    r_f5 = sum(max(0, j - 4) for j in range(1, N + 1))
    r_mfe = r_int + r_mlc + r_fml + r_f5
    r_pf = r_int + P_PAIR * sum((N - d) * (d - 1) for d in range(4, N)) + sum((N - d) * (d + 1) for d in range(4, N)) + r_f5
    return r_mfe, r_pf


def synth(L, B, rank=0):
    rng = np.random.default_rng(20240000 + L + 1000003 * rank)
    return rng.integers(0, 4, (B, L))


def to_strings(codes):
    lut = np.frombuffer(b"ACGU", np.uint8)
    return [bytes(lut[row]).decode() for row in codes]


def dump_outputs(path, out):
    """Write the arrays of `out` (name -> array, one row per sequence) as path/<name>.npy in float64, the structure bytes
    in float32.  When the batch exceeds DUMP_BYTES a fixed-seed sample of rows is written, with its indices as row.npy."""
    out = {k: a.astype(np.float32 if a.dtype == np.uint8 else np.float64) for k, a in out.items()}
    B = len(next(iter(out.values())))
    row_bytes = sum(a[0].nbytes for a in out.values()) + 8
    if B * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // row_bytes, replace=False))
        out = {k: a[rows] for k, a in out.items()}
        out["row"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ---------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------- reference arm (CPU oracle port)
def vienna_available():
    """BASELINE.md comparator A: DesiRNA's own ViennaRNA path, if the GPU host happens to have the module"""
    try:
        import RNA  # noqa: F401
        return True
    except Exception:
        return False


def _vienna_one(seq):
    import RNA
    md = RNA.md()
    md.compute_bpp = 0
    fc = RNA.fold_compound(seq, md)
    fc.pf()
    ss, _ = fc.mfe()
    return fc.eval_structure(ss)


def cpu_sample(L, budget_s, threads, fast=True):
    """Time the CPU arm (MFE + backtrack, PF inside, eval) on a bounded sample of the L-workload.
    fast: the tuned port (orc_mfe_fast / orc_pf_fast, bit-identical to the oracle, ~5x faster); else the clarity-first oracle.
    With ViennaRNA importable the sample runs get_mfe_e_ss's call sequence over a process pool instead (kind "reference")."""
    from oracle.pyoracle import Oracle   # loads the library build() made; compiles nothing into the tree
    O = Oracle(os.path.join(ROOT, "desirna_b200", "params", "turner1999_37C.par"))
    per_fold = (2.6e-8 * L ** 3 + 1.3e-6 * L ** 2) / (5.0 if fast else 1.0)  # rough single-thread seconds, only used to size the sample
    n = int(max(threads, min(65536, budget_s * threads / per_fold)))
    n = max(threads, (n // threads) * threads)
    seqs = to_strings(synth(L, n, rank=7))
    if fast and vienna_available():
        import multiprocessing as mp
        with mp.Pool(threads) as pool:
            pool.map(_vienna_one, seqs[:threads])
            t0 = time.perf_counter()
            pool.map(_vienna_one, seqs, chunksize=max(1, n // (4 * threads)))
            dt = time.perf_counter() - t0
        return n / dt, n, dt
    t0 = time.perf_counter()
    O.fold_batch(seqs, nthreads=threads, fast=fast)
    dt = time.perf_counter() - t0
    return n / dt, n, dt


def cpu_kind():
    return "reference" if vienna_available() else "port"


def cpu_desc(threads):
    if vienna_available():
        return f"ViennaRNA (import RNA): fc.pf(), fc.mfe(), fc.eval_structure() per sequence, multiprocessing.Pool({threads})"
    phys = physical_cores()
    return (f"oracle/orc_fold.c tuned arm (orc_mfe_fast / orc_pf_fast: bit-identical to the oracle, decomposed interior loops, AVX2) on {threads} threads"
            f" ({phys} physical cores); ViennaRNA 2.6.4 is not installable offline")


def physical_cores():
    try:
        cores = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    cores.add((phys, core))
                phys = core = None
        return len(cores) or None
    except Exception:
        return None


def run_reference(args):
    """The CPU arm on all host threads: the tuned port (or ViennaRNA when importable), each step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    L = args.L
    vals = []
    budget = max(1.0, min(20.0, 60.0 / max(1, args.steps)))
    for _ in range(min(args.warmup, 1)):
        cpu_sample(L, 0.5, threads)
    n_used = 0
    t_total = 0.0
    for _ in range(args.steps):
        v, n, dt = cpu_sample(L, budget, threads)
        vals.append(v); n_used = n; t_total += dt
    value = statistics.mean(vals)
    by = {}
    if not args.no_sweep:
        for l in SWEEP:
            by[str(l)] = value if l == L else cpu_sample(l, 8.0, threads)[0]
    # the clarity-first oracle on the same workload, and the cost of one counted relaxation on one core
    slow = cpu_sample(L, 4.0, threads, fast=False)[0]
    r_mfe, r_pf = relaxations(L)
    ns_per_relax = 1e9 * threads / value / (r_mfe + r_pf)
    line = {
        "impl": "reference", "metric": "MFE+PF folds/sec", "value": value, "unit": "folds/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
        "config": {"workload": f"synthetic batched fold sweep: random sequences x L={L}, MFE+backtrack+PF+eval, Turner 1999", "L": L,
                   "sample_per_step": n_used, "params": "turner1999"},
        "cpu_baseline": {"value": value, "unit": "folds/s", "cores": threads, "physical_cores": physical_cores(), "kind": cpu_kind(),
                         "sample": f"{n_used} random sequences of L={L} per step; " + cpu_desc(threads),
                         "oracle_port_value": slow, "ns_per_relaxation_per_thread": ns_per_relax,
                         "relaxations_per_fold": r_mfe + r_pf},
        "e2e": {"value": value, "unit": "folds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "by_length": by,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------- our arm
def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "hbm_src": "fallback", "int32_tops": 18.6, "fp64_tflops": 37.0, "smem_tbs": 37.2, "chip_src": "nominal"}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            peaks["hbm_gbs"] = float(json.load(open(p))["hbm_gbs"]); peaks["hbm_src"] = "measured"
        except Exception:
            pass
    return peaks


def run_ours(args):
    import torch
    import torch.distributed as dist
    from desirna_b200 import engine as eng

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng.init(local)
    eng.params_builtin(1999)
    dev = torch.device("cuda", local)
    tstream = torch.cuda.Stream(device=dev)  # timed work and its CUDA events share this stream
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    WANT = eng.WANT_MFE | eng.WANT_SS | eng.WANT_PF | eng.WANT_EVAL
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lut = torch.tensor(list(b"ACGU"), dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make(L, B):
        codes = synth(L, B, rank)
        seq = lut[torch.from_numpy(codes).to(dev)].contiguous()
        lens = torch.full((B,), L, dtype=torch.int32, device=dev)
        bufs = dict(seq=seq, lens=lens, mfe=torch.zeros(B, dtype=torch.int32, device=dev), ss=torch.zeros((B, L + 1), dtype=torch.uint8, device=dev),
                    pf=torch.zeros((B, 5), dtype=torch.float64, device=dev), ev=torch.zeros((B, 1), dtype=torch.int32, device=dev),
                    targets=torch.full((B, 1, L), ord("."), dtype=torch.uint8, device=dev))
        return codes, bufs

    def step(b):
        eng.score_batch_device(b["seq"], b["lens"], WANT, targets=b["targets"], mfe=b["mfe"], ss=b["ss"], pf=b["pf"], ev=b["ev"], stream=stream)

    def measure(L, B, steps, warmup):
        codes, b = make(L, B)
        # pass 0: the MFE structure of every sequence becomes its target (free invariant Ed == MFE)
        step(b)
        torch.cuda.synchronize()
        b["targets"][:, 0, :] = b["ss"][:, :L]
        for _ in range(warmup):
            step(b)
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kms = []
        for k in range(steps):
            flush.fill_(k & 0xff)  # L2 flush between timed steps
            ev[k][0].record()
            step(b)
            ev[k][1].record()
            ev[k][1].synchronize()
            kms.append(eng.last_kernel_ms())
        barrier()
        ms = [a.elapsed_time(c) for a, c in ev]
        total = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        ok = bool((b["ev"][:, 0] == b["mfe"]).all().item()) and bool((b["pf"][:, 4] <= b["mfe"].double() / 100.0 + 1e-9).all().item())
        kavg = [statistics.mean(x[i] for x in kms) for i in range(3)]
        return dict(total_ms=float(total.item()), ms=ms, kernel_ms=kavg, ok=ok, codes=codes, bufs=b)

    L, B = args.L, args.B
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches()
    main = measure(L, B, args.steps, args.warmup)
    launches = eng.kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # before the "+defect" column below reuses these buffers
        mb = main["bufs"]
        dump_outputs(args.dump_outputs, {"mfe_dcal": mb["mfe"].cpu().numpy(), "mfe_ss": mb["ss"].cpu().numpy(),
                                         "pf": mb["pf"].cpu().numpy(), "eval_dcal": mb["ev"].cpu().numpy()})
    value = world * B * args.steps / (main["total_ms"] * 1e-3)

    # ---- e2e: the host-buffer C-ABI call, H2D/D2H inside the timed region (pinned host memory)
    codes = main["codes"]
    seq_h = torch.from_numpy(np.frombuffer(b"ACGU", np.uint8)[codes].copy()).pin_memory()
    len_h = torch.full((B,), L, dtype=torch.int32).pin_memory()
    tg_h = main["bufs"]["targets"].cpu().pin_memory()
    mfe_h = torch.zeros(B, dtype=torch.int32).pin_memory(); ss_h = torch.zeros((B, L + 1), dtype=torch.uint8).pin_memory()
    pf_h = torch.zeros((B, 5), dtype=torch.float64).pin_memory(); ev_h = torch.zeros((B, 1), dtype=torch.int32).pin_memory()
    import ctypes as C
    bb, rr = eng.bf_batch_t(), eng.bf_result_t()
    bb.B, bb.stride, bb.seq, bb.len, bb.targets, bb.n_targets, bb.want = B, L, seq_h.data_ptr(), len_h.data_ptr(), tg_h.data_ptr(), 1, WANT
    rr.mfe_dcal, rr.mfe_ss, rr.pf, rr.eval_dcal = mfe_h.data_ptr(), ss_h.data_ptr(), pf_h.data_ptr(), ev_h.data_ptr()
    e2e_steps = max(1, args.steps)
    for _ in range(2):
        eng._check(eng.lib().bf_score_batch(C.byref(bb), C.byref(rr)))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng._check(eng.lib().bf_score_batch(C.byref(bb), C.byref(rr)))
    torch.cuda.synchronize()
    e2e_dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    e2e_val = world * B * e2e_steps / float(e2e_dt.item())
    e2e_ok = bool((ev_h[:, 0] == mfe_h).all().item()) and bool((mfe_h == main["bufs"]["mfe"].cpu()).all().item())
    h2d = seq_h.numel() + 4 * B + tg_h.numel()
    d2h = 4 * B + ss_h.numel() + 8 * 5 * B + 4 * B

    # ---- the other lengths of the sweep (fewer steps; same timing discipline)
    by = {str(L): world * B * args.steps / (main["total_ms"] * 1e-3)}
    kern = {str(L): main["kernel_ms"]}
    checks = {str(L): main["ok"]}
    if not args.no_sweep:
        for l in SWEEP:
            if l == L:
                continue
            m = measure(l, B, 10 if l == 400 else max(2, min(args.steps, 3)), 3)   # L = 400 is the second headline length: 10 steps
            by[str(l)] = world * B * len(m["ms"]) / (m["total_ms"] * 1e-3)
            kern[str(l)] = m["kernel_ms"]; checks[str(l)] = m["ok"]
            del m

    # ---- the "+defect" column: the same step plus the outside pass and the ensemble defect of the target (Edef scoring,
    # energy_scores.py:362-374), L-workload only
    WANTD = WANT | eng.WANT_DEFECT
    bD = main["bufs"]
    dfc = torch.zeros(B, dtype=torch.float64, device=dev)
    def stepD():
        eng.score_batch_device(bD["seq"], bD["lens"], WANTD, targets=bD["targets"], mfe=bD["mfe"], ss=bD["ss"], pf=bD["pf"], ev=bD["ev"],
                               stream=stream, defect=dfc)
    for _ in range(3):
        stepD()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nD = max(2, min(args.steps, 3))
    e0.record()
    for _ in range(nD):
        stepD()
    e1.record(); e1.synchronize()
    tD = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tD, op=dist.ReduceOp.MAX)
    with_defect = {"value": world * B * nD / (float(tD.item()) * 1e-3), "unit": "folds/s", "ms_per_step": float(tD.item()) / nD,
                   "defect_in_0_1": bool(((dfc >= -1e-9) & (dfc <= 1.0 + 1e-9)).all().item()), "defect_mean": float(dfc.mean().item())}
    # the same column at the second headline length (BASELINE config 5's Edef scoring is quoted on long targets): 1024 sequences of 400 nt
    if not args.no_sweep and L != 400:
        B4 = min(B, 1024)
        _c4, b4 = make(400, B4)
        d4 = torch.zeros(B4, dtype=torch.float64, device=dev)
        def stepD4():
            eng.score_batch_device(b4["seq"], b4["lens"], WANTD, targets=b4["targets"], mfe=b4["mfe"], ss=b4["ss"], pf=b4["pf"], ev=b4["ev"],
                                   stream=stream, defect=d4)
        for _ in range(2):
            stepD4()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(3):
            stepD4()
        f1.record(); f1.synchronize()
        t4 = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        with_defect["L400"] = {"value": world * B4 * 3 / (float(t4.item()) * 1e-3), "unit": "folds/s", "B_per_gpu": B4, "ms_per_step": float(t4.item()) / 3,
                               "defect_in_0_1": bool(((d4 >= -1e-9) & (d4 <= 1.0 + 1e-9)).all().item())}
        del b4, d4

    # ---- cofold sweep (SURVEY 8d): the same generator, L/2 + L/2 strands -- fc.mfe_dimer() / fc.pf_dimer() on the two-strand kernels
    cofold = None
    if not args.no_sweep:
        cofold = {}
        for l in (36, 100):
            _cc, bc = make(l, B)
            cut = torch.full((B,), l // 2 + 1, dtype=torch.int32, device=dev)
            def stepC():
                eng.score_batch_device(bc["seq"], bc["lens"], WANT, cut=cut, targets=bc["targets"], mfe=bc["mfe"], ss=bc["ss"], pf=bc["pf"], ev=bc["ev"], stream=stream)
            for _ in range(2):
                stepC()
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(3):
                stepC()
            c1.record(); c1.synchronize()
            tC = torch.tensor([c0.elapsed_time(c1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tC, op=dist.ReduceOp.MAX)
            pfc = bc["pf"]
            cofold[f"{l // 2}&{l - l // 2}"] = {"value": world * B * 3 / (float(tC.item()) * 1e-3), "unit": "folds/s", "ms_per_step": float(tC.item()) / 3,
                                                 "kernel_ms": eng.last_kernel_ms(),
                                                 "fab_le_fa_plus_fb": bool((pfc[:, 3] <= pfc[:, 0] + pfc[:, 1] + 1e-9).all().item())}
            del bc

    # ---- the path's caller: Monte-Carlo sub-steps of the device-resident replica-exchange design loop (N=1 only)
    design_blk = bench_design_loop() if world == 1 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (live CUDA-event kernel times of the L-workload)
    peaks = load_peaks()
    pk_path = os.path.join(ROOT, "profiles", "chip_peaks.json")
    if os.path.exists(pk_path):
        try:
            cp = json.load(open(pk_path))
            # shared memory: the microbenchmark's best-of-5 (38.2 TB/s) sits 2.6 % above 128 B/clk x 148 SMs x 1965 MHz = 37.2 TB/s, i.e.
            # within its timing error of the architectural ceiling -- the ceiling is what is reported
            smem_nominal = 128.0 * 148 * 1965e6 / 1e12
            peaks.update(int32_tops=cp["int32_ops_per_s"] / 1e12, fp64_tflops=cp["fp64_flops_per_s"] / 1e12,
                         smem_tbs=min(cp["smem_bytes_per_s"] / 1e12, smem_nominal), chip_src="measured (profiles/chip_peaks.json; shared memory capped at 128 B/clk/SM)")
        except Exception:
            pass
    r_mfe, r_pf = relaxations(L)
    mfe_ms, pf_ms, ev_ms = main["kernel_ms"]
    names = ["bf_k_mfe", "bf_k_pf", "bf_k_eval"]
    dom = int(np.argmax(main["kernel_ms"]))
    if dom == 1:
        ach = 2.0 * r_pf * B / (pf_ms * 1e-3) / 1e12
        roof = {"kernel": names[1], "bound": "fp64", "achieved": ach, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["fp64_tflops"],
                "traffic": None, "algorithmic": f"2 flops x {r_pf:.4g} relaxations/fold x {B} folds per launch", "peak_src": peaks["chip_src"]}
    else:
        ach = 2.0 * r_mfe * B / (mfe_ms * 1e-3) / 1e12
        roof = {"kernel": names[0], "bound": "int32", "achieved": ach, "peak": peaks["int32_tops"], "unit": "TOP/s", "frac": ach / peaks["int32_tops"],
                "traffic": None, "algorithmic": f"2 int32 ops x {r_mfe:.4g} relaxations/fold x {B} folds per launch", "peak_src": peaks["chip_src"]}
    # DRAM traffic of the dominant fill kernel per launch, from the committed `ncu --set full` capture of this workload (if any)
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        key = f"{'bf_k_pf_fill' if dom == 1 else 'bf_k_mfe_fill'}@L{L}xB{B}"
        if key in tr:
            roof["traffic"] = tr[key]["dram_bytes"]
            roof["traffic_src"] = tr[key]["src"]
        # executed thread-instructions per relaxation of both fill kernels at both headline lengths, from the same committed captures
        roof["thread_inst_per_relaxation"] = {k: {"value": v["thread_inst_per_relaxation"], "kernel": v.get("kernel"), "issue_active_pct": v.get("issue_active_pct")}
                                              for k, v in tr.items() if "thread_inst_per_relaxation" in v}
        roof["thread_inst_src"] = "profiles/ncu_traffic.json (smsp__inst_executed.sum x smsp__thread_inst_executed_per_inst_executed.ratio / (folds x closed-form relaxations))"
    except Exception:
        pass
    roof["kernel_ms"] = dict(zip(names, main["kernel_ms"]))
    roof["share_of_step"] = main["kernel_ms"][dom] / max(1e-9, sum(main["kernel_ms"]))
    # on-chip operand traffic view (4 B per interior candidate, 8 B per split candidate; fp64 doubles it)
    T = lambda m: (m + 1) * (m + 2) // 2 if m >= 0 else 0
    r_int = P_PAIR * sum((L - d) * T(min(30, d - 6)) for d in range(4, L))
    smem_mfe = (4 * r_int + 8 * (r_mfe - r_int)) * B / (mfe_ms * 1e-3) / 1e12
    smem_pf = (8 * r_int + 16 * (r_pf - r_int)) * B / (pf_ms * 1e-3) / 1e12
    roof["operand_tbs"] = {"bf_k_mfe": smem_mfe, "bf_k_pf": smem_pf, "peak_smem_tbs": peaks["smem_tbs"], "frac_mfe": smem_mfe / peaks["smem_tbs"], "frac_pf": smem_pf / peaks["smem_tbs"]}
    # HBM view: the path moves ~2L+60 bytes per fold over HBM by design
    hbm_bytes = (2 * L + 1 + 4 + 4 + 40 + 4 + L) * B
    roof["hbm"] = {"achieved_gbs": hbm_bytes / (sum(main["kernel_ms"]) * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"], "peak_src": peaks["hbm_src"], "algorithmic_bytes_per_launch": hbm_bytes}

    # the same two fractions for the other lengths of the sweep (kernel times of this run)
    roof["by_length"] = {}
    for l, (m_ms, p_ms, _e) in kern.items():
        rm, rp = relaxations(int(l))
        roof["by_length"][l] = {"mfe_int32_frac": 2.0 * rm * B / (m_ms * 1e-3) / 1e12 / peaks["int32_tops"],
                                "pf_fp64_frac": 2.0 * rp * B / (p_ms * 1e-3) / 1e12 / peaks["fp64_tflops"]}

    # relaxations the CPU restatement actually evaluates on sequences of THIS workload (it skips candidates whose inner pair cannot
    # form, the GPU kernels read them as +inf / 0 from the ring): reported next to the closed form the roofline uses (SURVEY 8d)
    if not args.no_cpu:
        try:
            from oracle.pyoracle import Oracle
            O = Oracle(os.path.join(ROOT, "desirna_b200", "params", "turner1999_37C.par"))
            cnt = np.array([O.mfe(sq, counts=True)[2] for sq in to_strings(synth(L, 32, rank=0))], dtype=np.float64)
            counted = float(cnt.sum(axis=1).mean())
            roof["relaxations_per_fold"] = {"closed_form_mfe": r_mfe, "closed_form_pf": r_pf, "counted_by_cpu_port_mfe": counted,
                                            "counted_parts": dict(zip(["interior", "ml_closing", "fml_split", "f5"], cnt.mean(axis=0).tolist())),
                                            "sample": "first 32 sequences of the workload",
                                            "mfe_int32_frac_on_counted": 2.0 * counted * B / (mfe_ms * 1e-3) / 1e12 / peaks["int32_tops"]}
        except Exception as exc:  # the count is auxiliary
            roof["relaxations_per_fold"] = {"error": str(exc)}

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        v, n, dt = cpu_sample(L, 12.0, threads)
        v400 = cpu_sample(400, 8.0, threads)[0] if L != 400 else v
        slow = cpu_sample(L, 4.0, threads, fast=False)[0]
        r_all = sum(relaxations(L))
        cpu = {"value": v, "unit": "folds/s", "cores": threads, "physical_cores": physical_cores(), "kind": cpu_kind(),
               "sample": f"{n} random sequences of L={L} ({dt:.1f} s); " + cpu_desc(threads),
               "value_L400": v400, "oracle_port_value": slow, "ns_per_relaxation_per_thread": 1e9 * threads / v / r_all}
    line = {
        "metric": "MFE+PF folds/sec", "value": value, "unit": "folds/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main["total_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32+f64", "data": "synthetic",
        "config": {"workload": f"synthetic batched fold sweep: {B} random sequences x L={L} per GPU, MFE+backtrack+PF+eval, Turner 1999",
                   "L": L, "B_per_gpu": B, "params": "turner1999", "parallelism": f"dp{world} (sequences sharded, no data-path collective)",
                   "l2": "256 MiB write between timed steps"},
        "e2e": {"value": e2e_val, "unit": "folds/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "timer": "host clock around the synchronous C-ABI call"},
        "gpu_launches": int(launches),
        "roofline": roof, "cpu_baseline": cpu, "by_length": by, "kernel_ms_by_length": kern, "with_ensemble_defect": with_defect,
        "cofold": cofold, "design_loop": design_blk,
        "checks": {"ed_equals_mfe_and_epf_le_mfe": checks, "e2e_matches_device_path": e2e_ok},
        "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_remc(args):
    """`--workload remc`: BASELINE.json config 3's shape through the lock-step replica loop of
    desirna_b200.utils.replica_exchange_monte_carlo (the reference's utils/replica_exchange_monte_carlo.py:233-271 re-plumbed):
    R = 64 replicas of one target, replica r on rank r mod G, every Monte-Carlo sub-step one engine call per rank for its R/G
    mutants, ONE all-gather of the packed replica records per global step (NCCL), neighbour swaps recomputed on every rank.
    Value = Monte-Carlo sub-steps of all replicas per second (R x RE_attempt x global steps / time), max time over ranks."""
    import random
    import torch
    import torch.distributed as dist
    from desirna_b200 import design, engine as eng
    from desirna_b200.utils import replica_exchange_monte_carlo as remc
    from desirna_b200.utils import sequence_utils as su
    from desirna_b200.utils import stats_inputs_outputs as sio

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng.init(local)
    eng.params_builtin(1999)
    rows = [json.loads(x) for x in open(os.path.join(ROOT, "tests", "golden", "E1.jsonl"))]
    targets = {"L104": next(r for r in rows if len(r["target"]) == 104), "L400": next(r for r in rows if len(r["target"]) == 400)}
    R, att = 64, args.re_attempt
    out = {}
    for tag, row in targets.items():
        random.seed(1234)                       # same start state and parent stream on every rank
        o = design.DesignOptions(replicas=R, RE_attempt=att)
        inp = sio.make_input(row["file"], row["target"])
        nts = su.get_nt_list(inp)
        objs = su.generate_initial_list(nts, inp, o)
        st = sio.Stats()
        def gstep(objs, st):
            objs, st = remc.mutate_sequence_re(objs, nts, st, o, inp, mutate=su.mutate_sequence)
            st.global_step += 1
            return remc.replica_exchange(objs, st, o)
        for _ in range(args.warmup):
            objs, st = gstep(objs, st)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            objs, st = gstep(objs, st)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        same = [x.sequence for x in objs]
        if world > 1:   # every rank must hold the same replica list after the all-gather + swaps
            gathered = [None] * world
            dist.all_gather_object(gathered, same)
            assert all(g == gathered[0] for g in gathered), "ranks disagree on the replica state"
        out[tag] = {"global_steps_per_s": args.steps / dt, "substeps_per_s": R * att * args.steps / dt, "ms_per_global_step": 1e3 * dt / args.steps,
                    "best_distance": min(sum(a != b for a, b in zip(x.mfe_ss, row["target"])) for x in objs)}
    if rank == 0:
        print(json.dumps({"metric": "REMC Monte-Carlo sub-steps/sec (R=64 replicas sharded r mod G, lock-step host loop, one all-gather per global step)",
                          "value": out["L104"]["substeps_per_s"], "unit": "sub-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "higher_is_better": True, "scaling": "strong", "data": "Eterna100-V1 targets of 104 and 400 nt (tests/golden/E1.jsonl)",
                          "config": {"workload": "remc", "replicas": R, "re_attempt": att, "scoring": "Ed-Epf:1.0", "params": "turner1999"},
                          "by_target": out,
                          "limiter": "per sub-step one engine call for R/G mutants: single-sequence latency of the fill kernels + Python move generator; the all-gather moves R x ~(2 L + 150) bytes once per global step"}))
    if world > 1:
        dist.destroy_process_group()


def bench_design_loop():
    """Sub-step cost of the replica-exchange design loop (bf_design_*: propose -> MFE + backtrack -> PF -> eval -> accept,
    all on the device).  (a) the shape of BASELINE.json's config 3 on one target: 64 replicas of one median-length Eterna
    puzzle; (b) the 100 Eterna V1 targets x 10 replicas advanced together, one loop per length bucket on its own stream."""
    import random
    from desirna_b200 import design
    from desirna_b200.utils import stats_inputs_outputs as sio
    rows = [json.loads(l) for l in open(os.path.join(ROOT, "tests", "golden", "E1.jsonl"))]
    one = min(rows, key=lambda r: (abs(len(r["target"]) - 104), r["file"]))
    random.seed(0)
    out = {}
    o = design.DesignOptions(replicas=64, RE_attempt=100)
    loop = design.DesignLoop([sio.make_input(one["file"], one["target"])], o, seed=1)
    loop.run(1); loop.sync()
    t0 = time.perf_counter()
    loop.run(2); loop.sync()
    dt = time.perf_counter() - t0
    loop.close()
    out["one_target_64_replicas"] = {"target": one["file"], "L": len(one["target"]), "ms_per_substep": dt / 200 * 1e3,
                                     "sequences_scored_per_s": 64 * 200 / dt}
    # (d) BASELINE config 1: the reference's standard example target (36 nt) with its default 10 replicas
    o = design.DesignOptions(replicas=10, RE_attempt=100)
    loop = design.DesignLoop([sio.make_input("Standard_design", "((((((.((((((((....))))).)).).))))))")], o, seed=4)
    loop.run(1); loop.sync()
    t0 = time.perf_counter()
    loop.run(3); loop.sync()
    dt = time.perf_counter() - t0
    loop.close()
    out["standard_36nt_10_replicas"] = {"ms_per_substep": dt / 300 * 1e3, "sequences_scored_per_s": 10 * 300 / dt,
                                        "reference_example_run": "1033 score calls/s on 10 processes (example_files/outputs/Standard_design*/*_stats)"}
    # (c) BASELINE config 4: the reference's two-strand example (17 & 18 nt), heterodimer scoring with the oligomerisation term
    o = design.DesignOptions(replicas=64, RE_attempt=100, oligo_state="heterodimer")
    loop = design.DesignLoop([sio.make_input("RNA_RNA_complex", "(((.(((((....))..&(((....)))..))))))", "NNNNNNNNNNNNNNNNN&NNNNNNNNNNNNNNNNNN")], o, seed=3)
    loop.run(1); loop.sync()
    t0 = time.perf_counter()
    loop.run(2); loop.sync()
    dt = time.perf_counter() - t0
    loop.close()
    out["heterodimer_17_18nt_64_replicas"] = {"ms_per_substep": dt / 200 * 1e3, "sequences_scored_per_s": 64 * 200 / dt,
                                              "reference_example_run": "933 score calls/s on 10 processes (example_files/outputs/RNA_RNA_complex*/*_stats)"}
    # (e) what the reference does per run: ONE target, its default 10 replicas -- here the longest Eterna V1 targets.  A sub-step
    # scores 10 sequences: the cluster-per-sequence kernels (csrc/bf_cluster.cu, a thread-block cluster per sequence) against the
    # single-CTA kernels (BF_CL=0 BF_EXT_WIDE=0)
    for L in (200, 400):
        one_long = min(rows, key=lambda r: (abs(len(r["target"]) - L), r["file"]))
        res = {"target": one_long["file"], "L": len(one_long["target"])}
        for tag, env in (("cluster_kernels", {}), ("single_cta_kernels", {"BF_CL": "0", "BF_EXT_WIDE": "0"})):
            os.environ.update(env)
            try:
                o = design.DesignOptions(replicas=10, RE_attempt=20)
                loop = design.DesignLoop([sio.make_input(one_long["file"], one_long["target"])], o, seed=5)
                loop.run(1); loop.sync()
                t0 = time.perf_counter()
                loop.run(2); loop.sync()
                dt = time.perf_counter() - t0
                loop.close()
                res[tag] = {"ms_per_substep": dt / 40 * 1e3, "sequences_scored_per_s": 10 * 40 / dt}
            finally:
                for k in env:
                    os.environ.pop(k, None)
        out["one_target_%dnt_10_replicas" % L] = res
    o = design.DesignOptions(replicas=10, RE_attempt=100)
    inputs = [sio.make_input(r["file"], r["target"]) for r in rows]
    groups = design.bucket_jobs([len(i.sec_struct) for i in inputs])
    loops = [design.DesignLoop([inputs[k] for k in g], o, seed=2 + b) for b, g in enumerate(groups)]
    for l in loops:
        l.run(1)
    for l in loops:
        l.sync()
    t0 = time.perf_counter()
    for l in loops:
        l.run(1)
    for l in loops:
        l.sync()
    dt = time.perf_counter() - t0
    for l in loops:
        l.close()
    out["eterna100_x_10_replicas"] = {"jobs": len(inputs), "buckets_stride_jobs": [(l.stride, l.J) for l in loops], "s_per_global_step": dt,
                                      "ms_per_substep": dt / 100 * 1e3, "sequences_scored_per_s": len(inputs) * 10 * 100 / dt}
    out["timer"] = "host clock around enqueue + stream synchronisation; sequences stay on the device"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--L", type=int, default=100)
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--workload", default="sweep", choices=["sweep", "remc"])
    ap.add_argument("--re-attempt", type=int, default=10, dest="re_attempt")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--peaks", action="store_true", help="measure INT32/FP64/smem chip peaks and write profiles/chip_peaks.json")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0's sequences)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.peaks or args.impl != "b200" or args.workload != "sweep"):
        ap.error("--dump-outputs applies to the sweep workload of --impl b200")
    args.warmup = max(3, args.warmup) if args.impl == "b200" else args.warmup
    if args.peaks:
        from desirna_b200 import engine as eng
        eng.init(0)
        pk = eng.microbench()
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        json.dump(pk, open(os.path.join(ROOT, "gpurun_out", "chip_peaks.json"), "w"), indent=1)
        print(json.dumps(pk))
        return
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "remc":
        run_remc(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE config 5 (the configuration the metric is quoted on):

    full PDAS s-path + 10-fold CV fits/sec  (and the dual-sweep HBM GB/s against the roofline)

Workload ("C5"): gaussian gen.data-shaped design n=1000, p=500000, true s=10, screening.num=5000, 10-fold CV,
sequential s.list=1..20  => one step = one full bessCpp call = 220 PDAS fits (20 levels x (1 full fit + 10 folds)).

  python bench.py --gpus 1 --steps K --warmup W            our arm, one GPU
  torchrun ... bench.py --gpus N ...                        our arm, N ranks: REPEATED 10-fold CV, one repetition per
                                                            rank (weak scaling, see below)
  python bench.py --impl reference ...                      the reference's own CPU code (oracle/_ref) on host cores
  python bench.py ... --dump-outputs DIR                    also write the last timed call's results as DIR/*.npy

N > 1.  A single C5 call is 2.3 ms of which only the 0.6 ms screening sweep is p-sized; the 220 fits behind it run on a
40 MB screened design as ONE resident launch whose length is the per-chain dependency chain, so one call cannot be made
shorter by more GPUs (measured, one call with the columns sharded over 1 / 2 / 4 / 8 GPUs: 2.3 / 2.1 / 2.0 / 2.0 ms).  What does shard is what north_star names first: "CV folds
and sparsity levels shard embarrassingly, with only per-fold losses reduced".  The N-GPU job is therefore repeated 10-fold
CV with N repetitions (rank r draws its folds from cv_seed + r): the columns of X are sharded over the ranks for the joint
screening sweep (local top-k + NCCL all-gather of candidates + all-reduce of the kept columns, inside the library), each
rank then runs its own repetition's 200 fold fits + the full-data chain on the replicated screened design, and one NCCL
all-reduce per step -- inside the library, on its own communicator (ext.cv_reduce_over_ranks) -- averages the per-level CV
losses so every rank chooses the same sparsity level and returns the same model.  Per-GPU work is fixed
as N grows => "scaling": "weak".  `value` counts UNIQUE fits only: the full-data chain is identical on every rank and is
counted once (20*(1 + 10*N) fits per step).  The strong-scaling numbers of the column-sharded path itself (C5 call and the
no-screening variant C5b, where every PDAS sweep is p = 500k wide) are reported next to it under "column_sharded", and
"fold_sharded_c2" is config 2 as ONE call whose fold chains are dealt over the ranks (ext.fold_shard) against the same call on
one GPU.  The N = 1 line carries "c2_glm_path": config 2 through the C ABI (the chain kernels: tensor-core Gram + Cholesky).

`value`  : whole-job fits/s with X already resident in HBM when the timed region starts.
`e2e`    : same metric through the reference-facing C-ABI call with X in pinned HOST memory (H2D inside the region).
Timing: CUDA events on the current stream around K steps, synchronize + barrier on both sides, max over ranks.
L2: the design is 4 GB (>> 126 MB L2), every step streams it from HBM again; no explicit flush needed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROWS, P_COLS, K_TRUE, SCREEN, NFOLDS, SMAX = 1000, 500000, 10, 5000, 10, 20
WORKLOAD = ("C5: gaussian gen.data n=1000 p=500000 true-s=10, screening.num=5000, 10-fold CV, sequential s.list=1..20 "
            "(220 PDAS fits per call)")
# CPU sample: a proportional slice of C5 (same n, folds, screening.num => same per-fit cost; 15% of the columns and the
# first 3 of 20 levels => same screening-to-fit ratio as the full call)
CPU_P, CPU_SMAX = 75000, 3


def make_c5_on_device(torch, device, p=P_COLS, seed=5, torch_design=False):
    """gen.data-shaped gaussian problem with the design born in HBM: x from the library's own generator
    (bess_b200_gen_design: rows ~ N(0, I), gen.data.R:110-118 with rho = 0), or torch.randn with --torch-design."""
    if torch_design:
        gen = torch.Generator(device=device).manual_seed(seed)
        X = torch.randn(N_ROWS, p, dtype=torch.float64, device=device, generator=gen)
    else:
        from bess_b200.gen_data import gen_design_device
        X = gen_design_device(N_ROWS, p, 0.0, seed, torch.device(device).index or 0)
    rng = np.random.default_rng(seed)
    nz = np.sort(rng.choice(p, K_TRUE, replace=False))
    m = 5 * np.sqrt(2 * np.log(p) / N_ROWS)
    beta = rng.uniform(m, 100 * m, K_TRUE)
    sigma = np.sqrt((beta @ beta) / 10.0)
    y = (X[:, torch.as_tensor(nz, device=device)] @ torch.as_tensor(beta, device=device)).cpu().numpy()
    y = y + rng.normal(0.0, sigma, N_ROWS)
    return X, y, nz


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _ref_sample(levels):
    """A proportional slice of C5 for the CPU arm: same n, folds and screening.num (=> same per-fit cost), `levels` of the
    20 sparsity levels and the same share of the 500000 columns (=> same screening-to-fit ratio as the full call)."""
    from bess_b200.gen_data import gen_data
    p = CPU_P * levels // CPU_SMAX
    d = gen_data(N_ROWS, p, "gaussian", K_TRUE, seed=5)
    return d, p


def _ref_call(d, levels):
    from oracle import ref
    w = np.ones(N_ROWS)
    seq = np.arange(1, levels + 1)
    t0 = time.perf_counter()
    ref.pywrap_bess(d.x, d.y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, NFOLDS, seq, 1, levels, True, SCREEN, cv_seed=123)
    return time.perf_counter() - t0


def _sample_text(p, levels, procs):
    return (f"oracle/_ref (reference src/*.cpp, -O2, single-threaded as shipped) on a {100 * levels // 20}% slice of C5: "
            f"n=1000, p={p}, screening.num=5000, 10-fold CV, s.list=1..{levels} ({levels * (1 + NFOLDS)} fits per call)"
            + (f"; {procs} independent calls side by side, one per process" if procs > 1 else ""))


def cpu_baseline(levels=CPU_SMAX):
    """The reference's own C++ (oracle/_ref, single thread as shipped) on a bounded slice of the workload."""
    from oracle import ref
    if not ref.available():
        return None
    d, p = _ref_sample(levels)
    dt = _ref_call(d, levels)
    fits = levels * (1 + NFOLDS)
    return {"value": fits / dt, "unit": "fits/s", "cores": 1, "kind": "reference", "seconds": dt,
            "sample": _sample_text(p, levels, 1)}


def _ref_worker(d, levels, nsteps, barrier, q):
    times = []
    for _ in range(nsteps):
        barrier.wait()
        times.append(_ref_call(d, levels))
    q.put(times)


def _mem_available_gb():
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                return float(ln.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


# one reference call on C5 holds its row-major input (shared with the parent, copy-on-write), the column-major copy of
# Pointer2MatrixXd (utilities.cpp:13-25) and the by-value copy of bessCpp (bess.h:20) until screening shrinks it: ~9-12 GB
REF_GB_PER_PROC, REF_GB_PARENT = 13.0, 6.0


def run_reference(args):
    """The reference arm: the reference's own CPU implementation (oracle/_ref = /root/reference/src compiled as shipped) on
    the box's host cores, ON CONFIG 5 ITSELF -- n=1000, p=500000, screening.num=5000, 10-fold CV, s.list=1..20, 220 fits per
    call, ~50-150 s per call.  The library is single-threaded (python/setup.py:38-40: no OpenMP), so "all the host threads it
    can use" = independent calls side by side, one process per core, as many as the host memory holds (~13 GB each).
    Every process makes ONE timed call (no warm-up: --steps/--warmup would cost tens of minutes and a CPU library has nothing
    to warm), all released together; the step time is the slowest process.  If the host cannot hold even one full call
    the arm falls back to the proportional slice of round 1 and says so in `reference_sample`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libbess_ref.so was not built"}))
        return
    ref.lib()  # mapped in THIS process before forking, so the loaded .so is visible to whoever inspects the arm
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    avail = _mem_available_gb()
    procs_full = int(min(cores, 16, (avail - REF_GB_PARENT) // REF_GB_PER_PROC))
    # test overrides (tests/test_bench_contract.py runs this arm on a tiny sample)
    force_levels = os.environ.get("BESS_BENCH_REF_LEVELS")
    full = procs_full >= 1 and force_levels is None
    if full:
        levels, procs, total, warm = SMAX, procs_full, 1, 0
        from bess_b200.gen_data import gen_data
        d, p = gen_data(N_ROWS, P_COLS, "gaussian", K_TRUE, seed=5), P_COLS
    else:
        total, warm = args.warmup + args.steps, args.warmup
        levels = int(max(1, min(CPU_SMAX, 150.0 / (max(total, 1) * 3.5))))  # keep the whole run within a few minutes
        levels = int(force_levels) if force_levels is not None else levels
        procs = int(os.environ.get("BESS_BENCH_REF_PROCS", max(1, min(cores, 16))))
        d, p = _ref_sample(levels)
    ctx = mp.get_context("fork")
    barrier, q = ctx.Barrier(procs), ctx.Queue()
    ws = [ctx.Process(target=_ref_worker, args=(d, levels, total, barrier, q)) for _ in range(procs)]
    for pr in ws:
        pr.start()
    per_proc = [q.get() for _ in ws]
    for pr in ws:
        pr.join()
    step_s = np.max(np.array(per_proc), axis=0)[warm:]  # slowest process of every timed step
    dt = float(np.mean(step_s))
    fits = levels * (1 + NFOLDS) * procs
    val = fits / dt
    if full:
        sample = (f"oracle/_ref (reference src/*.cpp, -O2, single-threaded as shipped) on config 5 ITSELF: n=1000, p=500000, "
                  f"screening.num=5000, 10-fold CV, s.list=1..20 (220 fits per call); {procs} independent calls side by side, one "
                  f"per process ({cores} cores, {avail:.0f} GB available, ~{REF_GB_PER_PROC:.0f} GB per call); one timed call per "
                  f"process, no warm-up (per-process call times {min(min(t) for t in per_proc):.1f}-{max(max(t) for t in per_proc):.1f} s)")
    else:
        sample = _sample_text(p, levels, procs) + (f" [fallback: {avail:.0f} GB of host memory cannot hold one full config-5 call]"
                                                   if force_levels is None else "")
    base = {"value": val, "unit": "fits/s", "cores": procs, "kind": "reference", "seconds": dt, "sample": sample}
    print(json.dumps({"impl": "reference", "metric": "pdas_path_cv_fits_per_sec", "value": val, "unit": "fits/s",
                      "n_gpus": args.gpus, "steps": len(step_s), "warmup": warm, "steps_requested": args.steps,
                      "warmup_requested": args.warmup, "ms_per_step": dt * 1e3,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                      "data": "synthetic", "config": {"workload": WORKLOAD, "reference_sample": sample,
                                                      "same_config_as_gpu_arm": bool(full)},
                      "cpu_baseline": base,
                      "e2e": {"value": val, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from bess_b200 import _lib, cbess
    from bess_b200 import dist as bdist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    _lib.require_gpu()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    dev = f"cuda:{local_rank}"
    X, y, nz = make_c5_on_device(torch, dev, torch_design=args.torch_design)
    w = np.ones(N_ROWS)
    seq = np.arange(1, SMAX + 1)
    lo, hi = (0, P_COLS) if world == 1 else bdist.shard_range(P_COLS, world, rank)
    # N > 1: rank 0 first runs the SAME calls on the whole design on its own GPU -- the answers the column-sharded calls
    # must reproduce (checked on the box, reported as parity_vs_single_gpu)
    single = None
    if world > 1 and rank == 0:
        one = lambda scr: cbess.fit(None, y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, NFOLDS, seq, 1, SMAX, scr > 0, max(scr, 1),
                                    cv_seed=123, device=local_rank, x_device_ptr=X.data_ptr(), n=N_ROWS, p=P_COLS, want_trace=False)
        single = {"c5": one(SCREEN), "c5b": None if args.no_c5b else one(0)}
    Xs = X if world == 1 else X[:, lo:hi].contiguous()
    del X
    torch.cuda.empty_cache()

    curve_dev = torch.zeros(SMAX, dtype=torch.float64, device=dev)

    def reduce_curve(o):
        # repeated CV: average the per-level CV losses over the repetitions (one 160-byte NCCL all-reduce per step)
        curve_dev.copy_(torch.from_numpy(o["ic_all"]), non_blocking=False)
        dist.all_reduce(curve_dev)
        mean = (curve_dev / world).cpu().numpy()
        o["cv_curve_mean"], o["s_joint"] = mean, int(o["s_all"][int(np.argmin(mean))])
        return o

    lib_reduce = not args.torch_cv_reduce  # the library averages the CV curves itself (ext.cv_reduce_over_ranks)

    def step(host_x=None, profile=False, seed_shift=True):
        if world == 1:
            if host_x is None:
                return cbess.fit(None, y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, NFOLDS, seq, 1, SMAX, True, SCREEN,
                                 cv_seed=123, device=local_rank, x_device_ptr=Xs.data_ptr(), n=N_ROWS, p=P_COLS,
                                 want_trace=False, profile=profile)
            return cbess.fit(host_x, y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, NFOLDS, seq, 1, SMAX, True, SCREEN,
                             cv_seed=123, device=local_rank, want_trace=False, profile=profile)
        seed = 123 + (rank if seed_shift else 0)
        if host_x is None:
            o = bdist.fit_column_sharded(None, lo, P_COLS, y, w, 1, True, 1, 20, 1, True, 1, True, NFOLDS, seq, 1, SMAX,
                                         SCREEN, cv_seed=seed, device=local_rank, x_shard_device_ptr=Xs.data_ptr(),
                                         n=N_ROWS, p_local=hi - lo, profile=profile, want_curve=seed_shift and not lib_reduce,
                                         cv_reduce_over_ranks=seed_shift and lib_reduce)
        else:
            o = bdist.fit_column_sharded(host_x, lo, P_COLS, y, w, 1, True, 1, 20, 1, True, 1, True, NFOLDS, seq, 1, SMAX,
                                         SCREEN, cv_seed=seed, device=local_rank, profile=profile,
                                         want_curve=seed_shift and not lib_reduce,
                                         cv_reduce_over_ranks=seed_shift and lib_reduce)
        if seed_shift and lib_reduce:
            o["s_joint"] = int(o["s"])  # chosen from the rank-averaged CV curve inside the library (one ncclAllReduce)
            return o
        return reduce_curve(o) if seed_shift else o

    def timed(nsteps, host_x=None, **kw):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(nsteps):
            out = step(host_x, **kw)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    # clocks are sampled from the warm-up to the end of the e2e region (the timed region alone lasts well under a second,
    # shorter than nvidia-smi's start-up); every sample is taken under load
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    ms, out = timed(args.steps)
    # unique fits per step: 20 levels x (the full-data chain once + 10 folds per CV repetition)
    fits_per_step = bdist.unique_fits_repeated_cv(world, SMAX, NFOLDS)
    value = fits_per_step * args.steps / (ms / 1e3)

    # ---- e2e: X in pinned host memory, H2D inside the timed region, results (beta, coef0, losses) read back
    Xh = torch.empty(Xs.shape, dtype=torch.float64, pin_memory=True)
    Xh.copy_(Xs)
    xh = Xh.numpy()
    step(xh)
    e2e_steps = max(1, min(args.steps, 5))
    ms_e2e, out_e = timed(e2e_steps, xh)
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region + e2e region"
    e2e_val = fits_per_step * e2e_steps / (ms_e2e / 1e3)
    st = out["stats"]
    d2h = st["n_batches"] * (16 * SMAX * 12 + 16 * 12) + st["n_sweeps"] * 16 * 8 + SCREEN * 4 + P_COLS * 0
    h2d = int(Xs.numel() * 8 + 2 * N_ROWS * 8)

    # ---- roofline of the dual-sweep kernel: CUDA events around every launch on the engine's own stream, over a
    # profiled repeat of the timed region (event recording costs ~1 ms per call, so it is kept out of `value`)
    ncat = len(cbess.PROF_CATS)
    prof_ms = np.zeros(ncat)
    prof_n = np.zeros(ncat)
    big_bytes = pdas_bytes = 0.0
    for _ in range(args.steps):
        o = step(profile=True)
        prof_ms += np.array(list(o["stats"]["prof_ms"].values()))
        prof_n += np.array(list(o["stats"]["prof_launches"].values()))
        big_bytes += o["stats"]["big_sweep_bytes"]
        pdas_bytes += o["stats"]["sweep_bytes"]
    # ---- the resident-path kernel (gaussian family on the screened, L2-resident design): the whole 20-level x 11-chain
    # PDAS path is ONE cooperative launch; its own clock64 phase timers say where that launch spends its time
    res = np.array(o["stats"]["resident"])
    resident = None
    if res[0] > 0:
        mhz = 1965.0
        sweeps = float(res[1])
        stream_us, reduce_us = float(res[17]) / mhz, float(res[18]) / mhz
        xbytes = 8.0 * N_ROWS * SCREEN
        own_names = ("prologue", "wait", "select_and_level_bookkeeping", "load_columns", "gram", "solve", "residual", "publish")
        resident = {
            "kernel": "lm_path_kernel<FT=6>: 137 sweeper CTAs (column slices of the screened 1000 x 5000 design, L2-resident) + 11 "
                      "chain-owner CTAs; PDAS iteration loop, top-k, Cholesky, cycle test, level loop and losses on the device",
            "launches_per_step": float(res[0]), "path_steps_per_launch": float(res[3]),
            "sweeps_per_launch": sweeps, "full_vector_select_fallbacks": float(res[2]), "level_starts_served_by_the_previous_sweep": float(res[4]),
            "sweep_us": (stream_us + reduce_us) / max(sweeps, 1.0),
            "sweep_x_bytes": xbytes,
            "sweep_stream_GBps_from_L2": xbytes / (stream_us / max(sweeps, 1.0) * 1e-6) / 1e9 if stream_us > 0 else None,
            "owner0_us_by_phase": {nm: float(v) / mhz for nm, v in zip(own_names, res[8:16])},
            "sweeper0_us": {"wait_for_owners": float(res[16]) / mhz, "stream_x": stream_us, "reduce_and_sacrifice": reduce_us},
            "note": "clock64 ticks of chain owner 0 / sweeper 0 at 1965 MHz, last profiled call",
        }
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    cat = dict(zip(cbess.PROF_CATS, range(ncat)))
    scr_ms, scr_n = prof_ms[cat["screen_sweep"]], max(prof_n[cat["screen_sweep"]], 1)
    hbm_gbs = big_bytes / (scr_ms * 1e-3) / 1e9 if scr_ms > 0 else None
    sweep_ms = scr_ms + prof_ms[cat["dual_sweep"]]
    sweep_n = max(scr_n + prof_n[cat["dual_sweep"]], 1)
    achieved = (big_bytes + pdas_bytes) / (sweep_ms * 1e-3) / 1e9 if sweep_ms > 0 else None
    total_kernel_ms = float(prof_ms.sum() - prof_ms[cat["upload"]])
    # DRAM traffic of the same kernel instantiation and grid, from the committed ncu --set full capture
    traffic = traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["screen_sweep_4GB"]
        traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
    except Exception:
        pass

    # ---- the p=500k PDAS dual sweep itself (config 5 with screening off, "C5b"): all 11 chains in one pass over X
    probe = None
    if world == 1:
        from bess_b200.engine import GpuEngine
        eng = GpuEngine(local_rank)
        eng.load(None, y, w, 1, x_device_ptr=Xs.data_ptr(), n=N_ROWS, p=P_COLS)
        eng.normalize(1, True)
        eng.setup_chains(NFOLDS, cbess.cv_fold_ids(N_ROWS, NFOLDS, 123), SMAX, 20, True)
        eng.run_batch(5, list(range(NFOLDS + 1)), True)
        pms, pbytes = eng.time_dual_sweep(20)
        eng.close()
        probe = {"what": "dual_sweep_tma_kernel<FT=12,MODE_D> (bulk-TMA pipeline): X^T r for 11 chains (full fit + 10 folds) in ONE pass over the "
                         "normalised 1000 x 500000 design (config 5 without screening)",
                 "ms_per_launch": pms, "achieved": pbytes / (pms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                 "frac": pbytes / (pms * 1e-3) / 1e9 / peak, "algorithmic_bytes": pbytes}
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["tma_sweep_F12_4GB"]
            probe["traffic"], probe["traffic_source"] = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
        except Exception:
            pass

    # ---- C5b: config 5 WITHOUT screening -- every PDAS dual sweep is p=500k-sized; at N > 1 each iteration is sharded by
    # columns (local sweep + local top-k, NCCL all-gather of candidates, all-reduce of the k active columns).  This is the
    # part of the path whose work grows with p and therefore the part that scales with GPUs.
    def c5b_call():
        if world == 1:
            return cbess.fit(None, y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, NFOLDS, seq, 1, SMAX, False, 1, cv_seed=123,
                             device=local_rank, x_device_ptr=Xs.data_ptr(), n=N_ROWS, p=P_COLS, want_trace=False)
        return bdist.fit_column_sharded(None, lo, P_COLS, y, w, 1, True, 1, 20, 1, True, 1, True, NFOLDS, seq, 1, SMAX, 0,
                                        cv_seed=123, device=local_rank, x_shard_device_ptr=Xs.data_ptr(), n=N_ROWS,
                                        p_local=hi - lo)
    c5b = None
    if not args.no_c5b:
        for _ in range(2):
            ob = c5b_call()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nb = 5
        e0.record()
        for _ in range(nb):
            ob = c5b_call()
        e1.record()
        torch.cuda.synchronize()
        tb = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        ms_b = float(tb.item()) / nb
        sb = ob["stats"]
        c5b = {"workload": "C5b: config 5 with screening off (PDAS dual sweeps over all 500000 columns, 11 chains per pass)",
               "ms_per_call": ms_b, "fits_per_s": 220 / (ms_b * 1e-3), "pdas_sweeps_per_call": sb["n_sweeps"],
               "chosen_s": int(ob["s"]), "aggregate_sweep_GBps_incl_all_other_work": world * sb["sweep_bytes"] / (ms_b * 1e-3) / 1e9,
               "parallelism": "single GPU" if world == 1 else f"columns sharded over {world} ranks, NCCL all-gather of "
                              "top-k candidates + all-reduce of active columns every PDAS iteration"}

    # ---- config 2 (binomial, n = 2000, p = 20000, golden section over s = 1..263, 10-fold CV): the call the chain kernels
    # (IRLS: weighted Gram on the FP64 tensor cores + Cholesky, chain_fit.cu) dominate -- the kernel the round-1 review
    # named as furthest below its roof.  Reported beside the headline, N = 1 only.
    c2 = None
    if world == 1 and not args.no_c2:
        from bess_b200.gen_data import gen_data as _gen
        d2 = _gen(2000, 20000, "binomial", 20, seed=2)
        w2 = np.ones(2000)
        for r2 in range(2):
            t0 = time.perf_counter()
            o2 = cbess.fit(d2.x, d2.y, 2, w2, True, 1, 2, 20, 2, 2, True, 1, True, 10, np.arange(1, 2), 1, 263, False, 1,
                           cv_seed=123, device=local_rank, profile=True, want_trace=False)
            t1 = time.perf_counter()
        s2 = o2["stats"]
        c2 = {"workload": "C2: binomial gen.data n=2000 p=20000 true-s=20, golden section s in [1, 263], 10-fold CV "
                          "(host design, 320 MB H2D inside the call)",
              "ms_per_call": (t1 - t0) * 1e3, "fits": s2["n_fits"], "pdas_iters": s2["n_pdas_iters"], "chosen_s": int(o2["s"]),
              "chain_kernel_ms": s2["prof_ms"]["chain"], "chain_kernel_launches": s2["prof_launches"]["chain"],
              "dual_sweep_ms": s2["prof_ms"]["dual_sweep"], "upload_ms": s2["prof_ms"]["upload"],
              "round1_ms_per_call": 1254.0,
              "evidence": "profiles/r02b_chain_fit_c2_full.md (ncu --set full of one chain_fit launch), "
                          "profiles/r02b_chain_fit_building_blocks.md (solver / Gram probes, FP64 issue rates)"}

    # ---- strong scaling of ONE C5 call with the columns sharded (same folds on every rank, no repetition): what the
    # column axis alone buys at config 5 (only the screening sweep is p-sized)
    col_sharded = None
    if world > 1:
        for _ in range(2):
            step(seed_shift=False)
        ns = max(3, min(args.steps, 20))
        ms_s, out_s = timed(ns, seed_shift=False)
        col_sharded = {"c5_one_call_strong": {"ms_per_call": ms_s / ns, "fits_per_s": 220 * ns / (ms_s * 1e-3),
                                              "chosen_s": int(out_s["s"]),
                                              "note": "one C5 call, columns sharded for the screening sweep, same folds on "
                                                      "every rank; the PDAS path on the screened design is replicated"},
                       "c5b_no_screening_strong": c5b}

    # ---- axis A inside ONE call (ext.fold_shard): config 2 (binomial, golden section, 10-fold CV; chain-kernel bound) with
    # the whole design on every rank and the fold chains dealt over the ranks; against the same call on one GPU, same run
    fold_sharded = None
    if world > 1 and not args.no_c2:
        from bess_b200.gen_data import gen_data as _gen
        d2 = _gen(2000, 20000, "binomial", 20, seed=2)
        w2 = np.ones(2000)
        X2 = torch.as_tensor(d2.x, device=dev)  # resident on every rank: the comparison is about the chains, not PCIe
        fold2 = cbess.cv_fold_ids(2000, 10, 123)
        seq2 = np.arange(1, 2)

        def c2_call(sharded):
            if sharded:
                return bdist.fit_fold_sharded(None, d2.y, w2, 2, True, 2, 20, 2, True, 1, 10, seq2, 1, 263, 0, fold_of_row=fold2,
                                              device=local_rank, x_device_ptr=X2.data_ptr(), n=2000, p=20000)
            return cbess.fit(None, d2.y, 2, w2, True, 1, 2, 20, 2, 2, True, 1, True, 10, seq2, 1, 263, False, 1, fold_of_row=fold2,
                             device=local_rank, x_device_ptr=X2.data_ptr(), n=2000, p=20000, want_trace=False)
        res = {}
        for mode in (False, True):
            if not mode and rank != 0:
                dist.barrier()
                continue
            c2_call(mode)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = c2_call(mode)
            torch.cuda.synchronize()
            res[mode] = ((time.perf_counter() - t0) * 1e3, o)
            if not mode:
                dist.barrier()
        tf = torch.tensor([res[True][0]], dtype=torch.float64, device=dev)
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
        if rank == 0:
            o1, oN = res[False][1], res[True][1]
            fold_sharded = {"workload": "C2 (binomial n=2000 p=20000, golden section s in [1, 263], 10-fold CV), design resident on "
                                        "every rank, fold chains dealt over the ranks (ext.fold_shard)",
                            "ms_per_call": float(tf.item()), "single_gpu_ms_per_call": res[False][0],
                            "fits_this_rank": int(oN["stats"]["n_fits"]), "fits_single_gpu": int(o1["stats"]["n_fits"]),
                            "same_support_and_s": bool(np.nonzero(oN["beta"])[0].tolist() == np.nonzero(o1["beta"])[0].tolist()
                                                       and oN["s"] == o1["s"]),
                            "beta_max_rel_diff": float(np.abs(oN["beta"] - o1["beta"]).max() / max(np.abs(o1["beta"]).max(), 1e-300)),
                            "note": "a rank runs its share of the 11 chains and gives each a 16-CTA cluster (8 CTAs when all 11 share "
                                    "one GPU): the Gram sums run over different row slices, hence last-bit differences"}
        del X2

    parity = None
    if world > 1 and rank == 0:
        def cmp(a, b):
            sa, sb = np.nonzero(a["beta"])[0], np.nonzero(b["beta"])[0]
            same = sa.tolist() == sb.tolist()
            rel = float(np.max(np.abs(a["beta"][sb] - b["beta"][sb]) / np.abs(b["beta"][sb]))) if same and sb.size else None
            return {"support_equal": bool(same), "chosen_s_equal": int(a["s"]) == int(b["s"]), "beta_max_rel_diff": rel,
                    "ic_rel_diff": abs(a["ic"] - b["ic"]) / abs(b["ic"])}
        parity = {"what": f"the column-sharded call on {world} GPUs against the same call on ONE GPU holding the whole design "
                          "(same folds, cv_seed 123), computed on this box in this run",
                  "c5_one_call": cmp(out_s, single["c5"]),
                  "c5b_no_screening": cmp(ob, single["c5b"]) if (single["c5b"] is not None and c5b is not None) else None}
        parity["ok"] = all(v is None or (v["support_equal"] and v["chosen_s_equal"] and v["beta_max_rel_diff"] <= 1e-9)
                           for k2, v in parity.items() if k2 in ("c5_one_call", "c5b_no_screening"))
    base = cpu_baseline() if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    if rank == 0:
        line = {
            "metric": "pdas_path_cv_fits_per_sec", "value": value, "unit": "fits/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic (gen.data recipe; design drawn in HBM by " + ("torch.randn" if args.torch_design else "bess_b200_gen_design") + ")",
            "config": {"workload": WORKLOAD if world == 1 else WORKLOAD + f" x {world} CV repetitions (repeated 10-fold CV, "
                       f"one repetition per rank; {fits_per_step} unique fits per step)",
                       "parallelism": "single GPU" if world == 1 else
                       f"{world} ranks: columns of X sharded for the joint screening sweep (local top-k + NCCL all-gather of "
                       f"candidates + all-reduce of the kept columns), CV repetitions sharded over the ranks (rank r: folds "
                       f"from cv_seed 123 + r) on the replicated 1000 x 5000 screened design, one NCCL all-reduce of the "
                       f"per-level CV losses per step ({'inside the library' if lib_reduce else 'torch.distributed in the bench'})",
                       "l2_policy": ("inputs larger than L2 (4 GB design streamed from HBM every step)" if world == 1 else
                                     f"inputs larger than L2 ({4.0 / world:.2f} GB column shard per rank streamed from HBM every step)"),
                       "cv_seed": 123, "chosen_s": int(out["s"]) if world == 1 else int(out["s_joint"]),
                       "support_recovered": int(np.isin(nz, np.nonzero(out["beta"])[0]).sum())},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "fits/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps},
            "gpu_launches": int(st["kernel_launches"] * args.steps),
            "roofline": {"bound": "hbm", "achieved": hbm_gbs, "peak": peak, "unit": "GB/s",
                         "frac": (hbm_gbs / peak) if hbm_gbs else None, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "dual_sweep_kernel<FT=1,MODE_DH,CPT=2>: the marginal-utility sweep over the "
                                   f"{N_ROWS} x {hi - lo} raw design (d = X^T y, h = (X.X)^T 1 in one pass)",
                         "algorithmic_bytes_per_launch": float(big_bytes / scr_n),
                         "peak_source": peak_src, "launches_per_step": float(scr_n / args.steps),
                         "ms_per_launch": float(scr_ms / scr_n),
                         "resident_path": resident,
                         "all_dual_sweep_launches": None if resident else {
                             "achieved": achieved, "launches_per_step": float(sweep_n / args.steps),
                             "note": "incl. the L2-resident 40 MB PDAS sweeps of the multi-kernel path"},
                         "kernel_ms_per_step": {k: float(v / args.steps) for k, v in zip(cbess.PROF_CATS, prof_ms)},
                         "kernel_share_of_step": float(total_kernel_ms / args.steps / (ms / args.steps)),
                         "p500k_pdas_sweep": probe},
            "cpu_baseline": base, "c5b_no_screening": c5b if world == 1 else None, "c2_glm_path": c2,
            "column_sharded": col_sharded, "fold_sharded_c2": fold_sharded,
            # the strong-scaling curve of ONE call (columns sharded) starts here: N = 1 of column_sharded.c5_one_call_strong /
            # c5b_no_screening_strong in the N > 1 lines
            "strong_scaling_n1": {"c5_one_call_ms": ms / args.steps, "c5b_no_screening_ms": c5b["ms_per_call"] if c5b else None}
            if world == 1 else None,
            "parity_vs_single_gpu": parity,
            "fits_per_step": fits_per_step, "n_boundary_ties": int(st["n_boundary_ties"]),
            "host_ms_last_call": {k: round(float(v), 4) for k, v in st["host_ms"].items()},
        }
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    return line if rank == 0 else None


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out, dirname):
    """Writes what the last timed call returned to its caller -- every array and number of the result, not the run
    statistics -- as <dirname>/<name>.npy in float64 (the index arrays are exact there).  The inputs are fixed by their
    seeds, so two builds of the library can be compared output for output."""
    arrays = {name: np.atleast_1d(np.asarray(v, dtype=np.float64)) for name, v in out.items() if name != "stats" and v is not None}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


class StdoutToStderr:
    """Everything libraries write to fd 1 while the benchmark runs (NCCL prints its version banner there) goes to
    stderr, so that stdout carries exactly one line: the JSON result."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5b", action="store_true")
    ap.add_argument("--no-c2", action="store_true", help="skip the config-2 (chain-kernel bound) block of the N = 1 line")
    ap.add_argument("--torch-cv-reduce", action="store_true",
                    help="N > 1: average the CV curves with torch.distributed in the bench instead of inside the library")
    ap.add_argument("--torch-design", action="store_true", help="draw the design with torch.randn instead of the library's generator")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed call returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        with StdoutToStderr():
            line = run_ours(args)
        if line is not None:
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()

"""Sparse (CSC) designs on one GPU: config-5-shaped calls with the design passed in CSC form against the same matrix passed
dense, and a design whose dense form does not fit in HBM.  Writes one JSON (default profiles/r03a_sparse_c5.json).

Designs (seeded, generated on the device with torch.Generator(seed)): every column holds exactly k = density * n non-zeros,
one per stratum of n / k consecutive rows (row = stratum * (n / k) + uniform offset), values N(0, 1).  y = X[:, true] @ beta
+ N(0, 1) noise with 10 true columns evenly spaced over the p columns and beta = 3, -3, 3, ... (gaussian).

  C5-shaped: n = 1000, p = 500000, density 1 % / 5 % / 20 %, screening 5000, 10-fold CV (cv_seed 123), s = 1..20.  Per
             density: the end-to-end call from host CSC arrays (pageable numpy) against the end-to-end call on the same
             matrix densified in pinned host memory; the same pair with the design already resident on the device; >= 5
             repetitions each (median, min, max); device time per category from a separate profiled call; the screening
             kernel's algorithmic bytes over its time as a share of 7.7 TB/s; and whether both arms returned the same
             screening set, chosen s and beta (bit for bit).
  capacity:  n = 10000, p = 4000000, 1 %, screening 5000, s = 1..20, EBIC: 320 GB dense, 4.8 GB of non-zeros.  Whether it
             runs, its time and the device memory high-water mark (the smallest free memory seen while the call ran,
             sampled every 2 ms, against the free memory before it).

Usage: python tools/gpu_sparse_bench.py [--reps 5] [--out profiles/r03a_sparse_c5.json] [--no-capacity | --capacity-only]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_BW = 7.7e12  # B200 HBM3e, data sheet (one GPU)
SEED = 20261020


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:  # noqa: BLE001
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def make_csc(torch, n, p, density, seed, dev, chunk=250000):
    """The stratified design of the module docstring, on the device: (colptr int64, rowidx int32, values float64)."""
    k = int(round(density * n))
    stride = n // k
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    colptr = torch.arange(p + 1, device=dev, dtype=torch.int64) * k
    rowidx = torch.empty(p * k, device=dev, dtype=torch.int32)
    base = torch.arange(k, device=dev, dtype=torch.int32) * stride
    for j0 in range(0, p, chunk):
        j1 = min(p, j0 + chunk)
        off = torch.randint(0, stride, (j1 - j0, k), device=dev, generator=g, dtype=torch.int32)
        rowidx[j0 * k:j1 * k] = (base[None, :] + off).reshape(-1)
    values = torch.randn(p * k, device=dev, dtype=torch.float64, generator=g)
    true = np.linspace(0, p - 1, 10).astype(np.int64)
    beta = np.array([3.0, -3.0] * 5)
    y = torch.randn(n, device=dev, dtype=torch.float64, generator=g)
    for j, b in zip(true, beta):
        lo, hi = int(j) * k, (int(j) + 1) * k
        y.index_add_(0, rowidx[lo:hi].long(), b * values[lo:hi])
    return colptr, rowidx, values, y.cpu().numpy()


def densify(torch, colptr, rowidx, values, n, p):
    k = int(colptr[1].item())
    X = torch.zeros((n, p), dtype=torch.float64, device=values.device)
    cols = torch.arange(p, device=values.device).repeat_interleave(k)
    X[rowidx.long(), cols] = values
    return X


class MemSampler:
    def __init__(self, torch):
        self.torch, self.stop, self.min_free = torch, False, None

    def __enter__(self):
        self.free0 = self.torch.cuda.mem_get_info()[0]
        self.min_free = self.free0
        self.th = threading.Thread(target=self.run, daemon=True)
        self.th.start()
        return self

    def run(self):
        while not self.stop:
            self.min_free = min(self.min_free, self.torch.cuda.mem_get_info()[0])
            time.sleep(0.002)

    def __exit__(self, *a):
        self.stop = True
        self.th.join()
        self.min_free = min(self.min_free, self.torch.cuda.mem_get_info()[0])

    @property
    def high_water_bytes(self):
        return int(self.free0 - self.min_free)


def timed(fn, reps):
    out, ts = None, []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()  # returns after the results are back on the host (the library synchronises)
        ts.append((time.perf_counter() - t0) * 1e3)
    return out, dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), max_ms=float(np.max(ts)), reps=reps,
                     all_ms=[round(t, 3) for t in ts])


def categories(o):
    pm = o["stats"]["prof_ms"]
    rest = sum(v for k, v in pm.items() if k not in ("upload", "screen_sweep"))
    return dict(upload_ms=pm["upload"], screening_ms=pm["screen_sweep"], rest_ms=rest)


def same(a, b):
    return dict(screening_A=bool(np.array_equal(a["screening_A"], b["screening_A"])), s=a["s"] == b["s"],
                beta=bool(np.array_equal(a["beta"], b["beta"])), coef0=a["coef0"] == b["coef0"], ic=a["ic"] == b["ic"])


def c5_case(torch, density, reps):
    from bess_b200 import cbess
    n, p, scr, K, smax = 1000, 500000, 5000, 10, 20
    colptr, rowidx, values, y = make_csc(torch, n, p, density, SEED, "cuda")
    nnz = int(values.numel())
    w = np.ones(n)
    seq = np.arange(1, smax + 1)
    args = (y, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, K, seq, 1, smax, True, scr)
    kw = dict(cv_seed=123, want_trace=False)
    host_csc = (colptr.cpu().numpy(), rowidx.cpu().numpy(), values.cpu().numpy(), (n, p))
    dev_csc = (colptr, rowidx, values, (n, p))
    Xd = densify(torch, colptr, rowidx, values, n, p)
    Xh = torch.empty((n, p), dtype=torch.float64, pin_memory=True)
    Xh.copy_(Xd)
    xh = Xh.numpy()
    arms = {
        "sparse_e2e_host_csc": lambda prof=False: cbess.fit(host_csc, *args, profile=prof, **kw),
        "dense_e2e_pinned_host": lambda prof=False: cbess.fit(xh, *args, profile=prof, **kw),
        "sparse_resident_device_csc": lambda prof=False: cbess.fit(dev_csc, *args, profile=prof, **kw),
        "dense_resident_device": lambda prof=False: cbess.fit(None, *args, x_device_ptr=Xd.data_ptr(), n=n, p=p, profile=prof,
                                                              **kw),
    }
    res = dict(n=n, p=p, density=density, nnz=nnz, csc_bytes=12 * nnz + 8 * (p + 1), dense_bytes=8 * n * p, arms={})
    outs = {}
    for name, fn in arms.items():
        fn()  # warm-up
        outs[name], t = timed(fn, reps)
        o = fn(True)
        sb = o["stats"]["big_sweep_bytes"]
        sms = o["stats"]["prof_ms"]["screen_sweep"]
        res["arms"][name] = dict(time=t, device_ms_by_category=categories(o), screening_bytes=sb,
                                 screening_share_of_7_7TBps=(sb / (sms * 1e-3)) / PEAK_BW if sms > 0 else None,
                                 chosen_s=int(outs[name]["s"]))
        print(f"density {density:.2f} {name}: median {t['median_ms']:.2f} ms  {res['arms'][name]['device_ms_by_category']}",
              flush=True)
    res["same_outputs_e2e"] = same(outs["sparse_e2e_host_csc"], outs["dense_e2e_pinned_host"])
    res["same_outputs_resident"] = same(outs["sparse_resident_device_csc"], outs["dense_resident_device"])
    res["same_outputs_sparse_host_vs_device"] = same(outs["sparse_e2e_host_csc"], outs["sparse_resident_device_csc"])
    del Xd, Xh, colptr, rowidx, values, dev_csc
    torch.cuda.empty_cache()
    return res


def capacity_case(torch):
    from bess_b200 import cbess
    n, p, density, scr, smax = 10000, 4000000, 0.01, 5000, 20
    colptr, rowidx, values, y = make_csc(torch, n, p, density, SEED + 1, "cuda")
    nnz = int(values.numel())
    host_csc = (colptr.cpu().numpy(), rowidx.cpu().numpy(), values.cpu().numpy(), (n, p))
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    total = torch.cuda.mem_get_info()[1]
    seq = np.arange(1, smax + 1)
    args = (y, 1, np.ones(n), True, 1, 1, 20, 2, 1, True, 4, False, 5, seq, 1, smax, True, scr)
    res = dict(n=n, p=p, density=density, nnz=nnz, dense_bytes=8 * n * p, csc_bytes=12 * nnz + 8 * (p + 1),
               device_total_bytes=int(total))
    try:
        with MemSampler(torch) as ms:
            t0 = time.perf_counter()
            o = cbess.fit(host_csc, *args, want_trace=False)
            res["first_call_ms"] = (time.perf_counter() - t0) * 1e3
        res["device_high_water_bytes_first_call"] = ms.high_water_bytes
        _, t = timed(lambda: cbess.fit(host_csc, *args, want_trace=False), 3)
        o2 = cbess.fit(host_csc, *args, want_trace=False, profile=True)
        res.update(ran=True, time=t, device_ms_by_category=categories(o2), chosen_s=int(o["s"]),
                   support=np.nonzero(o["beta"])[0].tolist(), true_columns=np.linspace(0, p - 1, 10).astype(int).tolist(),
                   screening_bytes=o2["stats"]["big_sweep_bytes"])
    except Exception as e:  # noqa: BLE001
        res.update(ran=False, error=repr(e))
    print(f"capacity: {res.get('ran')} {res.get('time')} high water {res.get('device_high_water_bytes_first_call')}", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03a_sparse_c5.json"))
    ap.add_argument("--no-capacity", action="store_true")
    ap.add_argument("--capacity-only", action="store_true",
                    help="only the capacity case, in a fresh process (the library's memory pool keeps what earlier calls "
                         "allocated, which would hide the case's own high-water mark)")
    a = ap.parse_args()
    import torch
    from bess_b200 import _lib
    _lib.require_gpu()
    rec = dict(gpu=gpu_info(), seed=SEED, generator=__doc__.split("\n\n")[1], cases=[])
    for d in () if a.capacity_only else (0.01, 0.05, 0.20):
        rec["cases"].append(c5_case(torch, d, a.reps))
    if not a.no_capacity:
        rec["capacity"] = capacity_case(torch)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f)
        f.write("\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()

"""Sparse designs without screening: the CSC sweep path against the same matrix passed dense (DESIGN 3.12).

Writes profiles/<tag>_sparse_path.json (default tag r03d) with the card's name and power limit read in the same run.
Per workload: call time (host clock around a synchronised call, median of 5 after a warm-up), PDAS sweep kernel time
(profile category 1, CUDA events) and its algorithmic bytes over that time against 7.7 TB/s, launches per category, and
for every pair of arms whether the supports, the chosen s and the per-level supports agree, with the largest relative
difference of beta / coef0 / IC.  The power-law workload has a few columns hundreds of times longer than the mean (swept by a
CTA each).  The n = 10 000, p = 4 000 000 capacity case is left to tests/test_sparse_path.py (a 200 GB-dense design):
drawing 400 M non-zeros on the host would dominate the run.  The sweep-level crossover (CSC sweep vs dense sweep, engine level, the same chains) is
measured at every density: it is what the selection rule's ratio rests on."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make(n, p, density, seed, family="gaussian", true=(3, 1000, 7000, 40001)):
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    m = sp.random(n, p, density=density, format="csc", random_state=rng, data_rvs=rng.standard_normal)
    m.sort_indices()
    true = [t for t in true if t < p]
    eta = np.asarray(m[:, true] @ np.linspace(1.5, 0.8, len(true))).ravel() + 0.0
    if family == "gaussian":
        y = eta + 0.3 * rng.standard_normal(n)
    elif family == "binomial":
        y = (rng.random(n) < 1.0 / (1.0 + np.exp(-eta))).astype(float)
    else:
        o = np.argsort(rng.exponential(1.0 / np.exp(0.5 * eta)))
        m = m[o, :].tocsc()
        m.sort_indices()
        y = (rng.random(n) < 0.8).astype(float)
    return m, y, true


def make_powerlaw(n, p, seed):
    """Power-law column lengths (text-like): length ~ 0.5 n / rank^0.9, at least 2, so most columns hold a few entries and
    the most frequent ones hundreds to all n rows.  (Columns with one entry are avoided: two of them in the same row are the
    same column after normalisation up to sign, an exact tie in every selection.)"""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    lens = np.minimum(n, np.maximum(2, (0.5 * n / (1.0 + rng.permutation(p)) ** 0.9).astype(np.int64)))
    indptr = np.concatenate([[0], np.cumsum(lens)])
    rows = np.empty(indptr[-1], dtype=np.int32)
    for j in range(p):
        k = lens[j]
        rows[indptr[j]:indptr[j + 1]] = np.sort(rng.choice(n, k, replace=False))
    m = sp.csc_matrix((rng.standard_normal(indptr[-1]), rows, indptr), shape=(n, p))
    y = np.asarray(m[:, [0, 1, 2]] @ np.array([1.0, -0.8, 0.6])).ravel() + 0.3 * rng.standard_normal(n)
    return m, y


def fit(x, y, family, is_cv, seq, **kw):
    from bess_b200 import cbess
    model, dt = {"gaussian": (1, 1), "binomial": (2, 2), "cox": (4, 3)}[family]
    n = y.size
    return cbess.fit(x, y, dt, np.ones(n), True, 1, model, 20, 2, 1, True, 1 if is_cv else 4, is_cv, 10, seq, 1,
                     int(max(seq)), False, 1, want_trace=True, **kw)


def timed(call, reps):
    import torch
    call()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = call()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def compare(a, b):
    def rel(u, v):
        u, v = np.asarray(u, float), np.asarray(v, float)
        return float(np.max(np.abs(u - v)) / max(np.max(np.abs(v)), 1e-300)) if u.size else 0.0
    same_levels = all(np.array_equal(x != 0, y != 0) for x, y in zip(a.get("beta_all", []), b.get("beta_all", [])))
    return dict(same_support=bool(np.array_equal(np.flatnonzero(a["beta"]), np.flatnonzero(b["beta"]))),
                same_s=a["s"] == b["s"], same_level_supports=bool(same_levels),
                max_rel_beta=rel(a["beta"], b["beta"]), rel_coef0=abs(a["coef0"] - b["coef0"]) / max(abs(b["coef0"]), 1e-300),
                rel_ic=abs(a["ic"] - b["ic"]) / max(abs(b["ic"]), 1e-300))


def arm_record(ms, out):
    st = out["stats"]
    sweep_ms = st["prof_ms"][list(st["prof_ms"])[1]]
    return dict(call_ms=ms, sparse_sweeps=st["sparse_sweeps"], sweep_kernel_ms=sweep_ms, sweep_bytes=st["sweep_bytes"],
                sweep_share_of_hbm=(st["sweep_bytes"] / (sweep_ms * 1e-3)) / HBM if sweep_ms > 0 else None,
                launches=st["prof_launches"], s=out["s"])


def workload(name, m, y, family, is_cv, seq, reps, dense=True):
    import torch
    rec = dict(name=name, n=m.shape[0], p=m.shape[1], nnz=int(m.nnz), density=m.nnz / (m.shape[0] * m.shape[1]),
               family=family, cv=is_cv)
    arms = {}
    ms, out_h = timed(lambda: fit(m, y, family, is_cv, seq), reps)
    prof = fit(m, y, family, is_cv, seq, profile=True)
    arms["csc_host"] = arm_record(ms, out_h) | {"profiled": arm_record(0.0, prof)}
    cp, ri, cv = (torch.as_tensor(v).cuda() for v in (m.indptr.astype(np.int64), m.indices.astype(np.int32), m.data))
    ms, out_d = timed(lambda: fit((cp, ri, cv, m.shape), y, family, is_cv, seq), reps)
    arms["csc_device"] = arm_record(ms, out_d)
    outs = {"csc_host": out_h, "csc_device": out_d}
    if dense:
        xd = torch.sparse_csc_tensor(torch.as_tensor(m.indptr.astype(np.int64)), torch.as_tensor(m.indices.astype(np.int64)),
                                     torch.as_tensor(m.data), size=m.shape).cuda().to_dense().contiguous()
        n, p = m.shape
        ms, out_x = timed(lambda: fit(None, y, family, is_cv, seq, x_device_ptr=xd.data_ptr(), n=n, p=p), reps)
        prof = fit(None, y, family, is_cv, seq, x_device_ptr=xd.data_ptr(), n=n, p=p, profile=True)
        arms["dense_device"] = arm_record(ms, out_x) | {"profiled": arm_record(0.0, prof)}
        outs["dense_device"] = out_x
        del xd
        torch.cuda.empty_cache()
    rec["arms"] = arms
    keys = list(outs)
    rec["pairs"] = {f"{a}|{b}": compare(outs[a], outs[b]) for i, a in enumerate(keys) for b in keys[i + 1:]}
    return rec


def sweep_crossover(n, p, density, K):
    """Engine level: one CSC sweep vs one dense sweep for 1 + K chain slots on the same matrix."""
    import torch
    from bess_b200.engine import GpuEngine
    m, y, _ = make(n, p, density, 3)
    fold = (np.arange(n) % K).astype(np.int32)
    e = GpuEngine()
    e.load_csc((m.indptr.astype(np.int64), m.indices.astype(np.int32), m.data, m.shape), y, np.ones(n), 1)
    e.normalize(1, True)
    e.setup_chains(K, fold, 4)
    cms, cby = e.time_dual_sweep(20)
    e.close()
    xd = torch.sparse_csc_tensor(torch.as_tensor(m.indptr.astype(np.int64)), torch.as_tensor(m.indices.astype(np.int64)),
                                 torch.as_tensor(m.data), size=m.shape).cuda().to_dense().contiguous()
    e = GpuEngine()
    e.load(None, y, np.ones(n), 1, x_device_ptr=xd.data_ptr(), n=n, p=p)
    e.normalize(1, True)
    e.setup_chains(K, fold, 4)
    dms, dby = e.time_dual_sweep(20)
    e.close()
    del xd
    torch.cuda.empty_cache()
    return dict(density=density, csc_sweep_ms=cms, csc_bytes=cby, csc_share_of_hbm=cby / (cms * 1e-3) / HBM,
                dense_sweep_ms=dms, dense_bytes=dby, dense_share_of_hbm=dby / (dms * 1e-3) / HBM,
                dense_over_csc_bytes=dby / cby, speedup=dms / cms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="r03d")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="profiles")
    a = ap.parse_args()
    from bess_b200 import _lib
    _lib.require_gpu()
    res = dict(card=card(), workloads=[], crossover=[])
    seq = np.arange(1, 21)
    for dens in (0.001, 0.01, 0.05, 0.2):
        res["crossover"].append(sweep_crossover(1000, 500_000, dens, 10))
        print(json.dumps(res["crossover"][-1]), flush=True)
    for dens in (0.001, 0.01, 0.05, 0.2):
        m, y, _ = make(1000, 500_000, dens, 1)
        res["workloads"].append(workload(f"c5b_gaussian_{dens}", m, y, "gaussian", True, seq, a.reps))
        print(json.dumps(res["workloads"][-1])[:400], flush=True)
    for fam in ("binomial", "cox"):
        m, y, _ = make(2000, 200_000, 0.01, 2, fam)
        res["workloads"].append(workload(f"{fam}_2000x200000", m, y, fam, True, np.arange(1, 11), a.reps))
        print(json.dumps(res["workloads"][-1])[:400], flush=True)
    m, y = make_powerlaw(20_000, 200_000, 5)
    res["workloads"].append(workload("powerlaw_gaussian_20000x200000", m, y, "gaussian", True, np.arange(1, 11), a.reps))
    print(json.dumps(res["workloads"][-1])[:400], flush=True)
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, f"{a.tag}_sparse_path.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1, default=float)
    print("wrote", path)


if __name__ == "__main__":
    main()

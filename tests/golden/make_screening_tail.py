"""Cases of tests/test_screening_tail.py and the maker of their golden, tests/golden/screening/screening_tail.npz.

Each case loads a seeded design into a GpuEngine, screens it (marginal utilities, top-`size`, kept columns gathered),
normalises it and reads back what the fit will see: the kept-column list, the column means and norms, and the screened,
normalised design (stored as its SHA-256, since at n = 1000 and size = 5000 it is 40 MB).  The shapes cover the screening
of the benchmark's largest configuration at a smaller p, an odd screening size (padded row length) with non-unit
weights, the binomial and poisson utilities, always_select pins, a design too tall for the gather to be staged in shared
memory, and no normalisation at all.  The golden holds what a build of the library returned, to be matched bit for bit.

  python tests/golden/make_screening_tail.py [--root TREE] [--out FILE]

--root picks the source tree whose bess_b200 package computes the golden (default: this repository).
"""
import argparse
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))

# name -> n, p, screening size, model_type, data_type, is_normal, unit weights, always_select
CASES = {
    "lm_n1000_p100k": (1000, 100_000, 5000, 1, 1, True, True, ()),
    "lm_odd_size_weights": (600, 20_000, 777, 1, 1, True, False, ()),
    "logit_weights_pins": (400, 9_000, 301, 2, 2, True, False, (5, 4000, 8999)),
    "poisson": (500, 6_000, 250, 3, 2, True, True, ()),
    "lm_tall_unfused": (4000, 3_000, 400, 1, 1, True, False, ()),
    "lm_not_normal": (300, 4_000, 123, 1, 1, False, True, ()),
}


def make_problem(name):
    n, p, _, model_type, _, _, unit_w, _ = CASES[name]
    rng = np.random.Generator(np.random.PCG64(1000 + sum(map(ord, name))))
    x = rng.standard_normal((n, p))
    cols = rng.choice(p, 10, replace=False)
    eta = x[:, cols] @ rng.uniform(0.5, 1.5, 10)
    if model_type == 1:
        y = eta + rng.standard_normal(n)
    elif model_type == 2:
        y = (rng.uniform(size=n) < 1.0 / (1.0 + np.exp(-0.5 * eta))).astype(np.float64)
    else:
        y = rng.poisson(np.exp(0.2 * eta / np.abs(eta).max())).astype(np.float64)
    w = np.ones(n) if unit_w else rng.uniform(0.5, 2.0, n)
    return x, y, w


def run_case(name, engine):
    _, _, size, model_type, data_type, is_normal, _, always = CASES[name]
    x, y, w = make_problem(name)
    eng = engine.GpuEngine()
    try:
        eng.load(x, y, w, model_type)
        sel = eng.screen(size, always)
        xm, xn, ym = eng.normalize(data_type, is_normal)
        xs = np.ascontiguousarray(eng.design())
    finally:
        eng.close()
    return {"sel": np.asarray(sel, dtype=np.int64), "x_mean": xm, "x_norm": xn, "y_mean": np.array([ym]),
            "design_sha256": np.frombuffer(hashlib.sha256(xs.tobytes()).digest(), dtype=np.uint8),
            "design_shape": np.array(xs.shape)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=REPO)
    ap.add_argument("--out", default=os.path.join(HERE, "screening", "screening_tail.npz"))
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    from bess_b200 import engine
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    blob = {}
    for name in CASES:
        res = run_case(name, engine)
        for k, v in res.items():
            blob[f"{name}/{k}"] = v
        print(name, "kept", res["sel"].size, "first", res["sel"][:5].tolist(), flush=True)
    np.savez_compressed(args.out, **blob)


if __name__ == "__main__":
    main()

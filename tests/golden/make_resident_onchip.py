"""Cases of tests/test_resident_onchip.py and the maker of their golden, tests/golden/onchip/resident_onchip.npz.

Each case is a seeded gen_data problem (gaussian, 10-fold CV, sequential path) that the resident PDAS kernel
(lm_path.cu) runs, shaped to cover the sweepers' on-chip slices: wholly on chip, partly on chip, almost nothing on chip
(n near the largest the owner budget admits), odd p with uneven and empty slices, many columns with alike sacrifices (long
candidate lists for the ranking to narrow), and duplicated columns whose sacrifices tie exactly.  The golden holds what a build of
the library returned for them, to be matched bit for bit.

  python tests/golden/make_resident_onchip.py [--root TREE] [--out FILE]

--root picks the source tree whose bess_b200 package computes the golden (default: this repository).
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))

# name -> n, p, support size of the truth, s_max, design transform
CASES = {
    "whole_slice": (200, 400, 5, 10, None),
    "part_slice": (1000, 5000, 10, 20, None),
    "large_n": (4700, 2100, 2, 2, None),
    "odd_p_empty_slices": (300, 301, 5, 10, None),
    "shared_factor": (300, 6000, 0, 20, None),
    "dup_columns": (400, 1200, 5, 5, "dup"),
}
OUTPUTS = ("beta", "coef0", "train_loss", "ic", "s", "beta_all", "coef0_all", "loss_all", "ic_all", "l_all")


def make_problem(name):
    from bess_b200.gen_data import gen_data
    n, p, k, _, tr = CASES[name]
    if k == 0:
        # no sparse truth: y follows a factor that 2000 columns share, so their sacrifices are alike and many of them pass
        # a candidate threshold
        rng = np.random.Generator(np.random.PCG64(7))
        x = rng.standard_normal((n, p))
        f = rng.standard_normal(n)
        x[:, :2000] = f[:, None] + 0.3 * x[:, :2000]
        return x, 2.0 * f + rng.standard_normal(n)
    if tr == "dup":
        # noise columns in identical pairs (their sacrifices tie bit for bit, so the candidate lists hold exact ties), the
        # k signal columns last and unique; s_max = k keeps the ties off the selection boundary, where the library would
        # repeat the call on the multi-kernel path to resolve them the reference's way
        rng = np.random.Generator(np.random.PCG64(11))
        x = rng.standard_normal((n, p))
        x[:, 1:p - k:2] = x[:, 0:p - k - 1:2]
        beta = rng.uniform(2.0, 4.0, k)
        return x, x[:, p - k:] @ beta + rng.standard_normal(n)
    d = gen_data(n, p, "gaussian", k, seed=100 + n + p)
    return d.x, d.y


def run_case(name, cbess):
    n, p, _, smax, _ = CASES[name]
    x, y = make_problem(name)
    out = cbess.fit(x, y, 1, np.ones(n), True, 1, 1, 20, 2, 1, True, 1, True, 10, np.arange(1, smax + 1), 1, smax, False, 1,
                    cv_seed=123)
    res = {k: np.atleast_1d(np.asarray(out[k], dtype=np.float64)) for k in OUTPUTS if out.get(k) is not None}
    resident = out["stats"]["resident"]
    res["resident_launches"] = np.array([resident[0]])
    res["select_fallbacks"] = np.array([resident[2]])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=REPO)
    ap.add_argument("--out", default=os.path.join(HERE, "onchip", "resident_onchip.npz"))
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    from bess_b200 import cbess
    blob = {}
    for name in CASES:
        res = run_case(name, cbess)
        for k, v in res.items():
            blob[f"{name}/{k}"] = v
        print(name, "resident launches", res["resident_launches"][0], "fallbacks", res["select_fallbacks"][0],
              "s", res["s"][0], flush=True)
    np.savez_compressed(args.out, **blob)


if __name__ == "__main__":
    main()

"""Cases of tests/test_resident_round.py and the maker of their golden, tests/golden/onchip/resident_round.npz.

Each seeded gaussian case runs the resident kernel (lm_path.cu) at one edge of its round: the sweepers' on-chip rows and
streamed rows, the phase barriers and the termination word that their waits read, chains that finish at different
phases.  The golden holds what the previous build returned (the termination word read by every thread after a second
barrier wait, the residual mirrored into G every phase), to be matched bit for bit:

  rows_all_streamed   n so large that almost no row stays on chip
  rows_all_on_chip    every row on chip, nothing streamed
  one_stream_group    every row on chip but the last few
  odd_n_many_groups   odd n, most rows streamed
  uneven_slices       p giving slices of different widths and sweepers without columns
  tied_columns        duplicated columns whose sacrifices tie exactly
  early_finisher      a short path on which chains finish while the other group is still being swept
  swapping_columns    columns with alike sacrifices that leave the active set and come back while still cached

  python tests/golden/make_resident_round.py [--root TREE] [--out FILE]

--root picks the source tree whose bess_b200 package computes the golden (default: this repository).
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))

# name -> n, p, support size of the truth, s_max, K (0: no CV), always_select, design transform
CASES = {
    "rows_all_streamed": (4720, 2000, 2, 2, 10, (), None),
    "rows_all_on_chip": (256, 400, 5, 10, 10, (), None),
    "one_stream_group": (200, 400, 5, 10, 10, (), None),
    "odd_n_many_groups": (999, 5000, 10, 20, 10, (), None),
    "uneven_slices": (301, 587, 5, 10, 10, (), None),
    "tied_columns": (400, 1200, 5, 5, 10, (), "dup"),
    "early_finisher": (600, 1500, 3, 4, 5, (), None),
    "swapping_columns": (400, 3000, 0, 15, 10, (), "factor"),
}
OUTPUTS = ("beta", "coef0", "train_loss", "ic", "s", "beta_all", "coef0_all", "loss_all", "ic_all", "l_all")


def make_problem(name):
    from bess_b200.gen_data import gen_data
    n, p, k, _, _, _, tr = CASES[name]
    if tr == "factor":
        # no sparse truth: 1000 columns share a factor of y, so their sacrifices are alike and the active sets churn
        rng = np.random.Generator(np.random.PCG64(17))
        x = rng.standard_normal((n, p))
        f = rng.standard_normal(n)
        x[:, :1000] = f[:, None] + 0.3 * x[:, :1000]
        return x, 2.0 * f + rng.standard_normal(n)
    if tr == "dup":
        # noise columns in identical pairs, the k signal columns last and unique (as in make_resident_onchip.py)
        rng = np.random.Generator(np.random.PCG64(13))
        x = rng.standard_normal((n, p))
        x[:, 1:p - k:2] = x[:, 0:p - k - 1:2]
        beta = rng.uniform(2.0, 4.0, k)
        return x, x[:, p - k:] @ beta + rng.standard_normal(n)
    d = gen_data(n, p, "gaussian", k, seed=300 + n + p)
    return d.x, d.y


def run_case(name, cbess):
    n, p, _, smax, K, always, _ = CASES[name]
    x, y = make_problem(name)
    out = cbess.fit(x, y, 1, np.ones(n), True, 1, 1, 20, 2, 1, True, 1, K > 0, max(K, 1), np.arange(1, smax + 1), 1, smax,
                    False, 1, always_select=always, cv_seed=123)
    res = {k: np.atleast_1d(np.asarray(out[k], dtype=np.float64)) for k in OUTPUTS if out.get(k) is not None}
    resident = out["stats"]["resident"]
    res["resident_launches"] = np.array([resident[0]])
    res["select_fallbacks"] = np.array([resident[2]])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=REPO)
    ap.add_argument("--out", default=os.path.join(HERE, "onchip", "resident_round.npz"))
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

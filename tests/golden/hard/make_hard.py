"""Generates tests/golden/hard/*.npz from the REAL reference (oracle/_ref/libbess_ref.so): the designs the first round's
goldens (iid N(0,1) columns) did not cover.

  ties_*   exactly duplicated NOISE columns: every noise pair has bit-equal sacrifices / screening utilities, so the first
           sparsity level past the true support -- and the screening cut -- is a BOUNDARY TIE that the reference leaves to
           std::nth_element (utilities.cpp:179-188).  s.list stops before both copies of a pair can enter the active set
           (a duplicated active column makes the Gram singular: a different row of the scope table).
  ar*_ / band_*  correlated designs: rows ~ MVN(0, Sigma), Sigma_jk = rho^|j-k| with rho = 0.5 / 0.9 (gen.data cortype 2,
           R/R/gen.data.R:110-118) and the banded design of the Python generator (python/bess/gen_data.py:25-30, rho = 0.5):
           small boundary gaps, ill-conditioned Grams.
  k20_ / iter_   20 CV folds; max_iter = 100 (more than the 64 the first round's workspaces allowed).

Run in the build container only:  python tests/golden/hard/make_hard.py [names...]"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, ROOT)
from bess_b200.gen_data import gen_data, gen_data_reference  # noqa: E402
from oracle import ref  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
FAM = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}  # family -> (model_type, data_type)


def ar1_design(n, p, rho, rng):
    z = rng.standard_normal((n, p))
    x = np.empty((n, p))
    x[:, 0] = z[:, 0]
    s = np.sqrt(1.0 - rho * rho)
    for j in range(1, p):
        x[:, j] = rho * x[:, j - 1] + s * z[:, j]
    return x


def banded_design(n, p, rho, rng):
    X = rng.standard_normal((n, p))
    X = X - X.mean(axis=0, keepdims=True)
    X = np.sqrt(n) * X / np.sqrt((X ** 2).sum(axis=0, keepdims=True))
    zero = np.zeros((n, 1))
    return X + rho * (np.hstack((zero, X[:, 0:(p - 2)], zero)) + np.hstack((zero, X[:, 2:p], zero)))


def dupsig_design(n, p_true, p_noise, rng):
    """[true columns | exact copies of the true columns | noise columns]: with COLD starts every level's first selection
    (beta = 0: the copies tie with the originals at the top of the ranking) puts both copies of a signal column into the
    active set -- a singular Gram that the reference's colPivHouseholderQr / pivoted ldlt truncate (Algorithm.h:1134, 1171)."""
    base = rng.standard_normal((n, p_true + p_noise))
    return np.ascontiguousarray(np.hstack((base[:, :p_true], base[:, :p_true], base[:, p_true:])))


def dup_design(n, p_true, p_noise, rng):
    """[true columns | noise columns | exact copies of the noise columns]"""
    base = rng.standard_normal((n, p_true + p_noise))
    return np.ascontiguousarray(np.hstack((base, base[:, p_true:])))


# name: (family, design, n, p, k, path_type, is_cv, K, ic_type, smax, screening, weighted, max_iter, seed)
CASES = {
    "ties_lm_seq_gic": ("gaussian", ("dup", 5, 60), 150, 125, 5, 1, False, 5, 3, 6, 0, False, 20, 101),
    "ties_lm_seq_cv": ("gaussian", ("dup", 4, 50), 160, 104, 4, 1, True, 5, 1, 5, 0, False, 20, 102),
    "ties_lm_screen": ("gaussian", ("dup", 5, 95), 150, 195, 5, 1, False, 5, 3, 6, 50, False, 20, 103),
    "ties_logit_seq_gic": ("binomial", ("dup", 3, 40), 200, 83, 3, 1, False, 5, 3, 4, 0, False, 20, 104),
    "ties_cox_seq_gic": ("cox", ("dup", 3, 40), 160, 83, 3, 1, False, 5, 3, 4, 0, False, 20, 105),
    "ties_lm_gs_cv": ("gaussian", ("dup", 6, 40), 160, 86, 6, 2, True, 4, 1, 7, 0, True, 20, 106),
    "ar5_lm_seq_cv": ("gaussian", ("ar", 0.5), 200, 400, 6, 1, True, 5, 1, 12, 0, False, 20, 111),
    "ar9_lm_seq_gic": ("gaussian", ("ar", 0.9), 200, 400, 6, 1, False, 5, 3, 12, 0, False, 20, 112),
    "ar9_lm_gs_cv": ("gaussian", ("ar", 0.9), 200, 300, 5, 2, True, 5, 1, 14, 0, True, 20, 113),
    "ar9_logit_seq_cv": ("binomial", ("ar", 0.9), 300, 250, 4, 1, True, 4, 1, 8, 0, False, 20, 114),
    "ar5_poisson_gs_gic": ("poisson", ("ar", 0.5), 250, 250, 4, 2, False, 5, 3, 10, 0, False, 20, 115),
    "ar9_cox_seq_cv": ("cox", ("ar", 0.9), 200, 200, 4, 1, True, 3, 1, 7, 0, False, 20, 116),
    "ar9_lm_screen": ("gaussian", ("ar", 0.9), 150, 1000, 5, 1, False, 5, 4, 8, 120, False, 20, 117),
    "band_lm_seq_cv": ("gaussian", ("band", 0.5), 200, 300, 5, 1, True, 5, 1, 10, 0, False, 20, 121),
    "band_logit_gs_cv": ("binomial", ("band", 0.5), 250, 200, 4, 2, True, 4, 1, 10, 0, False, 20, 122),
    "k20_lm_seq_cv": ("gaussian", ("ar", 0.5), 240, 200, 5, 1, True, 20, 1, 8, 0, False, 20, 131),
    "k20_logit_seq_cv": ("binomial", ("ar", 0.5), 300, 150, 4, 1, True, 20, 1, 6, 0, False, 20, 132),
    "iter_lm_seq_gic": ("gaussian", ("ar", 0.9), 150, 300, 8, 1, False, 5, 3, 14, 0, False, 100, 133),
    # rank-deficient active sets (cold starts; see dupsig_design).  Which copy of a duplicated column a singular solve keeps
    # follows the reference's pivot order (reproducible for these seeds: Eigen's positional LDLT pivoting; for other draws
    # the reference's choice between the two equivalent copies rides on rounding noise -- e.g. seed 12 with 4 signal
    # columns agrees on the chosen model but not on every level of the trace, poisson / cox not at all -- no golden there)
    "dupsig_lm_seq_gic": ("gaussian", ("dupsig", 3, 40), 150, 46, 3, 1, False, 4, 3, 7, 0, False, 20, 7),
    "dupsig_lm_gs_gic": ("gaussian", ("dupsig", 3, 40), 150, 46, 3, 2, False, 4, 3, 7, 0, False, 20, 7),
    "dupsig_lm_seq_cv": ("gaussian", ("dupsig", 3, 40), 150, 46, 3, 1, True, 4, 1, 7, 0, False, 20, 7),
    "dupsig_logit_seq_gic": ("binomial", ("dupsig", 3, 40), 150, 46, 3, 1, False, 4, 3, 7, 0, False, 20, 7),
    "dupsig_logit_seq_cv": ("binomial", ("dupsig", 3, 40), 150, 46, 3, 1, True, 4, 1, 7, 0, False, 20, 7),
}
COLD = {name for name in CASES if name.startswith("dupsig_")}


def build(name):
    fam, design, n, p, k, path_type, is_cv, K, ic_type, smax, scr, weighted, max_iter, seed = CASES[name]
    rng = np.random.Generator(np.random.PCG64(seed))
    if design[0] == "dupsig":
        base = rng.standard_normal((n, design[1] + design[2]))
        x = np.ascontiguousarray(np.hstack((base[:, :design[1]], base[:, :design[1]], base[:, design[1]:])))
        assert x.shape[1] == p
        d = gen_data(n, design[1], fam, k, seed=seed, x=np.ascontiguousarray(base[:, :design[1]]))
        return x, d.y
    if design[0] == "dup":
        x = dup_design(n, design[1], design[2], rng)
        assert x.shape[1] == p
        d = gen_data(n, design[1], fam, k, seed=seed, x=np.ascontiguousarray(x[:, :design[1]]))  # response from the true columns only
        y = d.y
        if fam == "cox":
            # rows must be time-sorted consistently for ALL columns: redo the draw on the full design
            tb = np.zeros(p)
            tb[:design[1]] = d.beta
            time = (-np.log(rng.uniform(size=n)) / np.exp(x @ tb)) ** 0.1
            ctime = 10.0 * rng.uniform(size=n)
            status = (time < ctime).astype(np.float64)
            order = np.argsort(np.minimum(time, ctime), kind="stable")
            x, y = np.ascontiguousarray(x[order]), status[order]
        elif fam == "poisson":
            x = x / 16.0
    else:
        x = ar1_design(n, p, design[1], rng) if design[0] == "ar" else banded_design(n, p, design[1], rng)
        d = gen_data(n, p, fam, k, seed=seed, x=x)
        x, y = d.x, d.y
    return x, y


def main():
    only = set(sys.argv[1:])
    for name, (fam, design, n, p, k, path_type, is_cv, K, ic_type, smax, scr, weighted, max_iter, seed) in CASES.items():
        if only and name not in only:
            continue
        model_type, data_type = FAM[fam]
        x, y = build(name)
        rng = np.random.Generator(np.random.PCG64(5000 + seed))
        w = rng.uniform(0.5, 1.5, n) if weighted else np.ones(n)
        seq = np.arange(1, smax + 1, dtype=np.int32)
        fold = ref.cv_fold_ids(n, K) if is_cv else np.zeros(n, dtype=np.int32)
        warm = name not in COLD
        r = ref.pywrap_bess(x, y, data_type, w, True, 1, model_type, max_iter, 2, path_type, warm, ic_type, is_cv, K,
                            seq, 1, smax, scr > 0, scr if scr > 0 else 1)
        out = dict(x=x, y=y, weight=w, fold_of_row=fold, beta=r["beta"], coef0=r["coef0"], train_loss=r["train_loss"], ic=r["ic"],
                   meta=np.array([model_type, data_type, path_type, int(is_cv), K, ic_type, smax, scr], dtype=np.int64),
                   max_iter=np.int64(max_iter), warm=np.int64(warm))
        if scr > 0:
            out["screening_A"] = ref.screening(x, y, w, model_type, scr)
        elif path_type == 1:
            t = ref.seq_trace(x, y, w, data_type, True, model_type, max_iter, warm, ic_type, is_cv, K, seq)
            out.update({k2: v for k2, v in t.items()})
        if x.nbytes > (1 << 20):  # too large to store: tests/helpers.py regenerates it with build() and checks the hash
            out["x_sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest())
            del out["x"]
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
        print(name, "support", np.nonzero(r["beta"])[0].tolist(), "ic", r["ic"], flush=True)


if __name__ == "__main__":
    main()

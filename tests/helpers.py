"""Shared helpers for the parity tests."""
import glob
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-8  # north_star: coefficients and losses within 1e-8 relative in fp64


def golden_names():
    return sorted(os.path.splitext(os.path.basename(f))[0] for f in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    m = g["meta"]
    g["model_type"], g["data_type"], g["path_type"], g["is_cv"], g["K"], g["ic_type"], g["smax"], g["scr"] = (
        int(m[0]), int(m[1]), int(m[2]), bool(m[3]), int(m[4]), int(m[5]), int(m[6]), int(m[7]))
    g["lambda_seq"] = g.get("lambda_seq", np.zeros(1))
    return g


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    scale = max(np.max(np.abs(b)) if b.size else 0.0, 1e-300)
    return float(np.max(np.abs(a - b)) / scale) if a.size else 0.0


def assert_same_support(beta_a, beta_b):
    sa = np.nonzero(beta_a)[0]
    sb = np.nonzero(beta_b)[0]
    assert sa.tolist() == sb.tolist(), f"support differs: {sa.tolist()} vs {sb.tolist()}"


# The five BASELINE configs at full size (tests/golden/full/*.npz, made by tests/golden/make_full_size.py from the real
# reference).  name -> family, n, p, k, path_type, is_cv, K, ic_type, s_min, s_max, screening_size, data seed
FULL_CONFIGS = {
    "c1": ("gaussian", 500, 1000, 10, 1, False, 5, 3, 1, 20, 0, 1),
    "c1cv": ("gaussian", 500, 1000, 10, 1, True, 10, 1, 1, 20, 0, 1),
    "c2": ("binomial", 2000, 20000, 20, 2, True, 10, 1, 1, 263, 0, 2),
    "c3": ("poisson", 5000, 50000, 30, 1, False, 5, 3, 1, 40, 0, 3),
    "c4": ("cox", 2000, 10000, 15, 1, True, 5, 1, 1, 30, 0, 4),
    "c5": ("gaussian", 1000, 500000, 10, 1, True, 10, 1, 1, 20, 5000, 5),
}


def full_checksum(d):
    """Cheap fingerprint of the regenerated inputs (guards against a numpy RNG stream change)."""
    return np.array([float(d.x[::7, ::13].sum()), float(np.abs(d.x[-1]).sum()), float(d.y.sum())])


def load_full_golden(name):
    path = os.path.join(GOLDEN_DIR, "full", name + ".npz")
    return dict(np.load(path)) if os.path.exists(path) else None


PGS_DIR = os.path.join(GOLDEN_DIR, "pgs")


def pgs_golden_names():
    return sorted(os.path.splitext(os.path.basename(f))[0] for f in glob.glob(os.path.join(PGS_DIR, "*.npz")))


def load_pgs_golden(name):
    """tests/golden/pgs/*.npz (made by tests/golden/pgs/make_pgs.py from the real reference's pgs_path)."""
    g = dict(np.load(os.path.join(PGS_DIR, name + ".npz")))
    (g["model_type"], g["data_type"], g["powell_path"], g["is_cv"], g["K"], g["ic_type"], g["s_min"], g["s_max"],
     g["n_lambda"], g["warm"]) = (int(v) for v in g["meta"])
    g["is_cv"], g["warm"] = bool(g["is_cv"]), bool(g["warm"])
    g["lambda_min"], g["lambda_max"] = (float(v) for v in g["lambda_range"])
    n = g["x"].shape[0]
    g["full_fits"] = g["fits"][g["fits"][:, 2] == n][:, :2]  # (sparsity level, lambda) of the full-data fits, in order
    return g


GROUP_DIR = os.path.join(GOLDEN_DIR, "group")


def group_golden_names():
    return sorted(os.path.splitext(os.path.basename(f))[0] for f in glob.glob(os.path.join(GROUP_DIR, "*.npz")))


def load_group_golden(name):
    """tests/golden/group/*.npz (made by tests/golden/group/make_group.py from the real reference, gsize > 1)."""
    g = dict(np.load(os.path.join(GROUP_DIR, name + ".npz")))
    (g["model_type"], g["data_type"], g["algorithm_type"], g["path_type"], g["is_cv"], g["K"], g["ic_type"], g["s_min"],
     g["s_max"], g["pgs"], g["n_lambda"], g["powell_path"]) = (int(v) for v in g["meta"])
    g["is_cv"], g["pgs"] = bool(g["is_cv"]), bool(g["pgs"])
    g["seq"] = np.arange(g["s_min"], g["s_max"] + 1)
    if g["pgs"]:
        g["kw"] = dict(lambda_min=float(g["lambdas"][0]), lambda_max=float(g["lambdas"][1]), n_lambda=g["n_lambda"],
                       powell_path=g["powell_path"])
    else:
        g["kw"] = dict(lambda_seq=g["lambdas"])
    return g


HARD_DIR = os.path.join(GOLDEN_DIR, "hard")


def hard_golden_names():
    return sorted(os.path.splitext(os.path.basename(f))[0] for f in glob.glob(os.path.join(HARD_DIR, "*.npz")))


def load_hard_golden(name):
    """tests/golden/hard/*.npz (made by tests/golden/hard/make_hard.py from the real reference): boundary ties from
    duplicated columns, correlated designs (rho = 0.5 / 0.9, banded), 20 folds, max_iter = 100, and dupsig_*: duplicated
    SIGNAL columns under cold starts -- both copies enter the active set, the Gram is singular, the reference's
    colPivHouseholderQr / pivoted ldlt truncate."""
    g = dict(np.load(os.path.join(HARD_DIR, name + ".npz")))
    if "x" not in g:  # a design too large to store: regenerated from its seed, checked against the stored hash
        g["x"] = _regenerate_hard_design(name, str(g["x_sha256"]))
    m = g["meta"]
    g["model_type"], g["data_type"], g["path_type"], g["is_cv"], g["K"], g["ic_type"], g["smax"], g["scr"] = (
        int(m[0]), int(m[1]), int(m[2]), bool(m[3]), int(m[4]), int(m[5]), int(m[6]), int(m[7]))
    g["max_iter"] = int(g["max_iter"])
    g["warm"] = bool(g["warm"]) if "warm" in g else True  # dupsig_*: cold starts (rank-deficient active sets)
    return g


def _regenerate_hard_design(name, sha256):
    import hashlib
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_hard", os.path.join(HARD_DIR, "make_hard.py"))
    make_hard = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(make_hard)
    x = np.ascontiguousarray(make_hard.build(name)[0])
    assert hashlib.sha256(x.tobytes()).hexdigest() == sha256, f"the regenerated design of {name} is not the stored one"
    return x


def fold_duplicates(x, beta):
    """Coefficients summed over exactly duplicated columns of x onto the first copy (the last axis of beta indexes the
    columns).  Two models that differ only in WHICH copy of a duplicated column carries the coefficient are the same
    function of the data; the reference's own choice rides on its pivot order (tests/golden/hard/make_hard.py)."""
    beta = np.array(beta, dtype=np.float64, copy=True)
    first = {}
    for j in range(x.shape[1]):
        key = x[:, j].tobytes()
        if key in first:
            beta[..., first[key]] += beta[..., j]
            beta[..., j] = 0.0
        else:
            first[key] = j
    return beta

"""CPU: the numpy oracle (oracle/pdas_oracle.py) against the golden vectors produced by the real reference."""
import subprocess

import numpy as np
import pytest

from oracle import pdas_oracle as orc
from tests.helpers import (RTOL, assert_same_support, fold_duplicates, golden_names, group_golden_names, hard_golden_names, load_golden,
                           load_group_golden, load_hard_golden, load_pgs_golden, pgs_golden_names, rel_err)


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_reference_golden(name):
    g = load_golden(name)
    seq = np.arange(1, g["smax"] + 1)
    out = orc.bess_cpp(g["x"], g["y"], g["data_type"], g["weight"], True, g["model_type"], 20, g["path_type"], True,
                       g["ic_type"], g["is_cv"], g["K"], seq, 1, g["smax"], g["scr"] > 0, max(g["scr"], 1),
                       fold_of_row=g["fold_of_row"], lambda_seq=g["lambda_seq"])
    assert_same_support(out["beta"], g["beta"])
    assert rel_err(out["beta"], g["beta"]) < RTOL
    assert abs(out["coef0"] - g["coef0"]) <= RTOL * max(1.0, abs(g["coef0"]))
    assert abs(out["train_loss"] - g["train_loss"]) <= RTOL * abs(g["train_loss"])
    assert abs(out["ic"] - g["ic"]) <= RTOL * abs(g["ic"])
    if "screening_A" in g:
        assert out["screening_A"].tolist() == g["screening_A"].tolist()
    if "beta_all" in g:  # per-level trace of the sequential path
        for lvl in range(len(seq)):
            assert_same_support(out["beta_all"][lvl], g["beta_all"][lvl])
        assert rel_err(out["beta_all"], g["beta_all"]) < RTOL
        assert rel_err(out["ic_all"], g["ic_all"]) < RTOL
        assert rel_err(out["loss_all"], g["loss_all"]) < RTOL
        assert out["l_all"].tolist() == g["l_all"].tolist()
    assert out["min_gap"] > 1e-9, "a top-k decision sits inside rounding noise"


@pytest.mark.parametrize("name", hard_golden_names())
def test_oracle_matches_reference_on_ties_and_correlated_designs(name):
    """Duplicated columns (boundary ties at the first level past the true support and at the screening cut: the oracle
    asks the compiled reference's max_k, utilities.cpp:179-188), rho = 0.5 / 0.9 and banded designs, 20 folds, max_iter 100."""
    g = load_hard_golden(name)
    seq = np.arange(1, g["smax"] + 1)
    orc.TIES["count"] = orc.TIES["unresolved"] = 0
    out = orc.bess_cpp(g["x"], g["y"], g["data_type"], g["weight"], True, g["model_type"], g["max_iter"], g["path_type"],
                       g["warm"], g["ic_type"], g["is_cv"], g["K"], seq, 1, g["smax"], g["scr"] > 0, max(g["scr"], 1),
                       fold_of_row=g["fold_of_row"])
    assert_same_support(out["beta"], g["beta"])
    assert rel_err(out["beta"], g["beta"]) < RTOL
    assert abs(out["coef0"] - g["coef0"]) <= RTOL * max(1.0, abs(g["coef0"]))
    assert abs(out["train_loss"] - g["train_loss"]) <= RTOL * abs(g["train_loss"])
    assert abs(out["ic"] - g["ic"]) <= RTOL * abs(g["ic"])
    if "screening_A" in g:
        assert out["screening_A"].tolist() == g["screening_A"].tolist()
    if "beta_all" in g and name.startswith("dupsig_"):
        # per level: the same model up to which copy of a duplicated column carries the coefficient
        ob, gb = fold_duplicates(g["x"], out["beta_all"]), fold_duplicates(g["x"], g["beta_all"])
        for lvl in range(len(seq)):
            assert_same_support(ob[lvl], gb[lvl])
        assert rel_err(ob, gb) < RTOL
    elif "beta_all" in g:
        for lvl in range(len(seq)):
            assert_same_support(out["beta_all"][lvl], g["beta_all"][lvl])
        assert rel_err(out["beta_all"], g["beta_all"]) < RTOL
        assert out["l_all"].tolist() == g["l_all"].tolist()
    if name.startswith("ties_"):
        assert orc.TIES["count"] > 0  # the case does exercise the reference's tie rule
    elif not name.startswith("dupsig_"):  # (a duplicated signal pair ties INSIDE the selection, not at its boundary ...
        assert orc.TIES["count"] == 0     #  ... but the copies' noise twins may)


def test_rank_revealing_solve_truncates_like_the_reference():
    """solve_rank_revealing on a Gram with an exactly duplicated column: one copy carries the coefficient of the reduced
    system, the other gets 0 (Eigen's pivoted ldlt skips the exactly zero pivot, LDLT.h:558-592; colPivHouseholderQr
    truncates, Algorithm.h:1134); a full-rank system is solved as before."""
    rng = np.random.default_rng(3)
    X = rng.standard_normal((80, 5))
    Xd = np.hstack([X, X[:, [1]]])
    y = rng.standard_normal(80)
    b = orc.solve_rank_revealing(Xd.T @ Xd, Xd.T @ y)
    full = np.linalg.solve(X.T @ X, X.T @ y)
    assert (b[1] == 0.0) != (b[5] == 0.0)
    assert np.allclose(np.r_[b[:5]] + np.r_[0, b[5], 0, 0, 0], full, rtol=1e-10)
    assert np.allclose(orc.solve_rank_revealing(X.T @ X, X.T @ y), full, rtol=1e-12)


def test_max_k_ties_follow_libstdcxx_nth_element(tmp_path):
    """The oracle's max_k resolves boundary ties by replaying std::nth_element; here the real one (compiled with g++, the
    reference's utilities.cpp:179-188 statement for statement) decides the same sets on tie-heavy keys of many sizes."""
    src = tmp_path / "max_k.cpp"
    src.write_text(r'''
#include <algorithm>
#include <cstdio>
#include <numeric>
#include <vector>
int main() {
    int n, k;
    while (std::scanf("%d %d", &n, &k) == 2) {
        std::vector<double> v(n);
        for (double &x : v) if (std::scanf("%lf", &x) != 1) return 1;
        std::vector<int> ind(n);
        std::iota(ind.begin(), ind.end(), 0);
        auto rule = [&v](int i, int j) -> bool { return v[i] > v[j]; };
        std::nth_element(ind.data(), ind.data() + k, ind.data() + ind.size(), rule);
        std::sort(ind.data(), ind.data() + k);
        for (int i = 0; i < k; i++) std::printf("%d ", ind[i]);
        std::printf("\n");
    }
    return 0;
}
''')
    exe = tmp_path / "max_k"
    r = subprocess.run(["g++", "-std=c++11", "-O2", str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    rng = np.random.default_rng(11)
    cases = []
    for t in range(1500):
        n = int(rng.integers(2, 12 if t % 3 == 0 else 600))
        cases.append((np.floor(rng.random(n) * rng.integers(1, 9)), int(rng.integers(1, n))))
    text = "".join(f"{v.size} {k} " + " ".join(repr(float(x)) for x in v) + "\n" for v, k in cases)
    run = subprocess.run([str(exe)], input=text, capture_output=True, text=True, timeout=120)
    lines = run.stdout.splitlines()
    assert run.returncode == 0 and len(lines) == len(cases)
    for (v, k), line in zip(cases, lines):
        assert orc.max_k(v, k).tolist() == [int(s) for s in line.split()], (v.tolist(), k)


# poisson_seq_gic is left to the GPU suite: its IRLS fits run away to huge counts and take a minute in numpy
@pytest.mark.parametrize("name", [n for n in pgs_golden_names() if n != "poisson_seq_gic"])
def test_oracle_pgs_path_matches_reference(name):
    """pgs_path (path.cpp:1138-1309): Powell search over (s, lambda).  The order of the evaluated (s, lambda) points is
    checked too -- the search is stateful (warm starts, stale records), so a wrong turn cannot cancel out."""
    g = load_pgs_golden(name)
    out = orc.bess_cpp(g["x"], g["y"], g["data_type"], g["weight"], True, g["model_type"], 20, 2, g["warm"], g["ic_type"],
                       g["is_cv"], g["K"], [1], g["s_min"], g["s_max"], False, 1, fold_of_row=g["fold_of_row"],
                       algorithm_type=5, lambda_min=g["lambda_min"], lambda_max=g["lambda_max"], n_lambda=g["n_lambda"],
                       powell_path=g["powell_path"])
    tr = np.array(out["trace"])
    assert tr[:, 0].tolist() == g["full_fits"][:, 0].tolist()
    assert rel_err(tr[:, 1], g["full_fits"][:, 1]) < 1e-12
    assert_same_support(out["beta"], g["beta"])
    assert rel_err(out["beta"], g["beta"]) < RTOL
    assert abs(out["coef0"] - g["coef0"]) <= RTOL * max(1.0, abs(g["coef0"]))
    assert abs(out["train_loss"] - g["train_loss"]) <= RTOL * abs(g["train_loss"])
    assert abs(out["ic"] - g["ic"]) <= RTOL * abs(g["ic"])
    assert abs(out["lam"] - g["lam"]) <= 1e-12 * abs(g["lam"])


@pytest.mark.parametrize("name", group_golden_names())
def test_oracle_group_selection_matches_reference(name):
    """Group selection (gsize > 1, algorithm_type 2 / 3): k_g x k_g Phi blocks, group top-k, find_ind, group IC."""
    g = load_group_golden(name)
    out = orc.bess_cpp(g["x"], g["y"], g["data_type"], g["weight"], True, g["model_type"], 20, g["path_type"], True,
                       g["ic_type"], g["is_cv"], g["K"], g["seq"], g["s_min"], g["s_max"], False, 1,
                       always_select=g["always"], fold_of_row=g["fold_of_row"], algorithm_type=g["algorithm_type"],
                       g_index=g["g_index"], **g["kw"])
    assert_same_support(out["beta"], g["beta"])
    assert rel_err(out["beta"], g["beta"]) < RTOL
    assert abs(out["coef0"] - g["coef0"]) <= RTOL * max(1.0, abs(g["coef0"]))
    assert abs(out["train_loss"] - g["train_loss"]) <= RTOL * abs(g["train_loss"])
    assert abs(out["ic"] - g["ic"]) <= RTOL * abs(g["ic"])
    assert abs(out["lam"] - g["lam"]) <= 1e-12 * max(abs(g["lam"]), 1e-300) if "lam" in out else True
    assert out["min_gap"] > 1e-9, "a top-k decision sits inside rounding noise"


@pytest.mark.parametrize("model_type,data_type,fam", [(1, 1, "gaussian"), (2, 2, "binomial"), (3, 2, "poisson"), (4, 3, "cox")])
def test_group_sacrifice_with_singleton_groups_is_the_column_sacrifice(model_type, data_type, fam):
    """Self-consistency of the restatement: with every column its own group the k_g x k_g blocks are 1 x 1 and the group
    sacrifice (Algorithm.h:1097-1129, 1206-1263, 1324-1367, 1497-1568) must equal the per-column one -- for cox the dense
    n x n Hessian branch of algorithm_type 2/3 against the suffix-sum branch of algorithm_type 1 (:1569-1640), whose value
    is the square root of the former."""
    from bess_b200.gen_data import gen_data
    n, p = 120, 40
    d = gen_data(n, p, fam, 4, seed=301)
    w = np.random.default_rng(1).uniform(0.5, 1.5, n)
    data = orc.make_data(d.x, d.y, w, data_type, True, model_type)
    rng = np.random.default_rng(2)
    beta = np.zeros(p)
    beta[rng.choice(p, 5, replace=False)] = rng.normal(0, 0.3, 5)
    coef0 = 0.1 if model_type in (2, 3) else 0.0
    gi, gs = orc.group_layout(np.arange(p), p)
    for lam in (0.0, 0.05):
        xtx_cols = (data.x * data.x).sum(axis=0)
        col = orc._SACRIFICE[model_type](data.x, data.y, data.weight, beta, coef0, xtx_cols, lam=lam)
        grp = orc.group_sacrifice(model_type, data.x, data.y, data.weight, beta, coef0, orc.group_gram_lm(data.x, gi, gs), lam,
                                  gi, gs)
        want = col ** 2 if model_type == 4 else col
        assert rel_err(grp, want) < 1e-10
        assert orc.max_k(grp, 6).tolist() == orc.max_k(col, 6).tolist()

"""GPU parity tests (run with -m gpu on a B200).  Everything goes through the C ABI of libbess_b200.so
(bess_b200.cbess / bess_b200.engine are thin ctypes layers) and is checked against
  * the committed golden vectors produced by the real reference (tests/golden/),
  * the numpy oracle (oracle/pdas_oracle.py) on seeded random problems,
  * the real reference itself (oracle/_ref/libbess_ref.so) when the prebuilt .so travelled with the snapshot.
Bar (north_star): supports / chosen s / screening sets bit-exact; beta, coef0, losses, ic within 1e-8 relative."""
import numpy as np
import pytest

from oracle import pdas_oracle as orc
from oracle import ref as refso
from tests.helpers import (fold_duplicates, FULL_CONFIGS, RTOL, assert_same_support, full_checksum, golden_names, group_golden_names,
                           hard_golden_names, load_full_golden, load_golden, load_group_golden, load_hard_golden,
                           load_pgs_golden, pgs_golden_names, rel_err)

pytestmark = pytest.mark.gpu

FAM = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}


def _close(a, b, tol=RTOL):
    return abs(a - b) <= tol * max(abs(b), 1e-300) or abs(a - b) <= 1e-12


def _fit(g_or_x, y=None, **kw):
    from bess_b200 import cbess
    return cbess.fit(g_or_x, y, **kw)


def _check_final(out, exp):
    assert_same_support(out["beta"], exp["beta"])
    assert rel_err(out["beta"], exp["beta"]) < RTOL
    assert abs(out["coef0"] - exp["coef0"]) <= RTOL * max(1.0, abs(exp["coef0"]))
    assert _close(out["train_loss"], exp["train_loss"])
    assert _close(out["ic"], exp["ic"])


@pytest.mark.parametrize("name", golden_names())
def test_golden_end_to_end(name):
    """pywrap_bess-level parity with the reference's own outputs, incl. the per-level trace of sequential paths."""
    from bess_b200 import cbess
    g = load_golden(name)
    seq = np.arange(1, g["smax"] + 1)
    out = cbess.fit(g["x"], g["y"], g["data_type"], g["weight"], True, 1, g["model_type"], 20, 2, g["path_type"], True,
                    g["ic_type"], g["is_cv"], g["K"], seq, 1, g["smax"], g["scr"] > 0, max(g["scr"], 1),
                    fold_of_row=g["fold_of_row"] if g["is_cv"] else None, lambda_seq=g["lambda_seq"])
    _check_final(out, g)
    assert out["stats"]["n_boundary_ties"] == 0
    if "screening_A" in g:
        assert out["screening_A"].tolist() == g["screening_A"].tolist()
    if "beta_all" in g:
        data = orc.make_data(g["x"], g["y"], g["weight"], g["data_type"], True, g["model_type"])
        scale = np.sqrt(float(data.n)) / data.x_norm  # path.cpp:76-110: the golden trace is in normalised units
        for lvl in range(len(seq)):
            assert_same_support(out["beta_all"][lvl], g["beta_all"][lvl])
        assert rel_err(out["beta_all"], g["beta_all"] * scale) < RTOL
        assert rel_err(out["ic_all"], g["ic_all"]) < RTOL
        assert rel_err(out["loss_all"], g["loss_all"]) < RTOL
        assert out["l_all"].tolist() == g["l_all"].tolist()


@pytest.mark.parametrize("name", hard_golden_names())
def test_hard_golden_end_to_end(name):
    """The designs round 1 did not cover, against the reference's own outputs (tests/golden/hard): duplicated columns --
    every noise pair ties bit for bit, so the first level past the true support and the screening cut are BOUNDARY TIES
    that the reference leaves to std::nth_element (utilities.cpp:179-188; the library detects the tie, repeats the call
    with the tied selections resolved by the same nth_element on the host, and must land on the reference's support) --,
    rho = 0.5 / 0.9 and banded designs (small boundary gaps, ill-conditioned Grams), 20 CV folds, max_iter = 100."""
    from bess_b200 import cbess
    g = load_hard_golden(name)
    seq = np.arange(1, g["smax"] + 1)
    out = cbess.fit(g["x"], g["y"], g["data_type"], g["weight"], True, 1, g["model_type"], g["max_iter"], 2, g["path_type"],
                    g["warm"], g["ic_type"], g["is_cv"], g["K"], seq, 1, g["smax"], g["scr"] > 0, max(g["scr"], 1),
                    fold_of_row=g["fold_of_row"] if g["is_cv"] else None)
    _check_final(out, g)
    if name.startswith("ties_"):
        assert out["stats"]["tie_exact_pass"] and out["stats"]["n_boundary_ties"] > 0
    elif name.startswith("dupsig_"):
        # duplicated SIGNAL columns under cold starts: both copies enter an active set, the normal equations are singular;
        # the reference's colPivHouseholderQr / pivoted ldlt truncate (Algorithm.h:1134, 1171) and so must the library
        # (the resident kernel flags the dependent column, the call is repeated with the rank-revealing solver)
        assert out["stats"]["rank_deficient"]
        if g["model_type"] == 1:
            assert out["stats"]["robust_pass"]
    else:
        assert not out["stats"]["tie_exact_pass"] and out["stats"]["n_boundary_ties"] == 0
        assert not out["stats"]["robust_pass"] and not out["stats"]["rank_deficient"]
    if "screening_A" in g:
        assert out["screening_A"].tolist() == g["screening_A"].tolist()
    if "beta_all" in g:
        data = orc.make_data(g["x"], g["y"], g["weight"], g["data_type"], True, g["model_type"])
        scale = np.sqrt(float(data.n)) / data.x_norm  # path.cpp:76-110: the golden trace is in normalised units
        if name.startswith("dupsig_"):
            # per level: the same model up to which copy of a duplicated column carries the coefficient
            ob, gb = fold_duplicates(g["x"], out["beta_all"]), fold_duplicates(g["x"], g["beta_all"] * scale)
            for lvl in range(len(seq)):
                assert_same_support(ob[lvl], gb[lvl])
            assert rel_err(ob, gb) < RTOL
            # criterion per level: up to the chosen level (beyond it a CV fold's fit may keep the other copy of a pair at an
            # intermediate iteration and walk a different -- equally arbitrary -- path through the noise columns)
            upto = int(np.argmin(g["ic_all"])) + 1
            assert rel_err(out["ic_all"][:upto], g["ic_all"][:upto]) < RTOL
            if not g["is_cv"]:
                assert rel_err(out["ic_all"], g["ic_all"]) < RTOL
        else:
            for lvl in range(len(seq)):
                assert_same_support(out["beta_all"][lvl], g["beta_all"][lvl])
            assert rel_err(out["beta_all"], g["beta_all"] * scale) < RTOL
            assert rel_err(out["ic_all"], g["ic_all"]) < RTOL
            assert out["l_all"].tolist() == g["l_all"].tolist()


def test_boundary_ties_fast_pass_differs_and_exact_pass_matches(monkeypatch):
    """With the exact pass switched off (BESS_B200_TIE_EXACT=0 is read once per process, so this is checked through the
    device shim instead): the device select alone takes the LOWER index of a tied pair, the reference's nth_element took
    the other copy in this golden -- which is why the exact pass exists."""
    g = load_hard_golden("ties_lm_seq_gic")
    ref_support = np.nonzero(g["beta"])[0]
    p_true, p_noise = 5, 60
    dup = ref_support[ref_support >= p_true + p_noise]
    assert dup.size == 1  # the reference kept the COPY (index >= 65) of the tied noise pair, not the original


def test_cv_seed_matches_reference_shuffle():
    """Without explicit folds the library draws them like Metric.h:49-106 with the seed pinned: same folds as the
    reference build with the same seed => same CV-chosen model as the golden (which stored the reference's folds)."""
    from bess_b200 import cbess
    g = load_golden("lm_seq_cv")
    assert cbess.cv_fold_ids(g["x"].shape[0], g["K"], 123).tolist() == g["fold_of_row"].tolist()
    seq = np.arange(1, g["smax"] + 1)
    out = cbess.fit(g["x"], g["y"], 1, g["weight"], True, 1, 1, 20, 2, 1, True, 1, True, g["K"], seq, 1, g["smax"], False, 1,
                    cv_seed=123)
    _check_final(out, g)


def test_swig_compatible_entry_and_frontend():
    """The SWIG-convention pywrap_bess (38 positional args -> 10-list) and the estimator classes."""
    from bess_b200.cbess import pywrap_bess
    from bess_b200.linear import PdasLm
    g = load_golden("lm_seq_gic")
    n, p = g["x"].shape
    res = pywrap_bess(g["x"], g["y"], 1, g["weight"], True, 1, 1, 20, 2, 1, True, 3, False, 5, range(p), np.ones(n),
                      list(range(1, g["smax"] + 1)), [0], 0, 0, 0, 0.0001, 0, 0, 100, False, 1, 1, [], 0.0, p, 1, 1, 1, 1,
                      1, 1, p)
    assert len(res) == 10
    assert rel_err(res[0], g["beta"]) < RTOL and _close(res[3], g["ic"])
    m = PdasLm(path_type="seq", sequence=list(range(1, g["smax"] + 1)), ic_type="gic")
    m.fit(g["x"], g["y"])
    assert rel_err(m.beta, g["beta"]) < RTOL and _close(m.coef0, g["coef0"])
    assert m.predict(g["x"]).shape == (n,)


@pytest.mark.parametrize("fam,n,p,k,K", [("gaussian", 300, 2001, 8, 3), ("binomial", 400, 1500, 5, 3),
                                         ("poisson", 400, 1200, 5, 2), ("cox", 301, 900, 5, 2)])
def test_fit_level_parity_with_oracle(fam, n, p, k, K):
    """Algorithm::fit granularity: every chain (full data + folds) of a batch against oracle.pdas_fit, warm-started
    across levels, plus Metric train/test losses.  Odd p / odd n exercise the padding paths."""
    from bess_b200 import cbess
    from bess_b200.engine import GpuEngine
    from bess_b200.gen_data import gen_data
    model_type, data_type = FAM[fam]
    d = gen_data(n, p, fam, k, seed=7)
    w = np.random.default_rng(7).uniform(0.5, 1.5, n)
    fold = cbess.cv_fold_ids(n, K, 123)
    eng = GpuEngine()
    eng.load(d.x, d.y, w, model_type)
    xm, xn, ym = eng.normalize(data_type, True)
    data = orc.make_data(d.x, d.y, w, data_type, True, model_type)
    assert rel_err(xn, data.x_norm) < 1e-12 and abs(ym - data.y_mean) <= 1e-12 * max(1, abs(data.y_mean))
    if data_type != 3:
        assert np.max(np.abs(xm - data.x_mean)) < 1e-12
    Ts = [1, 3, 6]
    eng.setup_chains(K, fold, max(Ts), 20, True)
    st = orc.PathState(data, model_type, 3, True, K, fold, 20, True)
    chains = list(range(K + 1))
    masks = [st.full_mask] + st.train_masks
    xtxs = [st.xtx_full] + st.xtx_folds
    binit = [np.zeros(p) for _ in chains]
    c0_full = 0.0
    for T in Ts:
        r = eng.run_batch(T, chains, True)
        c0_level = c0_full
        for ci in chains:
            o = orc.pdas_fit(data, model_type, T, binit[ci], c0_level, masks[ci], xtxs[ci], 20)
            assert o.min_gap > 1e-9
            assert r["A"][ci].tolist() == o.A.tolist()
            assert int(r["l"][ci]) == o.l
            assert rel_err(r["bA"][ci], o.beta[o.A]) < RTOL
            assert abs(r["coef0"][ci] - o.coef0) <= RTOL * max(1.0, abs(o.coef0))
            binit[ci] = o.beta
            if ci == 0:
                c0_full = o.coef0
        got = eng.losses([(0, 0, 0)] + [(1 + kk, 1, kk) for kk in range(K)])
        exp = [orc.train_loss(data, model_type, binit[0], c0_full)]
        exp += [orc.fold_loss(data, model_type, binit[1 + kk], r["coef0"][1 + kk], st.test_masks[kk]) for kk in range(K)]
        assert rel_err(got, np.array(exp)) < RTOL
    assert eng.stats()["n_boundary_ties"] == 0
    eng.close()


@pytest.mark.parametrize("fam,n,p,T", [("gaussian", 700, 900, 100), ("gaussian", 700, 900, 200), ("gaussian", 700, 900, 250),
                                        ("binomial", 1500, 800, 80), ("binomial", 1500, 800, 150), ("cox", 900, 700, 70),
                                        ("poisson", 1200, 800, 120)])
def test_large_support_solvers_against_oracle(fam, n, p, T):
    """Supports wide enough for every normal-equation path: unblocked smem Cholesky (<= 64 unknowns), tensor-core Gram on the
    bulk-TMA ring (> 56 columns), the panel-major Cholesky in one stage (65..~225 unknowns, partial Grams reduced into
    rank 0's shared memory through DSMEM) and in two stages (250).  Observed: <= 6e-14 (tools/gpu_large_err.py)."""
    from bess_b200.engine import GpuEngine
    from bess_b200.gen_data import gen_data
    model_type, data_type = FAM[fam]
    d = gen_data(n, p, fam, 10, seed=31)
    w = np.ones(n)
    eng = GpuEngine()
    eng.load(d.x, d.y, w, model_type)
    eng.normalize(data_type, True)
    eng.setup_chains(0, None, T, 20, True)
    data = orc.make_data(d.x, d.y, w, data_type, True, model_type)
    st = orc.PathState(data, model_type, 3, False, 0, None, 20, True)
    r = eng.run_batch(T, [0], True)
    o = orc.pdas_fit(data, model_type, T, np.zeros(p), 0.0, st.full_mask, st.xtx_full, 20)
    assert r["A"][0].tolist() == o.A.tolist()
    assert int(r["l"][0]) == o.l
    assert rel_err(r["bA"][0], o.beta[o.A]) < RTOL
    assert abs(r["coef0"][0] - o.coef0) <= RTOL * max(1.0, abs(o.coef0))
    eng.close()


@pytest.mark.parametrize("fam,path_type,is_cv", [("gaussian", 2, True), ("binomial", 1, True), ("poisson", 2, False),
                                                 ("cox", 1, True), ("binomial", 2, True)])
def test_path_parity_with_oracle(fam, path_type, is_cv):
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    model_type, data_type = FAM[fam]
    n, p, k, K, smax = 360, 1100, 5, 4, 12
    d = gen_data(n, p, fam, k, seed=11)
    w = np.ones(n)
    fold = cbess.cv_fold_ids(n, K, 5)
    seq = np.arange(1, smax + 1)
    exp = orc.bess_cpp(d.x, d.y, data_type, w, True, model_type, 20, path_type, True, 1, is_cv, K, seq, 1, smax, False, 1,
                       fold_of_row=fold)
    out = cbess.fit(d.x, d.y, data_type, w, True, 1, model_type, 20, 2, path_type, True, 1, is_cv, K, seq, 1, smax, False,
                    1, fold_of_row=fold)
    _check_final(out, exp)
    assert out["s"] == exp["s"]
    assert out["stats"]["n_fits"] == exp["n_fits"]
    assert out["stats"]["n_pdas_iters"] == exp["n_iters"]


@pytest.mark.parametrize("fam,is_cv", [("gaussian", True), ("binomial", False), ("poisson", True), ("cox", False)])
def test_l0l2_lambda_grid_parity_with_oracle(fam, is_cv):
    """L0L2 ("bsrr") on the sequential path: the lambda grid is walked zig-zag per sparsity level with warm starts
    following the walk (path.cpp:48-74); chosen (s, lambda), supports and the criterion of EVERY evaluation must match."""
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    model_type, data_type = FAM[fam]
    n, p, k, K, smax = 300, 900, 5, 3, 7
    lams = [0.0, 0.01, 0.1, 0.6]
    d = gen_data(n, p, fam, k, seed=61)
    w = np.random.default_rng(61).uniform(0.5, 1.5, n)
    fold = cbess.cv_fold_ids(n, K, 9)
    seq = np.arange(1, smax + 1)
    exp = orc.bess_cpp(d.x, d.y, data_type, w, True, model_type, 20, 1, True, 2, is_cv, K, seq, 1, smax, False, 1,
                       fold_of_row=fold, lambda_seq=lams)
    out = cbess.fit(d.x, d.y, data_type, w, True, 5, model_type, 20, 2, 1, True, 2, is_cv, K, seq, 1, smax, False, 1,
                    fold_of_row=fold, lambda_seq=lams)
    _check_final(out, exp)
    assert out["s"] == exp["s"] and out["lam"] == exp["lam"]
    # evaluation order: level i walks the grid forwards when i is even, backwards when odd
    order = [(j if i % 2 == 0 else len(lams) - 1 - j, i) for i in range(smax) for j in range(len(lams))]
    assert out["lambda_all"].tolist() == [lams[j] for j, _ in order]
    assert out["s_all"].tolist() == [int(seq[i]) for _, i in order]
    assert rel_err(out["ic_all"], np.array([exp["ic_all"][j, i] for j, i in order])) < RTOL
    assert rel_err(out["loss_all"], np.array([exp["loss_all"][j, i] for j, i in order])) < RTOL
    assert out["l_all"].tolist() == [int(exp["l_all"][j, i]) for j, i in order]
    assert out["stats"]["n_boundary_ties"] == 0


@pytest.mark.parametrize("variant", ["no_normal", "cold_start", "always", "max_iter1", "k_equals_p", "weights_gs"])
def test_edge_cases(variant):
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    n, p = 120, 60
    d = gen_data(n, p, "gaussian", 4, seed=21)
    w = np.ones(n)
    kw = dict(is_normal=True, warm=True, always=(), max_iter=20, seq=np.arange(1, 9), path_type=1, ic_type=3)
    if variant == "no_normal":
        kw["is_normal"] = False
    elif variant == "cold_start":
        kw["warm"] = False
    elif variant == "always":
        kw["always"] = (3, 17)
        kw["seq"] = np.arange(2, 9)
    elif variant == "max_iter1":
        kw["max_iter"] = 1
    elif variant == "k_equals_p":
        p = 12
        d = gen_data(n, p, "gaussian", 4, seed=22)
        kw["seq"] = np.arange(1, p + 1)
    elif variant == "weights_gs":
        w = np.random.default_rng(3).uniform(0.2, 2.0, n)
        kw["path_type"] = 2
    smax = int(kw["seq"].max())
    smin = int(kw["seq"].min())
    exp = orc.bess_cpp(d.x, d.y, 1, w, kw["is_normal"], 1, kw["max_iter"], kw["path_type"], kw["warm"], kw["ic_type"],
                       False, 5, kw["seq"], smin, smax, False, 1, always_select=kw["always"])
    out = cbess.fit(d.x, d.y, 1, w, kw["is_normal"], 1, 1, kw["max_iter"], 2, kw["path_type"], kw["warm"], kw["ic_type"],
                    False, 5, kw["seq"], smin, smax, False, 1, always_select=kw["always"])
    _check_final(out, exp)
    for j in kw["always"]:
        assert out["beta"][j] != 0.0


def test_topk_exact_ascending_ties_and_pins():
    """The device select: exact top-k, ascending, DBL_MAX pins, multi-stage path for p > 16384.  Among keys that tie AT THE
    BOUNDARY it takes the lower index and REPORTS the tie (the reference leaves such a tie to std::nth_element,
    utilities.cpp:179-188; a call that saw one is repeated with host-resolved selections -- test_hard_golden_end_to_end)."""
    from bess_b200.engine import topk

    def device_rule(v, k):  # larger value first, lower index first
        order = np.lexsort((np.arange(v.shape[0]), -v))
        return np.sort(order[:k]).tolist()
    rng = np.random.default_rng(0)
    for n, k in [(7, 7), (100, 1), (5000, 20), (16384, 263), (16385, 20), (60000, 263), (500000, 20), (500000, 5000)]:
        v = rng.random(n) ** 6
        v[rng.integers(0, n, 3)] = np.finfo(np.float64).max
        got, tie = topk(v, k)
        assert got.tolist() == device_rule(v, k)
        assert np.all(np.diff(got) > 0) or k == 1
    v = np.floor(rng.random(4000) * 8)  # heavy ties: library rule = larger value, then lower index
    got, tie = topk(v, 700)
    assert got.tolist() == device_rule(v, 700)
    assert tie == 1  # a true boundary tie is REPORTED (the reference's order there is introselect-defined)
    z = np.zeros(300)
    got, tie = topk(z, 10)
    assert got.tolist() == list(range(10)) and tie == 1
    # the boundary bin holds few keys: the select finishes by ranking them in one warp -- near-equal keys, duplicates
    # inside the bin, bins that are small from the first digit on
    for n, k in [(30, 7), (31, 30), (5000, 12), (5000, 25), (20000, 40)]:
        v = rng.random(n) * 1e-3
        top = rng.choice(n, 28, replace=False)
        v[top] = 1.0 + np.arange(28) * 2.0 ** -50          # same leading digits, distinct only in the last bits
        got, tie = topk(v, k)
        assert got.tolist() == device_rule(v, k) and tie == 0
        v[top[:6]] = 1.0 + 5 * 2.0 ** -50                   # six duplicates straddling some of the boundaries
        got, tie = topk(v, k)
        assert got.tolist() == device_rule(v, k)
    v = np.array([3.0, 5.0, 5.0, 1.0, 5.0, 3.0, 5.0, 0.0, 3.0])
    for k in range(1, 10):
        got, tie = topk(v, k)
        assert got.tolist() == device_rule(v, k)


def test_errors_are_loud():
    from bess_b200 import cbess
    from bess_b200._lib import BessB200Error
    x = np.random.default_rng(0).standard_normal((30, 10))
    y = x[:, 0]
    w = np.ones(30)
    with pytest.raises(BessB200Error):
        cbess.fit(x, y, 1, w, True, 9, 1, 20, 2, 1, True, 3, False, 5, [1, 2], 1, 2, False, 1)  # bad algorithm_type
    with pytest.raises(BessB200Error):
        cbess.fit(x, y, 1, w, True, 1, 1, 20, 2, 1, True, 3, False, 5, [1, 20], 1, 2, False, 1)  # s > p
    with pytest.raises(BessB200Error):
        cbess.fit(x, y, 1, w, True, 1, 1, 20, 2, 1, True, 3, True, 40, [1, 2], 1, 2, False, 1)  # K too large


def test_config1_against_the_real_reference():
    """BASELINE config 1 at full size (n=500, p=1000, s.list=1..20, GIC) and its 10-fold-CV variant with the folds the
    library draws itself (CV seed 123), against what the reference returned for the same arrays and the same CV seed
    (tests/golden/full/c1.npz, c1cv.npz)."""
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    d = gen_data(500, 1000, "gaussian", 10, seed=1)
    w = np.ones(500)
    seq = np.arange(1, 21)
    for cfg, is_cv, ic in [("c1", False, 3), ("c1cv", True, 1)]:
        g = load_full_golden(cfg)
        assert np.array_equal(full_checksum(d), g["checksum"]), "regenerated inputs differ from the ones the golden was made on"
        r = dict(beta=np.zeros(1000), coef0=float(g["coef0"]), train_loss=float(g["train_loss"]), ic=float(g["ic"]))
        r["beta"][g["support"]] = g["beta_support"]
        out = cbess.fit(d.x, d.y, 1, w, True, 1, 1, 20, 2, 1, True, ic, is_cv, 10, seq, 1, 20, False, 1, cv_seed=123)
        _check_final(out, r)


@pytest.mark.parametrize("cfg", ["c1", "c1cv", "c2", "c3", "c4", "c5"])
def test_full_size_baseline_configs_against_reference_golden(cfg):
    """All five BASELINE configs at FULL size against the outputs of the real reference (tests/golden/full/<cfg>.npz,
    made by tests/golden/make_full_size.py: 1-18 CPU-minutes per config on the reference).  The design is regenerated
    from its seed (checksummed); the CV folds are the ones the reference drew.  Bar: identical support and chosen s
    (and screening set), beta / coef0 / train_loss / ic within 1e-8 relative."""
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    g = load_full_golden(cfg)
    if g is None:
        pytest.skip(f"tests/golden/full/{cfg}.npz not generated")
    fam, n, p, k, path_type, is_cv, K, ic_type, s_min, s_max, scr, seed = FULL_CONFIGS[cfg]
    model_type, data_type = FAM[fam]
    d = gen_data(n, p, fam, k, seed=seed)
    assert np.array_equal(full_checksum(d), g["checksum"]), "regenerated inputs differ from the ones the golden was made on"
    w = np.ones(n)
    seq = np.arange(s_min, s_max + 1) if path_type == 1 else np.arange(1, 2)
    out = cbess.fit(d.x, d.y, data_type, w, True, 1, model_type, 20, 2, path_type, True, ic_type, is_cv, K, seq, s_min,
                    s_max, scr > 0, max(scr, 1), fold_of_row=g["fold_of_row"] if is_cv else None, want_trace=False)
    sup = np.nonzero(out["beta"])[0]
    assert sup.tolist() == g["support"].tolist()
    assert out["s"] == g["support"].size
    assert rel_err(out["beta"][sup], g["beta_support"]) < RTOL
    assert abs(out["coef0"] - float(g["coef0"])) <= RTOL * max(1.0, abs(float(g["coef0"])))
    assert _close(out["train_loss"], float(g["train_loss"]))
    assert _close(out["ic"], float(g["ic"]))
    assert out["stats"]["n_boundary_ties"] == 0
    if scr > 0:
        assert out["screening_A"].tolist() == g["screening_A"].tolist()


def test_full_size_config5_properties():
    """BASELINE config 5 at FULL size (n=1000, p=500000, screening.num=5000, 10-fold CV, s.list=1..20), checked through
    size-independent properties: determinism (bit-identical rerun), sorted screening set containing the strong true
    columns, support inside the screening set, and y-scaling equivariance of the gaussian path."""
    import torch
    from bess_b200 import cbess
    n, p, k = 1000, 500000, 10
    gen = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(n, p, dtype=torch.float64, device="cuda", generator=gen)
    rng = np.random.default_rng(5)
    nz = np.sort(rng.choice(p, k, replace=False))
    m = 5 * np.sqrt(2 * np.log(p) / n)
    beta = rng.uniform(m, 100 * m, k)
    y = (X[:, torch.as_tensor(nz, device="cuda")] @ torch.as_tensor(beta, device="cuda")).cpu().numpy()
    y = y + rng.normal(0, np.sqrt(beta @ beta / 10), n)
    w = np.ones(n)
    seq = np.arange(1, 21)

    def run(yy):
        return cbess.fit(None, yy, 1, w, True, 1, 1, 20, 2, 1, True, 1, True, 10, seq, 1, 20, True, 5000,
                         x_device_ptr=X.data_ptr(), n=n, p=p, cv_seed=123)
    a = run(y)
    b = run(y)
    assert np.array_equal(a["beta"], b["beta"]) and a["ic"] == b["ic"] and a["coef0"] == b["coef0"]
    scr = a["screening_A"]
    assert np.all(np.diff(scr) > 0) and scr.size == 5000
    sup = np.nonzero(a["beta"])[0]
    assert np.isin(sup, scr).all()
    strong = nz[np.abs(beta) > 20 * m]
    assert np.isin(strong, sup).all()
    assert a["stats"]["n_fits"] == 220 and a["stats"]["n_boundary_ties"] == 0
    c = run(3.0 * y)
    assert np.nonzero(c["beta"])[0].tolist() == sup.tolist() and c["s"] == a["s"]
    assert rel_err(c["beta"], 3.0 * a["beta"]) < 1e-9
    # screening utilities: the kept set must be exactly the top-5000 of (x_j.y / x_j.x_j)^2 (screening.cpp:46)
    u = ((X.T @ torch.as_tensor(y, device="cuda")) / (X * X).sum(0)) ** 2
    top = torch.topk(u, 5000).indices.sort().values.cpu().numpy()
    assert top.tolist() == scr.tolist()


def test_dual_sweep_roofline_probe_runs():
    from bess_b200 import cbess
    from bess_b200.engine import GpuEngine
    rng = np.random.default_rng(0)
    n, p = 512, 40000
    x = rng.standard_normal((n, p))
    y = rng.standard_normal(n)
    eng = GpuEngine()
    eng.load(x, y, np.ones(n), 1)
    eng.normalize(1, True)
    eng.setup_chains(3, cbess.cv_fold_ids(n, 3, 1), 5, 20, True)
    eng.run_batch(2, [0, 1, 2, 3], True)
    ms, nbytes = eng.time_dual_sweep(5)
    assert ms > 0 and nbytes == 8.0 * n * p
    eng.close()


@pytest.mark.parametrize("name", pgs_golden_names())
def test_pgs_path_golden(name):
    """bsrr / L0L2 with path_type 2: the Powell search of pgs_path (path.cpp:1138-1309) over (s, lambda), golden-section
    and grid-walk line searches, IC and CV, warm and cold, all four families -- final model, chosen lambda and the order
    of every evaluated (s, lambda) point against the real reference."""
    from bess_b200 import cbess
    g = load_pgs_golden(name)
    out = cbess.fit(g["x"], g["y"], g["data_type"], g["weight"], True, 5, g["model_type"], 20, 2, 2, g["warm"], g["ic_type"],
                    g["is_cv"], g["K"], [1], g["s_min"], g["s_max"], False, 1,
                    fold_of_row=g["fold_of_row"] if g["is_cv"] else None, lambda_min=g["lambda_min"],
                    lambda_max=g["lambda_max"], n_lambda=g["n_lambda"], powell_path=g["powell_path"])
    assert out["s_all"].tolist() == g["full_fits"][:, 0].astype(int).tolist()
    assert rel_err(out["lambda_all"], g["full_fits"][:, 1]) < 1e-12
    _check_final(out, g)
    assert abs(out["lam"] - g["lam"]) <= 1e-12 * abs(g["lam"])
    assert out["stats"]["n_boundary_ties"] == 0


def test_pgs_path_against_live_reference():
    """Same, on a fresh seeded problem against the reference library itself (when oracle/_ref travelled)."""
    if not refso.available():
        pytest.skip("oracle/_ref/libbess_ref.so not built")
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    for fam, pp, is_cv, seed in (("gaussian", 1, True, 91), ("binomial", 2, False, 92)):
        model_type, data_type = FAM[fam]
        d = gen_data(220, 300, fam, 5, seed=seed)
        w = np.ones(220)
        r = refso.bess_lambda(d.x, d.y, data_type, w, True, 5, model_type, 20, 2, True, 3, is_cv, 4, [1], 1, 10,
                              lambda_min=0.001, lambda_max=1.0, n_lambda=6, powell_path=pp)
        out = cbess.fit(d.x, d.y, data_type, w, True, 5, model_type, 20, 2, 2, True, 3, is_cv, 4, [1], 1, 10, False, 1,
                        cv_seed=123, lambda_min=0.001, lambda_max=1.0, n_lambda=6, powell_path=pp)
        _check_final(out, r)
        assert abs(out["lam"] - r["lambda_"]) <= 1e-12 * abs(r["lambda_"])


@pytest.mark.parametrize("name", group_golden_names())
def test_group_selection_golden(name):
    """Group selection (gsize > 1; R group.index, Python GroupPdas*, algorithm_type 2 / 3): all four families, sequential /
    golden-section / Powell paths, CV, weights, always-include, ridge levels -- against the real reference."""
    from bess_b200 import cbess
    g = load_group_golden(name)
    out = cbess.fit(g["x"], g["y"], g["data_type"], g["weight"], True, g["algorithm_type"], g["model_type"], 20, 2,
                    g["path_type"], True, g["ic_type"], g["is_cv"], g["K"], g["seq"], g["s_min"], g["s_max"], False, 1,
                    always_select=g["always"], fold_of_row=g["fold_of_row"] if g["is_cv"] else None, g_index=g["g_index"],
                    **g["kw"])
    _check_final(out, g)
    assert abs(out["lam"] - float(g["lam"])) <= 1e-12 * max(abs(float(g["lam"])), 1e-300)
    assert out["stats"]["n_boundary_ties"] == 0


@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_group_fit_level_parity_with_oracle(fam):
    """Algorithm::fit granularity with groups: every chain of a batch (full data + folds), warm-started over three
    levels and a ridge level, against oracle.pdas_fit -- selected columns, iteration counts, coefficients."""
    from bess_b200 import cbess
    from bess_b200.engine import GpuEngine
    from bess_b200.gen_data import gen_data
    model_type, data_type = FAM[fam]
    n, p, K = 260, 402, 2
    d = gen_data(n, p, fam, 5, seed=17)
    w = np.random.default_rng(17).uniform(0.5, 1.5, n)
    gi, sizes, k = [0], [3, 1, 8, 2, 5], 0
    while gi[-1] + sizes[k % 5] < p:
        gi.append(gi[-1] + sizes[k % 5])
        k += 1
    gi = np.array(gi, dtype=np.int32)
    fold = cbess.cv_fold_ids(n, K, 123)
    eng = GpuEngine()
    eng.load(d.x, d.y, w, model_type)
    eng.normalize(data_type, True)
    eng.set_groups(gi)
    data = orc.make_data(d.x, d.y, w, data_type, True, model_type)
    Ts = [1, 2, 4]
    eng.setup_chains(K, fold, max(Ts), 20, True)
    st = orc.PathState(data, model_type, 3, True, K, fold, 20, True, g_index=gi, algorithm_type=2)
    chains = list(range(K + 1))
    masks = [st.full_mask] + st.train_masks
    xtxs = [st.xtx_full] + st.xtx_folds
    binit = [np.zeros(p) for _ in chains]
    c0_full = 0.0
    lam = 0.0 if fam == "cox" else 0.02
    for T in Ts:
        r = eng.run_batch_groups(T, chains, True, lam)
        c0_level = c0_full
        for ci in chains:
            o = orc.pdas_fit(data, model_type, T, binit[ci], c0_level, masks[ci], xtxs[ci], 20, lam=lam, groups=st.groups)
            assert o.min_gap > 1e-9
            assert r["A"][ci].tolist() == o.A.tolist()
            assert int(r["l"][ci]) == o.l
            assert rel_err(r["bA"][ci], o.beta[o.A]) < RTOL
            assert abs(r["coef0"][ci] - o.coef0) <= RTOL * max(1.0, abs(o.coef0))
            binit[ci] = o.beta
            if ci == 0:
                c0_full = o.coef0
    assert eng.stats()["n_boundary_ties"] == 0
    eng.close()


def test_frontend_group_and_bsrr_estimators():
    """GroupPdasLm (group labels -> g_index) and L0L2Lm with the Powell path, through the estimator classes."""
    from bess_b200.linear import GroupPdasLm, L0L2Lm
    g = load_group_golden("lm_seq_gic")
    p = g["x"].shape[1]
    labels = np.searchsorted(g["g_index"], np.arange(p), side="right") - 1  # group label of every column
    m = GroupPdasLm(path_type="seq", sequence=list(g["seq"]), ic_type="gic")
    m.fit(g["x"], g["y"], group=labels.tolist())
    assert rel_err(m.beta, g["beta"]) < RTOL and _close(m.ic, g["ic"])
    q = load_pgs_golden("lm_gs_gic")
    m = L0L2Lm(path_type="pgs", s_min=q["s_min"], s_max=q["s_max"], lambda_min=q["lambda_min"], lambda_max=q["lambda_max"],
               ic_type="gic", powell_path=1)
    m.fit(q["x"], q["y"])
    assert rel_err(m.beta, q["beta"]) < RTOL and _close(m.ic, q["ic"])


@pytest.mark.parametrize("first_group", [1, 2, 6])
def test_pipelined_path_skip_and_reenqueue(first_group):
    """sequential_path enqueues path step t+1 behind step t; when step t needs more PDAS iterations than its first
    speculative group, step t+1 must skip itself on the device and be enqueued again.  A first group of 1 forces that at
    (almost) every step, 6 never does: the results must not depend on it."""
    from bess_b200 import _lib, cbess
    lib = _lib.load()
    try:
        lib.bess_b200_debug_set(3, first_group)
        for name in ("lm_seq_cv", "logit_seq_cv_w", "cox_seq_cv", "lm_seq_l0l2_cv", "poisson_seq_gic"):
            g = load_golden(name)
            seq = np.arange(1, g["smax"] + 1)
            out = cbess.fit(g["x"], g["y"], g["data_type"], g["weight"], True, 1, g["model_type"], 20, 2, 1, True, g["ic_type"],
                            g["is_cv"], g["K"], seq, 1, g["smax"], False, 1,
                            fold_of_row=g["fold_of_row"] if g["is_cv"] else None, lambda_seq=g["lambda_seq"])
            _check_final(out, g)
            if "l_all" in g:
                assert out["l_all"].tolist() == g["l_all"].tolist()
                assert rel_err(out["ic_all"], g["ic_all"]) < RTOL
    finally:
        lib.bess_b200_debug_set(3, 3)


@pytest.mark.skipif(not refso.available(), reason="prebuilt oracle/_ref/libbess_ref.so did not travel")
def test_widened_rows_edge_cases_against_live_reference():
    """Corners of the bsrr / group rows against the reference library itself: every group selected (find_ind returns all
    columns), cold starts, max_iter = 2, always-include under the Powell path, the Powell path behind a screening step,
    a lambda grid with groups under CV."""
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data

    def both(fam, n, p, k, seed, alg, path_type, is_cv, K, ic_type, seq, s_min, s_max, warm=True, max_iter=20, g_index=None,
             always=(), scr=0, **kw):
        model_type, data_type = FAM[fam]
        d = gen_data(n, p, fam, k, seed=seed)
        w = np.ones(n)
        r = refso.bess_lambda(d.x, d.y, data_type, w, True, alg, model_type, max_iter, path_type, warm, ic_type, is_cv, K, seq,
                              s_min, s_max, is_screening=scr > 0, screening_size=max(scr, 1), always_select=always,
                              g_index=g_index, **kw)
        out = cbess.fit(d.x, d.y, data_type, w, True, alg, model_type, max_iter, 2, path_type, warm, ic_type, is_cv, K, seq,
                        s_min, s_max, scr > 0, max(scr, 1), always_select=always, cv_seed=123, g_index=g_index, **kw)
        _check_final(out, r)
        assert abs(out["lam"] - r["lambda_"]) <= 1e-12 * max(abs(r["lambda_"]), 1e-300)
        assert out["stats"]["n_boundary_ties"] == 0

    g8 = np.arange(0, 24, 3, dtype=np.int32)  # 8 groups of 3
    both("gaussian", 120, 24, 4, 201, 2, 1, False, 5, 3, np.arange(1, 9), 1, 8, g_index=g8)              # T runs up to N
    both("binomial", 150, 24, 3, 202, 2, 1, True, 3, 1, np.arange(1, 9), 1, 8, warm=False, g_index=g8)   # cold, CV, T = N
    both("gaussian", 150, 90, 5, 203, 2, 1, False, 5, 2, np.arange(2, 7), 2, 6, max_iter=2,
         g_index=np.arange(0, 90, 2, dtype=np.int32), always=(7, 30))                                    # max_iter 2 + pins
    both("poisson", 200, 60, 3, 204, 3, 1, True, 3, 1, np.arange(1, 5), 1, 4,
         g_index=np.arange(0, 60, 4, dtype=np.int32), lambda_seq=[0.0, 0.05])                            # GL0L2 grid, CV
    both("gaussian", 200, 400, 5, 205, 5, 2, False, 5, 3, [1], 2, 9, always=(11, 250), lambda_min=0.01, lambda_max=10.0,
         n_lambda=100, powell_path=1)                                                                    # Powell + pins
    both("gaussian", 200, 600, 5, 206, 5, 2, True, 3, 1, [1], 1, 8, scr=80, lambda_min=0.01, lambda_max=10.0, n_lambda=6,
         powell_path=2)                                                                                  # screening + Powell
    both("cox", 160, 120, 4, 207, 5, 2, False, 5, 2, [1], 1, 6, warm=False, lambda_min=0.001, lambda_max=0.05, n_lambda=100,
         powell_path=1)                                                                                  # cold Powell, cox

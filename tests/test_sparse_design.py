"""Sparse (CSC) designs: bess_b200_ext.x_csc, bessgpu_load_csc, cbess.fit / the estimators on scipy.sparse input.

The bar: a sparse call sees exactly the matrix X.toarray() holds, so screening sets, chosen s, coefficients, losses, criteria
and the per-level trace are IDENTICAL to the dense call on the same matrix (the kept columns are densified into the same
n x screening_size buffer the dense gather fills).  The one computation that adds in a different order is the gaussian
screening utility (a sweep over the non-zeros instead of all n rows): equal within 1e-12 relative, and the same screening set
on these problems."""
import numpy as np
import pytest

from tests.helpers import RTOL, assert_same_support, load_golden, load_hard_golden, rel_err

sp = pytest.importorskip("scipy.sparse")

FAM = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}


def _problem(family, n=160, p=400, density=0.08, seed=0):
    """Seeded sparse design with the awkward corners: empty columns, empty rows, explicitly stored zeros, columns whose only
    non-zero sits in row 0 or in row n-1.  Returns the dense matrix, the raw CSC triple (explicit zeros kept), y, weight."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, p)) * (rng.random((n, p)) < density)
    x[:, 5] = 0.0
    x[:, 17] = 0.0
    x[7, :] = 0.0
    x[n - 3, :] = 0.0
    x[:, 9] = 0.0
    x[0, 9] = 1.5
    x[:, 11] = 0.0
    x[n - 1, 11] = -2.0
    true = [1, 3, 20, 40]
    for j in true:
        x[:, j] = rng.standard_normal(n) * (rng.random(n) < 0.5)
    eta = x[:, true] @ np.array([1.5, -1.0, 1.2, 0.8])
    if family == "gaussian":
        y = eta + 0.3 * rng.standard_normal(n)
    elif family == "binomial":
        y = (rng.random(n) < 1.0 / (1.0 + np.exp(-eta))).astype(float)
    elif family == "poisson":
        y = rng.poisson(np.exp(0.3 * eta)).astype(float)
    else:
        y = (rng.random(n) < 0.7).astype(float)  # status; rows already in time order (cbess-level calls)
    m = sp.csc_matrix(x)
    # explicit zeros: store a zero in a few columns without changing the matrix
    indptr, indices, data = m.indptr.astype(np.int64), m.indices.astype(np.int32), m.data.copy()
    extra_cols = [2, 30, 31]
    cols = [indices[indptr[j]:indptr[j + 1]] for j in range(p)]
    vals = [data[indptr[j]:indptr[j + 1]] for j in range(p)]
    for j in extra_cols:
        free = np.setdiff1d(np.arange(n), cols[j])[:2]
        r = np.concatenate([cols[j], free])
        v = np.concatenate([vals[j], np.zeros(free.size)])
        o = np.argsort(r)
        cols[j], vals[j] = r[o].astype(np.int32), v[o]
    indptr = np.concatenate([[0], np.cumsum([c.size for c in cols])]).astype(np.int64)
    triple = (indptr, np.concatenate(cols).astype(np.int32), np.concatenate(vals), (n, p))
    return x, triple, y, np.ones(n)


# ---- CPU --------------------------------------------------------------------------------------------------------------
def test_canonical_csc_sorts_sums_and_widens():
    from bess_b200.cbess import canonical_csc
    row = np.array([3, 0, 3, 1, 0, 2])
    col = np.array([0, 0, 0, 2, 2, 1])
    val = np.array([1.0, 2.0, 0.5, -1.0, 4.0, 3.0], dtype=np.float32)
    coo = sp.coo_matrix((val, (row, col)), shape=(4, 3))
    before = coo.copy()
    m = canonical_csc(coo)
    assert m.indptr.dtype == np.int64 and m.indices.dtype == np.int32 and m.data.dtype == np.float64
    assert m.has_sorted_indices and m.has_canonical_format
    assert m.indptr.tolist() == [0, 2, 3, 5]
    assert m.indices.tolist() == [0, 3, 2, 0, 1]
    assert m.data.tolist() == [2.0, 1.5, 3.0, 4.0, -1.0]
    np.testing.assert_array_equal(m.toarray(), coo.toarray().astype(np.float64))
    np.testing.assert_array_equal(coo.toarray(), before.toarray())  # the caller's matrix is untouched
    for fmt in ("csr", "csc", "lil", "dok"):
        np.testing.assert_array_equal(canonical_csc(coo.asformat(fmt)).toarray(), m.toarray())


def test_cox_row_permutation_of_a_sparse_design_matches_the_dense_one(monkeypatch):
    """PdasCox sorts the rows by time (linear.py:257-263); on sparse input it permutes the CSC rows and must hand the
    library the same matrix, response and arguments as the dense call."""
    from bess_b200 import cbess, linear
    rng = np.random.default_rng(3)
    n, p = 40, 12
    x = rng.standard_normal((n, p)) * (rng.random((n, p)) < 0.3)
    y = np.column_stack([rng.permutation(n) + 0.5, (rng.random(n) < 0.7).astype(float)])
    seen = {}

    def fake_pywrap(X, yy, *args):
        seen["dense"] = (np.array(X), np.array(yy), args)
        return [np.zeros(p), 0.0, 0.0, 0.0]

    def fake_fit(X, yy, *args, **kw):
        seen["sparse"] = (X, np.array(yy), args, kw)
        return dict(beta=np.zeros(p), coef0=0.0, train_loss=0.0, ic=0.0)

    monkeypatch.setattr(linear, "pywrap_bess", fake_pywrap)
    monkeypatch.setattr(cbess, "fit", fake_fit)
    linear.PdasCox(sequence=[1, 2]).fit(x, y)
    linear.PdasCox(sequence=[1, 2]).fit(sp.csr_matrix(x), y)
    xd, yd, args_d = seen["dense"]
    xs, ys, args_s, kw = seen["sparse"]
    assert sp.isspmatrix_csc(xs) and xs.has_sorted_indices and xs.indptr.dtype == np.int64
    np.testing.assert_array_equal(xs.toarray(), xd)
    np.testing.assert_array_equal(ys, yd)
    for a, b in zip(args_s[:12], args_d[:12]):  # data_type .. K sit at the same positions in both entries
        assert np.array_equal(a, b)
    assert list(kw["always_select"]) == [] and kw["g_index"] is None


def _raw_fit(triple, **kw):
    from bess_b200 import cbess
    y = np.zeros(triple[3][0])
    args = dict(is_screening=False, screening_size=1)
    args.update(kw)
    return cbess.fit(triple, y, 1, np.ones(y.size), True, 1, 1, 20, 2, 1, True, 3, False, 5, [1], 1, 1,
                     args.pop("is_screening"), args.pop("screening_size"), **args)


def test_csc_with_a_dense_x_or_several_gpus_is_refused_before_any_device_work():
    from bess_b200 import _lib
    n, p = 6, 3
    triple = (np.array([0, 1, 2, 3]), np.array([0, 1, 2]), np.ones(3), (n, p))
    with pytest.raises(_lib.BessB200Error, match="both given"):
        _raw_fit(triple, x_device_ptr=1 << 20)
    with pytest.raises(_lib.BessB200Error, match="single-GPU"):
        _raw_fit(triple, world=2, rank=0, col_lo=0, p_total=p, nccl_id=bytes(128))
    with pytest.raises(_lib.BessB200Error, match="single-GPU"):
        _raw_fit(triple, world=2, rank=0, nccl_id=bytes(128), fold_shard=True)


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _fit(x, g, seq, scr):
    from bess_b200 import cbess
    return cbess.fit(x, g["y"], g["data_type"], g["weight"], True, 1, g["model_type"], g.get("max_iter", 20), 2,
                     g["path_type"], g.get("warm", True), g["ic_type"], g["is_cv"], g["K"], seq, 1, g["smax"], scr > 0,
                     max(scr, 1), fold_of_row=g["fold_of_row"] if g["is_cv"] else None,
                     lambda_seq=g.get("lambda_seq", (0.0,)))


def _golden(name):
    return load_hard_golden(name[5:]) if name.startswith("hard/") else load_golden(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lm_seq_ebic_screen", "logit_seq_screen", "poisson_seq_screen", "cox_seq_screen",
                                  "hard/ar9_lm_screen", "hard/ties_lm_screen"])
def test_screening_goldens_through_csc(name):
    """The reference's own outputs, reached with x passed as CSC: screening set exact, supports exact, values within 1e-8."""
    from oracle import pdas_oracle as orc
    g = _golden(name)
    seq = np.arange(1, g["smax"] + 1)
    out = _fit(sp.csc_matrix(g["x"]), g, seq, g["scr"])
    assert_same_support(out["beta"], g["beta"])
    assert rel_err(out["beta"], g["beta"]) < RTOL
    assert abs(out["coef0"] - g["coef0"]) <= RTOL * max(1.0, abs(g["coef0"]))
    for k in ("train_loss", "ic"):
        assert abs(out[k] - g[k]) <= RTOL * max(abs(g[k]), 1e-300) or abs(out[k] - g[k]) <= 1e-12
    assert out["screening_A"].tolist() == g["screening_A"].tolist()
    if name.startswith("hard/ties_"):
        assert out["stats"]["tie_exact_pass"] and out["stats"]["n_boundary_ties"] > 0
    else:
        assert not out["stats"]["tie_exact_pass"] and out["stats"]["n_boundary_ties"] == 0
    if "beta_all" in g:
        data = orc.make_data(g["x"], g["y"], g["weight"], g["data_type"], True, g["model_type"])
        scale = np.sqrt(float(data.n)) / data.x_norm
        for lvl in range(len(seq)):
            assert_same_support(out["beta_all"][lvl], g["beta_all"][lvl])
        assert rel_err(out["beta_all"], g["beta_all"] * scale) < RTOL


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAM))
def test_screening_utilities_equal_the_dense_ones(family):
    from bess_b200.engine import GpuEngine
    x, triple, y, w = _problem(family, seed=11)
    n, p = x.shape
    model = FAM[family][0]
    e = GpuEngine()
    e.load(x, y, w, model)
    vd, idd = e.screen_local(p)
    vs, ids = e.load_csc(triple, y, w, model).screen_local(p)
    assert idd.tolist() == list(range(p)) and ids.tolist() == list(range(p))
    if family == "gaussian":
        np.testing.assert_allclose(vs, vd, rtol=1e-12, atol=0, equal_nan=True)
        assert np.isnan(vs[5]) and np.isnan(vd[5])  # an empty column: 0 / 0 in both
    else:
        np.testing.assert_array_equal(vs, vd)  # same reads, same arithmetic, same order
    e.close()


def _pair(x, y, family, scr, is_cv, K=4, fold=None, **kw):
    from bess_b200 import cbess
    model, dt = FAM[family]
    n, p = x.shape
    args = (y, dt, np.ones(n), True, kw.pop("alg", 1), model, 20, 2, kw.pop("path", 1), True, 4 if not is_cv else 1,
            is_cv, K, kw.pop("seq", np.arange(1, 7)), kw.pop("smin", 1), kw.pop("smax", 6), scr > 0, max(scr, 1))
    d = cbess.fit(x, *args, fold_of_row=fold, **kw)
    s = cbess.fit(sp.csc_matrix(x), *args, fold_of_row=fold, **kw)
    return d, s


def _assert_identical(d, s):
    for k in ("s", "coef0", "train_loss", "ic", "lam"):
        assert d[k] == s[k] or (np.isnan(d[k]) and np.isnan(s[k])), k
    np.testing.assert_array_equal(s["beta"], d["beta"])
    if "screening_A" in d:
        np.testing.assert_array_equal(s["screening_A"], d["screening_A"])
    for k in ("s_all", "l_all", "coef0_all", "loss_all", "ic_all", "beta_all", "lambda_all"):
        if d.get(k) is not None:
            np.testing.assert_array_equal(s[k], d[k], err_msg=k)


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAM))
@pytest.mark.parametrize("mode", ["screen_ic", "screen_cv", "plain_ic"])
def test_sparse_call_equals_dense_call(family, mode):
    x, _, y, _ = _problem(family, n=200, p=600, density=0.1, seed=5)
    n = x.shape[0]
    fold = np.random.default_rng(1).integers(0, 4, n).astype(np.int32) if mode == "screen_cv" else None
    scr = 0 if mode == "plain_ic" else 60
    d, s = _pair(x, y, family, scr, mode == "screen_cv", fold=fold)
    _assert_identical(d, s)
    if scr:
        assert s["stats"]["big_sweep_bytes"] < d["stats"]["big_sweep_bytes"]


@pytest.mark.gpu
def test_sparse_call_equals_dense_call_for_groups_and_pgs():
    x, _, y, _ = _problem("gaussian", n=200, p=90, density=0.15, seed=8)
    g_index = np.arange(0, 90, 3, dtype=np.int32)
    d, s = _pair(x, y, "gaussian", 0, False, alg=2, g_index=g_index)
    _assert_identical(d, s)
    d, s = _pair(x, y, "binomial", 0, True, fold=(np.arange(200) % 4).astype(np.int32), alg=5, path=2, seq=[1], smin=1,
                 smax=5, lambda_min=1e-3, lambda_max=1.0, n_lambda=10, powell_path=1)
    _assert_identical(d, s)


@pytest.mark.gpu
def test_device_resident_csc_equals_host_csc():
    import torch
    from bess_b200 import cbess
    x, triple, y, w = _problem("binomial", n=200, p=500, density=0.1, seed=21)
    args = (y, 2, w, True, 1, 2, 20, 2, 1, True, 4, False, 5, np.arange(1, 6), 1, 5, True, 40)
    h = cbess.fit(triple, *args)
    dev = tuple(torch.as_tensor(a).cuda() for a in triple[:3]) + (triple[3],)
    d = cbess.fit(dev, *args)
    _assert_identical(h, d)
    # and without screening (the whole design densified from the borrowed device arrays)
    args = args[:16] + (False, 1)
    _assert_identical(cbess.fit(triple, *args), cbess.fit(dev, *args))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["unsorted", "duplicate", "row_out_of_range", "negative_row", "colptr_decreasing",
                                  "colptr_end", "colptr_start", "device_colptr"])
def test_malformed_csc_is_refused(case):
    from bess_b200 import _lib
    n, p = 6, 3
    indptr, indices = np.array([0, 2, 3, 5]), np.array([1, 4, 2, 0, 5])
    if case == "unsorted":
        indices = np.array([4, 1, 2, 0, 5])
    elif case == "duplicate":
        indices = np.array([1, 1, 2, 0, 5])
    elif case == "row_out_of_range":
        indices = np.array([1, 6, 2, 0, 5])
    elif case == "negative_row":
        indices = np.array([1, 4, -1, 0, 5])
    elif case in ("colptr_decreasing", "device_colptr"):
        indptr = np.array([0, 3, 2, 5])
    elif case == "colptr_end":
        indptr = np.array([0, 2, 3, 4])
    elif case == "colptr_start":
        indptr = np.array([1, 2, 3, 5])
    triple = (indptr, indices, np.arange(1.0, 6.0), (n, p))
    if case == "device_colptr":
        import torch
        triple = (torch.as_tensor(indptr, dtype=torch.int64).cuda(), torch.as_tensor(indices, dtype=torch.int32).cuda(),
                  torch.arange(1.0, 6.0, dtype=torch.float64).cuda(), (n, p))
    with pytest.raises(_lib.BessB200Error, match="x_csc"):
        _raw_fit(triple)


ESTIMATORS = [a + m for a in ("Pdas", "L0L2", "GroupPdas") for m in ("Lm", "Logistic", "Poisson", "Cox")]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ESTIMATORS)
def test_estimators_on_sparse_input_equal_dense(name):
    from bess_b200 import linear
    model = name.replace("GroupPdas", "").replace("Pdas", "").replace("L0L2", "")
    family = {"Lm": "gaussian", "Logistic": "binomial", "Poisson": "poisson", "Cox": "cox"}[model]
    x, _, y, _ = _problem(family, n=150, p=60, density=0.2, seed=31)
    rng = np.random.default_rng(2)
    if family == "cox":  # unsorted times: the estimator sorts the rows
        y = np.column_stack([rng.permutation(x.shape[0]) + 1.0, y])
    kw = dict(sequence=[1, 2, 3, 4])
    if name.startswith("L0L2"):
        kw["lambda_sequence"] = [0.1, 0.01]
    fit_kw = dict(group=np.repeat(np.arange(20), 3)) if name.startswith("GroupPdas") else {}
    est = getattr(linear, name)
    dense = est(**kw).fit(x, y, **fit_kw)
    for fmt in ("csr", "csc", "coo"):
        s = est(**kw).fit(sp.csc_matrix(x).asformat(fmt), y, **fit_kw)
        np.testing.assert_array_equal(s.beta, dense.beta)
        assert (s.coef0, s.train_loss, s.ic) == (dense.coef0, dense.train_loss, dense.ic)
    if family != "cox":
        pd, ps = dense.predict(x), s.predict(sp.csr_matrix(x))
        for a, b in (zip(pd.values(), ps.values()) if isinstance(pd, dict) else [(pd, ps)]):
            np.testing.assert_allclose(b, a, rtol=1e-13, atol=1e-13)  # X @ beta summed in another order

"""Sparse designs without screening: the PDAS sweeps run on the CSC arrays and only the active columns are expanded.

The sparse path sees the implicit normalised design x~ = ((x - m) mul) rowmul with the statistics summed over the stored
entries.  Only summation orders differ from the dense path, so supports and iteration counts are identical and values
agree to rounding; the selection rule (path.cpp keep_sparse) decides between the two paths from the shape alone."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

sp = pytest.importorskip("scipy.sparse")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAM = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}


# ---- CPU: the public struct ---------------------------------------------------------------------------------------------
def test_ext_layout_keeps_every_offset_and_appends_sparse_sweeps_out(tmp_path):
    from bess_b200 import _lib
    names = [f[0] for f in _lib.Ext._fields_]
    assert names[-1] == "sparse_sweeps_out"
    src = tmp_path / "off.cpp"
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "bess_b200.h"\nint main() {\n' +
                   "".join(f'  std::printf("%zu\\n", offsetof(bess_b200_ext, {nm}));\n' for nm in names) +
                   '  std::printf("%zu\\n", sizeof(bess_b200_ext));\n  return 0;\n}\n')
    exe = tmp_path / "off"
    r = subprocess.run(["g++", "-std=c++11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    offs, size = got[:-1], got[-1]
    assert offs == [getattr(_lib.Ext, nm).offset for nm in names]  # the ctypes mirror agrees
    assert size == C.sizeof(_lib.Ext)
    assert offs[-1] == size - C.sizeof(C.c_void_p)  # the new field is last

    class Parent(C.Structure):  # the struct before the field was added: every earlier offset is unchanged
        _fields_ = _lib.Ext._fields_[:-1]
    assert [getattr(Parent, nm).offset for nm in names[:-1]] == offs[:-1]


# ---- CPU: references of the implicit-centring sweep ---------------------------------------------------------------------
LD_EPS = float(np.finfo(np.longdouble).eps)


def csc_sweep_ref(rows, vals, n, m, mul, G, W):
    """The CSC sweep's D and DH sums of one column in long double, in the kernel's form:
    d = mul (sum_stored x G - m sum G), h = mul^2 (sum_stored (x - m)^2 W + m^2 (sum W - sum_stored W)).
    Returns (d, h, first-order error bound of d, of h).  The bound carries the |m| sum|G| and m^2 sum W terms that the dense
    sweep over centred columns does not have."""
    L = np.longdouble
    x, g, w = vals.astype(L), G.astype(L)[rows], W.astype(L)[rows]
    m, mul = L(m), L(mul)
    sg, sw = np.sum(G.astype(L)), np.sum(W.astype(L))
    xc = x - m
    d = mul * (np.sum(x * g) - m * sg)
    h = mul * mul * (np.sum(xc * xc * w) + m * m * (sw - np.sum(w)))
    k = len(rows) + n + 4
    ed = k * LD_EPS * abs(mul) * (np.sum(np.abs(x * g)) + abs(m) * np.sum(np.abs(G.astype(L))))
    eh = k * LD_EPS * mul * mul * (np.sum(xc * xc * w) + (abs(m) + np.max(np.abs(xc), initial=0)) ** 2 * sw)
    return d, h, ed, eh


def _exact_dense(xcol, m, mul, G, W):
    import mpmath as mp
    mp.mp.dps = 60
    xt = [(mp.mpf(float(v)) - mp.mpf(float(m))) * mp.mpf(float(mul)) for v in xcol]
    d = mp.fsum(a * mp.mpf(float(g)) for a, g in zip(xt, G))
    h = mp.fsum(a * a * mp.mpf(float(w)) for a, w in zip(xt, W))
    return d, h


@pytest.mark.parametrize("shift", [0.0, 1.0, 1e4, -3e6])
def test_implicit_centring_references_within_their_bounds(shift):
    """Against the dense definition sum_i x~_i G_i / x~_i^2 W_i in 60 digits, on columns whose mean dwarfs their spread
    (shift): the long-double references stay inside their first-order bounds, and W >= 0 keeps every term of h >= 0."""
    rng = np.random.default_rng(7)
    n = 300
    for trial in range(6):
        rows = np.sort(rng.choice(n, size=int(rng.integers(0, n + 1)), replace=False))
        vals = shift + rng.standard_normal(rows.size)
        if trial == 1 and rows.size:
            vals[0] = 0.0  # an explicitly stored zero
        xcol = np.zeros(n)
        xcol[rows] = vals
        w = rng.random(n) + 0.1
        m = float(np.dot(xcol, w / n))
        mul = 0.37
        G, W = rng.standard_normal(n), rng.random(n)
        d, h, ed, eh = csc_sweep_ref(rows, vals, n, m, mul, G, W)
        de, he = _exact_dense(xcol, m, mul, G, W)
        assert abs(float(d) - float(de)) <= float(ed) + 1e-300
        assert abs(float(h) - float(he)) <= float(eh) + 1e-300
        assert h >= 0


def cox_r_ref(rows, vals, th, c2, mul):
    """The CSC sweep's Cox R of one column in long double, in the kernel's form R = mul^2 sum_t (P_{i_t} - P_{i_{t-1}}) S_t^2
    (P the row prefix of C2, S_t the suffix of th x over the column's entries), and its first-order error bound.  The
    difference of prefix sums is exact in value but carries the rounding of P_{i_t} and P_{i_{t-1}} themselves: the bound
    grows with the prefix, i.e. when an early C2 term dominates the later ones."""
    L = np.longdouble
    P = np.cumsum(c2.astype(L))
    v = vals.astype(L) * th.astype(L)[rows]
    S = np.cumsum(v[::-1])[::-1]
    Sa = np.cumsum(np.abs(v)[::-1])[::-1]
    Pp = np.concatenate([[L(0)], P[rows[:-1]]]) if rows.size else np.zeros(0, dtype=L)
    dP = P[rows] - Pp
    R = L(mul) * L(mul) * np.sum(dP * S * S)
    k = c2.size + rows.size + 8
    eR = k * LD_EPS * L(mul) * L(mul) * np.sum((P[rows] + Pp + dP) * Sa * Sa)
    return R, eR


@pytest.mark.parametrize("early", [1.0, 1e6, 1e12])
def test_cox_r_reference_within_its_bound(early):
    """Against the dense definition sum_k C2_k s1_k^2 (s1_k = sum_{i >= k} th_i x_i) in 60 digits, with the first C2 term
    `early` times the others: the row-0 and row n-1 edges, an explicit zero and a full column included."""
    import mpmath as mp
    mp.mp.dps = 60
    rng = np.random.default_rng(5)
    n = 200
    c2 = rng.random(n) + 0.1
    c2[0] *= early
    th = rng.random(n) + 0.5
    cases = [np.array([0]), np.array([n - 1]), np.array([0, 7, n - 1]), np.arange(n),
             np.sort(rng.choice(n, 40, replace=False))]
    for rows in cases:
        vals = rng.standard_normal(rows.size)
        vals[rows.size // 2] = 0.0 if rows.size > 2 else vals[rows.size // 2]
        R, eR = cox_r_ref(rows, vals, th, c2, 0.9)
        x = np.zeros(n)
        x[rows] = vals
        s1 = mp.mpf(0)
        exact = mp.mpf(0)
        for k in range(n - 1, -1, -1):
            s1 += mp.mpf(float(x[k])) * mp.mpf(float(th[k]))
            exact += mp.mpf(float(c2[k])) * s1 * s1
        exact *= mp.mpf(0.9) ** 2
        assert abs(float(R) - float(exact)) <= float(eR) + 1e-300, (rows.size, early)
        assert R >= 0


# ---- GPU: engine level --------------------------------------------------------------------------------------------------
def _small(family, seed=0, n=160, p=300, weights=True):
    """_problem's design with its explicitly stored zeros kept, plus a fully stored column with a large mean (60) and a
    column whose entries sit in row 0 and one inner row (13: the first-entry edge of the Cox suffix)."""
    from tests.test_sparse_design import _problem
    x, (indptr, indices, data, _), y, _ = _problem(family, n=n, p=p, seed=seed)
    rng = np.random.default_rng(seed)
    cols = [[indices[indptr[j]:indptr[j + 1]], data[indptr[j]:indptr[j + 1]]] for j in range(p)]
    cols[60] = [np.arange(n, dtype=np.int32), rng.standard_normal(n) + 4.0]
    cols[13] = [np.array([0, n // 2], dtype=np.int32), np.array([1.3, -0.7])]
    if family == "cox":
        # a Cox column whose only entry is the first row of the risk order has l2 = h - R equal to rounding noise on
        # either path (its one term in h and in R coincide), so which of such columns a fit selects is undefined
        cols[9] = [np.zeros(0, dtype=np.int32), np.zeros(0)]
    x = np.zeros((n, p))
    for j, (r, v) in enumerate(cols):
        x[r, j] = v
    ip = np.concatenate([[0], np.cumsum([c[0].size for c in cols])]).astype(np.int64)
    triple = (ip, np.concatenate([c[0] for c in cols]).astype(np.int32), np.concatenate([c[1] for c in cols]), (n, p))
    assert (triple[2] == 0).sum() >= 3  # the stored zeros survive
    w = rng.random(n) + 0.5 if weights else np.ones(n)
    return x, triple, y, w


def _skewed(family, seed, n=700, p=400):
    """Power-law column lengths: most columns hold 1-3 entries, a few hold hundreds, three are fully stored (the frequent
    terms of text data); explicit zeros included."""
    rng = np.random.default_rng(seed)
    lens = np.minimum(n, np.maximum(1, (0.3 * n / (1.0 + rng.permutation(p)) ** 1.1).astype(int)))
    lens[[5, 77, 301]] = n
    # one-entry columns at distinct rows, never row 0: two one-entry columns in the same row normalise to the same column
    # up to sign (an exact tie that rounding breaks either way), and for Cox a row-0 one has l2 = rounding noise (_small)
    single = iter(rng.permutation(np.arange(1, n)))
    rows = [np.sort(rng.choice(n, size=k, replace=False) if k > 1 else [next(single)]).astype(np.int32) for k in lens]
    vals = [rng.standard_normal(k) for k in lens]
    vals[7][0] = 0.0
    x = np.zeros((n, p))
    for j in range(p):
        x[rows[j], j] = vals[j]
    eta = 0.8 * x[:, 5] - 0.6 * x[:, 1] + 0.5 * x[:, 77]
    if family == "gaussian":
        y = eta + 0.3 * rng.standard_normal(n)
    elif family == "binomial":
        y = (rng.random(n) < 1.0 / (1.0 + np.exp(-eta))).astype(float)
    elif family == "poisson":
        y = rng.poisson(np.exp(0.3 * eta)).astype(float)
    else:
        y = (rng.random(n) < 0.7).astype(float)
    ip = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    return x, (ip, np.concatenate(rows), np.concatenate(vals), (n, p)), y, rng.random(n) + 0.5


def _engines(family, is_normal, K, seed=0, kcap=6, design=None):
    from bess_b200.engine import GpuEngine
    model, dt = FAM[family]
    x, triple, y, w = (design or _small)(family, seed)
    n = x.shape[0]
    folds = (np.arange(n) % K).astype(np.int32) if K else None
    ed, es = GpuEngine(), GpuEngine()
    ed.load(x, y, w, model)
    ed.normalize(dt, is_normal)
    es.load_csc(triple, y, w, model)
    stats = es.normalize(dt, is_normal)
    es.case = dict(y=y, w=w, ym=stats[2] if stats is not None else 0.0)
    return x, ed, es, folds


def _rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)) if a.size else 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAM))
@pytest.mark.parametrize("is_normal", [True, False])
def test_engine_design_and_statistics_equal_the_dense_ones(family, is_normal):
    """Normalised design and column statistics: summation order only, so within 16 ulps (relative 4e-15) of the dense
    engine on every entry, empty and explicitly stored zero columns included."""
    x, ed, es, _ = _engines(family, is_normal, 0)
    Xd, Xs = ed.design(), es.design()
    ok = np.isfinite(Xd)  # an empty column normalises to 0/0 on both paths
    assert np.array_equal(ok, np.isfinite(Xs))
    np.testing.assert_allclose(Xs[ok], Xd[ok], rtol=4e-15, atol=4e-15 * np.max(np.abs(Xd[ok])))
    ed.close()
    es.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAM))
@pytest.mark.parametrize("K", [0, 3, 5, 7, 11, 15, 23, 31])
def test_engine_fits_losses_and_sacrifice_equal_the_dense_ones(family, K):
    """run_batch: same supports and PDAS iteration counts, coefficients within 1e-10; losses within 1e-12; the sacrifice
    of every chain through the CSC sweep (FS = 1 .. 32) within 1e-9 of the dense sweep's."""
    x, ed, es, folds = _engines(family, True, K, seed=K)
    n, p = x.shape
    always = ()
    for e in (ed, es):
        e.setup_chains(K, folds, 6, always_select=always)
    chains = list(range(K + 1))
    for T in (1, 3, 6):
        rd, rs = ed.run_batch(T, chains), es.run_batch(T, chains)
        assert np.array_equal(rd["A"], rs["A"]) and np.array_equal(rd["l"], rs["l"])
        assert _rel(rs["bA"], rd["bA"]) < 1e-10
        assert _rel(rs["coef0"], rd["coef0"]) < 1e-10 or np.max(np.abs(rs["coef0"] - rd["coef0"])) < 1e-12
        jobs = [(0, 0, 0)] + [(c, 1, c - 1) for c in range(1, K + 1)]
        assert _rel(es.losses(jobs), ed.losses(jobs)) < 1e-12
    bd, info = ed.sacrifice(chains)
    bs, info_s = es.sacrifice(chains)
    assert info_s["kernel"] == "csc" and info_s["FS"] == info["FS"] and info_s["S"] == 1
    # a column without entries in a chain's train rows has 0 / 0 on both paths (e.g. the row n-1 column in its fold)
    assert np.array_equal(np.isfinite(bs), np.isfinite(bd))
    ok = np.isfinite(bd)
    assert np.max(np.abs(bs[ok] - bd[ok])) <= 1e-9 * np.max(np.abs(bd[ok]))
    ed.close()
    es.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAM))
@pytest.mark.parametrize("K", [0, 3, 5, 7, 11, 15, 23, 31])
@pytest.mark.parametrize("design", ["small", "skewed"])
def test_engine_sacrifice_within_the_long_double_references(family, K, design):
    """The sacrifice of every chain and column through the CSC sweep (every FS the engine instantiates) against the
    long-double references of test_sacrifice.py on the normalised design, within their bounds.  The skewed design puts
    its long columns on the one-CTA-per-column kernel."""
    from tests.test_sacrifice import LD, sacrifice_ref
    x, ed, es, folds = _engines(family, True, K, seed=100 + K, design=_skewed if design == "skewed" else None)
    ed.close()
    n, p = x.shape
    es.setup_chains(K, folds, 4)
    chains = list(range(K + 1))
    X = es.design().astype(LD)
    y, w = es.case["y"], es.case["w"]
    yf = (y - es.case["ym"]) * np.sqrt(w) if family == "gaussian" else y
    for T in (1, 3):
        r = es.run_batch(T, chains)
        bd, info = es.sacrifice(chains)
        assert info["kernel"] == "csc" and info["S"] == 1
        if design == "skewed":
            assert info["long_columns"] >= 3
        for i, c in enumerate(chains):
            rows = np.arange(n) if c == 0 else np.flatnonzero(folds != c - 1)
            beta = np.zeros(p)
            beta[r["A"][i]] = r["bA"][i]
            ok = np.all(np.isfinite(X[rows]), axis=0)  # an empty column normalises to 0 / 0
            ref, bound = sacrifice_ref(family, X[rows][:, ok], yf[rows], w[rows], beta[ok], float(r["coef0"][i]),
                                       len(r["A"][i]), 0.0)
            # a column without entries in the chain's train rows: 0 / 0 in the reference and in the kernel
            fin = np.isfinite(ref.astype(np.float64))
            assert np.array_equal(fin, np.isfinite(bd[i][ok]))
            err = np.abs(bd[i][ok].astype(LD) - ref).astype(np.float64)
            bad = np.flatnonzero(fin & ~(err <= bound))
            assert bad.size == 0, (family, K, T, c, np.flatnonzero(ok)[bad[:6]].tolist(), err[bad[:6]].tolist(),
                                   bound[bad[:6]].tolist())
    es.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAM))
def test_engine_skewed_design_equals_the_dense_one(family):
    x, ed, es, folds = _engines(family, True, 5, seed=3, design=_skewed)
    for e in (ed, es):
        e.setup_chains(5, folds, 6)
    for T in (1, 3, 6):
        rd, rs = ed.run_batch(T, list(range(6))), es.run_batch(T, list(range(6)))
        assert np.array_equal(rd["A"], rs["A"]) and np.array_equal(rd["l"], rs["l"])
        assert _rel(rs["bA"], rd["bA"]) < 1e-10
    ed.close()
    es.close()


# ---- GPU: public call ---------------------------------------------------------------------------------------------------
def _big(family, seed, n=2000, p=70000, density=0.01, weights=False):
    """A design whose dense form is just over 1 GiB at 1 % density, with a planted support."""
    rng = np.random.default_rng(seed)
    m = sp.random(n, p, density=density, format="csc", random_state=rng, data_rvs=rng.standard_normal)
    true = [j for j in (3, 500, 7000, 40001, 69999) if j < p]
    coef = np.array([1.5, -1.2, 1.0, 0.9, -1.1])[:len(true)]
    lil = m.tolil()
    for j in true:
        lil[:, j] = (rng.standard_normal(n) * (rng.random(n) < 0.3)).reshape(-1, 1)
    m = lil.tocsc()
    m.sort_indices()
    eta = m[:, true] @ coef
    if family == "gaussian":
        y = eta + 0.3 * rng.standard_normal(n)
    elif family == "binomial":
        y = (rng.random(n) < 1.0 / (1.0 + np.exp(-eta))).astype(float)
    elif family == "poisson":
        y = rng.poisson(np.exp(0.3 * eta)).astype(float)
    else:
        t = rng.exponential(1.0 / np.exp(0.5 * eta))
        o = np.argsort(t)
        m = m[o, :].tocsc()
        m.sort_indices()
        y = (rng.random(n) < 0.8).astype(float)
    w = rng.random(n) + 0.5 if weights else np.ones(n)
    return m, y, w, true


def _call(x, y, w, family, **kw):
    from bess_b200 import cbess
    model, dt = FAM[family]
    kw = dict(kw)
    path = kw.pop("path", 1)
    is_cv = kw.pop("is_cv", False)
    K = kw.pop("K", 10)
    seq = kw.pop("seq", np.arange(1, 9))
    return cbess.fit(x, y, dt, w, True, kw.pop("alg", 1), model, 20, 2, path, True, kw.pop("ic", 3), is_cv, K, seq,
                     kw.pop("smin", 1), kw.pop("smax", 8), False, 1, fold_of_row=kw.pop("fold", None), **kw)


def _assert_same(a, b, tol=1e-10):
    assert a["s"] == b["s"]
    assert np.array_equal(np.flatnonzero(a["beta"]), np.flatnonzero(b["beta"]))
    assert _rel(a["beta"], b["beta"]) < tol
    for k in ("coef0", "train_loss", "ic"):
        assert abs(a[k] - b[k]) <= tol * max(abs(b[k]), 1e-12)
    for k in ("s_all", "l_all"):
        if b.get(k) is not None:
            assert np.array_equal(a[k], b[k])
    for k in ("beta_all",):
        if b.get(k) is not None:
            assert np.array_equal(a[k] != 0, b[k] != 0)
            assert _rel(a[k], b[k]) < tol
    if b.get("ic_all") is not None:
        assert _rel(a["ic_all"], b["ic_all"]) < tol


CASES = [
    ("gaussian", dict()), ("binomial", dict()), ("poisson", dict()), ("cox", dict()),
    ("gaussian", dict(is_cv=True, ic=1)), ("binomial", dict(is_cv=True, ic=1)),
    ("poisson", dict(is_cv=True, ic=1)), ("cox", dict(is_cv=True, ic=1)),
    ("gaussian", dict(is_cv=True, ic=1, path=2)), ("binomial", dict(is_cv=True, ic=1, path=2)),
    ("poisson", dict(is_cv=True, ic=1, path=2)), ("cox", dict(is_cv=True, ic=1, path=2)),
    ("gaussian", dict(alg=5, lambda_seq=(0.0, 0.1, 1.0))),
    ("binomial", dict(alg=5, path=2, lambda_min=0.01, lambda_max=1.0, n_lambda=3, powell_path=2, is_cv=True, ic=1, K=5)),
    ("gaussian", dict(always_select=(10, 20))),
    ("gaussian", dict(is_cv=True, ic=1, K=31, weights=True)),
    ("poisson", dict(weights=True)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("family,kw", CASES, ids=[f"{f}-{i}" for i, (f, _) in enumerate(CASES)])
def test_public_call_equals_the_dense_call(family, kw):
    kw = dict(kw)
    m, y, w, true = _big(family, seed=len(kw) * 7 + list(FAM).index(family), weights=kw.pop("weights", False))
    s = _call(m, y, w, family, want_trace=True, **kw)
    assert s["stats"]["sparse_sweeps"] == 1
    d = _call(m.toarray(), y, w, family, want_trace=True, **kw)
    assert d["stats"]["sparse_sweeps"] == 0
    _assert_same(s, d)


@pytest.mark.gpu
def test_public_call_is_reproducible_and_device_arrays_agree():
    import torch
    m, y, w, true = _big("gaussian", seed=5)
    a = _call(m, y, w, "gaussian", is_cv=True, ic=1)
    b = _call(m, y, w, "gaussian", is_cv=True, ic=1)
    cp, ri, cv = (torch.as_tensor(v).cuda() for v in (m.indptr.astype(np.int64), m.indices.astype(np.int32), m.data))
    c = _call((cp, ri, cv, m.shape), y, w, "gaussian", is_cv=True, ic=1)
    for r in (b, c):
        assert r["stats"]["sparse_sweeps"] == 1
        assert np.array_equal(a["beta"], r["beta"]) and a["s"] == r["s"]
        for k in ("coef0", "train_loss", "ic"):
            assert a[k] == r[k]
    assert set(np.flatnonzero(a["beta"])) == set(true)


@pytest.mark.gpu
def test_both_sides_of_the_rule():
    # under 1 GiB dense: densified, bit for bit the dense call
    m, y, w, _ = _big("gaussian", seed=9, p=20000)
    s, d = _call(m, y, w, "gaussian"), _call(m.toarray(), y, w, "gaussian")
    assert s["stats"]["sparse_sweeps"] == 0
    assert np.array_equal(s["beta"], d["beta"]) and s["ic"] == d["ic"] and s["coef0"] == d["coef0"]
    # over 1 GiB but denser than 1 / 24 of the dense bytes (12 nnz > dense / 24 above ~ 2.8 %): densified
    m, y, w, _ = _big("gaussian", seed=10, p=70000, density=0.04)
    assert _call(m, y, w, "gaussian")["stats"]["sparse_sweeps"] == 0
    # a large grouped call keeps today's behaviour (densified, group kernels)
    m, y, w, _ = _big("gaussian", seed=11)
    g = np.arange(0, 70000, 2, dtype=np.int32)
    out = _call(m, y, w, "gaussian", alg=2, g_index=g, seq=np.arange(1, 4), smax=3)
    assert out["stats"]["sparse_sweeps"] == 0


@pytest.mark.gpu
def test_capacity_dense_form_larger_than_the_device():
    """200 GB dense, 600 MB CSC: runs without screening on the sparse path and recovers its planted support."""
    rng = np.random.default_rng(21)
    n, p, per = 5000, 5_000_000, 10
    gap = n // per
    true = np.array([11, 2_000_003, 4_999_990])
    counts = np.full(p, per, dtype=np.int64)
    counts[true] = n  # the planted columns are fully stored
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    rows = (rng.integers(0, gap, size=(p, 1)) + gap * np.arange(per)).astype(np.int32)  # distinct, increasing
    ri = np.empty(indptr[-1], dtype=np.int32)
    cv = rng.standard_normal(indptr[-1])
    mask = np.ones(p, dtype=bool)
    mask[true] = False
    sparse_pos = (indptr[:-1][mask][:, None] + np.arange(per)).ravel()
    ri[sparse_pos] = rows[mask].ravel()
    eta = np.zeros(n)
    for j, c in zip(true, (2.0, -1.5, 1.8)):
        ri[indptr[j]:indptr[j + 1]] = np.arange(n, dtype=np.int32)
        eta += c * cv[indptr[j]:indptr[j + 1]]
    y = eta + 0.5 * rng.standard_normal(n)
    out = _call((indptr, ri, cv, (n, p)), y, np.ones(n), "gaussian", seq=np.arange(1, 6), smax=5, ic=4)
    assert out["stats"]["sparse_sweeps"] == 1
    assert set(np.flatnonzero(out["beta"])) == set(true.tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["gaussian", "binomial"])
def test_public_call_against_the_reference_arithmetic(family):
    """The reference's own algorithm (oracle.pdas_oracle.bess_cpp) on the same matrix, few levels: support exact, values
    within RTOL."""
    from oracle import pdas_oracle as orc
    from tests.helpers import RTOL, assert_same_support, rel_err
    m, y, w, _ = _big(family, seed=31)
    model, dt = FAM[family]
    seq = np.arange(1, 4)
    out = _call(m, y, w, family, seq=seq, smax=3)
    assert out["stats"]["sparse_sweeps"] == 1
    exp = orc.bess_cpp(m.toarray(), y, dt, w, True, model, 20, 1, True, 3, False, 10, seq, 1, 3, False, 1)
    assert_same_support(out["beta"], exp["beta"])
    assert rel_err(out["beta"], exp["beta"]) < RTOL
    assert abs(out["coef0"] - exp["coef0"]) <= RTOL * max(1.0, abs(exp["coef0"]))
    for k in ("train_loss", "ic"):
        assert abs(out[k] - exp[k]) <= RTOL * max(abs(exp[k]), 1e-300)

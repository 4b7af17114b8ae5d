"""CPU restatement (numpy, fp64) of the BeSS primal-dual active-set hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``bess_b200/`` may import this module;
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline leg do,
and only as the *checker*.

Parity status: PINNED.  ``tests/test_oracle_golden.py`` checks every function here
against outputs of the real reference (Mamba413/bess ``src/*.cpp`` compiled unmodified
into ``oracle/_ref/libbess_ref.so`` by ``oracle/Makefile``; fixtures committed under
``tests/golden/`` by ``tests/golden/make_golden.py``).  The reference itself ships no
golden vectors or tests (SURVEY.md section 4).

All ``file:line`` citations are into ``/root/reference/src``.  Everything is the
gsize==1, lambda==0 specialisation that ``bessCpp`` reaches for ``type="bss"``.

``max_k`` boundary ties: the reference's order among *exactly equal* keys that
straddle the k-th position is whatever libstdc++'s introselect leaves
(utilities.cpp:179-188); ``nth_element`` below replays that algorithm step for step.

Known, deliberate deviation from the reference (none changes a result):
  * CV fold assignment is an *input* (``fold_of_row``) because it comes from
    ``std::shuffle(mt19937)`` (Metric.h:49-106); the golden fixtures store it.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

DBL_MAX = np.finfo(np.float64).max


# --------------------------------------------------------------------------------------
# Data + normalisation: Data.h:41-77, normalize.cpp:20-86
# --------------------------------------------------------------------------------------
@dataclass
class Data:
    x: np.ndarray  # n x p, normalised (and sqrt(w)-row-scaled for gaussian)
    y: np.ndarray
    weight: np.ndarray
    x_mean: np.ndarray
    x_norm: np.ndarray
    y_mean: float
    data_type: int
    is_normal: bool
    n: int = 0
    p: int = 0


def make_data(x, y, weight, data_type, is_normal, model_type):
    """Data ctor (Data.h:41-68) + Normalize/Normalize3/Normalize4 (normalize.cpp:20-86)
    + add_weight for gaussian (Data.h:70-77, called from bess.cpp:97)."""
    x = np.array(x, dtype=np.float64, order="F", copy=True)
    y = np.array(y, dtype=np.float64, copy=True)
    w = np.array(weight, dtype=np.float64, copy=True)
    n, p = x.shape
    x_mean = np.zeros(p)
    x_norm = np.zeros(p)
    y_mean = 0.0
    if is_normal:
        if data_type in (1, 2):
            x_mean = (w @ x) / float(n)  # normalize.cpp:25-28 / 52-55
            x = x - x_mean
        if data_type == 1:
            y_mean = float(y @ w) / float(n)  # normalize.cpp:29
            y = y - y_mean
        x_norm = np.sqrt(w @ (x * x))  # normalize.cpp:36-41
        x = math.sqrt(float(n)) * x / x_norm  # normalize.cpp:42-45
    if model_type == 1:
        sw = np.sqrt(w)  # Data.h:70-77
        x = x * sw[:, None]
        y = y * sw
    return Data(np.asfortranarray(x), y, w, x_mean, x_norm, y_mean, data_type, is_normal, n, p)


# --------------------------------------------------------------------------------------
# Selection: utilities.cpp:179-199
# --------------------------------------------------------------------------------------
TIES = {"count": 0}  # boundary ties met by max_k since import (tests reset and read it)


def _sift_down(a, first, hole, length, value, comp):
    """libstdc++ std::__adjust_heap + std::__push_heap on a[first:first + length]."""
    top, child = hole, hole
    while child < (length - 1) // 2:
        child = 2 * (child + 1)
        if comp(a[first + child], a[first + child - 1]):
            child -= 1
        a[first + hole] = a[first + child]
        hole = child
    if length % 2 == 0 and child == (length - 2) // 2:
        child = 2 * (child + 1)
        a[first + hole] = a[first + child - 1]
        hole = child - 1
    parent = (hole - 1) // 2
    while hole > top and comp(a[first + parent], value):
        a[first + hole] = a[first + parent]
        hole = parent
        parent = (hole - 1) // 2
    a[first + hole] = value


def nth_element(a, nth, comp):
    """std::nth_element(a.begin(), a.begin() + nth, a.end(), comp) as libstdc++ implements it (bits/stl_algo.h:
    __introselect with depth limit 2 * floor(log2(n)), median-of-three pivot, unguarded partition, insertion sort of the
    last <= 3 elements, heap select once the depth limit is spent), on the Python list `a` in place.  Which of several
    keys equal under `comp` end up in front of `nth` is fixed by these steps alone."""
    first, last = 0, len(a)
    if first == last or nth == last:
        return
    depth = 2 * ((last - first).bit_length() - 1)
    while last - first > 3:
        if depth == 0:
            middle = nth + 1
            length = middle - first
            for parent in range((length - 2) // 2, -1, -1) if length >= 2 else ():
                _sift_down(a, first, parent, length, a[first + parent], comp)
            for i in range(middle, last):
                if comp(a[i], a[first]):
                    value, a[i] = a[i], a[first]
                    _sift_down(a, first, 0, length, value, comp)
            a[first], a[nth] = a[nth], a[first]
            return
        depth -= 1
        mid = first + (last - first) // 2
        x, y, z = first + 1, mid, last - 1  # __move_median_to_first
        if comp(a[x], a[y]):
            m = y if comp(a[y], a[z]) else (z if comp(a[x], a[z]) else x)
        else:
            m = x if comp(a[x], a[z]) else (z if comp(a[y], a[z]) else y)
        a[first], a[m] = a[m], a[first]
        lo, hi = first + 1, last  # __unguarded_partition around a[first]
        while True:
            while comp(a[lo], a[first]):
                lo += 1
            hi -= 1
            while comp(a[first], a[hi]):
                hi -= 1
            if not lo < hi:
                break
            a[lo], a[hi] = a[hi], a[lo]
            lo += 1
        if lo <= nth:
            first = lo
        else:
            last = lo
    for i in range(first + 1, last):  # __insertion_sort
        v = a[i]
        if comp(v, a[first]):
            a[first + 1:i + 1] = a[first:i]
            a[first] = v
        else:
            j = i
            while comp(v, a[j - 1]):
                a[j] = a[j - 1]
                j -= 1
            a[j] = v


def max_k(vec, k):
    """Indices of the k largest entries, returned ascending (utilities.cpp:179-188).
    Tie rule at the boundary: see module docstring."""
    p = vec.shape[0]
    order = np.lexsort((np.arange(p), -vec))  # primary: value desc; secondary: index asc
    if k < p and vec[order[k - 1]] == vec[order[k]]:
        # a boundary tie: the reference leaves its resolution to std::nth_element over the index array 0..p-1 with the
        # comparator vec(i) > vec(j), then sorts the first k -- replayed step for step
        TIES["count"] += 1
        v = vec.tolist()
        ind = list(range(p))
        nth_element(ind, k, lambda i, j: v[i] > v[j])
        return np.sort(np.array(ind[:k], dtype=np.int32))
    return np.sort(order[:k]).astype(np.int32)


def boundary_gap(vec, k):
    """Relative gap between the k-th and (k+1)-th largest sacrifice (SURVEY 8c: margin logging)."""
    if k >= vec.shape[0]:
        return np.inf
    s = np.sort(vec)[::-1]
    return float((s[k - 1] - s[k]) / max(abs(s[k - 1]), 1e-300))


# --------------------------------------------------------------------------------------
# log-likelihoods: logistic.cpp:15-59, poisson.cpp:15-82, coxph.cpp:16-40
# --------------------------------------------------------------------------------------
def _clip(v, c):
    return np.minimum(np.maximum(v, -c), c)


def loglik_cox(X, status, beta, weights):
    """coxph.cpp:16-40 (rows time-sorted; suffix sums are the risk sets)."""
    eta = _clip(X @ beta, 30.0)
    e = np.exp(eta)
    cum = np.cumsum(e[::-1])[::-1]
    return float((np.log(e / cum) * status) @ weights)


def _log_factorial_term(y):
    """poisson.cpp:29-44: sum_{j=1..y} log(j), with y==1 short-circuited to 0."""
    out = np.zeros_like(y)
    for i, yi in enumerate(y):
        if yi == 1:
            out[i] = 0.0
        else:
            t = 0.0
            j = 1.0
            while j <= yi:
                t += math.log(j)
                j += 1.0
            out[i] = t
    return out


def loglik_poisson(x, y, coef, weights):
    """poisson.cpp:15-47 (coef[0] is the intercept; includes the -log y! term)."""
    eta = _clip(x @ coef[1:] + coef[0], 30.0)
    return float((y * eta - np.exp(eta) - _log_factorial_term(y)) @ weights)


def loglik_poiss(x, y, coef, weights):
    """poisson.cpp:67-82 (no factorial term)."""
    eta = _clip(x @ coef[1:] + coef[0], 30.0)
    return float((y * eta - np.exp(eta)) @ weights)


# --------------------------------------------------------------------------------------
# primary_model_fit x4: Algorithm.h:1131-1135, 1148-1204, 1273-1322, 1377-1490
# --------------------------------------------------------------------------------------
PIVOT_TOL = 1e-13


def solve_rank_revealing(G, b):
    """The normal-equation solve of primary_model_fit on a system that may be singular.  The reference factors with
    colPivHouseholderQr (Algorithm.h:1134) / Eigen's pivoted ldlt (:1171, :1299); on an active set that holds an EXACTLY
    duplicated column both drop the second copy -- the QR truncates at its rank threshold, the LDLT meets an exactly zero
    pivot that its solve() skips (Eigen/src/Cholesky/LDLT.h:558-592) -- and the unknown gets a zero coefficient.
    Full-rank systems take numpy's LU; a system whose Cholesky pivots fall to PIVOT_TOL of the column's own diagonal is
    solved by LDL^T with Eigen's diagonal pivoting that stops when no remaining pivot passes that bound and leaves the
    remaining unknowns at 0."""
    G = np.asarray(G, dtype=np.float64)
    dg = np.diag(G)
    try:
        L = np.linalg.cholesky(G)
        if np.all(np.diag(L) ** 2 > PIVOT_TOL * dg):
            return np.linalg.solve(G, b)
    except np.linalg.LinAlgError:
        pass
    m = G.shape[0]
    S = G.copy()
    y = np.asarray(b, dtype=np.float64).copy()
    # Eigen's pivoting (LDLT.h:300-330): at step k the FIRST largest diagonal entry in the current positional order of the
    # remaining unknowns, which is then swapped into position k -- the unknown that sat at k moves back to where the
    # pivot came from.  Which copy of a duplicated column is met first therefore depends on the swaps made so far.
    perm = list(range(m))
    mult = {}
    rank = 0
    for k in range(m):
        best, bpos = -1.0, -1
        for pos in range(k, m):
            p = perm[pos]
            if S[p, p] > PIVOT_TOL * dg[p] and S[p, p] > best:
                best, bpos = S[p, p], pos
        if bpos < 0:
            break
        perm[k], perm[bpos] = perm[bpos], perm[k]
        p = perm[k]
        rest = np.zeros(m, dtype=bool)
        rest[perm[k + 1:]] = True
        l = np.where(rest, S[:, p] / S[p, p], 0.0)
        S[np.ix_(rest, rest)] -= np.outer(l[rest], S[p, rest])
        y[rest] -= l[rest] * y[p]
        mult[p] = l
        rank += 1
    x = np.zeros(m)
    for k in range(rank - 1, -1, -1):
        p = perm[k]
        x[p] = y[p] / S[p, p] - sum(mult[p][q] * x[q] for q in perm[k + 1:rank])
    return x


def fit_lm(XA, y, w, coef0, lam=0.0):
    """Algorithm.h:1131-1135.  coef0 untouched.  lam: X'X + lambda*I (:1134, not 2*lambda, not scaled by n)."""
    G = XA.T @ XA + lam * np.eye(XA.shape[1])
    beta = solve_rank_revealing(G, XA.T @ y)
    return beta, coef0


def _pi(X1, coef):
    """logistic.cpp:15-59 with the intercept column already in X1."""
    eta = _clip(X1 @ coef, 30.0)
    e = np.exp(eta)
    return e / (1.0 + e)


def fit_logistic(XA, y, w, coef0, floor_w=True, lam=0.0):
    """Algorithm.h:1148-1204 (floor_w=True) and logistic.cpp:61-157 ``logit_fit`` (floor_w=False).
    Starts from 0, returns the iterate *before* the last solve."""
    n, k = XA.shape
    X = np.hstack([np.ones((n, 1)), XA])
    beta0 = np.zeros(k + 1)
    lmat = 2.0 * lam * np.eye(k + 1)  # 2*lambda*lambdamat, lambdamat(0,0) = 0 (:1158-1159, :1171)
    lmat[0, 0] = 0.0
    Pi = _pi(X, beta0)
    ll0 = float((y * np.log(Pi) + (1 - y) * np.log(1 - Pi)) @ w)
    W = Pi * (1 - Pi)
    Z = X @ beta0 + (y - Pi) / W
    W = W * w
    beta1 = solve_rank_revealing(lmat + (X * W[:, None]).T @ X, (X * W[:, None]).T @ Z)
    for _ in range(30):
        Pi = _pi(X, beta1)
        ll1 = float((y * np.log(Pi) + (1 - y) * np.log(1 - Pi)) @ w)
        if abs(ll0 - ll1) / (0.1 + abs(ll1)) < 1e-6:
            break
        beta0 = beta1
        ll0 = ll1
        W = Pi * (1 - Pi)
        if floor_w:
            W = np.maximum(W, 0.001)
        Z = X @ beta0 + (y - Pi) / W
        W = W * w
        beta1 = solve_rank_revealing(lmat + (X * W[:, None]).T @ X, (X * W[:, None]).T @ Z)
    return beta0[1:].copy(), float(beta0[0])


def fit_poisson(XA, y, w, coef0, lam=0.0):
    """Algorithm.h:1273-1322.  Intercept warm-started from coef0, slopes from 0."""
    n, k = XA.shape
    X = np.hstack([np.ones((n, 1)), XA])
    beta0 = np.zeros(k + 1)
    beta0[0] = coef0
    lmat = 2.0 * lam * np.eye(k + 1)  # :1299
    lmat[0, 0] = 0.0
    eta = X @ beta0
    expeta = np.exp(eta)
    ll0 = 1e5
    for _ in range(50):
        ww = expeta * w
        z = eta + (y - expeta) / expeta
        XtW = (X * ww[:, None]).T
        beta0 = solve_rank_revealing(lmat + XtW @ X, XtW @ z)
        eta = _clip(X @ beta0, 30.0)
        expeta = np.maximum(np.exp(eta), 0.001)
        ll1 = float((y * eta - expeta) @ w)
        if abs(ll0 - ll1) / abs(0.1 + ll0) < 1e-6:
            break
        ll0 = ll1
    return beta0[1:].copy(), float(beta0[0])


def fit_cox(XA, status, w, coef0, clamp=30.0, lam=0.0):
    """Algorithm.h:1377-1490 (clamp 30) and coxph.cpp:42-109 ``cox_fit`` (clamp 50).
    theta has NO weights here; first Newton step is always d/32 (ll0 starts at 1e5)."""
    n, k = XA.shape
    beta0 = np.zeros(k)
    ll0 = 1e5
    ws = w * status
    for _ in range(30):
        theta = np.exp(_clip(XA @ beta0, clamp))
        cum = np.cumsum(theta[::-1])[::-1]
        xt = np.cumsum((XA * theta[:, None])[::-1], axis=0)[::-1] / cum[:, None]
        g = (XA - xt).T @ ws + 2.0 * lam * beta0  # :1429
        h = np.empty((k, k))
        for a in range(k):
            for b in range(a, k):
                s = np.cumsum((theta * XA[:, a] * XA[:, b])[::-1])[::-1]
                h[a, b] = h[b, a] = -float((s / cum - xt[:, a] * xt[:, b]) @ ws)
        h = h + 2.0 * lam * np.eye(k)  # :1472 (added to the NEGATIVE-definite h, as the reference does)
        d = np.linalg.solve(h, g)
        m = 1
        beta1 = beta0 - 0.5 ** m * d
        ll1 = loglik_cox(XA, status, beta1, w)
        while ll0 > ll1 and m < 5:
            m += 1
            beta1 = beta0 - 0.5 ** m * d
            ll1 = loglik_cox(XA, status, beta1, w)
        if abs(ll0 - ll1) / abs(0.1 + ll0) < 1e-5:
            break
        beta0 = beta1
        ll0 = ll1
    return beta0, coef0


# --------------------------------------------------------------------------------------
# get_A x4 (sacrifices): Algorithm.h:1097-1129, 1206-1263, 1324-1367, 1569-1640
# --------------------------------------------------------------------------------------
def sacrifice_lm(X, y, w, beta, coef0, xtx, lam=0.0):
    n = X.shape[0]
    d = X.T @ (y - X @ beta - coef0) / float(n) - 2.0 * lam * beta  # :1109
    phi = np.sqrt(2.0 * lam + xtx / float(n))  # utilities.cpp:142-151 (1x1 sqrt)
    inv = 1.0 / phi  # utilities.cpp:167-177 (1x1 ldlt inverse)
    return (phi * beta + inv * d) ** 2  # :1116-1122


def sacrifice_logistic(X, y, w, beta, coef0, xtx=None, lam=0.0):
    eta = _clip(X @ beta + coef0, 30.0)  # :1223-1231
    e = np.exp(eta)
    pr = e / (e + 1.0)
    g = w * (y - pr)
    h = w * pr * (1 - pr)
    d = X.T @ g - 2.0 * lam * beta  # :1236
    phi = np.sqrt((X * X).T @ h + 2.0 * lam)  # :1238-1250
    return (phi * beta + d / phi) ** 2


def sacrifice_poisson(X, y, w, beta, coef0, xtx=None, lam=0.0):
    eta = X @ beta + coef0  # :1338 (NOT clamped)
    e = np.exp(eta)
    g = (y - e) * w
    d = X.T @ g - 2.0 * lam * beta  # :1341
    phi = np.sqrt((X * X).T @ (e * w) + 2.0 * lam)  # :1342-1350
    return (phi * beta + d / phi) ** 2


def sacrifice_cox(X, y, w, beta, coef0=0.0, xtx=None, lam=0.0):
    """Algorithm.h:1569-1640 (algorithm_type 1 branch).  y is the 0/1 status, rows time-sorted."""
    theta = w * np.exp(_clip(X @ beta, 30.0))  # :1579-1587
    cum = np.cumsum(theta[::-1])[::-1]
    xth = np.cumsum((X * theta[:, None])[::-1], axis=0)[::-1] / cum[:, None]
    x2th = np.cumsum((X * X * theta[:, None])[::-1], axis=0)[::-1] / cum[:, None]
    x2th = x2th - xth ** 2
    xth = X - xth
    ev = (y != 0.0)  # :1618-1625 rows with status 0 are zeroed
    l1 = -(xth[ev].T @ w[ev]) + 2.0 * lam * beta  # :1629
    l2 = x2th[ev].T @ w[ev] + 2.0 * lam  # :1630
    d = -l1 / l2
    return np.abs(beta + d) * np.sqrt(l2)  # :1631-1634 (not squared)


_SACRIFICE = {1: sacrifice_lm, 2: sacrifice_logistic, 3: sacrifice_poisson, 4: sacrifice_cox}
_FIT = {1: fit_lm, 2: fit_logistic, 3: fit_poisson, 4: fit_cox}


# --------------------------------------------------------------------------------------
# Group selection (gsize > 1; R: bess(..., group.index=), Python: GroupPdas*): the same get_A functions with real
# k_g x k_g Phi / invPhi blocks.  Algorithm.h:1097-1129 (lm), :1206-1263 (logistic), :1324-1367 (poisson),
# :1497-1568 (cox, dense n x n Hessian branch of algorithm_type 2 / 3); utilities.cpp:113-177.
# --------------------------------------------------------------------------------------
def group_layout(g_index, p):
    """Data ctor, Data.h:53-61: g_index holds the first column of every group (ascending), sizes by difference."""
    g_index = np.asarray(g_index, dtype=np.int64)
    g_size = np.diff(np.append(g_index, p))
    return g_index, g_size


def _sqrtm_spd(M):
    """Principal square root of a symmetric positive-definite block (the reference calls Eigen's Schur-based
    MatrixBase::sqrt(), utilities.cpp:147; for an SPD argument that is U diag(sqrt(ev)) U^T)."""
    ev, U = np.linalg.eigh(M)
    return (U * np.sqrt(ev)) @ U.T


def group_gram_lm(X, g_index, g_size):
    """utilities.cpp:153-165 group_XTX: X_g^T X_g per group (over the rows handed in)."""
    return [X[:, a:a + k].T @ X[:, a:a + k] for a, k in zip(g_index, g_size)]


def find_ind(A, g_index, g_size, p):
    """utilities.cpp:113-130."""
    if len(A) == len(g_index):
        return np.arange(p)
    return np.concatenate([np.arange(g_index[g], g_index[g] + g_size[g]) for g in A]).astype(np.int64)


def group_sacrifice(model_type, X, y, w, beta, coef0, xtx, lam, g_index, g_size):
    n = X.shape[0]
    N = len(g_index)
    if model_type == 1:
        d = X.T @ (y - X @ beta - coef0) / float(n) - 2.0 * lam * beta
        blocks = [2.0 * lam * np.eye(k) + xtx[i] / float(n) for i, k in enumerate(g_size)]
    elif model_type in (2, 3):
        if model_type == 2:
            e = np.exp(_clip(X @ beta + coef0, 30.0))
            pr = e / (e + 1.0)
            g, h = w * (y - pr), w * pr * (1 - pr)
        else:
            e = np.exp(X @ beta + coef0)
            g, h = (y - e) * w, e * w
        d = X.T @ g - 2.0 * lam * beta
        blocks = []
        for a, k in zip(g_index, g_size):
            XG = X[:, a:a + k]
            blocks.append((XG * h[:, None]).T @ XG + 2.0 * lam * np.eye(k))
    else:
        theta = w * np.exp(_clip(X @ beta, 30.0))
        cum = np.cumsum(theta[::-1])[::-1]
        c2 = np.cumsum(y * w / cum)
        c3 = np.cumsum(y * w / cum ** 2)
        idx = np.minimum.outer(np.arange(n), np.arange(n))
        H = -c3[idx] * np.outer(theta, theta)  # :1535-1545: upper triangle mirrored
        H[np.diag_indices(n)] += c2 * theta
        g = w * y - c2 * theta
        d = X.T @ g - 2.0 * lam * beta
        blocks = [X[:, a:a + k].T @ H @ X[:, a:a + k] + 2.0 * lam * np.eye(k) for a, k in zip(g_index, g_size)]
    bd = np.zeros(N)
    for i, (a, k) in enumerate(zip(g_index, g_size)):
        phi = _sqrtm_spd(blocks[i])
        t = phi @ beta[a:a + k] + np.linalg.solve(phi, d[a:a + k])
        bd[i] = float(t @ t) / k
    return bd


# --------------------------------------------------------------------------------------
# Algorithm::fit  (Algorithm.h:113-171)
# --------------------------------------------------------------------------------------
@dataclass
class FitResult:
    beta: np.ndarray
    coef0: float
    l: int
    A: np.ndarray
    A_hist: list = field(default_factory=list)
    min_gap: float = np.inf
    G: np.ndarray = None  # selected groups (== A without group structure)


def pdas_fit(data: Data, model_type, T0, beta_init, coef0_init, train_mask, xtx, max_iter=20, always_select=(),
             lam=0.0, groups=None):
    """groups: None, or (g_index, g_size) -- then T0 counts GROUPS, xtx is the list of per-group Grams (lm) and
    FitResult.A holds the selected columns (find_ind), FitResult.G the selected groups."""
    X = data.x[train_mask] if len(train_mask) != data.n else data.x
    y = data.y[train_mask] if len(train_mask) != data.n else data.y
    w = data.weight[train_mask] if len(train_mask) != data.n else data.weight
    p = data.p
    beta = beta_init.copy()
    coef0 = float(coef0_init)
    seen = [np.zeros(T0, dtype=np.int32)]  # A_list.col(0) = 0  (:142-143)
    res = FitResult(beta, coef0, 0, seen[0])
    for l in range(1, max_iter + 1):
        if groups is None:
            bd = _SACRIFICE[model_type](X, y, w, beta, coef0, xtx, lam=lam)
        else:
            bd = group_sacrifice(model_type, X, y, w, beta, coef0, xtx, lam, groups[0], groups[1])
        if len(always_select):
            bd[np.asarray(always_select)] = DBL_MAX  # slice_assignment, utilities.cpp:190-199
        res.min_gap = min(res.min_gap, boundary_gap(bd, T0))
        A = max_k(bd, T0)
        ind = A if groups is None else find_ind(A, groups[0], groups[1], p)
        beta_A, coef0 = _FIT[model_type](X[:, ind], y, w, coef0, lam=lam)  # beta_A reset to 0 before the fit (:157)
        beta = np.zeros(p)
        beta[ind] = beta_A
        res.A_hist.append(A)
        res.l = l
        if any(np.array_equal(A, s) for s in seen):  # :164-170
            break
        seen.append(A)
    else:
        res.l = max_iter + 1  # loop variable after a non-returning for (:151)
    res.beta, res.coef0, res.A = beta, coef0, ind
    res.G = A
    return res


# --------------------------------------------------------------------------------------
# Metric: Metric.h:138-676
# --------------------------------------------------------------------------------------
def train_loss(data: Data, model_type, beta, coef0):
    if model_type == 1:
        return float(((data.y - data.x @ beta) ** 2).sum() / data.n)  # :145-148
    if model_type == 2:  # :266-290
        e = np.exp(_clip(data.x @ beta + coef0, 30.0))
        pr = e / (e + 1.0)
        return float(-2 * (data.weight * (data.y * np.log(pr) + (1 - data.y) * np.log(1 - pr))).sum())
    if model_type == 3:  # :426-440
        return -2 * loglik_poisson(data.x, data.y, np.concatenate([[coef0], beta]), data.weight)
    return -2 * loglik_cox(data.x, data.y, beta, data.weight)  # :565-568


def fold_loss(data: Data, model_type, beta, coef0, test_mask):
    X, y, w = data.x[test_mask], data.y[test_mask], data.weight[test_mask]
    if model_type == 1:
        return float(((y - X @ beta) ** 2).sum() / float(2 * len(test_mask)))  # :190
    if model_type == 2:  # :336-351 (clamp 25!)
        e = np.exp(_clip(X @ beta + coef0, 25.0))
        pr = e / (e + 1.0)
        return float(-2 * (w * (y * np.log(pr) + (1 - y) * np.log(1 - pr))).sum())
    if model_type == 3:  # :489 (factor 1, not 2)
        return -loglik_poisson(X, y, np.concatenate([[coef0], beta]), w)
    return -2 * loglik_cox(X, y, beta, w)  # :609


def ic_penalty(ic_type, n, p, s):
    if ic_type == 1:
        return 2.0 * s
    if ic_type == 2:
        return math.log(float(n)) * s
    if ic_type == 3:
        return math.log(float(p)) * math.log(math.log(float(n))) * s
    if ic_type == 4:
        return (math.log(float(n)) + 2 * math.log(float(p))) * s
    return None


class PathState:
    """The mutable state the reference keeps in Algorithm + Metric between calls."""

    def __init__(self, data, model_type, ic_type, is_cv, K, fold_of_row, max_iter, warm_start, always_select=(),
                 g_index=None, algorithm_type=1):
        self.data, self.model_type, self.ic_type, self.is_cv, self.K = data, model_type, ic_type, is_cv, K
        self.max_iter, self.warm, self.always = max_iter, warm_start, tuple(always_select)
        n, p = data.n, data.p
        self.algorithm_type = algorithm_type
        self.groups = None
        if g_index is not None and len(g_index) != p:
            self.groups = group_layout(g_index, p)
        self.g_num = p if self.groups is None else len(self.groups[0])
        self.full_mask = np.arange(n)
        if model_type != 1:
            self.xtx_full = None
        elif self.groups is None:
            self.xtx_full = (data.x * data.x).sum(axis=0)  # utilities.cpp:153-165
        else:
            self.xtx_full = group_gram_lm(data.x, *self.groups)
        self.alg_coef0_init = 0.0
        self.lam = 0.0  # Algorithm::lambda_level
        self.alg_beta = np.zeros(p)
        self.alg_coef0 = 0.0
        self.T = 0
        self.n_fits = 0
        self.n_iters = 0
        self.min_gap = np.inf
        if is_cv:
            fold_of_row = np.asarray(fold_of_row)
            self.test_masks = [np.nonzero(fold_of_row == k)[0] for k in range(K)]
            self.train_masks = [np.nonzero(fold_of_row != k)[0] for k in range(K)]
            self.cv_param = np.zeros((K, p))  # Metric.h:39-42
            if model_type != 1:
                self.xtx_folds = [None] * K
            elif self.groups is None:
                self.xtx_folds = [(data.x[m] ** 2).sum(axis=0) for m in self.train_masks]  # Metric.h:108-129
            else:
                self.xtx_folds = [group_gram_lm(data.x[m], *self.groups) for m in self.train_masks]

    def _fit(self, T, beta_init, coef0_init, mask, xtx):
        r = pdas_fit(self.data, self.model_type, T, beta_init, coef0_init, mask, xtx, self.max_iter, self.always,
                     lam=self.lam, groups=self.groups)
        self.n_fits += 1
        self.n_iters += min(r.l, self.max_iter)
        self.min_gap = min(self.min_gap, r.min_gap)
        self.alg_beta, self.alg_coef0, self.last = r.beta, r.coef0, r
        self.alg_beta_init = beta_init  # what update_beta_init was last handed (path.cpp:56 / Metric.h:179)
        return r

    def full_fit(self, T, beta_init, coef0_init):
        self.T = T
        self.alg_coef0_init = coef0_init  # update_coef0_init, path.cpp:57
        return self._fit(T, beta_init, coef0_init, self.full_mask, self.xtx_full)

    def train_loss(self):
        return train_loss(self.data, self.model_type, self.alg_beta, self.alg_coef0)

    def ic(self):
        if self.is_cv:  # Metric::test_loss
            losses = []
            for k in range(self.K):
                binit = self.cv_param[k].copy() if self.warm else np.zeros(self.data.p)
                # NB: the reference never resets beta_init when warm_start is false either: it keeps
                # whatever update_beta_init last set (the path's beta_init).  With warm_start=false the
                # path's beta_init stays zero, so zeros is the same thing.
                r = self._fit(self.T, binit, self.alg_coef0_init, self.train_masks[k], self.xtx_folds[k])
                if self.warm:
                    self.cv_param[k] = r.beta
                losses.append(fold_loss(self.data, self.model_type, r.beta, r.coef0, self.test_masks[k]))
            return float(np.mean(losses))
        tl = self.train_loss()
        # algorithm_type 2 / 3 (GPDAS / GL0L2): g_num and group_df (= sparsity level) replace p and s (Metric.h:230-254)
        pen = ic_penalty(self.ic_type, self.data.n, self.g_num if self.algorithm_type in (2, 3) else self.data.p, self.T)
        if pen is None:
            return 0.0
        if self.model_type == 1:
            return float(self.data.n) * math.log(tl) + pen  # Metric.h:205-229
        return tl + pen  # Metric.h:365-388 etc.


def _denormalise(data: Data, beta, coef0, gs):
    """path.cpp:76-110 (sequential) / :330-343 (gs: the non-gaussian branch also subtracts beta.x_mean
    for data_type 3, where x_mean is all zero)."""
    n = data.n
    if not data.is_normal:
        return beta, coef0
    beta = math.sqrt(float(n)) * beta / data.x_norm
    if data.data_type == 1:
        coef0 = data.y_mean - float(beta @ data.x_mean)
    elif data.data_type == 2 or gs:
        coef0 = coef0 - float(beta @ data.x_mean)
    return beta, coef0


def sequential_path(st: PathState, sequence, lambda_seq=(0.0,)):
    """path.cpp:25-132: for every sparsity level the lambda grid is walked zig-zag (:50), warm starts follow the walk,
    the criterion matrix ic[s][lambda] is minimised with Eigen's minCoeff (column-major visit: lambda outer, s inner)."""
    p = st.data.p
    S, L = len(sequence), len(lambda_seq)
    beta_init, coef0_init = np.zeros(p), 0.0
    betas = np.zeros((L, S, p))
    coef0s, losses, ics = np.zeros((L, S)), np.zeros((L, S)), np.zeros((L, S))
    ls = np.zeros((L, S), dtype=np.int64)
    for i, s in enumerate(sequence):
        js = range(L) if i % 2 == 0 else range(L - 1, -1, -1)
        for j in js:
            st.lam = float(lambda_seq[j])
            r = st.full_fit(int(s), beta_init, coef0_init)
            if st.warm:
                beta_init, coef0_init = r.beta.copy(), r.coef0
            betas[j, i] = r.beta
            coef0s[j, i] = r.coef0
            ls[j, i] = r.l
            losses[j, i] = st.train_loss()
            ics[j, i] = st.ic()
    flat = int(np.argmin(ics.reshape(-1)))  # [lambda][s] row-major == Eigen column-major visit of ic(s, lambda)
    bj, bi = divmod(flat, S)
    beta, coef0 = _denormalise(st.data, betas[bj, bi], coef0s[bj, bi], gs=False)
    out = dict(beta=beta, coef0=coef0, train_loss=float(losses[bj, bi]), ic=float(ics[bj, bi]), best=bi,
               s=int(sequence[bi]), lam=float(lambda_seq[bj]))
    if L == 1:
        out.update(beta_all=betas[0], coef0_all=coef0s[0], loss_all=losses[0], ic_all=ics[0], l_all=ls[0])
    else:
        out.update(beta_all=betas, coef0_all=coef0s, loss_all=losses, ic_all=ics, l_all=ls)
    return out


def gs_path(st: PathState, s_min, s_max):
    """path.cpp:134-389, including the double ic() evaluation and the read-after-ic() of beta."""
    p = st.data.p
    beta_init, coef0_init = np.zeros(p), 0.0

    def rnd(v):  # C round(): half away from zero
        return int(math.floor(v + 0.5)) if v >= 0 else -int(math.floor(-v + 0.5))

    def ev(T):
        nonlocal beta_init, coef0_init
        r = st.full_fit(T, beta_init, coef0_init)
        if st.warm:
            beta_init, coef0_init = r.beta.copy(), r.coef0
        return r

    Tmin, Tmax = s_min, s_max
    T1 = rnd(0.618 * Tmin + 0.382 * Tmax)
    T2 = rnd(0.382 * Tmin + 0.618 * Tmax)
    ic_seq = [0.0] * 4
    trace = []
    ev(T1); st.train_loss(); ic_seq[1] = st.ic(); icT1 = ic_seq[1]; trace.append(T1)
    ev(T2); st.train_loss(); ic_seq[2] = st.ic(); icT2 = st.ic(); trace.append(T2)
    while T1 != T2:
        if icT1 < icT2:
            Tmax = T2
            ic_seq[3] = ic_seq[2]
            T2 = T1
            ic_seq[2] = ic_seq[1]
            icT2 = ic_seq[1]
            T1 = rnd(0.618 * Tmin + 0.382 * Tmax)
            ev(T1); ic_seq[1] = st.ic(); icT1 = st.ic(); trace.append(T1)
        else:
            Tmin = T1
            ic_seq[0] = ic_seq[1]
            T1 = T2
            ic_seq[1] = ic_seq[2]
            icT1 = ic_seq[2]
            T2 = rnd(0.382 * Tmin + 0.618 * Tmax)
            ev(T2); ic_seq[2] = st.ic(); icT2 = st.ic(); trace.append(T2)
    best_ic, best = DBL_MAX, None
    for T in range(Tmin, Tmax + 1):
        ev(T)
        v = st.ic()
        if v < best_ic:
            # algorithm->get_beta() AFTER ic(): under CV this is the last fold's fit (path.cpp:314-319)
            best = (st.alg_beta.copy(), st.alg_coef0, st.train_loss(), T)
            best_ic = v
    beta, coef0 = _denormalise(st.data, best[0], best[1], gs=True)
    return dict(beta=beta, coef0=coef0, train_loss=best[2], ic=best_ic, s=best[3], trace=trace,
                Tmin=Tmin, Tmax=Tmax)


# --------------------------------------------------------------------------------------
# pgs_path: path.cpp:391-1309 (Powell search over (s, log lambda); "bsrr")
# --------------------------------------------------------------------------------------
def _c_round(v):
    return math.floor(v + 0.5) if v >= 0 else -math.floor(-v + 0.5)


def _sign(a):
    return 1 if a > 0 else (-1 if a < 0 else 0)


def _det(a, b):
    return a[0] * b[1] - a[1] * b[0]


def _line_intersection(l1, l2):
    """path.cpp:414-440; None when parallel."""
    xdiff = (l1[0][0] - l1[1][0], l2[0][0] - l2[1][0])
    ydiff = (l1[0][1] - l1[1][1], l2[0][1] - l2[1][1])
    div = _det(xdiff, ydiff)
    if div == 0:
        return None
    d = (_det(l1[0], l1[1]), _det(l2[0], l2[1]))
    return [_det(d, xdiff) / div, _det(d, ydiff) / div]


def _cal_intersections(p, u, s_min, s_max, lmin, lmax):
    """path.cpp:445-577."""
    line0 = ((p[0], p[1]), (p[0] + u[0], p[1] + u[1]))
    ls = [((s_min, lmin), (s_min, lmax)), ((s_max, lmin), (s_max, lmax)), ((s_min, lmin), (s_max, lmin)),
          ((s_min, lmax), (s_max, lmax))]
    ls = [tuple(tuple(float(v) for v in pt) for pt in ln) for ln in ls]
    xs = [_line_intersection(line0, ln) for ln in ls]
    need = [x is not None for x in xs]
    for i in range(4):
        if need[i] and (xs[i][0] < s_min - 0.0001 or xs[i][0] > s_max + 0.0001 or xs[i][1] < lmin - 0.001
                        or xs[i][1] > lmax + 0.001):
            need[i] = False
    for i in range(4):
        if need[i]:
            for j in range(i + 1, 4):
                if need[j] and abs(xs[i][0] - xs[j][0]) < 0.0001 and abs(xs[i][1] - xs[j][1]) < 0.0001:
                    need[j] = False
    pts = [xs[i] for i in range(4) if need[i]]
    if len(pts) < 2:
        raise ValueError("pgs_path: search line does not cross the box twice (uninitialised end points in the reference)")
    return list(pts[0]), list(pts[1])


class _PgsRec:
    __slots__ = ("beta", "coef0", "train_loss", "ic", "T", "lam")


def pgs_path(st: PathState, s_min, s_max, lmin, lmax, powell_path, nlambda):
    """path.cpp:1138-1309.  lmin/lmax are LOG lambda bounds (bess.cpp:171-172).  Returns the de-normalised winner, the
    chosen lambda and the (T, lambda) trace of the full-data fits."""
    p_cols = st.data.p
    trace = []
    state = dict(beta_init=np.zeros(p_cols), coef0_init=0.0)

    def ev(Td, loglam):
        """fit + ic() + get_beta()/train_loss() AFTER ic() (path.cpp:633-650)."""
        T = int(Td)
        st.lam = math.exp(loglam)
        r = st.full_fit(T, state["beta_init"], state["coef0_init"])
        if st.warm:
            state["beta_init"], state["coef0_init"] = r.beta.copy(), r.coef0
        trace.append((T, st.lam))
        rec = _PgsRec()
        rec.ic = st.ic()
        rec.beta, rec.coef0, rec.train_loss, rec.T, rec.lam = st.alg_beta.copy(), st.alg_coef0, st.train_loss(), T, st.lam
        return rec

    def golden(p, u):
        state["beta_init"], state["coef0_init"] = np.zeros(p_cols), 0.0
        s_tol, tol = 2, (lmax - lmin) / 200
        invphi, invphi2 = (5 ** 0.5 - 1.0) / 2.0, (3.0 - 5 ** 0.5) / 2.0
        a, b = _cal_intersections(p, u, s_min, s_max, lmin, lmax)
        h = [b[0] - a[0], b[1] - a[1]]
        c = [a[0] + invphi2 * h[0], a[1] + invphi2 * h[1]]
        d = [a[0] + invphi * h[0], a[1] + invphi * h[1]]
        if h[0] > 0.0001:
            c[0], d[0] = float(int(c[0])), float(math.ceil(d[0]))
        elif h[0] < -0.0001:
            c[0], d[0] = float(math.ceil(c[0])), float(int(d[0]))
        else:
            c[0], d[0] = float(_c_round(c[0])), float(_c_round(d[0]))
        t1 = ev(c[0], c[1]); closs = t1.ic
        t2 = ev(d[0], d[1]); dloss = t2.ic

        def small():
            return abs((invphi2 - invphi) * h[0]) <= s_tol and abs((invphi2 - invphi) * h[1]) < tol

        def finish():
            if closs < dloss:
                arg, best, min_loss = [c[0], c[1]], t1, closs
            else:
                arg, best, min_loss = [d[0], d[1]], t2, dloss
            best = _copy_rec(best, min_loss)
            i = 1
            while i < abs((invphi2 - invphi) * h[0]):
                e = ev(float(int(c[0] + _sign(h[0]) * i)), c[1])
                if e.ic < min_loss:
                    arg, min_loss, best = [c[0] + _sign(h[0]) * i, c[1]], e.ic, e
                i += 1
            return arg, best

        if small():
            return finish()
        tt = 0
        while tt < 100:
            tt += 1
            if closs < dloss:
                b = [d[0], d[1]]
                d = [c[0], c[1]]
                dloss = closs
                h = [b[0] - a[0], b[1] - a[1]]
                c = [a[0] + invphi2 * h[0], a[1] + invphi2 * h[1]]
                c[0] = float(int(c[0])) if h[0] > 0.0001 else (float(math.ceil(c[0])) if h[0] < -0.0001 else float(_c_round(c[0])))
                t1 = ev(c[0], c[1]); closs = t1.ic
            else:
                a = [c[0], c[1]]
                c = [d[0], d[1]]
                closs = dloss
                h = [b[0] - a[0], b[1] - a[1]]
                d = [a[0] + invphi * h[0], a[1] + invphi * h[1]]
                d[0] = float(math.ceil(d[0])) if h[0] > 0.0001 else (float(int(d[0])) if h[0] < -0.0001 else float(_c_round(d[0])))
                t2 = ev(d[0], d[1]); dloss = t2.ic
            if small() or tt == 50:
                return finish()
        raise AssertionError("unreachable")

    def gdc(a, b):
        mx = max(a, b)
        mn = b if a == mx else a
        if mn == 0:
            raise ValueError("pgs_path: degenerate direction (integer division by zero in the reference)")
        z = mn
        while mx % mn != 0:
            z = mx % mn
            mx, mn = mn, z
        return z

    def seqs(p, u):
        """u is rescaled in place (the caller's U row changes, path.cpp:971-992)."""
        state["beta_init"], state["coef0_init"] = np.zeros(p_cols), 0.0
        dl = (lmax - lmin) / (nlambda - 1)
        k_lambda = int(abs(_c_round(u[1] / dl)))
        if abs(u[0]) != 1 and k_lambda != 1:
            if k_lambda == 0 and u[0] != 0:
                u[0] = u[0] / abs(u[0])
            elif u[0] == 0 and k_lambda != 0:
                u[1] = u[1] / k_lambda
            else:
                g = gdc(k_lambda, abs(int(u[0])))
                if g:
                    u[0] = float(_c_round(u[0] / g))
                    u[1] = u[1] / g
        p0, p1 = p[0], p[1]

        def inside(s, l):
            return s <= s_max and l <= lmax + dl * 1e-4 and s >= s_min and l >= lmin - dl * 1e-4

        fwd = [ev(p0, p1)]
        bwd = [fwd[0]]
        warm = (state["beta_init"].copy(), state["coef0_init"])
        i = 1
        while inside(p0 + i * u[0], p1 + i * u[1]):
            fwd.append(ev(p0 + i * u[0], p1 + i * u[1]))
            i += 1
        state["beta_init"], state["coef0_init"] = warm[0].copy(), warm[1]
        j = 1
        while inside(p0 - j * u[0], p1 - j * u[1]):
            bwd.append(ev(p0 - j * u[0], p1 - j * u[1]))
            j += 1
        m1 = int(np.argmin([e.ic for e in fwd]))
        m2 = int(np.argmin([e.ic for e in bwd]))
        if fwd[m1].ic < bwd[m2].ic:
            pos, best = m1, fwd[m1]
        else:
            pos, best = -m2, bwd[m2]
        return [p0 + pos * u[0], p1 + pos * u[1]], best

    if powell_path == 1:
        nlambda = 100
    search = golden if powell_path == 1 else seqs
    P = [[float(s_min), lmin], [0.0, 0.0], [0.0, 0.0]]
    U = [[0.0, (lmax - lmin) / (nlambda - 1)], [1.0, 0.0]]
    recs, lams = {}, {}
    ttt = 0
    P[0], recs[0] = search(P[0], U[1])
    lams[0] = math.exp(P[0][1])
    while ttt < 11:
        ttt += 1
        for i in range(2):
            P[i + 1], recs[ttt] = search(P[i], U[i])
            lams[ttt] = math.exp(P[i + 1][1])
            ttt += 1
        U[0] = [U[1][0], U[1][1]]
        U[1] = [P[2][0] - P[0][0], P[2][1] - P[0][1]]
        if not (abs(U[1][0]) <= 0.0001 and abs(U[1][1]) <= 0.0001) and ttt < 11:
            P[0], recs[ttt] = search(P[0], U[1])
            lams[ttt] = math.exp(P[0][1])
        else:
            # closing fit: no update_beta_init / update_coef0_init (path.cpp:1212-1217)
            T = int(P[0][0])
            st.lam = math.exp(P[0][1])
            st.T = T
            r = st._fit(T, st.alg_beta_init, st.alg_coef0_init, st.full_mask, st.xtx_full)
            trace.append((T, st.lam))
            rec = _PgsRec()
            rec.beta, rec.coef0, rec.train_loss, rec.T, rec.lam = r.beta.copy(), r.coef0, st.train_loss(), T, st.lam
            rec.ic = st.ic()
            recs[ttt] = rec
            lams[ttt] = math.exp(P[0][1])
            ttt += 1
            ics = [recs[i].ic for i in range(ttt)]
            mi = int(np.argmin(ics))
            if ics[mi] == ics[ttt - 1]:
                mi = ttt - 1
            best = recs[mi]
            beta, coef0 = _denormalise(st.data, best.beta, best.coef0, gs=False)
            return dict(beta=beta, coef0=coef0, train_loss=best.train_loss, ic=best.ic, lam=lams[mi], trace=trace,
                        s=int(np.count_nonzero(best.beta)))
    raise ValueError("pgs_path: no result (empty list in the reference)")


def _copy_rec(r, ic):
    o = _PgsRec()
    o.beta, o.coef0, o.train_loss, o.T, o.lam, o.ic = r.beta, r.coef0, r.train_loss, r.T, r.lam, ic
    return o


# --------------------------------------------------------------------------------------
# Screening: screening.cpp:26-105 + marginal fits
# --------------------------------------------------------------------------------------
def poisson_fit_marginal(xj, y, w):
    """poisson.cpp:84-137, *literally*, including the vector*vector product that (asserts off)
    evaluates to X.col(i)*expeta_w(0) (:117) and the wrong-sign step (:122,:128)."""
    n = xj.shape[0]
    X = np.column_stack([np.ones(n), xj])
    beta0 = np.zeros(2)
    for _ in range(100):
        eta = _clip(X @ beta0, 30.0)
        expeta = np.exp(eta)
        ew0 = expeta[0] * w[0]
        temp = X * ew0
        g = X.T @ ((y - expeta) * w)
        h = X.T @ temp
        d = np.linalg.solve(h, g)
        m = 0
        beta1 = beta0 - 0.2 ** m * d
        ll0 = loglik_poiss(xj[:, None], y, beta0, w)
        ll1 = loglik_poiss(xj[:, None], y, beta1, w)
        while ll0 >= ll1 and m < 10:
            m += 1
            beta1 = beta0 - 0.2 ** m * d
            ll1 = loglik_poiss(xj[:, None], y, beta1, w)
        beta0 = beta1
        if abs(ll0 - ll1) / abs(ll0) < 1e-8:
            break
    return beta0


def screening_utility(x, y, w, model_type):
    """coef_norm of screening.cpp:40-61 on RAW x (gsize 1): squared marginal slope."""
    n, p = x.shape
    u = np.empty(p)
    if model_type == 1:
        u[:] = ((x.T @ y) / (x * x).sum(axis=0)) ** 2  # 1-column colPivHouseholderQr().solve(y)
        return u
    for j in range(p):
        xj = x[:, j]
        if model_type == 2:
            b, _ = fit_logistic(xj[:, None], y, w, 0.0, floor_w=False)
            u[j] = b[0] ** 2
        elif model_type == 3:
            u[j] = poisson_fit_marginal(xj, y, w)[1] ** 2
        else:
            b, _ = fit_cox(xj[:, None], y, w, 0.0, clamp=50.0)
            u[j] = b[0] ** 2
    return u


def screening(x, y, w, model_type, screening_size, always_select=()):
    u = screening_utility(np.asarray(x, dtype=np.float64), y, w, model_type)
    if len(always_select):
        u[np.asarray(always_select)] = DBL_MAX
    return max_k(u, screening_size)


# --------------------------------------------------------------------------------------
# bessCpp: bess.cpp:37-214
# --------------------------------------------------------------------------------------
def bess_cpp(x, y, data_type, weight, is_normal, model_type, max_iter, path_type, is_warm_start, ic_type, is_cv, K,
             sequence, s_min, s_max, is_screening, screening_size, always_select=(), fold_of_row=None,
             lambda_seq=(0.0,), algorithm_type=1, lambda_min=0.0, lambda_max=0.0, n_lambda=100, powell_path=1,
             g_index=None):
    x = np.asarray(x, dtype=np.float64)
    p0 = x.shape[1]
    always = np.asarray(always_select, dtype=np.int64)
    scr = None
    if is_screening:
        scr = screening(x, y, weight, model_type, screening_size, always)
        x = x[:, scr]
        always = np.searchsorted(scr, always) if len(always) else always  # screening.cpp:91-102
    data = make_data(x, y, weight, data_type, is_normal, model_type)
    if g_index is not None and len(g_index) != x.shape[1] and is_screening:
        raise ValueError("screening with groups un-screens by group id in the reference (bess.cpp:186-209): not restated")
    st = PathState(data, model_type, ic_type, is_cv, K, fold_of_row, max_iter, is_warm_start, always, g_index=g_index,
                   algorithm_type=algorithm_type)
    if path_type == 1:
        out = sequential_path(st, sequence, lambda_seq)
    elif algorithm_type in (5, 3):  # bess.cpp:167-175
        out = pgs_path(st, s_min, s_max, math.log(max(lambda_min, 1e-5)), math.log(max(lambda_max, 1e-5)), powell_path,
                       n_lambda)
    else:
        out = gs_path(st, s_min, s_max)
    if is_screening:
        b = np.zeros(p0)
        b[scr] = out["beta"]
        out["beta"] = b
        out["screening_A"] = scr
    out["n_fits"], out["n_iters"], out["min_gap"] = st.n_fits, st.n_iters, st.min_gap
    return out

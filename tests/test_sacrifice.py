"""The selection half of a PDAS iteration -- the sacrifice ``bd`` of every column or group that get_A ranks -- against
high-precision references, through ``GpuEngine.sacrifice`` (bessgpu_sacrifice): the probe publishes the gradient vectors
of every chain of a batch again from the chain's current (A, beta_A, coef0) and runs the dispatch a fit of that batch
runs (column sweep + finish, or the group kernels), reporting which code ran.

References are computed here in np.longdouble from the engine's own normalised design, the response and weights as the
fits see them and each chain's train rows, written independently of the kernels' algebra (cox from the per-row risk-set
form, groups from the closed form with a refined solve).  Tolerances are first-order error bounds the references compute
from absolute-value sums; the CPU tests check the references against mpmath.  Then whole fits at every chain-slot count
against oracle.pdas_fit."""
import collections

import numpy as np
import pytest

from oracle import pdas_oracle as orc
from tests.helpers import RTOL, rel_err

LD = np.longdouble
U = 2.0 ** -53
FAM = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}
MODE = {"gaussian": "D", "binomial": "DH", "poisson": "DH", "cox": "COX"}
FS_ALL = [1, 4, 6, 8, 12, 16, 24, 32]  # FS = 2 needs K = 1, which setup_chains refuses (a fold without train rows)
GSAC_SERIAL, GSAC_WARP, GSAC_B2, GSAC_B4, GSAC_B8, GSAC_WIDE = 1, 2, 4, 8, 16, 32

SEEN = set()                             # (kernel, FS, CPT, mode) reported by the probe
SEEN_GROUP = 0                           # group kernel bits reported by the probe
SPLITS = collections.defaultdict(set)    # family -> row-split counts S reported
WORST = collections.defaultdict(float)   # family -> largest err / bound


def k_of_fs(fs):
    return 0 if fs == 1 else fs - 1


def tma_cpt(fs, mode):
    """columns per thread of dual_sweep_tma_kernel (sweep_tma.cu tma_cpt)"""
    if fs <= 6:
        return 2
    if fs <= 12:
        return 1 if mode == "COX" else 2
    if fs == 16:
        return 2 if mode == "D" else 1
    return 1


def expected_sweeps():
    out = {("stream", 1, 2, m) for m in ("D", "DH", "COX")}
    out |= {("tma", fs, tma_cpt(fs, m), m) for fs in FS_ALL[1:] for m in ("D", "DH", "COX")}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# references (long double) and their first-order error bounds
# ---------------------------------------------------------------------------------------------------------------------
def _gamma(n):
    return 4.0 * (n + 8) * U


def published(fam, Xm, y, w, beta, coef0, ks):
    """Per train row: the gradient vectors the chain kernels publish for (beta, coef0) and a bound on their error.
    Returns dict(g, dg, h, dh) (gaussian: h = None) or, for cox, the risk-set quantities."""
    nt = Xm.shape[0]
    b = beta.astype(LD)
    eta = Xm @ b + LD(coef0)
    # the chain kernels form eta in fp64 over the ks support columns (+ the intercept)
    deta = 2.0 * (ks + 2) * U * (np.abs(Xm) @ np.abs(b) + abs(coef0)).astype(np.float64)
    yl, wl = y.astype(LD), w.astype(LD)
    if fam == "gaussian":
        g = (yl - eta) / nt
        dg = (deta + 2 * U * np.abs((yl.astype(np.float64)) - eta.astype(np.float64)) + 2 * U * np.abs(y)) / nt
        return dict(g=g, dg=dg, eta=eta)
    if fam == "binomial":
        clamped = np.abs(eta) >= 30
        e = np.exp(np.clip(eta, -30, 30))
        pr = e / (1 + e)
        g = wl * (yl - pr)
        h = wl * pr * (1 - pr)
        hf = h.astype(np.float64)
        dg = np.where(clamped, 0.0, hf * deta) + 8 * U * w * (np.abs(y) + pr.astype(np.float64))
        dh = np.where(clamped, 0.0, hf * deta) + 10 * U * hf
        return dict(g=g, dg=dg, h=h, dh=dh, eta=eta)
    if fam == "poisson":
        e = np.exp(eta)
        g = (yl - e) * wl
        h = e * wl
        hf = h.astype(np.float64)
        dg = hf * deta + 6 * U * w * (np.abs(y) + e.astype(np.float64))
        dh = hf * (deta + 6 * U)
        return dict(g=g, dg=dg, h=h, dh=dh, eta=eta)
    # cox: rows in time order; theta, the risk-set sums S_k, e_k = w_k on event rows
    clamped = np.abs(eta) >= 30
    th = wl * np.exp(np.clip(eta, -30, 30))
    S = np.cumsum(th[::-1])[::-1]
    ev = (y != 0.0)
    e = np.where(ev, wl, LD(0))
    gn = _gamma(nt)
    r1 = float(np.max(np.where(clamped, 0.0, deta))) + 3 * U    # relative error of theta
    rS = r1 + gn                                                  # ... of the suffix sums
    rc = rS + gn + 3 * U                                          # ... of the prefix sums of e / S
    rho = r1 + rc + 2 * U                                         # ... of omega, TH, C2 (C2 = e / S^2: 2 rS)
    return dict(th=th, S=S, e=e, ev=ev, r1=r1, rho=max(rho, 2 * rS + 3 * U), eta=eta)


def sacrifice_ref(fam, Xm, y, w, beta, coef0, ks, lam):
    """bd of every column and its error bound over the chain's train rows Xm (long double, n_t x p)."""
    nt, p = Xm.shape
    gn = _gamma(nt)
    ax = np.abs(Xm).astype(np.float64)
    b = beta.astype(LD)
    bf = np.abs(beta)
    lam2 = LD(2.0 * lam)
    pv = published(fam, Xm, y, w, beta, coef0, ks)
    if fam != "cox":
        g = pv["g"]
        d = Xm.T @ g
        Dbar = ax.T @ np.abs(g).astype(np.float64)
        dd = gn * Dbar + ax.T @ pv["dg"] + 2 * U * np.abs(d.astype(np.float64))
        dp = d - lam2 * b
        ddp = dd + 4 * U * np.abs(2 * lam * bf) + U * np.abs(dp.astype(np.float64))
        if fam == "gaussian":
            xtx = (Xm * Xm).sum(axis=0)  # x_j.x_j over the chain's train rows
            phi2 = lam2 + xtx / nt
            dphi2 = (gn + 4 * U) * (xtx / nt).astype(np.float64) + 2 * U * phi2.astype(np.float64)
        else:
            hs = (Xm * Xm).T @ pv["h"]
            phi2 = hs + lam2
            dphi2 = (gn + 3 * U) * hs.astype(np.float64) + (ax * ax).T @ pv["dh"] + 2 * U * phi2.astype(np.float64)
        phi = np.sqrt(phi2)
        t = phi * b + dp / phi
        bd = t * t
        ph, dpf, tf = phi.astype(np.float64), np.abs(dp.astype(np.float64)), np.abs(t.astype(np.float64))
        dphi = dphi2 / (2 * ph) + U * ph
        dt = bf * dphi + ddp / ph + dpf * dphi / ph ** 2 + 4 * U * (ph * bf + dpf / ph)
        bound = 2 * tf * dt + dt * dt + 4 * U * tf * tf
        return bd, bound
    th, S, e, rho, r1 = pv["th"], pv["S"], pv["e"], pv["rho"], pv["r1"]
    xth = np.cumsum((Xm * th[:, None])[::-1], axis=0)[::-1] / S[:, None]
    x2th = np.cumsum((Xm * Xm * th[:, None])[::-1], axis=0)[::-1] / S[:, None]
    ev = pv["ev"]
    wl = w.astype(LD)
    l1 = -((Xm[ev] - xth[ev]).T @ wl[ev]) + lam2 * b
    l2 = (x2th[ev] - xth[ev] ** 2).T @ wl[ev] + lam2
    # absolute-value quantities of the device's arrangement d = X^T (e - omega), l2 = sum x^2 omega - sum C2 s1^2
    cc = np.cumsum(e / S)
    om = (th * cc).astype(np.float64)
    G = np.abs((e - th * cc).astype(np.float64))
    Dbar = ax.T @ G
    Hbar = (ax * ax).T @ om
    s1bar = np.cumsum((ax * th.astype(np.float64)[:, None])[::-1], axis=0)[::-1]
    C2 = (e / (S * S)).astype(np.float64)
    Rbar = C2 @ (s1bar * s1bar)
    dpl = -l1
    dd = gn * Dbar + ax.T @ (rho * om + U * G) + 2 * U * np.abs(dpl.astype(np.float64)) + 4 * U * np.abs(2 * lam * bf)
    dl2 = (gn + rho + 2 * U) * Hbar + (4 * gn + 2 * r1 + rho + 6 * U) * Rbar + 2 * U * np.abs(l2.astype(np.float64))
    q = b + dpl / l2
    bd = np.abs(q) * np.sqrt(l2)
    l2f, qf, dplf = l2.astype(np.float64), np.abs(q.astype(np.float64)), np.abs(dpl.astype(np.float64))
    dq = dd / l2f + dplf * dl2 / l2f ** 2 + 2 * U * (bf + dplf / l2f)
    bound = dq * np.sqrt(l2f) + qf * dl2 / (2 * np.sqrt(l2f)) + 4 * U * bd.astype(np.float64)
    return bd, bound


def refine_solve(A, b):
    """A^{-1} b to long-double accuracy: fp64 LU, iterative refinement on long-double residuals"""
    import scipy.linalg
    lu = scipy.linalg.lu_factor(A.astype(np.float64))
    x = scipy.linalg.lu_solve(lu, b.astype(np.float64)).astype(LD)
    for _ in range(8):
        x = x + scipy.linalg.lu_solve(lu, (b - A @ x).astype(np.float64)).astype(LD)
    return x


def group_sacrifice_ref(fam, Xm, y, w, beta, coef0, ks, lam, gidx, gsz):
    """bd_g = (b'A b + 2 b'd' + d'A^{-1}d') / k_g with A = M_g + 2 lambda I, d' = d_g - 2 lambda b_g, and its bound"""
    nt, p = Xm.shape
    gn = _gamma(nt)
    pv = published(fam, Xm, y, w, beta, coef0, ks)
    ax = np.abs(Xm).astype(np.float64)
    lam2 = LD(2.0 * lam)
    if fam == "cox":
        th, S, e, rho, r1 = pv["th"], pv["S"], pv["e"], pv["rho"], pv["r1"]
        cc = np.cumsum(e / S)
        om = th * cc
        C2 = e / (S * S)
        g = e - om
        dg = rho * om.astype(np.float64) + U * np.abs(g.astype(np.float64))
        s = np.cumsum((Xm * th[:, None])[::-1], axis=0)[::-1]
        sbar = np.cumsum((ax * th.astype(np.float64)[:, None])[::-1], axis=0)[::-1]
        crel = 4 * gn + 2 * r1 + 2 * rho + 8 * U
    else:
        g, dg = pv["g"], pv["dg"]
        if fam == "gaussian":
            h = np.full(nt, LD(1) / nt)
            dh = np.zeros(nt)
        else:
            h, dh = pv["h"], pv["dh"]
        crel = gn + 4 * U
    d = Xm.T @ g
    dd = gn * (ax.T @ np.abs(g).astype(np.float64)) + ax.T @ dg + 2 * U * np.abs(d.astype(np.float64))
    bd = np.zeros(len(gidx), dtype=LD)
    bound = np.zeros(len(gidx))
    for q, (a, k) in enumerate(zip(gidx, gsz)):
        sl = slice(a, a + k)
        Xg, axg = Xm[:, sl], ax[:, sl]
        if fam == "cox":
            M = (Xg * om[:, None]).T @ Xg - (s[:, sl] * C2[:, None]).T @ s[:, sl]
            Mbar = (axg * om.astype(np.float64)[:, None]).T @ axg + (sbar[:, sl] * C2.astype(np.float64)[:, None]).T @ sbar[:, sl]
            dM = crel * Mbar
        else:
            M = (Xg * h[:, None]).T @ Xg
            Mbar = (axg * h.astype(np.float64)[:, None]).T @ axg
            dM = crel * Mbar + (axg * dh[:, None]).T @ axg
        A = M + lam2 * np.eye(k, dtype=LD)
        bg = beta[sl].astype(LD)
        dp = d[sl] - lam2 * bg
        z = refine_solve(A, dp)
        val = (bg @ A @ bg + 2 * bg @ dp + dp @ z) / k
        bd[q] = val
        bgf, zf, dpf = np.abs(bg.astype(np.float64)), np.abs(z.astype(np.float64)), np.abs(dp.astype(np.float64))
        Af = A.astype(np.float64)
        nA = np.linalg.norm(Af, 2)
        lmin = max(np.linalg.eigvalsh(Af)[0], 1e-300)
        ddp = dd[sl] + 4 * U * np.abs(2 * lam * bgf) + U * dpf
        J = 16 * k * U  # Jacobi / Cholesky backward error, relative to ||A||
        nb, nz, nd = np.linalg.norm(bgf), np.linalg.norm(zf), np.linalg.norm(dpf)
        err = bgf @ dM @ bgf + 2 * bgf @ ddp + 2 * zf @ ddp + zf @ dM @ zf
        err += J * (nA * nb * nb + 2 * nb * nd + nz * nz * nA + np.sqrt(k * abs(float(val))) * (np.sqrt(nA) * nb + nd / np.sqrt(lmin)))
        err += 8 * k * U * (bgf @ np.abs(Af) @ bgf + 2 * bgf @ dpf + zf @ np.abs(Af) @ zf)
        bound[q] = err / k + 4 * U * abs(float(val))
    return bd, bound


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the references against mpmath
# ---------------------------------------------------------------------------------------------------------------------
def _mp_sacrifice(fam, X, y, w, beta, coef0, lam, groups=None):
    import mpmath as mp
    mp.mp.dps = 50
    n, p = X.shape
    Xm = [[mp.mpf(float(X[i, j])) for j in range(p)] for i in range(n)]
    b = [mp.mpf(float(v)) for v in beta]
    eta = [mp.fsum(Xm[i][j] * b[j] for j in range(p)) + mp.mpf(coef0) for i in range(n)]
    W = [mp.mpf(float(v)) for v in w]
    Y = [mp.mpf(float(v)) for v in y]
    M = None
    if fam == "gaussian":
        g = [(Y[i] - eta[i]) / n for i in range(n)]
        hr = [mp.mpf(1) / n] * n
    elif fam == "binomial":
        pr = [mp.exp(min(max(e, -30), 30)) / (1 + mp.exp(min(max(e, -30), 30))) for e in eta]
        g = [W[i] * (Y[i] - pr[i]) for i in range(n)]
        hr = [W[i] * pr[i] * (1 - pr[i]) for i in range(n)]
    elif fam == "poisson":
        g = [(Y[i] - mp.exp(eta[i])) * W[i] for i in range(n)]
        hr = [mp.exp(eta[i]) * W[i] for i in range(n)]
    else:
        th = [W[i] * mp.exp(min(max(eta[i], -30), 30)) for i in range(n)]
        S = [mp.fsum(th[i:]) for i in range(n)]
        def M(cols):  # risk-set Hessian block from its definition: sum over events of w_k (x2th - xth xth')
            out = mp.zeros(len(cols), len(cols))
            for k in range(n):
                if y[k] == 0:
                    continue
                xt = [mp.fsum(th[i] * Xm[i][a] for i in range(k, n)) / S[k] for a in cols]
                for u, a in enumerate(cols):
                    for v, c in enumerate(cols):
                        out[u, v] += W[k] * (mp.fsum(th[i] * Xm[i][a] * Xm[i][c] for i in range(k, n)) / S[k] - xt[u] * xt[v])
            return out
        d = [mp.fsum(W[k] * (Xm[k][j] - mp.fsum(th[i] * Xm[i][j] for i in range(k, n)) / S[k]) for k in range(n) if y[k] != 0)
             for j in range(p)]
    if M is None:
        d = [mp.fsum(Xm[i][j] * g[i] for i in range(n)) for j in range(p)]
        def M(cols):
            return mp.matrix([[mp.fsum(hr[i] * Xm[i][a] * Xm[i][c] for i in range(n)) for c in cols] for a in cols])
    if groups is None:
        groups = (list(range(p)), [1] * p)
    out = []
    for a, k in zip(*groups):
        cols = list(range(a, a + k))
        A = M(cols) + 2 * mp.mpf(lam) * mp.eye(k)
        bg = mp.matrix([b[c] for c in cols])
        dp = mp.matrix([d[c] for c in cols]) - 2 * mp.mpf(lam) * bg
        if fam == "cox" and k == 1:  # the reference's cox form: |beta + d / l2| sqrt(l2)
            out.append(abs(bg[0] + dp[0] / A[0, 0]) * mp.sqrt(A[0, 0]))
            continue
        z = mp.lu_solve(A, dp)
        out.append(((bg.T * A * bg)[0] + 2 * (bg.T * dp)[0] + (dp.T * z)[0]) / k)
    return out


@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_references_against_mpmath(fam):
    import mpmath as mp
    rng = np.random.default_rng(5)
    n, p = 9, 4
    X = rng.standard_normal((n, p)) * np.array([1e-3, 1.0, 3.0, 1e2])
    y = {"gaussian": rng.standard_normal(n), "binomial": (rng.random(n) < 0.5) * 1.0,
         "poisson": rng.poisson(3.0, n) * 1.0, "cox": (rng.random(n) < 0.7) * 1.0}[fam]
    w = rng.uniform(0.5, 1.5, n)
    beta = np.array([0.0, 0.3, -0.2, 0.0]) if fam != "poisson" else np.array([0.0, 0.1, -0.05, 0.0])
    for lam in (0.0, 0.07):
        ref, bound = sacrifice_ref(fam, X.astype(LD), y, w, beta, 0.2 if fam in ("binomial", "poisson") else 0.0, 2, lam)
        ex = _mp_sacrifice(fam, X, y, w, beta, 0.2 if fam in ("binomial", "poisson") else 0.0, lam)
        for j in range(p):
            got = mp.mpf(np.format_float_scientific(ref[j], precision=30))
            assert abs(got - ex[j]) <= 0.01 * bound[j], (fam, lam, j)
            assert bound[j] < 1e-8 * abs(float(ex[j]))
    gidx, gsz = [0, 1], [1, 3]
    for lam in (0.0, 0.05):
        ref, bound = group_sacrifice_ref(fam, X.astype(LD), y, w, beta, 0.2 if fam in ("binomial", "poisson") else 0.0, 2,
                                         lam, gidx, gsz)
        ex = _mp_sacrifice(fam, X, y, w, beta, 0.2 if fam in ("binomial", "poisson") else 0.0, lam, (gidx, gsz))
        for q in range(2):
            got = mp.mpf(np.format_float_scientific(ref[q], precision=30))
            exq = ex[q] if not (fam == "cox" and gsz[q] == 1) else None
            if exq is None:  # a width-1 cox group: the group form (b'Ab + 2b'd + d^2/A), i.e. the square of the column form
                exq = ex[q] ** 2
            assert abs(got - exq) <= 0.01 * bound[q], (fam, lam, q)


def test_references_catch_a_dropped_row():
    """The tolerance is far below what one missing train row changes."""
    rng = np.random.default_rng(3)
    X = rng.standard_normal((300, 20)).astype(LD)
    y = rng.standard_normal(300)
    w = np.ones(300)
    beta = np.zeros(20)
    beta[[2, 7]] = [0.5, -1.0]
    for fam in ("gaussian", "cox"):
        yy = y if fam == "gaussian" else (y > -0.5) * 1.0
        a, bound = sacrifice_ref(fam, X, yy, w, beta, 0.0, 2, 0.0)
        b, _ = sacrifice_ref(fam, X[1:], yy[1:], w[1:], beta, 0.0, 2, 0.0)
        assert np.median(np.abs((a[:20] - b[:20]).astype(np.float64)) / bound) > 1e6


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the probe against the references
# ---------------------------------------------------------------------------------------------------------------------
def _data(fam, n, p, seed, kind=None):
    from bess_b200.gen_data import gen_data
    rng = np.random.default_rng(seed)
    d = gen_data(n, p, fam, min(5, p), seed=seed)
    x, y = d.x, d.y
    w = rng.uniform(0.5, 1.5, n)
    if kind == "separable":  # |eta| of the fitted model runs past the +-30 clamp
        z = rng.standard_normal(n)
        z += np.sign(z) * 0.5
        x[:, 0] = z
        y = (z > 0) * 1.0
    elif kind == "large_counts":
        x[:, 0] = rng.standard_normal(n)
        y = rng.poisson(np.exp(np.clip(10.0 + 0.7 * x[:, 0], -30, 13))).astype(np.float64)
    elif kind == "cox_hard":  # theta over ~e^+-30, an event in row 0, none in the last third, uncentred columns
        z = np.sort(rng.standard_normal(n))[::-1] * 12.0
        x[:, 0] = z + 0.01 * rng.standard_normal(n)
        x = x + 5.0
        y = (rng.random(n) < 0.7) * 1.0
        y[0] = 1.0
        y[(2 * n) // 3:] = 0.0
    elif kind == "collinear":  # column 7 = column 6 + 1e-4 of its spread: the block of group [4, 8) has condition ~1e8
        x[:, 7] = x[:, 6] + 1e-4 * np.std(x[:, 6]) * rng.standard_normal(n)
    return x, y, w


class Case:
    """one engine: load, normalise, chains; fit levels and probe them"""

    def __init__(self, fam, n, p, K, seed, kcap, max_iter=20, kind=None, g_index=None):
        from bess_b200 import cbess
        from bess_b200.engine import GpuEngine
        self.fam, self.K = fam, K
        model_type, data_type = FAM[fam]
        x, y, w = _data(fam, n, p, seed, kind)
        self.eng = GpuEngine()
        self.eng.load(x, y, w, model_type)
        xm, xn, ym = self.eng.normalize(data_type, True)
        self.X = self.eng.design().astype(LD)
        self.y = (y - ym) * np.sqrt(w) if fam == "gaussian" else y
        self.w = w
        self.n, self.p = n, p
        self.fold = cbess.cv_fold_ids(n, K, seed) if K else None
        self.groups = None
        if g_index is not None:
            self.eng.set_groups(np.asarray(g_index, dtype=np.int32))
            self.groups = (np.asarray(g_index), np.diff(np.append(g_index, p)))
        self.eng.setup_chains(K, self.fold, kcap, max_iter, True)

    def rows(self, c):
        return np.arange(self.n) if c == 0 else np.nonzero(self.fold != c - 1)[0]

    def fit_and_probe(self, T, chains, lam=0.0, ridge_api=False, well_conditioned=True):
        if ridge_api or self.groups is not None:
            r = self.eng.run_batch_groups(T, chains, True, lam)
        else:
            r = self.eng.run_batch(T, chains, True)
        bd, info = self.eng.sacrifice(chains, lam)
        global SEEN_GROUP
        if self.groups is not None:
            SEEN_GROUP |= info["groups"]
        else:
            SEEN.add((info["kernel"], info["FS"], info["CPT"], MODE[self.fam]))
            SPLITS[self.fam].add(info["S"])
        etas = []
        for i, c in enumerate(chains):
            A, bA = np.asarray(r["A"][i]), np.asarray(r["bA"][i])
            beta = np.zeros(self.p)
            beta[A] = bA
            rows = self.rows(c)
            Xm = self.X[rows]
            args = (self.fam, Xm, self.y[rows], self.w[rows], beta, float(r["coef0"][i]), len(A), lam)
            ref, bound = group_sacrifice_ref(*args, *self.groups) if self.groups is not None else sacrifice_ref(*args)
            err = np.abs(bd[i].astype(LD) - ref).astype(np.float64)
            ratio = err / np.maximum(bound, 1e-300)
            WORST[self.fam] = max(WORST[self.fam], float(np.max(ratio)))
            bad = np.nonzero(~(err <= bound))[0]
            assert bad.size == 0, (self.fam, T, c, info, bad[:8].tolist(), bd[i][bad[:4]].tolist(),
                                   ref[bad[:4]].astype(np.float64).tolist(), bound[bad[:4]].tolist())
            if well_conditioned:  # the bound is not vacuous: below 1e-10 of |bd| for most columns.  Poisson: the error of
                # eta reaches g = (y - e^eta) w amplified by e^eta / |y - e^eta| ~ sqrt(counts), a real sensitivity
                lim = max(1e-9, 1e-12 * np.sqrt(np.max(self.y))) if self.fam == "poisson" else 1e-10
                rel = bound / np.maximum(np.abs(ref.astype(np.float64)), 1e-300)
                assert np.median(rel) < lim, (self.fam, T, c, np.median(rel), lim)
            etas.append(Xm @ beta.astype(LD) + LD(r["coef0"][i]))
        return r, info, etas

    def close(self):
        self.eng.close()


def _cols_per_cta(fs, fam):
    mode = MODE[fam]
    cpt = 2 if fs == 1 else tma_cpt(fs, mode)
    return 128 * cpt


@pytest.mark.gpu
@pytest.mark.parametrize("fs", FS_ALL)
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_column_sacrifice_every_chain_slot_count(fam, fs):
    """Full-data chain + K folds, non-uniform weights, at two shapes per chain-slot count: n = 97 (one row split) with
    p one column more than a CTA's columns, and n = 389 (several splits, n not a multiple of 8) with p one less."""
    K = k_of_fs(fs)
    chains = list(range(K + 1))
    cols = _cols_per_cta(fs, fam)
    for n, p, seed in ((97, cols + 1, 10 + fs), (389, cols - 1, 20 + fs)):
        cs = Case(fam, n, p, K, seed, kcap=3)
        for T in (1, 3):
            _, info, _ = cs.fit_and_probe(T, chains)
            assert info["FS"] == fs and info["kernel"] == ("stream" if fs == 1 else "tma")
            assert (info["S"] == 1) == (n < 128), info
            assert info["rows_per_split"] % 2 == 0 and (info["S"] - 1) * info["rows_per_split"] < n <= info["S"] * info["rows_per_split"]
        cs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_column_sacrifice_tiny_p(fam):
    """p = 1, and p smaller than the chain-slot count (p = 5 with 8 slots); odd n around the 64-row chunk"""
    for n, p, K, seed in ((150, 1, 3, 31), (203, 5, 7, 32), (65, 3, 5, 33)):
        cs = Case(fam, n, p, K, seed, kcap=1)
        cs.fit_and_probe(1, list(range(K + 1)))
        cs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_sacrifice_is_recomputed_for_the_returned_model(fam):
    """max_iter = 1: the last sacrifice a fit computed belongs to the model before its only fit, not the returned one."""
    cs = Case(fam, 260, 300, 3, 41, kcap=4, max_iter=1)
    r, _, _ = cs.fit_and_probe(4, [0, 1, 2, 3])
    assert all(int(v) == 2 for v in r["l"])  # max_iter + 1: the stopping rule did not fire
    cs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_ridge_sacrifice(fam):
    """lambda > 0 through run_batch_groups without groups, probed at the same level"""
    cs = Case(fam, 301, 400, 5, 51, kcap=4)
    for T in (2, 4):
        cs.fit_and_probe(T, list(range(6)), lam=0.05, ridge_api=True)
    cs.close()


@pytest.mark.gpu
def test_hard_numerics():
    """logistic past the eta clamp, poisson with large counts, cox with theta over ~e^+-30 and no event in the last row
    split (several splits, so the risk-set sums of the later splits carry into the earlier ones)"""
    cs = Case("binomial", 300, 40, 3, 61, kcap=2, kind="separable")
    _, _, etas = cs.fit_and_probe(1, [0, 1, 2, 3], well_conditioned=False)
    cs.fit_and_probe(2, [0, 1, 2, 3], well_conditioned=False)
    assert max(float(np.max(np.abs(e))) for e in etas) > 30.0
    cs.close()
    cs = Case("poisson", 300, 40, 3, 62, kcap=2, kind="large_counts")
    cs.fit_and_probe(1, [0, 1, 2, 3], well_conditioned=False)
    cs.fit_and_probe(2, [0, 1, 2, 3], well_conditioned=False)
    cs.close()
    for K in (0, 5, 11):
        cs = Case("cox", 389, 60, K, 63, kcap=2, kind="cox_hard")
        for T in (1, 2):
            _, info, etas = cs.fit_and_probe(T, list(range(K + 1)), well_conditioned=False)
            assert info["S"] >= 3 and (info["S"] - 1) * info["rows_per_split"] >= (2 * 389) // 3, info
        assert float(np.max(etas[0]) - np.min(etas[0])) > 20.0
        cs.close()


def _gindex(widths, p):
    gi, k = [0], 0
    while gi[-1] + widths[k % len(widths)] < p:
        gi.append(gi[-1] + widths[k % len(widths)])
        k += 1
    return np.array(gi, dtype=np.int32)


def _group_mask(fam, nch, sizes):
    if fam == "cox":
        m = GSAC_SERIAL
    elif nch == 1:
        m = GSAC_WARP
    else:
        m = 0
        m |= GSAC_B2 if np.any(sizes <= 2) else 0
        m |= GSAC_B4 if np.any((sizes > 2) & (sizes <= 4)) else 0
        m |= GSAC_B8 if np.any((sizes > 4) & (sizes <= 8)) else 0
    return m | (GSAC_WIDE if np.any(sizes > 8) else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_group_sacrifice(fam):
    """widths 1..8 mixed (all three batched classes in one call, 6 and 12 chain slots: not powers of two), a single-chain
    batch, widths 9..20 beside narrow groups, ridge levels"""
    cases = [(389, 301, 5, [1, 2, 3, 4, 5, 6, 7, 8], (0.0, 0.03)), (200, 250, 11, [3, 1, 8, 2, 5, 4, 7, 6], (0.0,)),
             (97, 140, 3, [9, 2, 20, 1, 13, 6], (0.0, 0.02))]
    for n, p, K, widths, lams in cases:
        gi = _gindex(widths, p)
        cs = Case(fam, n, p, K, 70 + K, kcap=3, g_index=gi)
        sizes = cs.groups[1]
        for chains in (list(range(K + 1)), [0]):
            for lam in lams:
                for T in (1, 3):
                    _, info, _ = cs.fit_and_probe(T, chains, lam=lam)
                    assert info["kernel"] == "group" and info["groups"] == _group_mask(fam, len(chains), sizes), info
        cs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_group_sacrifice_nearly_collinear_block(fam):
    """one group of four whose last column is the third plus 1e-4 noise: a block condition number of about 1e8"""
    cs = Case(fam, 300, 48, 3, 81, kcap=2, kind="collinear", g_index=np.arange(0, 48, 4))
    for chains in ([0, 1, 2, 3], [0]):
        for T in (1, 2):
            cs.fit_and_probe(T, chains, lam=0.0, well_conditioned=False)
    Xg = cs.X[:, 4:8].astype(np.float64)
    assert np.linalg.cond(Xg.T @ Xg) > 1e6
    cs.close()


# ---------------------------------------------------------------------------------------------------------------------
# whole fits at every chain-slot count
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("K", [5, 7, 11, 15, 23, 31])
@pytest.mark.parametrize("fam", ["gaussian", "binomial", "poisson", "cox"])
def test_fit_level_parity_every_chain_slot_count(fam, K):
    """Algorithm::fit granularity at K + 1 chains (6 .. 32 chain slots): every chain against oracle.pdas_fit, warm-started
    across levels, plus Metric train / test losses.  For gaussian this runs the resident kernel at 8 / 16 chain slots."""
    from bess_b200 import cbess
    from bess_b200.engine import GpuEngine
    from bess_b200.gen_data import gen_data
    model_type, data_type = FAM[fam]
    n, p = (301, 503) if fam == "cox" else (300, 501)
    d = gen_data(n, p, fam, 5, seed=90 + K)
    w = np.random.default_rng(90 + K).uniform(0.5, 1.5, n)
    fold = cbess.cv_fold_ids(n, K, 7 + K)
    eng = GpuEngine()
    eng.load(d.x, d.y, w, model_type)
    eng.normalize(data_type, True)
    data = orc.make_data(d.x, d.y, w, data_type, True, model_type)
    Ts = [1, 3, 5]
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
            assert r["A"][ci].tolist() == o.A.tolist(), (T, ci)
            assert int(r["l"][ci]) == o.l, (T, ci)
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


@pytest.mark.gpu
def test_every_reachable_sacrifice_kernel_ran():
    """Last in the module: every (kernel, chain slots, columns per thread, mode) of the column sweep, one and several row
    splits per family, and every group kernel were reported by the probe above."""
    want = expected_sweeps()
    assert want <= SEEN, sorted(want - SEEN)
    for fam in FAM:
        assert 1 in SPLITS[fam] and max(SPLITS[fam]) > 1, (fam, sorted(SPLITS[fam]))
    allg = GSAC_SERIAL | GSAC_WARP | GSAC_B2 | GSAC_B4 | GSAC_B8 | GSAC_WIDE
    assert SEEN_GROUP == allg, bin(SEEN_GROUP)
    print("largest err / bound per family:", {f: float(f"{v:.3g}") for f, v in sorted(WORST.items())},
          "row splits:", {f: sorted(s) for f, s in sorted(SPLITS.items())})

"""The chain fit's numerical core (bess_b200/csrc/chain_fit.cu) against high-precision references, one building block at a
time: the weighted Gram (register-blocked FMA and FP64 tensor-core paths) and the bordered normal-equation solve, through
probes that run the production code at the placement a fit uses (bess_b200_debug_gram_rows / _debug_solve_path), then
whole fits at every cluster size.

References are computed here, from the fp64 inputs, in np.longdouble (the CPU tests check them against mpmath).  Size
boundaries of the solver dispatch are found by asking the solve probe which solver finished, not written down."""
import ctypes as C
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pdas_oracle as orc
from tests.helpers import RTOL, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
FIT_SMEM_MS = 64
# path codes of bess_b200_debug_solve_path (chain_fit.cu SOLVE_*)
WARP, WARP_LDLT, SMEM, SMEM_LDLT, PANEL, PACKED = 1, 2, 3, 4, 10, 30
SENTINEL = -7.77e300
PATHS_SEEN = set()


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def gram_ref(V, w, r0, r1, mm):
    """S = sum_r w_r v_a v_b and the bound sum_r |w_r v_a v_b|, both in long double."""
    X = V[r0:r1, :mm].astype(np.longdouble)
    ww = np.ones(r1 - r0, dtype=np.longdouble) if w is None else w[r0:r1].astype(np.longdouble)
    S = (X * ww[:, None]).T @ X
    B = (np.abs(X) * np.abs(ww)[:, None]).T @ np.abs(X)
    return S, B


def solve_ref(A, b):
    """x of A x = b to long-double accuracy: fp64 LU with iterative refinement on long-double residuals (converges for
    condition numbers well below 1 / 2^-53)."""
    import scipy.linalg
    lu = scipy.linalg.lu_factor(A)
    Al = np.asarray(A, dtype=np.longdouble)
    bl = np.asarray(b, dtype=np.longdouble)
    x = scipy.linalg.lu_solve(lu, b).astype(np.longdouble)
    for _ in range(6):
        x = x + scipy.linalg.lu_solve(lu, (bl - Al @ x).astype(np.float64)).astype(np.longdouble)
    return x


def spd_system(nu, kappa, seed):
    """A = Q diag(sigma) Q^T (fp64) with condition ~kappa, a right-hand side, and the bordered (nu + 1)^2 matrix."""
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((nu, nu)))
    sig = np.logspace(0, -np.log10(kappa), nu) if nu > 1 else np.ones(1)
    A = (Q * sig) @ Q.T
    A = 0.5 * (A + A.T)
    b = rng.standard_normal(nu)
    return A, b


def bordered(A, b, c=1.0):
    nu = A.shape[0]
    S = np.zeros((nu + 1, nu + 1))
    S[:nu, :nu] = A
    S[nu, :nu] = b
    S[:nu, nu] = b
    S[nu, nu] = c
    return S


def normal_eq(V, y):
    """V^T V and V^T y, exactly symmetric, with the rows of identical columns made bit-identical (a BLAS product may round
    them differently, and which copy a pivoted solver keeps would then ride on that)"""
    G, b = V.T @ V, V.T @ y
    G = 0.5 * (G + G.T)
    for j in range(V.shape[1]):
        for i in range(j):
            if np.array_equal(V[:, i], V[:, j]):
                G[j, :] = G[i, :]
                G[:, j] = G[:, i]
                G[j, j] = G[i, i]
                b[j] = b[i]
                break
    return G, b


# ---------------------------------------------------------------------------------------------------------------------
# probes
# ---------------------------------------------------------------------------------------------------------------------
def _lib():
    from bess_b200 import _lib as L
    lib = L.load()
    L.require_gpu()
    lib.bess_b200_debug_solve_path.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.bess_b200_debug_gram_rows.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                              C.c_int, C.c_int]
    lib.bess_b200_debug_solve.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    return lib, L


def solve_path(S, kcap):
    """-> x, path code, truncated-solve count, wide-singular count"""
    lib, L = _lib()
    S = np.ascontiguousarray(S, dtype=np.float64)
    mm = S.shape[0] - 1
    x = np.zeros(mm)
    po = np.zeros(3, dtype=np.int32)
    L.check(lib.bess_b200_debug_solve_path(S.ctypes.data, S.shape[1], mm, kcap, x.ctypes.data, po.ctypes.data))
    PATHS_SEEN.add(int(po[0]))
    return x, int(po[0]), int(po[1]), int(po[2])


def path_of(nu, kcap):
    return solve_path(bordered(2.0 * np.eye(nu), np.ones(nu)), kcap)[1]


def gram_rows(V, r0, r1, mm, w, kcap, impl):
    lib, L = _lib()
    V = np.ascontiguousarray(V, dtype=np.float64)
    ldv = V.shape[1]
    ldo = FIT_SMEM_MS if mm <= FIT_SMEM_MS else ldv
    S = np.full((ldo, ldo), SENTINEL)
    wp = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
    L.check(lib.bess_b200_debug_gram_rows(V.ctypes.data, ldv, r0, r1, mm, None if wp is None else wp.ctypes.data,
                                          S.ctypes.data, kcap, impl))
    return S


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the references themselves
# ---------------------------------------------------------------------------------------------------------------------
def test_references_against_mpmath():
    import mpmath
    mpmath.mp.dps = 60
    rng = np.random.default_rng(1)
    V = rng.standard_normal((9, 5)) * np.array([1e-6, 1.0, 1e6, 3.0, 1e3])
    w = 10.0 ** rng.uniform(-8, 8, 9)
    w[2] = 0.0
    S, B = gram_ref(V, w, 2, 9, 5)
    for a in range(5):
        for b in range(5):
            ex = mpmath.fsum(mpmath.mpf(w[r]) * mpmath.mpf(V[r, a]) * mpmath.mpf(V[r, b]) for r in range(2, 9))
            got = mpmath.mpf(np.format_float_scientific(S[a, b], precision=30))  # every bit of the long double
            assert abs(got - ex) <= mpmath.mpf(2.0 ** -60) * mpmath.mpf(float(B[a, b]))
    for kappa in (1.0, 1e8):
        A, b = spd_system(7, kappa, 3)
        x = solve_ref(A, b)
        ex = mpmath.lu_solve(mpmath.matrix(A.tolist()), mpmath.matrix(b.tolist()))
        for i in range(7):
            assert abs(mpmath.mpf(float(x[i])) - ex[i]) <= mpmath.mpf(1e-15) * kappa * mpmath.norm(ex, mpmath.inf)


def test_rank_revealing_oracle_truncates_duplicates():
    rng = np.random.default_rng(2)
    V = rng.standard_normal((40, 6))
    V[:, 4] = V[:, 1]
    G, b = normal_eq(V, rng.standard_normal(40))
    x = orc.solve_rank_revealing(G, b)
    assert (x[1] == 0.0) != (x[4] == 0.0) and np.count_nonzero(x) == 5
    assert np.allclose(V @ x, V @ np.linalg.lstsq(V, V @ x, rcond=None)[0])


# ---------------------------------------------------------------------------------------------------------------------
# Gram
# ---------------------------------------------------------------------------------------------------------------------
GRAM_MM = [1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 55, 56, 57, 60, 63, 64, 65, 96, 97, 144, 145, 203, 265]
GRAM_ROWS = [1, 2, 3, 4, 5, 63, 64, 65, 129, 193, 1800]


def _gram_case(mm, rows, r0, wkind, narrow, seed):
    rng = np.random.default_rng(seed)
    kcap = max(mm - 2, 1)
    mp = (mm + 3) // 4 * 4
    ldv = (kcap + 3) & ~1
    if narrow and ldv >= mp and mm < ldv:  # ldv < mp: the row is shorter than the padded tile width
        ldv = mm + (mm & 1)
    if ldv < mm:
        ldv = mm + (mm & 1)
    V = rng.standard_normal((r0 + rows, ldv)) * 10.0 ** rng.uniform(-6, 6, ldv)
    if mm >= 4:
        V[:, mm - 1] = V[:, 1]        # an exact duplicate
        V[:, mm // 2] = 0.0           # a zero column
    if wkind == "null":
        w = None
    else:
        w = 10.0 ** rng.uniform(-8, 8, r0 + rows)
        w[rng.random(r0 + rows) < 0.1] = 0.0
    return V, w, kcap, ldv


def _check_gram(S, V, w, r0, r1, mm, dup=True):
    ref, B = gram_ref(V, w, r0, r1, mm)
    got = S[:mm, :mm]
    err = np.abs(got.astype(np.longdouble) - ref)
    bound = (r1 - r0 + 4) * U * B
    assert np.all(err <= bound), f"max excess {np.max(err - bound)}"
    assert np.array_equal(got, got.T)
    out = np.ones(S.shape, dtype=bool)
    out[:mm, :mm] = False
    assert np.all(S[out] == SENTINEL), "write outside the mm x mm output"
    if dup and mm >= 4:  # columns 1 and mm-1 are identical: their Gram entries on the same side of both are bit-equal
        j1, j2 = 1, mm - 1
        assert got[j1, j1] == got[j2, j2] == got[j1, j2] == got[j2, j1]
        side = [c for c in range(mm) if c < j1 or c > j2]
        assert np.array_equal(got[j1, side], got[j2, side])


@pytest.mark.gpu
@pytest.mark.parametrize("mm", GRAM_MM)
def test_gram_against_long_double(mm):
    """Every width around the 4-column blocks, the FMA / DMMA switch (56 / 57), the Ssm output limit (64) and the DMMA pass
    count, at row counts around the 4-row steps and the 64-row ring stages, from row 0 and from row 37 (a cluster slice),
    weighted (zeros, 1e-8..1e8) or not, with the row as long as the padded tile or shorter."""
    impls = [0, 1, 2] if mm <= 97 else [0, 2]
    case = 0
    for rows in GRAM_ROWS:
        for r0 in (0, 37):
            wkind = "null" if case % 3 == 2 else "w"
            V, w, kcap, ldv = _gram_case(mm, rows, r0, wkind, case % 2 == 1, 1000 * mm + case)
            case += 1
            for impl in impls:
                S = gram_rows(V, r0, r0 + rows, mm, w, kcap, impl)
                _check_gram(S, V, w, r0, r0 + rows, mm)


@pytest.mark.gpu
def test_gram_dmma_ring_beside_ssm_in_minimal_arena():
    """57..64 columns on the tensor cores with a support cap small enough for the minimal arena: the ring must stay clear
    of the output in sm.Ssm."""
    for mm in (57, 60, 64):
        for kcap in (mm - 2, mm + 40):
            rng = np.random.default_rng(mm + kcap)
            ldv = (kcap + 3) & ~1
            V = rng.standard_normal((900, ldv))
            w = rng.uniform(0.1, 2.0, 900)
            for impl in (0, 2):
                _check_gram(gram_rows(V, 11, 900, mm, w, kcap, impl), V, w, 11, 900, mm, dup=False)


# ---------------------------------------------------------------------------------------------------------------------
# SPD solves through the production dispatcher
# ---------------------------------------------------------------------------------------------------------------------
def _largest(lo, hi, pred):
    """largest n in [lo, hi] with pred(n) (pred monotone: true then false), lo assumed true"""
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if pred(mid):
            lo = mid
        else:
            hi = mid - 1
    return lo


KCAP_BIG = 510


@functools.lru_cache(maxsize=None)
def stage_boundaries():
    """smallest size of every panel-major stage count at the largest support cap, and the largest panel-major size"""
    top = 511
    code_top = path_of(top, KCAP_BIG)
    panel_max = top if code_top < PACKED else _largest(65, top, lambda n: path_of(n, KCAP_BIG) < PACKED)
    nmax = path_of(panel_max, KCAP_BIG) - PANEL
    first = {1: 64}
    for s in range(2, nmax + 1):
        first[s] = _largest(64, panel_max, lambda n: path_of(n, KCAP_BIG) - PANEL < s) + 1
    return first, panel_max, panel_max < top and path_of(panel_max + 1, KCAP_BIG) == PACKED


def _check_spd(nu, kappa, kcap, seed):
    A, b = spd_system(nu, kappa, seed)
    x, code, rd, ws = solve_path(bordered(A, b), kcap)
    assert rd == 0 and ws == 0 and code not in (WARP_LDLT, SMEM_LDLT)
    xr = solve_ref(A, b)
    xl = x.astype(np.longdouble)
    res = np.linalg.norm((b.astype(np.longdouble) - A.astype(np.longdouble) @ xl).astype(np.float64))
    berr = res / (np.linalg.norm(A, 2) * np.linalg.norm(x) + np.linalg.norm(b))
    ferr = float(np.linalg.norm((xl - xr).astype(np.float64)) / np.linalg.norm(xr.astype(np.float64)))
    assert berr <= 8 * nu * U, (nu, kappa, kcap, code, berr)
    assert ferr <= 8 * nu * kappa * U, (nu, kappa, kcap, code, ferr)
    return code


@pytest.mark.gpu
def test_spd_solves_every_path():
    first, panel_max, packed = stage_boundaries()
    sizes = {1, 2, 15, 16, 17, 30, 31, 32, 33, 47, 62, 63, 64, 65, 80, 128, 129, panel_max}
    for s, n0 in first.items():
        sizes |= {n0, n0 - 1} if s > 1 else set()
    for nu in sorted(sizes):
        for kcap in sorted({max(nu - 1, 1), KCAP_BIG}):
            for kappa in (1.0, 1e4, 1e8, 1e12):
                code = _check_spd(nu, kappa, kcap, seed=nu)
                if nu <= 31 and kcap == KCAP_BIG:
                    assert code == WARP
                elif nu <= 63:
                    assert code in (WARP, SMEM)
                else:
                    assert code > PANEL
    if packed:
        _check_spd(panel_max + 1, 1e4, KCAP_BIG, seed=5)


@pytest.mark.gpu
def test_spd_solves_old_probe():
    """bess_b200_debug_solve: the panel-major (impl 0) and packed (impl 1) solvers called directly."""
    lib, L = _lib()
    for nu, impls in ((65, (0, 1)), (130, (0, 1)), (200, (0, 1)), (300, (0,)), (480, (0,))):
        for kappa in (1.0, 1e8):
            A, b = spd_system(nu, kappa, nu)
            lds = (nu + 3) & ~1
            S = np.zeros((nu + 1, lds))
            S[:nu, :nu] = A
            S[nu, :nu] = b
            xr = solve_ref(A, b)
            for impl in impls:
                x = np.zeros(nu)
                L.check(lib.bess_b200_debug_solve(S.ctypes.data, lds, nu, x.ctypes.data, impl, 1, None))
                ferr = float(np.linalg.norm((x.astype(np.longdouble) - xr).astype(np.float64)) / np.linalg.norm(xr.astype(np.float64)))
                assert ferr <= 8 * nu * kappa * U, (nu, kappa, impl, ferr)


# ---------------------------------------------------------------------------------------------------------------------
# rank-deficient systems
# ---------------------------------------------------------------------------------------------------------------------
def _near_dup(rng, n, nu, j1, j2, ratio):
    """column j2 = column j1 + eps z with the Schur pivot of j2 ~ ratio x its diagonal"""
    V = rng.standard_normal((n, nu))
    z = rng.standard_normal(n)
    z -= V[:, j1] * (V[:, j1] @ z) / (V[:, j1] @ V[:, j1])
    V[:, j2] = V[:, j1] + np.sqrt(ratio) * np.linalg.norm(V[:, j1]) / np.linalg.norm(z) * z
    return V


def deficient_cases(nu, rng):
    n = 3 * nu + 20
    out = []
    V = rng.standard_normal((n, nu)); V[:, nu - 1] = V[:, 0]; out.append(("dup", V))
    if nu >= 4:
        V = rng.standard_normal((n, nu)); V[:, 2] = V[:, 0]; V[:, nu - 1] = V[:, 1]; out.append(("two_dups", V))
    for a, b in ((15, 16), (30, 31), (31, 32), (16, 40), (0, 32)):
        if b < nu:
            V = rng.standard_normal((n, nu)); V[:, b] = V[:, a]; out.append((f"dup_{a}_{b}", V))
    if nu >= 33:  # the largest diagonal, twice, in the same lane of the pivot search: the first copy must win
        V = rng.standard_normal((n, nu)); V[:, 0] *= 3.0; V[:, 32] = V[:, 0]; out.append(("dup_max_0_32", V))
    V = rng.standard_normal((n, nu)); V[:, nu // 2] = 0.0; out.append(("zero_col", V))
    if nu >= 3:
        out.append(("few_rows", rng.standard_normal((nu - 2, nu))))
    if nu >= 2:
        out.append(("pivot_100x_above", _near_dup(rng, n, nu, 0, nu - 1, 1e-11)))
        out.append(("pivot_100x_below", _near_dup(rng, n, nu, 0, nu - 1, 1e-15)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [2, 3, 5, 16, 17, 31, 32, 33, 47, 63])
def test_rank_deficient_small_matches_rank_revealing_oracle(nu):
    rng = np.random.default_rng(nu)
    for name, V in deficient_cases(nu, rng):
        G, b = normal_eq(V, rng.standard_normal(V.shape[0]))
        xo = orc.solve_rank_revealing(G, b)
        trunc = np.count_nonzero(xo) < nu
        for kcap in sorted({max(nu - 1, 1), 200}):
            x, code, rd, ws = solve_path(bordered(G, b), kcap)
            assert ws == 0
            assert (code in (WARP_LDLT, SMEM_LDLT)) == trunc, (name, kcap, code)
            assert rd == (1 if trunc else 0), (name, kcap, rd)
            assert np.array_equal(x == 0.0, xo == 0.0), (name, kcap)
            # a full-rank but nearly singular system (pivot 100x above the tolerance) agrees to its conditioning only
            tol = 1e-10 if trunc else max(1e-10, 8 * nu * np.linalg.cond(G) * U)
            assert np.max(np.abs(x - xo)) <= tol * np.linalg.norm(xo), (name, kcap)


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [64, 65, 100, 200, 300])
def test_rank_deficient_wide_never_finite_and_wrong(nu):
    """No rank-revealing solver above 63 unknowns: a singular system must come back non-finite and counted."""
    rng = np.random.default_rng(nu)
    cases = [c for c in deficient_cases(nu, rng) if c[0] != "pivot_100x_above"]
    for name, V in cases:
        G, b = normal_eq(V, rng.standard_normal(V.shape[0]))
        for kcap in sorted({nu - 1, KCAP_BIG}):
            x, code, rd, ws = solve_path(bordered(G, b), kcap)
            assert code > PANEL
            assert ws == 1 and np.all(np.isnan(x)), (name, kcap, ws, x[:4])


# ---------------------------------------------------------------------------------------------------------------------
# whole fits at every cluster size
# ---------------------------------------------------------------------------------------------------------------------
FIT_CASES = [("gaussian", 2048, 300, 100), ("gaussian", 2048, 400, 250), ("binomial", 2048, 300, 80),
             ("cox", 2048, 300, 70), ("poisson", 2048, 300, 30)]
FAMS = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}

_WORKER = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from bess_b200.engine import GpuEngine
from bess_b200.gen_data import gen_data
cases = json.loads(sys.argv[2])
res = []
for fam, n, p, T, model_type, data_type in cases:
    d = gen_data(n, p, fam, 10, seed=31)
    eng = GpuEngine()
    eng.load(d.x, d.y, np.ones(n), model_type)
    eng.normalize(data_type, True)
    eng.setup_chains(0, None, T, 20, True)
    r = eng.run_batch(T, [0], True)
    res.append(dict(A=r["A"][0].tolist(), l=int(r["l"][0]), bA=r["bA"][0].tolist(), coef0=float(r["coef0"][0]),
                    cl=eng.stats()["max_cluster"]))
    eng.close()
print("RESULT" + json.dumps(res))
"""


def _run_cl(cl):
    env = dict(os.environ, BESS_B200_CL_MAX=str(cl), BESS_B200_CL_WORK="1")
    cases = [(f, n, p, T, *FAMS[f]) for f, n, p, T in FIT_CASES]
    out = subprocess.run([sys.executable, "-c", _WORKER, ROOT, json.dumps(cases)], env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT")][-1]
    return json.loads(line[6:])


@pytest.mark.gpu
def test_fit_level_every_cluster_size():
    from bess_b200.gen_data import gen_data
    runs = {cl: _run_cl(cl) for cl in (1, 2, 4, 8, 16)}
    for i, (fam, n, p, T) in enumerate(FIT_CASES):
        model_type, data_type = FAMS[fam]
        d = gen_data(n, p, fam, 10, seed=31)
        w = np.ones(n)
        data = orc.make_data(d.x, d.y, w, data_type, True, model_type)
        st = orc.PathState(data, model_type, 3, False, 0, None, 20, True)
        o = orc.pdas_fit(data, model_type, T, np.zeros(p), 0.0, st.full_mask, st.xtx_full, 20)
        base = runs[1][i]
        for cl, res in runs.items():
            r = res[i]
            assert r["A"] == o.A.tolist() and r["l"] == o.l, (fam, T, cl)
            assert rel_err(np.array(r["bA"]), o.beta[o.A]) < RTOL, (fam, T, cl)
            assert abs(r["coef0"] - o.coef0) <= RTOL * max(1.0, abs(o.coef0))
            assert rel_err(np.array(r["bA"]), np.array(base["bA"])) < 1e-12, (fam, T, cl)
            assert abs(r["coef0"] - base["coef0"]) <= 1e-12 * max(1.0, abs(base["coef0"]))
    missing = [(cl, FIT_CASES[i]) for cl, res in runs.items() for i, r in enumerate(res) if r["cl"] != cl]
    if missing:
        pytest.skip(f"the device did not schedule the forced cluster size for {missing} (stats()[7] differs)")


@pytest.mark.gpu
@pytest.mark.parametrize("is_cv", [False, True])
def test_supports_wider_than_train_rows_fail_loudly(is_cv):
    """n = 60 rows, s.list = 1..70: every level >= 60 (>= 48 in a CV fold) is singular; levels >= 64 are wide systems."""
    from bess_b200 import _lib as L, cbess
    from bess_b200.gen_data import gen_data
    d = gen_data(60, 200, "gaussian", 5, seed=4)
    seq = np.arange(1, 71)
    try:
        out = cbess.fit(d.x, d.y, 1, np.ones(60), True, 1, 1, 20, 2, 1, True, 1, is_cv, 5, seq, 1, 70, False, 1)
    except L.BessB200Error as e:
        assert "rank-deficient wide system" in str(e)
        return
    assert np.all(np.isfinite(out["ic_all"])) and np.all(np.isfinite(out["loss_all"]))


@pytest.mark.gpu
def test_every_reachable_solver_path_ran():
    """Last in the module: every solver the probe can reach finished at least one solve above."""
    first, panel_max, packed = stage_boundaries()
    want = {WARP, WARP_LDLT, SMEM, SMEM_LDLT} | {PANEL + s for s in first} | ({PACKED} if packed else set())
    assert want <= PATHS_SEEN, sorted(want - PATHS_SEEN)

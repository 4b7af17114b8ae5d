"""CPU-only checks of the boundary: the shared library loads, exports every symbol include/bess_b200.h declares (and the
reference's C++-mangled pywrap_bess), refuses loudly to compute without a GPU, and its pure-host helpers are right."""
import os
import re
import subprocess

import numpy as np
import pytest

from tests.helpers import golden_names, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MANGLED = "_Z11pywrap_bessPdiiS_iiS_ibiiiiibibiPiiS_iS0_iS_iiiidddibiiS0_idS_iS_iS_iS_iS_S_iS_iS_iS0_iS0_"


def _lib():
    from bess_b200 import _lib
    return _lib.load()


def test_library_exports_every_declared_symbol():
    lib = _lib()
    hdr = open(os.path.join(ROOT, "include", "bess_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b((?:bess_b200|bessgpu)_[a-z0-9_]+|pywrap_bess)\s*\(", hdr))
    assert {"pywrap_bess", "bess_b200_fit", "bessgpu_run_batch", "bess_b200_merge_candidates"} <= names
    for nm in sorted(names):
        assert hasattr(lib, nm), f"{nm} declared in include/bess_b200.h but not exported"
    assert lib.bess_b200_version() == 100


def test_reference_cxx_linkage_symbol_is_exported():
    """The reference's pywrap_bess has C++ linkage (bess.h:35-51); a SWIG module built from its bess.i must link."""
    from bess_b200 import _lib
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.SO_PATH], capture_output=True, text=True).stdout
    assert MANGLED in out
    assert re.search(r"\bT pywrap_bess\b", out)


def test_no_cpu_fallback_without_a_gpu():
    from bess_b200 import _lib, cbess
    lib = _lib.load()
    if lib.bess_b200_device_count() > 0:
        pytest.skip("a GPU is present")
    x = np.random.default_rng(0).standard_normal((20, 8))
    with pytest.raises(_lib.BessB200Error):
        cbess.fit(x, x[:, 0], 1, np.ones(20), True, 1, 1, 20, 2, 1, True, 3, False, 5, [1, 2], 1, 2, False, 1)
    with pytest.raises(_lib.BessB200Error):
        from bess_b200.engine import GpuEngine
        GpuEngine()


def test_product_never_imports_the_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "bess_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".cuh")):
                src = open(os.path.join(root, f)).read()
                assert "oracle" not in src.replace("the oracle", "").replace("numpy oracle", ""), f


@pytest.mark.parametrize("name", [n for n in golden_names() if "cv" in n])
def test_cv_folds_match_the_reference_draw(name):
    """Metric.h:49-106 restated in path.cpp: same mt19937 + std::shuffle + chunking => the folds the reference drew."""
    from bess_b200 import cbess
    g = load_golden(name)
    assert cbess.cv_fold_ids(g["x"].shape[0], g["K"], 123).tolist() == g["fold_of_row"].tolist()


def test_shard_ranges_cover_columns_contiguously():
    import ctypes as C
    lib = _lib()
    for p in (1, 2, 7, 5000, 500000, 500001):
        for world in (1, 2, 3, 4, 8):
            prev = 0
            for r in range(world):
                lo, hi = C.c_longlong(), C.c_longlong()
                lib.bess_b200_shard_range(p, world, r, C.byref(lo), C.byref(hi))
                assert lo.value == prev and hi.value >= lo.value and (lo.value % 2 == 0 or lo.value == p)
                prev = hi.value
            assert prev == p
    assert [lib.bess_b200_chain_owner(c, 4) for c in range(6)] == [0, 1, 2, 3, 0, 1]


def test_merge_candidates_is_exact_topk():
    from bess_b200._lib import dp, ip
    lib = _lib()
    rng = np.random.default_rng(1)
    v = np.floor(rng.random(1000) * 50)
    idx = rng.permutation(1000).astype(np.int32)
    k = 37
    out = np.zeros(k, dtype=np.int32)
    assert lib.bess_b200_merge_candidates(v.ctypes.data_as(dp), idx.ctypes.data_as(ip), 1000, k, out.ctypes.data_as(ip)) == 0
    order = np.lexsort((idx, -v))
    assert out.tolist() == sorted(idx[order[:k]].tolist())


def test_frontend_argument_surface(monkeypatch):
    """family/method/s.list/nfolds/IC/screening.num -> the integer codes of the reference (linear.py:138-324)."""
    from bess_b200 import linear
    seen = {}

    def fake(*args):
        seen["args"] = args
        p = args[0].shape[1]
        return [np.zeros(p), 0.0, 0.0, 0.0, 0.0, None, None, None, None, 0]
    monkeypatch.setattr(linear, "pywrap_bess", fake)
    x = np.random.default_rng(0).standard_normal((50, 30))
    m = linear.PdasLogistic(path_type="pgs", ic_type="gic", is_cv=True, K=7, is_screening=True, screening_size=20)
    m.fit(x, (x[:, 0] > 0).astype(float))
    a = seen["args"]
    assert a[2] == 2 and a[5] == 1 and a[6] == 2 and a[9] == 2 and a[11] == 3 and a[12] is True and a[13] == 7
    assert a[18] == 1 and a[19] == 30 and a[25] is True and a[26] == 20 and a[30] == 30
    m = linear.PdasCox(path_type="seq", sequence=[1, 2, 3])
    t = np.random.default_rng(1).random(50)
    m.fit(x, np.column_stack([t, np.ones(50)]))
    a = seen["args"]
    assert a[2] == 3 and a[6] == 4 and a[9] == 1 and list(a[16]) == [1, 2, 3]
    assert np.allclose(a[0], x[np.argsort(t)])  # rows time-sorted (linear.py:257-263)
    with pytest.raises(ValueError):
        linear.PdasLm(is_screening=True, screening_size=2, sequence=[1, 2, 3]).fit(x, x[:, 0])
    with pytest.raises(ValueError):
        linear.bess_base("Nope", "Lm", "seq")
    # the twelve estimator classes of the reference (linear.py:434-925) and their codes
    for alg, code in (("Pdas", 1), ("L0L2", 5), ("GroupPdas", 2)):
        for model, (mt, dt) in {"Lm": (1, 1), "Logistic": (2, 2), "Poisson": (3, 2), "Cox": (4, 3)}.items():
            est = getattr(linear, alg + model)()
            assert (est.algorithm_type_int, est.model_type_int, est.data_type) == (code, mt, dt)
    # bsrr: Powell search arguments travel unchanged (linear.py:360-372)
    m = linear.L0L2Lm(path_type="pgs", s_min=2, s_max=9, lambda_min=0.01, lambda_max=10, powell_path=2)
    m.fit(x, x[:, 0])
    a = seen["args"]
    assert a[5] == 5 and a[9] == 2 and (a[18], a[19]) == (2, 9) and (a[22], a[23], a[24]) == (0.01, 10, 100) and a[27] == 2
    # sequential lambda grid
    m = linear.L0L2Poisson(sequence=[1, 2], lambda_sequence=[0.1, 1.0])
    m.fit(x, np.ones(50))
    assert list(seen["args"][17]) == [0.1, 1.0] and list(seen["args"][16]) == [1, 2]
    # GroupPdas: group labels -> first column of each group (linear.py:238-254)
    m = linear.GroupPdasLm(sequence=[1, 2])
    with pytest.raises(ValueError):
        m.fit(x, x[:, 0])
    m.fit(x, x[:, 0], group=list(range(30)))
    assert list(seen["args"][14]) == list(range(30)) and seen["args"][5] == 2
    m.fit(x, x[:, 0], group=[i // 3 for i in range(30)])
    assert list(seen["args"][14]) == list(range(0, 30, 3))
    with pytest.raises(ValueError):
        m.fit(x, x[:, 0], group=[0, 1])


def test_pgs_line_box_matches_the_oracle():
    """Host logic of the Powell path (path.cpp:414-577) without a GPU: the library's line/box intersection against the
    numpy restatement on random lines through random points of the (s, log lambda) box, incl. axis-parallel directions."""
    import ctypes as C
    from bess_b200._lib import dp
    from oracle import pdas_oracle as orc
    lib = _lib()
    rng = np.random.default_rng(5)
    s_min, s_max, lmin, lmax = 2, 17, float(np.log(1e-3)), float(np.log(50.0))
    dirs = [(1.0, 0.0), (0.0, 0.1), (3.0, -0.7), (-2.0, 1.3), (5.0, 2.0)]
    for t in range(200):
        p = np.array([float(rng.integers(s_min, s_max + 1)), rng.uniform(lmin, lmax)])
        u = np.array(dirs[t % len(dirs)]) if t < 100 else np.array([float(rng.integers(-6, 7)), rng.normal()])
        if u[0] == 0.0 and abs(u[1]) < 1e-3:
            continue
        a, b = np.zeros(2), np.zeros(2)
        n = lib.bess_b200_pgs_line_box(p.ctypes.data_as(dp), u.ctypes.data_as(dp), s_min, s_max, lmin, lmax,
                                       a.ctypes.data_as(dp), b.ctypes.data_as(dp))
        try:
            ea, eb = orc._cal_intersections(p, u, s_min, s_max, lmin, lmax)
        except ValueError:
            assert n < 2
            continue
        assert n >= 2 and np.array_equal(a, np.array(ea)) and np.array_equal(b, np.array(eb))


@pytest.mark.parametrize("compiler,std,ext", [("gcc", "-std=c99", "c"), ("g++", "-std=c++11", "cpp")])
def test_public_header_is_self_contained(tmp_path, compiler, std, ext):
    """include/bess_b200.h is what a maintainer binds against (cgo / Rcpp / SWIG): it must compile on its own as C and C++."""
    src = tmp_path / f"hdr.{ext}"
    src.write_text('#include "bess_b200.h"\nint main(void) { return 0; }\n')
    r = subprocess.run([compiler, std, "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_plain_c_program_links_and_calls_the_library(tmp_path):
    """The boundary is a C ABI: a C99 program compiled with gcc links against libbess_b200.so and calls host-only entry
    points (no GPU here); a compute entry fails loudly with a status code and a message instead of falling back."""
    src = tmp_path / "client.c"
    src.write_text(r"""
#include <stdio.h>
#include <string.h>
#include "bess_b200.h"
int main(void) {
    long long lo = -1, hi = -1;
    double p[2] = {3.0, 0.5}, u[2] = {1.0, 0.0}, a[2], b[2];
    if (bess_b200_version() != BESS_B200_VERSION) return 10;
    bess_b200_shard_range(1001, 4, 3, &lo, &hi);
    if (!(lo >= 0 && hi == 1001 && lo < hi)) return 11;
    if (bess_b200_pgs_line_box(p, u, 1, 9, 0.0, 2.0, a, b) != 2 || a[0] != 1.0 || b[0] != 9.0) return 12;
    if (bess_b200_device_count() == 0) {
        double x[6] = {1, 2, 3, 4, 5, 7}, y[3] = {1, 2, 3}, w[3] = {1, 1, 1}, beta[2], c0, tl, ic;
        int seq[1] = {1};
        double lam[1] = {0.0}, st[1] = {0.0};
        int rc = bess_b200_fit(x, 3, 2, y, 3, 1, w, 3, 1, 1, 1, 20, 2, 1, 1, 3, 0, 5, NULL, 0, st, 1, seq, 1, lam, 1, 1, 1, 10,
                               10.0, 0.0, 0.0, 1, 0, 1, 1, NULL, 0, 1.1, beta, 2, &c0, &tl, &ic, NULL);
        if (rc == 0 || strlen(bess_b200_last_error()) == 0) return 13;   /* no GPU: must fail loudly, never fall back */
    }
    printf("ok\n");
    return 0;
}
""")
    exe = tmp_path / "client"
    libdir = os.path.join(ROOT, "bess_b200")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L", libdir,
                        "-lbess_b200", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, (r.returncode, r.stdout, r.stderr)


def test_reference_module_names_resolve_to_this_library():
    """bess_b200.compat.install_as_bess(): `from bess.linear import PdasLm` / `from bess.cbess import pywrap_bess` of
    unmodified user code land in this package (python/bess/linear.py:434-925, python/bess/cbess.py:65-66)."""
    import importlib
    import sys
    from bess_b200 import compat
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "bess" or k.startswith("bess.")}
    try:
        compat.install_as_bess()
        lin = importlib.import_module("bess.linear")
        from bess.cbess import pywrap_bess  # noqa: F401
        from bess.linear import GroupPdasCox, L0L2Logistic, PdasLm
        import bess_b200.linear
        assert lin is bess_b200.linear and PdasLm is bess_b200.linear.PdasLm
        assert L0L2Logistic().algorithm_type_int == 5 and GroupPdasCox().model_type_int == 4
        sys.modules["bess"] = type(sys)("bess")  # somebody else's bess
        with pytest.raises(ImportError):
            compat.install_as_bess()
    finally:
        for k in [k for k in sys.modules if k == "bess" or k.startswith("bess.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_compat_gen_data_has_the_reference_signature_and_shapes():
    """`bess.gen_data.gen_data` served by install_as_bess takes the reference's arguments (python/bess/gen_data.py:22:
    rho=, sigma=, beta=, censoring=, c=, scal=) and returns its `data` record; cox y is the unsorted [time, status] array
    PdasCox.fit sorts itself (linear.py:257-263)."""
    import importlib
    import inspect
    import sys
    from bess_b200 import compat
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "bess" or k.startswith("bess.")}
    try:
        compat.install_as_bess()
        gd = importlib.import_module("bess.gen_data")
        assert list(inspect.signature(gd.gen_data).parameters) == ["n", "p", "family", "k", "rho", "sigma", "beta", "censoring",
                                                                   "c", "scal"]
        np.random.seed(3)
        d = gd.gen_data(60, 20, "gaussian", 3, rho=0.3, sigma=0.5)
        assert isinstance(d, gd.data) and d.x.shape == (60, 20) and d.y.shape == (60,) and np.count_nonzero(d.beta) == 3
        # banded design: column j is X_j + rho (X_{j-1} + X_{j+1}) of a centred, sqrt(n)-normalised X => neighbours correlate
        c01 = np.corrcoef(d.x[:, 5], d.x[:, 6])[0, 1]
        assert 0.2 < c01 < 0.8
        dc = gd.gen_data(50, 10, "cox", 2, 0, 1, None, True, 10, 10)  # positional, as the reference's docs call it
        assert dc.y.shape == (50, 2) and set(np.unique(dc.y[:, 1])) <= {0.0, 1.0}
        assert not np.all(np.diff(dc.y[:, 0]) >= 0)  # rows are NOT time-sorted: the estimator sorts
        dp = gd.gen_data(40, 8, "poisson", 2)
        assert dp.y.dtype.kind in "iu" or np.all(dp.y == np.round(dp.y))
    finally:
        for k in [k for k in sys.modules if k == "bess" or k.startswith("bess.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_gen_data_does_not_modify_a_supplied_design():
    from bess_b200.gen_data import gen_data
    x = np.random.default_rng(0).standard_normal((30, 12))
    x0 = x.copy()
    gen_data(30, 12, "poisson", 3, seed=2, x=x)
    gen_data(30, 12, "poisson", 3, seed=2, x=x)
    assert np.array_equal(x, x0)


def test_group_index_accepts_any_sortable_labels(monkeypatch):
    """linear.py:238-254 builds g_index by walking list(set(group)) in hash order, which runs off the list for string,
    float or large labels; here the first position of every distinct label of the sorted list is taken."""
    import bess_b200.linear as lin
    seen = {}

    def fake(*args):
        seen["g"] = list(args[14])
        return [np.zeros(args[0].shape[1]), 0.0, 0.0, 0.0, 0.0, None, None, None, None, 0]

    monkeypatch.setattr(lin, "pywrap_bess", fake)
    x = np.random.default_rng(1).standard_normal((20, 6))
    y = x[:, 0] + 0.1
    for labels in (["b", "a", "a", "c", "c", "b"], [1000003, 7, 7, -5, -5, 1000003], [0.5, 0.25, 0.25, 2.0, 2.0, 0.5]):
        lin.GroupPdasLm(sequence=[1]).fit(x, y, group=list(labels))
        assert seen["g"] == [0, 2, 4]


# Eigen 3 headers (the reference vendors 3.3.4 under python/include); none ship with this repository
EIGEN_INC = os.environ.get("EIGEN3_INCLUDE_DIR", "/usr/include/eigen3")


@pytest.mark.skipif(not os.path.isdir(os.path.join(EIGEN_INC, "Eigen")),
                    reason="no Eigen 3 headers: set EIGEN3_INCLUDE_DIR to a directory holding Eigen/")
def test_bessCpp_eigen_adaptor_compiles_and_links_against_the_vendored_eigen(tmp_path):
    """include/bess_b200_eigen.hpp: `bessCpp` with the reference's thirty by-value arguments (src/bess.h:20-33) and a
    List-shaped result (src/List.h), header-only over bess_b200_fit.  Compiled here as C++11 against the reference's own
    Eigen 3.3.4, linked against the library and run: without a GPU the call must fail loudly (std::runtime_error carrying
    the library's message), never fall back to a CPU path."""
    src = tmp_path / "client.cpp"
    src.write_text(r'''
#include <bess_b200_eigen.hpp>
#include <cstdio>
int main() {
    const int n = 40, p = 12;
    Eigen::MatrixXd x = Eigen::MatrixXd::Random(n, p);
    Eigen::VectorXd y = x.col(0) * 2.0 + Eigen::VectorXd::Random(n) * 0.01, w = Eigen::VectorXd::Ones(n), state = Eigen::VectorXd::Ones(n);
    Eigen::VectorXi seq(3); seq << 1, 2, 3;
    Eigen::VectorXd lam(1); lam << 0.0;
    Eigen::VectorXi g = Eigen::VectorXi::LinSpaced(p, 0, p - 1), always(0);
    bess_b200::List r0;
    Eigen::VectorXd z3 = Eigen::VectorXd::Zero(3), o2 = Eigen::VectorXd::Ones(2);
    r0.add("beta", z3); r0.add("beta", o2); r0.add("ic", 1.5);
    Eigen::VectorXd b; double ic = 0; r0.get_value_by_name("beta", b); r0.get_value_by_name("ic", ic);
    if (b.size() != 2 || ic != 1.5 || r0.has("nope")) return 3;
    try {
        bess_b200::List r = bess_b200::bessCpp(x, y, 1, w, true, 1, 1, 20, 2, 1, true, 3, false, 5, state, seq, lam, 1, 3, 10, 10.0,
                                               0.0, 0.0, 1, false, 1, 1, g, always, 1.1);
        Eigen::VectorXd beta; r.get_value_by_name("beta", beta);
        std::printf("fit ok nnz=%d\n", (int)(beta.array() != 0.0).count());
    } catch (const std::runtime_error &e) {
        std::printf("loud failure: %s\n", e.what());
    }
    return 0;
}
''')
    exe = tmp_path / "client"
    so_dir = os.path.join(ROOT, "bess_b200")
    r = subprocess.run(["g++", "-std=c++11", "-O1", "-w", "-I", os.path.join(ROOT, "include"), "-I", EIGEN_INC, str(src), "-o", str(exe),
                        "-L", so_dir, "-l:libbess_b200.so", "-Wl,-rpath," + so_dir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, run.stdout + run.stderr
    assert ("fit ok" in run.stdout) or ("loud failure" in run.stdout and "bess_b200" in run.stdout), run.stdout

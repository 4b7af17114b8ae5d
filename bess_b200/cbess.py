"""Stand-in for the reference's SWIG module ``bess.cbess`` (python/bess/cbess.py:65-66, generated from
python/src/bess.i:17-30).  Same Python-visible calling convention: 38 positional arguments (arrays as ndarrays or
sequences, then the 8 ARGOUT lengths) -> a 10-element list ``[beta, coef0, train_loss, ic, nullloss, aic, bic, gic,
A_out, l_out]``, of which the reference only fills the first four (bess.cpp:277-280)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import BessB200Error, Ext, dp, ip


PROF_CATS = ("screen_sweep", "dual_sweep", "finish", "topk", "chain", "other", "normalize", "upload")


def _lazy_zeros(n):
    """A zero float64 vector of length n whose pages are only materialised when touched.  np.zeros(500000) is a 4 MB memset
    once glibc has raised its mmap threshold (every call after the first): 0.2 ms, a tenth of a whole config-5 call, for a
    result with ten non-zero entries.  An anonymous mapping starts as copy-on-write zero pages."""
    if n < (1 << 16):
        return np.zeros(n)
    import mmap
    return np.frombuffer(mmap.mmap(-1, n * 8), dtype=np.float64)


def _d(a):
    return a.ctypes.data_as(dp)


def _i(a):
    return a.ctypes.data_as(ip)


def is_sparse(x):
    """A scipy.sparse matrix or array (scipy is only imported by the caller that made one)."""
    return type(x).__module__.startswith("scipy.sparse")


def _is_raw_csc(x):
    """An ``(indptr, indices, data, shape)`` tuple: three arrays (numpy or torch) and a shape tuple.  Nested sequences of
    numbers stay a dense design."""
    return (isinstance(x, tuple) and len(x) == 4 and isinstance(x[3], tuple) and len(x[3]) == 2
            and all(hasattr(a, "ndim") for a in x[:3]))


def canonical_csc(x):
    """A scipy.sparse matrix in any format -> a new CSC matrix with float64 values, int64 indptr, int32 row indices sorted
    inside every column and duplicates summed (the form bess_b200_csc requires).  The caller's matrix is not modified."""
    import scipy.sparse as sp
    if x.ndim != 2:
        raise ValueError("x must be 2-D")
    m = sp.csc_matrix(x, dtype=np.float64, copy=True)
    m.sum_duplicates()
    m.sort_indices()
    m.indptr = m.indptr.astype(np.int64, copy=False)
    m.indices = m.indices.astype(np.int32, copy=False)
    return m


def csc_arrays(x):
    """The three CSC arrays of a sparse design, passed to the library as (colptr, rowidx, values, nnz, (n, p), on_device,
    keep-alive).  ``x`` is a scipy.sparse matrix (canonicalised by canonical_csc) or a raw ``(indptr, indices, data, shape)``
    tuple taken as given -- host arrays (converted to int64 / int32 / float64) or torch CUDA tensors of exactly those
    dtypes (device-resident, read in place)."""
    if is_sparse(x):
        m = canonical_csc(x)
        arrs, shape = (m.indptr, m.indices, m.data), m.shape
    else:
        if not _is_raw_csc(x):
            raise TypeError("a sparse x is a scipy.sparse matrix or an (indptr, indices, data, shape) tuple")
        arrs, shape = tuple(x[:3]), tuple(x[3])
    n, p = int(shape[0]), int(shape[1])
    if all(getattr(a, "is_cuda", False) for a in arrs):
        want = ("torch.int64", "torch.int32", "torch.float64")
        for a, dt in zip(arrs, want):
            if str(a.dtype) != dt or not a.is_contiguous():
                raise TypeError(f"device CSC arrays must be contiguous {want} tensors")
        ptrs = [C.c_void_p(a.data_ptr()) for a in arrs]
        return ptrs[0], ptrs[1], ptrs[2], int(arrs[2].numel()), (n, p), True, arrs
    host = (np.ascontiguousarray(arrs[0], dtype=np.int64).ravel(), np.ascontiguousarray(arrs[1], dtype=np.int32).ravel(),
            np.ascontiguousarray(arrs[2], dtype=np.float64).ravel())
    if host[0].size != p + 1 or host[1].size != host[2].size:
        raise ValueError("CSC arrays: indptr needs p + 1 entries and indices / data the same length")
    ptrs = [a.ctypes.data_as(C.c_void_p) for a in host]
    return ptrs[0], ptrs[1], ptrs[2], int(host[2].size), (n, p), False, host


def _prep(x, y, weight, g_index, state, sequence, lambda_sequence, always_select):
    x = np.ascontiguousarray(x, dtype=np.float64)
    if x.ndim != 2:
        raise ValueError("x must be 2-D")
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    w = np.ascontiguousarray(weight, dtype=np.float64).ravel()
    g = np.ascontiguousarray(list(g_index) if not isinstance(g_index, np.ndarray) else g_index, dtype=np.int32)
    st = np.ascontiguousarray(state, dtype=np.float64).ravel()
    seq = np.ascontiguousarray(sequence, dtype=np.int32).ravel()
    lam = np.ascontiguousarray(lambda_sequence, dtype=np.float64).ravel()
    alw = np.ascontiguousarray(list(always_select), dtype=np.int32).ravel()
    if st.size == 0:
        st = np.zeros(1)
    if lam.size == 0:
        lam = np.zeros(1)
    return x, y, w, g, st, seq, lam, alw


def pywrap_bess(x, y, data_type, weight, is_normal, algorithm_type, model_type, max_iter, exchange_num, path_type,
                is_warm_start, ic_type, is_cv, K, g_index, state, sequence, lambda_sequence, s_min, s_max, K_max,
                epsilon, lambda_min, lambda_max, n_lambda, is_screening, screening_size, powell_path, always_select, tao,
                beta_len, coef0_len=1, train_loss_len=1, ic_len=1, aic_len=1, bic_len=1, gic_len=1, A_len=None):
    """Drop-in for ``bess.cbess.pywrap_bess`` (SWIG typemaps of python/src/bess.i)."""
    lib = _lib.load()
    x, y, w, g, st, seq, lam, alw = _prep(x, y, weight, g_index, state, sequence, lambda_sequence, always_select)
    n, p = x.shape
    beta = np.zeros(int(beta_len))
    c0, tl, ic = np.zeros(1), np.zeros(1), np.zeros(1)
    nullloss, aic, bic, gic = np.zeros(1), np.zeros(aic_len), np.zeros(bic_len), np.zeros(gic_len)
    A_out = np.zeros(int(A_len if A_len is not None else beta_len), dtype=np.int32)
    l_out = np.zeros(1, dtype=np.int32)
    lib.pywrap_bess(_d(x), n, p, _d(y), y.size, int(data_type), _d(w), w.size, bool(is_normal), int(algorithm_type),
                    int(model_type), int(max_iter), int(exchange_num), int(path_type), bool(is_warm_start),
                    int(ic_type), bool(is_cv), int(K), _i(g), g.size, _d(st), st.size, _i(seq), seq.size, _d(lam),
                    lam.size, int(s_min), int(s_max), int(K_max), float(epsilon), float(lambda_min), float(lambda_max),
                    int(n_lambda), bool(is_screening), int(screening_size), int(powell_path), _i(alw), alw.size,
                    float(tao), _d(beta), beta.size, _d(c0), 1, _d(tl), 1, _d(ic), 1, _d(nullloss), _d(aic), aic.size,
                    _d(bic), bic.size, _d(gic), gic.size, _i(A_out), A_out.size, _i(l_out))
    err = _lib.last_error()
    if err:
        raise BessB200Error(err)
    return [beta, c0[0], tl[0], ic[0], nullloss[0], aic, bic, gic, A_out, l_out[0]]


def fit(x, y, data_type, weight, is_normal, algorithm_type, model_type, max_iter, exchange_num, path_type,
        is_warm_start, ic_type, is_cv, K, sequence, s_min, s_max, is_screening, screening_size, always_select=(),
        fold_of_row=None, cv_seed=None, device=-1, x_device_ptr=None, n=None, p=None, want_trace=True, profile=False,
        world=1, rank=0, col_lo=0, p_total=None, nccl_id=None, lambda_seq=(0.0,), lambda_min=0.0, lambda_max=0.0,
        n_lambda=None, powell_path=1, want_curve=False, g_index=None, cv_reduce_over_ranks=False, fold_shard=False):
    """``bess_b200_fit``: pywrap_bess + status code + extensions.  Returns a dict.
    ``x`` is a host ndarray, or pass ``x_device_ptr`` (int, row-major n x p fp64 in HBM) with ``n``/``p``.
    A sparse ``x`` -- a scipy.sparse matrix in any format, or a raw ``(indptr, indices, data, shape)`` tuple of host arrays
    or of torch CUDA tensors (device-resident) -- goes to the library as a CSC design (``bess_b200_csc``); see
    ``csc_arrays``.
    ``world > 1``: column-sharded multi-GPU call -- ``x`` is this rank's column shard ``[col_lo, col_lo + p)`` of a
    ``p_total``-column design, ``nccl_id`` the job's 128-byte NCCL unique id (``bess_b200.dist.nccl_unique_id``); beta
    and always_select use global column numbers.
    ``path_type == 2`` with ``algorithm_type`` 5 / 3 runs the Powell search over (s, lambda) in
    ``[s_min, s_max] x [lambda_min, lambda_max]`` (pgs_path, path.cpp:1138); ``powell_path`` 1 = golden-section line
    searches, 2 = walks on an ``n_lambda``-point log grid."""
    lib = _lib.load()
    csc = None
    if is_sparse(x) or _is_raw_csc(x):
        cp, ri, cv, nnz, (n, p), csc_on_device, _csc_arrays_alive = csc_arrays(x)
        csc = _lib.Csc(cp, ri, cv, nnz)
        xptr = None if x_device_ptr is None else C.cast(C.c_void_p(int(x_device_ptr)), dp)  # both: the library refuses
    elif x_device_ptr is None:
        x = np.ascontiguousarray(x, dtype=np.float64)
        n, p = x.shape
        xptr = _d(x)
    else:
        xptr = C.cast(C.c_void_p(int(x_device_ptr)), dp)
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    w = np.ascontiguousarray(weight, dtype=np.float64).ravel()
    # group selection: first column of every group (linear.py:238-254); None = no group structure
    # (no p-sized work on the call path when there are no groups: gindex = NULL means "every column its own group")
    g = None if g_index is None else np.ascontiguousarray(g_index, dtype=np.int32).ravel()
    st = np.zeros(1)
    lam = np.ascontiguousarray(lambda_seq, dtype=np.float64).ravel()
    seq = np.ascontiguousarray(sequence, dtype=np.int32).ravel()
    alw = np.ascontiguousarray(list(always_select), dtype=np.int32).ravel()
    fold_sharded = bool(fold_shard) and world > 1  # axis A inside one call: whole design on every rank, folds dealt out
    sharded = world > 1 and not fold_sharded
    p_all = int(p_total) if sharded else p
    beta = _lazy_zeros(p_all)
    c0, tl, ic = C.c_double(0), C.c_double(0), C.c_double(0)
    ext = Ext()
    if fold_sharded:
        if nccl_id is None or len(nccl_id) != 128:
            raise ValueError("fold-sharded fit needs the 128-byte NCCL unique id")
        idbuf = C.create_string_buffer(bytes(nccl_id), 128)
        ext.world, ext.rank, ext.fold_shard = int(world), int(rank), 1
        ext.nccl_unique_id = C.cast(idbuf, C.c_void_p)
    if sharded:
        if nccl_id is None or len(nccl_id) != 128:
            raise ValueError("sharded fit needs the 128-byte NCCL unique id")
        idbuf = C.create_string_buffer(bytes(nccl_id), 128)
        ext.world, ext.rank, ext.col_lo, ext.p_total = int(world), int(rank), int(col_lo), p_all
        ext.nccl_unique_id = C.cast(idbuf, C.c_void_p)
        want_trace = False
    fold = None
    if fold_of_row is not None:
        fold = np.ascontiguousarray(fold_of_row, dtype=np.int32)
        ext.fold_of_row = _i(fold)
    ext.cv_seed = int(cv_seed) if cv_seed is not None else 0  # None: $BESS_CV_SEED or 123
    ext.cv_seed_set = 1 if cv_seed is not None else 0
    ext.x_on_device = 1 if x_device_ptr is not None else 0
    if csc is not None:
        ext.x_csc = C.pointer(csc)
        ext.x_on_device = 1 if csc_on_device else 0
    ext.device = int(device)
    scrA = np.zeros(max(int(screening_size), 1), dtype=np.int32)
    ext.screening_A_out = _i(scrA)
    chosen = C.c_int(0)
    ext.chosen_s_out = C.pointer(chosen)
    chosen_lam = C.c_double(0.0)
    ext.chosen_lambda_out = C.pointer(chosen_lam)
    stats = np.zeros(32)
    ext.stats_out = _d(stats)
    resident = np.zeros(152)
    tie_exact = C.c_int(0)
    ext.tie_exact_out = C.pointer(tie_exact)
    ext.resident_out = _d(resident)
    sparse_sweeps = C.c_int(0)
    ext.sparse_sweeps_out = C.pointer(sparse_sweeps)
    ext.profile = 1 if profile else 0
    ext.beta_out_zeroed = 1  # `beta` comes from np.zeros (calloc): untouched pages stay untouched
    ext.cv_reduce_over_ranks = 1 if (cv_reduce_over_ranks and sharded) else 0
    rc = lib.bess_b200_fit(xptr, n, p, _d(y), y.size, int(data_type), _d(w), w.size, bool(is_normal),
                           int(algorithm_type), int(model_type), int(max_iter), int(exchange_num), int(path_type),
                           bool(is_warm_start), int(ic_type), bool(is_cv), int(K), _i(g) if g is not None else None,
                           g.size if g is not None else 0, _d(st), 1, _i(seq),
                           seq.size, _d(lam), lam.size, int(s_min), int(s_max), 10, 10.0, float(lambda_min), float(lambda_max),
                           int(n_lambda) if n_lambda is not None else lam.size, bool(is_screening),
                           int(screening_size), int(powell_path), _i(alw), alw.size, 1.1, _d(beta), p_all, C.byref(c0), C.byref(tl),
                           C.byref(ic), C.byref(ext))
    _lib.check(rc)
    out = dict(beta=beta, coef0=c0.value, train_loss=tl.value, ic=ic.value, s=chosen.value, lam=chosen_lam.value,
               stats=dict(n_fits=int(stats[0]), n_pdas_iters=int(stats[1]), n_sweeps=int(stats[2]),
                          n_batches=int(stats[3]), n_boundary_ties=int(stats[4]), sweep_bytes=float(stats[5]),
                          kernel_launches=int(stats[6]), big_sweep_bytes=float(stats[24]),
                          sweep_splits=int(stats[25]), norm_bytes=float(stats[26]),
                          host_ms=dict(zip(("load", "screen", "normalize", "setup_chains", "path"), stats[27:32].tolist())),
                          resident=resident.tolist(), tie_exact_pass=bool(tie_exact.value & 1),
                          robust_pass=bool(tie_exact.value & 2), rank_deficient=bool(tie_exact.value & 4),
                          sparse_sweeps=int(sparse_sweeps.value),
                          prof_ms=dict(zip(PROF_CATS, stats[8:16].tolist())),
                          prof_launches=dict(zip(PROF_CATS, [int(v) for v in stats[16:24]]))))
    if is_screening:
        out["screening_A"] = scrA[:int(screening_size)].copy()
    L = int(stats[7])
    if want_curve and L > 0 and not want_trace:  # criterion per evaluated level only (cheap)
        s_all, i_all = np.zeros(L, dtype=np.int32), np.zeros(L)
        lib.bess_b200_trace(_i(s_all), None, None, None, _d(i_all), None, 0)
        out.update(s_all=s_all, ic_all=i_all)
    if want_trace and L > 0:
        s_all, l_all = np.zeros(L, dtype=np.int32), np.zeros(L, dtype=np.int32)
        c_all, t_all, i_all = np.zeros(L), np.zeros(L), np.zeros(L)
        full = path_type == 1 or algorithm_type in (3, 5)  # sequential_path and pgs_path keep every evaluated model
        b_all = np.zeros((L, p)) if full else None
        lib.bess_b200_trace(_i(s_all), _i(l_all), _d(c_all) if full else None, _d(t_all), _d(i_all),
                            _d(b_all) if b_all is not None else None, p)
        lam_all = np.zeros(L)
        lib.bess_b200_trace_lambda(_d(lam_all))
        out.update(s_all=s_all, l_all=l_all, coef0_all=c_all, loss_all=t_all, ic_all=i_all, beta_all=b_all,
                   lambda_all=lam_all)
    return out


def cv_fold_ids(n, K, seed=123):
    lib = _lib.load()
    out = np.zeros(n, dtype=np.int32)
    _lib.check(lib.bess_b200_cv_fold_ids(int(n), int(K), int(seed), _i(out)))
    return out

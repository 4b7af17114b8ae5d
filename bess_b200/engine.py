"""Python handle on the ``bessgpu_*`` device shim (include/bess_b200.h, section 2) -- used by the parity tests and by
bench.py's roofline probe.  One ``GpuEngine`` = one design matrix resident in HBM plus its chain state."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import dp, ip


def _d(a):
    return a.ctypes.data_as(dp)


def _i(a):
    return a.ctypes.data_as(ip)


class GpuEngine:
    def __init__(self, device: int = -1):
        self._lib = _lib.load()
        _lib.require_gpu()
        self._h = C.c_void_p()
        _lib.check(self._lib.bessgpu_create(C.byref(self._h), device))
        self.n = self.p = 0

    def close(self):
        if self._h:
            self._lib.bessgpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load(self, x, y, weight, model_type, x_device_ptr=None, n=None, p=None):
        y = np.ascontiguousarray(y, dtype=np.float64)
        w = np.ascontiguousarray(weight, dtype=np.float64)
        if x_device_ptr is None:
            x = np.ascontiguousarray(x, dtype=np.float64)
            n, p = x.shape
            ptr = x.ctypes.data_as(C.c_void_p)
            on_dev = 0
        else:
            ptr = C.c_void_p(int(x_device_ptr))
            on_dev = 1
        _lib.check(self._lib.bessgpu_load(self._h, ptr, n, p, on_dev, _d(y), _d(w), model_type))
        self.n, self.p = n, p

    def load_csc(self, x, y, weight, model_type):
        """``load`` for a sparse design: a scipy.sparse matrix (canonicalised) or a raw ``(indptr, indices, data, shape)``
        tuple of host arrays or torch CUDA tensors (see ``cbess.csc_arrays``).  Returns self."""
        from .cbess import csc_arrays
        y = np.ascontiguousarray(y, dtype=np.float64)
        w = np.ascontiguousarray(weight, dtype=np.float64)
        cp, ri, cv, nnz, (n, p), on_dev, keep = csc_arrays(x)
        _lib.check(self._lib.bessgpu_load_csc(self._h, cp, ri, cv, n, p, nnz, int(on_dev), _d(y), _d(w), model_type))
        self._csc_arrays = keep  # device tensors are read in place until screening
        self.n, self.p = n, p
        return self

    def screen(self, size, always_select=()):
        alw = np.ascontiguousarray(list(always_select), dtype=np.int32)
        out = np.zeros(size, dtype=np.int32)
        _lib.check(self._lib.bessgpu_screen(self._h, size, _i(alw), alw.size, _i(out)))
        self.p = size
        return out

    def screen_local(self, size, always_select=()):
        alw = np.ascontiguousarray(list(always_select), dtype=np.int32)
        size = min(size, self.p)
        vals = np.zeros(size)
        idx = np.zeros(size, dtype=np.int32)
        cnt = C.c_int(0)
        _lib.check(self._lib.bessgpu_screen_local(self._h, size, _i(alw), alw.size, _d(vals), _i(idx), C.byref(cnt)))
        return vals[:cnt.value], idx[:cnt.value]

    def gather_columns(self, cols, pos, dst_device_ptr, ld):
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        _lib.check(self._lib.bessgpu_gather_columns(self._h, _i(cols), _i(pos), cols.size, C.c_void_p(int(dst_device_ptr)),
                                                    int(ld)))

    def normalize(self, data_type, is_normal=True):
        _lib.check(self._lib.bessgpu_normalize(self._h, data_type, int(is_normal)))
        xm, xn = np.zeros(self.p), np.zeros(self.p)
        ym = C.c_double(0)
        _lib.check(self._lib.bessgpu_get_norm(self._h, _d(xm), _d(xn), C.byref(ym)))
        return xm, xn, ym.value

    def design(self):
        """A host copy of the engine's current dense design (n x p): the kept columns after ``screen``, normalised after
        ``normalize``."""
        x = np.zeros((self.n, self.p))
        _lib.check(self._lib.bessgpu_design(self._h, _d(x)))
        return x

    def set_groups(self, g_index):
        """Group selection: g_index = first column of every group; levels / kcap / always_select then count groups."""
        g = np.ascontiguousarray(g_index, dtype=np.int32)
        _lib.check(self._lib.bessgpu_set_groups(self._h, _i(g), g.size))
        self._group_sizes = np.diff(np.append(g, self.p))

    def run_batch_groups(self, T, chains, new_path_step=True, lam=0.0):
        """run_batch for grouped designs (and / or a ridge level): supports come back as per-chain lists."""
        ch = np.ascontiguousarray(chains, dtype=np.int32)
        nch = ch.size
        sizes = getattr(self, "_group_sizes", np.ones(self.p, dtype=np.int64))
        ld = int(np.sort(sizes)[::-1][:T].sum())
        l, ks = np.zeros(nch, dtype=np.int32), np.zeros(nch, dtype=np.int32)
        c0 = np.zeros(nch)
        A = np.zeros((nch, ld), dtype=np.int32)
        bA = np.zeros((nch, ld))
        _lib.check(self._lib.bessgpu_run_batch_groups(self._h, T, _i(ch), nch, int(new_path_step), float(lam), _i(l),
                                                      _d(c0), _i(ks), _i(A), _d(bA), ld))
        return dict(l=l, coef0=c0, A=[A[i, :ks[i]].copy() for i in range(nch)], bA=[bA[i, :ks[i]].copy() for i in range(nch)])

    def setup_chains(self, K, fold_of_row, kcap, max_iter=20, warm_start=True, always_select=()):
        f = np.ascontiguousarray(fold_of_row if fold_of_row is not None else np.zeros(self.n), dtype=np.int32)
        alw = np.ascontiguousarray(list(always_select), dtype=np.int32)
        _lib.check(self._lib.bessgpu_setup_chains(self._h, K, _i(f), kcap, max_iter, int(warm_start), _i(alw), alw.size))

    def run_batch(self, T, chains, new_path_step=True):
        ch = np.ascontiguousarray(chains, dtype=np.int32)
        nch = ch.size
        l = np.zeros(nch, dtype=np.int32)
        c0 = np.zeros(nch)
        A = np.zeros((nch, T), dtype=np.int32)
        bA = np.zeros((nch, T))
        _lib.check(self._lib.bessgpu_run_batch(self._h, T, _i(ch), nch, int(new_path_step), _i(l), _d(c0), _i(A), _d(bA)))
        return dict(l=l, coef0=c0, A=A, bA=bA)

    def losses(self, jobs):
        ch = np.ascontiguousarray([j[0] for j in jobs], dtype=np.int32)
        kd = np.ascontiguousarray([j[1] for j in jobs], dtype=np.int32)
        fd = np.ascontiguousarray([j[2] for j in jobs], dtype=np.int32)
        out = np.zeros(len(jobs))
        _lib.check(self._lib.bessgpu_losses(self._h, _i(ch), _i(kd), _i(fd), len(jobs), _d(out)))
        return out

    def time_dual_sweep(self, reps=20):
        ms = C.c_float(0)
        by = C.c_double(0)
        _lib.check(self._lib.bessgpu_time_dual_sweep(self._h, reps, C.byref(ms), C.byref(by)))
        return ms.value, by.value

    def sacrifice(self, chains, lam=0.0):
        """Test probe after a batch: the sacrifice of every chain in ``chains`` for its current model, recomputed through
        the kernels a fit of this batch runs -> (bd [nch][p] or [nch][n_groups], dict of what ran)."""
        ch = np.ascontiguousarray(chains, dtype=np.int32)
        N = len(self._group_sizes) if hasattr(self, "_group_sizes") else self.p
        bd = np.zeros((ch.size, N))
        info = np.zeros(8, dtype=np.int32)
        _lib.check(self._lib.bessgpu_sacrifice(self._h, _i(ch), ch.size, float(lam), _d(bd), _i(info)))
        kind = {1: "stream", 2: "tma", 3: "group", 4: "csc"}[int(info[0])]
        return bd, dict(kernel=kind, FS=int(info[1]), CPT=int(info[2]), S=int(info[3]), rows_per_split=int(info[4]),
                        groups=int(info[5]), long_columns=int(info[5]) if kind == "csc" else 0)

    def stats(self):
        o = np.zeros(8)
        _lib.check(self._lib.bessgpu_stats(self._h, _d(o)))
        return dict(n_fits=int(o[0]), n_pdas_iters=int(o[1]), n_sweeps=int(o[2]), n_batches=int(o[3]),
                    n_boundary_ties=int(o[4]), sweep_bytes=float(o[5]), kernel_launches=int(o[6]),
                    max_cluster=int(o[7]))


def topk(vals, k):
    lib = _lib.load()
    _lib.require_gpu()
    v = np.ascontiguousarray(vals, dtype=np.float64)
    out = np.zeros(k, dtype=np.int32)
    tie = C.c_int(0)
    _lib.check(lib.bessgpu_topk(_d(v), v.size, k, _i(out), C.byref(tie)))
    return out, tie.value


def screen_select(vals, k):
    """``topk`` by the screening's select (device-wide when there are more than 16384 values): same result."""
    lib = _lib.load()
    _lib.require_gpu()
    v = np.ascontiguousarray(vals, dtype=np.float64)
    out = np.zeros(k, dtype=np.int32)
    tie = C.c_int(0)
    _lib.check(lib.bessgpu_screen_select(_d(v), v.size, k, _i(out), C.byref(tie)))
    return out, tie.value

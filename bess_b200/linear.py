"""Host-side mirror of the reference's Python front-end (python/bess/linear.py): same estimator names, constructor
arguments, code mapping and ValueErrors, so the parity tests read like calls into the reference.  All computation goes
through ``bess_b200.cbess.pywrap_bess`` (the SWIG-compatible entry over the C ABI) -- there is no numpy fallback.

Mapping (linear.py:138-202): algorithm_type "Pdas"->1 / "GroupPdas"->2 / "L0L2"->5; model_type "Lm","Logistic",
"Poisson","Cox" -> 1..4; path_type "seq"->1 / "pgs"->2; ic_type "aic","bic","gic","ebic" -> 1..4;
data_type 1 (Lm) / 2 (Logistic, Poisson) / 3 (Cox) (linear.py:475,517,559,597).
All twelve estimator classes of the reference are here: Pdas* (best-subset selection), L0L2* (best-subset ridge, "bsrr":
sequential lambda grids and the Powell search path_type="pgs") and GroupPdas* (group selection: sparsity levels count groups of up to 64 variables)."""
from __future__ import annotations

import math

import numpy as np

from . import cbess
from .cbess import pywrap_bess

_ALG = {"Pdas": 1, "GroupPdas": 2, "L0L2": 5}
_MODEL = {"Lm": 1, "Logistic": 2, "Poisson": 3, "Cox": 4}
_PATH = {"seq": 1, "pgs": 2}
_IC = {"aic": 1, "bic": 2, "gic": 3, "ebic": 4}


class bess_base:
    """See python/bess/linear.py:36-136 for the meaning of every argument (identical here)."""

    def __init__(self, algorithm_type, model_type, path_type, max_iter=20, exchange_num=0, is_warm_start=True,
                 sequence=None, lambda_sequence=None, s_min=None, s_max=None, K_max=None, epsilon=0.0001, lambda_min=0,
                 lambda_max=0, ic_type="ebic", is_cv=False, K=5, is_screening=False, screening_size=None, powell_path=1,
                 always_select=(), tao=0.):
        self.algorithm_type, self.model_type, self.path_type = algorithm_type, model_type, path_type
        self.max_iter, self.exchange_num, self.is_warm_start = max_iter, exchange_num, is_warm_start
        self.sequence, self.lambda_sequence = sequence, lambda_sequence
        self.s_min, self.s_max, self.K_max, self.epsilon = s_min, s_max, K_max, epsilon
        self.lambda_min, self.lambda_max, self.n_lambda = lambda_min, lambda_max, 100
        self.ic_type, self.is_cv, self.K = ic_type, is_cv, K
        self.is_screening, self.screening_size, self.powell_path = is_screening, screening_size, powell_path
        self.always_select, self.tao = list(always_select), tao
        self.path_len = self.p = self.data_type = None
        self.beta = self.coef0 = self.train_loss = self.ic = None
        self._arg_check()

    def _arg_check(self):
        if self.algorithm_type not in _ALG:
            raise ValueError("algorithm_type should not be " + str(self.algorithm_type))
        if self.model_type not in _MODEL:
            raise ValueError("model_type should not be " + str(self.model_type))
        if self.path_type not in _PATH:
            raise ValueError("path_type should be 'seq' or 'pgs'")
        if self.ic_type not in _IC:
            raise ValueError('ic_type should be "aic", "bic", "ebic" or "gic"')
        self.algorithm_type_int = _ALG[self.algorithm_type]
        self.model_type_int = _MODEL[self.model_type]
        self.path_type_int = _PATH[self.path_type]
        self.ic_type_int = _IC[self.ic_type]

    def fit(self, X, y, is_weight=False, is_normal=True, weight=None, state=None, group=None):
        """X: an n x p array, or a scipy.sparse matrix in any format (sent to the library in CSC form; the fit sees the
        same values as on X.toarray())."""
        sparse = cbess.is_sparse(X)
        X = cbess.canonical_csc(X) if sparse else np.asarray(X, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        if np.isnan(X.data if sparse else X).any():
            raise ValueError("There is NAN value in X")
        if np.isnan(y).any():
            raise ValueError("There is NAN value in y")
        n, p = X.shape
        self.p = p
        if self.algorithm_type_int == 2:  # linear.py:238-254
            if group is None:
                raise ValueError("When you choose GroupPdas algorithm, the group information should be given")
            if len(group) != p:
                raise ValueError("The length of group should be equal to the number of variables")
            group = sorted(group)  # the reference sorts the caller's list in place; a copy is sorted here
            # first position of every distinct label of the sorted list (the reference walks `list(set(group))`, whose
            # order is hash order: labels other than small non-negative ints run it off the end of the list)
            g_index = np.unique(np.asarray(group), return_index=True)[1].astype(np.int32)
        else:
            g_index = np.arange(p, dtype=np.int32)
        if self.model_type_int == 4:
            order = y[:, 0].argsort()  # linear.py:257-263: rows sorted by time, y <- status
            X = cbess.canonical_csc(X.tocsr()[order]) if sparse else X[order]
            y = y[order][:, 1].reshape(-1)
        if n != y.size:
            raise ValueError("X.shape(0) should be equal to y.size")
        if is_weight:
            if weight is None:
                raise ValueError("When you choose is_weight is True, the parameter weight should be given")
            weight = np.asarray(weight, dtype=np.float64)
            if n != weight.size:
                raise ValueError("X.shape(0) should be equal to weight.size")
        else:
            weight = np.ones(n)
        if state is None:
            state = np.ones(n)
        if self.path_type_int == 1:
            if self.sequence is None:
                self.sequence = [i + 1 for i in range(min(p, int(n / np.log(n))))]
            if self.lambda_sequence is None:
                self.lambda_sequence = [0]
            self.s_min = self.s_max = self.K_max = 0
            self.lambda_min = self.lambda_max = 0
            self.path_len = int(len(self.sequence))
        else:
            self.sequence = [1]
            self.lambda_sequence = [0]
            if self.s_min is None:
                self.s_min = 1
            if self.s_max is None:
                self.s_max = p
            if self.K_max is None:
                self.K_max = int(math.log(p, 2 / (math.sqrt(5) - 1)))
            if self.lambda_min is None:
                self.lambda_min = 0
            if self.lambda_max is None:
                self.lambda_max = 0
            self.path_len = self.K_max + 2
        if self.is_screening:
            if self.screening_size:
                if self.screening_size < max(self.sequence):
                    raise ValueError("screening size should be more than max(sequence).")
            else:
                self.screening_size = max(p, int(n / np.log(n)))  # linear.py:321 (a no-op size, SURVEY Q20)
            screening_size = min(self.screening_size, p)
        else:
            self.screening_size = screening_size = 1
        if sparse:  # the extended entry takes the CSC design; the arguments pywrap_bess ignores are left out
            out = cbess.fit(X, y, self.data_type, weight, is_normal, self.algorithm_type_int, self.model_type_int,
                            self.max_iter, self.exchange_num, self.path_type_int, self.is_warm_start, self.ic_type_int,
                            self.is_cv, self.K, self.sequence, self.s_min, self.s_max, self.is_screening, screening_size,
                            always_select=self.always_select, want_trace=False, lambda_seq=self.lambda_sequence,
                            lambda_min=self.lambda_min or 0, lambda_max=self.lambda_max or 0, n_lambda=self.n_lambda,
                            powell_path=self.powell_path, g_index=g_index if self.algorithm_type_int == 2 else None)
            self.beta, self.coef0, self.train_loss, self.ic = out["beta"], out["coef0"], out["train_loss"], out["ic"]
            return self
        result = pywrap_bess(X, y, self.data_type, weight, is_normal, self.algorithm_type_int, self.model_type_int,
                             self.max_iter, self.exchange_num, self.path_type_int, self.is_warm_start, self.ic_type_int,
                             self.is_cv, self.K, g_index, state, self.sequence, self.lambda_sequence, self.s_min,
                             self.s_max, self.K_max, self.epsilon, self.lambda_min or 0, self.lambda_max or 0,
                             self.n_lambda, self.is_screening, screening_size, self.powell_path, self.always_select,
                             self.tao, p, 1, 1, 1, 1, 1, 1, p)
        self.beta, self.coef0, self.train_loss, self.ic = result[0], result[1], result[2], result[3]
        return self

    def predict(self, X):
        """X: an array or a scipy.sparse matrix."""
        X = cbess.canonical_csc(X) if cbess.is_sparse(X) else np.asarray(X, dtype=np.float64)
        if X.shape[1] != self.p:
            raise ValueError("X.shape[1] should be " + str(self.p))
        eta = np.asarray(X @ self.beta).ravel() + self.coef0
        if self.model_type_int == 1:
            return eta
        if self.model_type_int == 2:
            yhat = (eta > 0).astype(np.float64)
            e = np.exp(np.clip(eta, -25, 25))
            return {"Y": yhat, "pr": e / (e + 1)}
        if self.model_type_int == 3:
            return {"lam": np.exp(eta)}
        return None  # the reference defines no prediction for Cox (linear.py:389-430)


def _make(name, algorithm, model, data_type):
    def __init__(self, max_iter=20, exchange_num=0, path_type="seq", is_warm_start=True, sequence=None,
                 lambda_sequence=None, s_min=None, s_max=None, K_max=None, epsilon=0.0001, lambda_min=None,
                 lambda_max=None, ic_type="ebic", is_cv=False, K=5, is_screening=False, screening_size=None,
                 powell_path=1, always_select=(), tao=0.):
        bess_base.__init__(self, algorithm, model, path_type, max_iter, exchange_num, is_warm_start, sequence,
                           lambda_sequence, s_min, s_max, K_max, epsilon, lambda_min, lambda_max, ic_type, is_cv, K,
                           is_screening, screening_size, powell_path, always_select, tao)
        self.data_type = data_type
    return type(name, (bess_base,), {"__init__": __init__,
                                     "__doc__": f"{algorithm} estimator, model {model} "
                                                f"(reference: python/bess/linear.py class {name})."})


_DATA_TYPE = {"Lm": 1, "Logistic": 2, "Poisson": 2, "Cox": 3}  # linear.py:475,517,559,597
for _alg in ("Pdas", "L0L2", "GroupPdas"):
    for _model, _dt in _DATA_TYPE.items():
        globals()[_alg + _model] = _make(_alg + _model, _alg, _model, _dt)
del _alg, _model, _dt
__all__ = ["bess_base"] + [a + m for a in ("Pdas", "L0L2", "GroupPdas") for m in _DATA_TYPE]

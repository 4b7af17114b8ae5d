"""Outputs of BASELINE configs 1-4 (the ones whose fits run through the chain kernels) for bitwise comparisons of two
builds of the library.

  python tools/chain_outputs.py dump DIR [SO]      write DIR/<cfg>.npz (beta, coef0, ic, and the per-level traces),
                                                   with the library at SO (default: the in-tree build)
  python tools/chain_outputs.py compare DIR1 DIR2  exit 1 unless every array is bitwise equal"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = ("c1", "c1cv", "c2", "c3", "c4")
FAM = {"gaussian": (1, 1), "binomial": (2, 2), "poisson": (3, 2), "cox": (4, 3)}
KEYS = ("beta", "coef0", "ic", "train_loss", "s_all", "l_all", "coef0_all", "loss_all", "ic_all", "beta_all")


def dump(dirname, so=None):
    from bess_b200 import _lib
    if so:
        _lib.SO_PATH = os.path.abspath(so)
    from bess_b200 import cbess
    from bess_b200.gen_data import gen_data
    from tests.helpers import FULL_CONFIGS
    os.makedirs(dirname, exist_ok=True)
    for cfg in CONFIGS:
        fam, n, p, k, path_type, is_cv, K, ic_type, s_min, s_max, scr, seed = FULL_CONFIGS[cfg]
        model_type, data_type = FAM[fam]
        d = gen_data(n, p, fam, k, seed=seed)
        seq = np.arange(s_min, s_max + 1) if path_type == 1 else np.arange(1, 2)
        out = cbess.fit(d.x, d.y, data_type, np.ones(n), True, 1, model_type, 20, 2, path_type, True, ic_type, is_cv, K, seq,
                        s_min, s_max, scr > 0, max(scr, 1), cv_seed=123)
        np.savez(os.path.join(dirname, cfg + ".npz"), **{k_: np.asarray(out[k_]) for k_ in KEYS if k_ in out})
        print(f"{cfg}: s {out['s']} ic {out['ic']!r}", flush=True)


def compare(d1, d2):
    bad = 0
    for cfg in CONFIGS:
        a, b = np.load(os.path.join(d1, cfg + ".npz")), np.load(os.path.join(d2, cfg + ".npz"))
        for k_ in sorted(set(a.files) | set(b.files)):
            same = k_ in a.files and k_ in b.files and a[k_].shape == b[k_].shape and a[k_].dtype == b[k_].dtype and \
                a[k_].tobytes() == b[k_].tobytes()
            bad += not same
            print(f"{cfg}.{k_}: {'bitwise equal' if same else 'DIFFERENT'}")
    return bad


if __name__ == "__main__":
    if sys.argv[1] == "dump":
        dump(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else None)
    else:
        sys.exit(1 if compare(sys.argv[2], sys.argv[3]) else 0)

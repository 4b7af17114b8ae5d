"""The resident gaussian kernel (lm_path.cu) reads the termination word once per CTA inside its barrier waits and
mirrors a chain's residual into the engine's G only when the chain finishes.  Neither may change a single bit: each case
of tests/golden/make_resident_round.py is compared bit for bit with the golden made by the previous build, and against
the multi-kernel path (BESS_B200_RESIDENT=0): same supports and same chosen s."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_spec = importlib.util.spec_from_file_location("make_resident_round", os.path.join(HERE, "golden", "make_resident_round.py"))
mk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mk)


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(HERE, "golden", "onchip", "resident_round.npz")))


@pytest.mark.parametrize("name", list(mk.CASES))
def test_bitwise_equal_to_golden(name, golden):
    from bess_b200 import cbess
    res = mk.run_case(name, cbess)
    assert res["resident_launches"][0] > 0, "the resident kernel did not run"
    for k, v in res.items():
        g = golden[f"{name}/{k}"]
        assert v.shape == g.shape and np.array_equal(v, g), f"{name}: {k} differs from the golden"


@pytest.mark.parametrize("name", list(mk.CASES))
def test_same_supports_as_multi_kernel_path(name, golden, tmp_path):
    out = tmp_path / "mk.npz"
    code = ("import sys, numpy as np; sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2]);"
            "import make_resident_round as mk; from bess_b200 import cbess;"
            "np.savez(sys.argv[4], **mk.run_case(sys.argv[3], cbess))")
    env = dict(os.environ, BESS_B200_RESIDENT="0")
    subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(HERE, "golden"), name, str(out)], env=env, check=True)
    m = dict(np.load(out))
    assert m["resident_launches"][0] == 0
    assert m["s"][0] == golden[f"{name}/s"][0]
    assert np.nonzero(m["beta"])[0].tolist() == np.nonzero(golden[f"{name}/beta"])[0].tolist()
    ga = golden[f"{name}/beta_all"]
    for lvl in range(ga.shape[0]):
        assert np.nonzero(m["beta_all"][lvl])[0].tolist() == np.nonzero(ga[lvl])[0].tolist(), f"{name}: level {lvl + 1}"

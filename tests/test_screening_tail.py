"""Screening's gather of the kept columns is deferred to the normalisation, which reads them from the raw design inside
its one launch (or, where that launch does not apply, runs the plain gather first).  Neither may change a bit of what
the fit sees: each case of tests/golden/make_screening_tail.py -- the kept list, the column means and norms and the
screened, normalised design -- is compared bit for bit with the golden made by the previous build, which gathered the
kept columns into a design of their own before normalising it."""
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_screening_tail", os.path.join(HERE, "golden", "make_screening_tail.py"))
mk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mk)


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(HERE, "golden", "screening", "screening_tail.npz")))


@pytest.mark.parametrize("name", list(mk.CASES))
def test_bitwise_equal_to_golden(name, golden):
    from bess_b200 import engine
    res = mk.run_case(name, engine)
    for k, v in res.items():
        g = golden[f"{name}/{k}"]
        assert v.shape == g.shape and np.array_equal(v, g), f"{name}: {k} differs from the golden"

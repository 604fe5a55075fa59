"""CPU tests of the R binding of resident batches (r-package/TADpoleB200/src/r_shim.c: C_tp_ctx_set, C_tp_batch_recall,
C_tp_batch_dendro) through the stand-in R runtime of tests/mock_r: registration and arity, and R errors with balanced
PROTECTs for released handles."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


@pytest.fixture(scope="module")
def R():
    import __graft_entry__ as g
    g.build()
    from mock_r.driver import MockR
    r = MockR()
    yield r
    r.reset()


def test_resident_routines_are_registered_with_their_arity(R):
    from mock_r.driver import RError
    for name, nargs in (("C_tp_ctx_set", 3), ("C_tp_batch_recall", 6), ("C_tp_batch_dendro", 4)):
        assert R.registered(name) == nargs
        with pytest.raises(RError, match=f"takes {nargs} arguments"):
            R.call(name, *([0] * (nargs - 1)))


def test_released_handles_are_r_errors(R):
    from mock_r.driver import RError
    one, minus = np.array([0], np.int32), np.array([-1], np.int32)
    # an object that is no external pointer reads as a released one
    with pytest.raises(RError, match="resident batch has been released"):
        R.call("C_tp_batch_dendro", 0, 0, -1, 1)
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_batch_recall", 0, 0, one, minus, 200, 2)
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_ctx_set", 0, "batch_resident", 1.0)

"""cuadmm_solver_update_data without a GPU: the call on a solver that was never initialised fails with an error code,
and the Python wrapper checks the shapes of its arguments before it reaches the library."""
import ctypes as C

import numpy as np
import pytest

import cuadmm_b200 as cu
from cuadmm_b200 import capi

CUADMM_EINVAL = -1


def test_update_before_init_returns_einval():
    s = cu.Solver(verbose=False)
    bi, bv = np.array([0, 1], np.int32), np.array([1.0, 2.0])
    ci, cv = np.array([0], np.int32), np.array([3.0])
    for keep in (0, 1):
        rc = capi.lib.cuadmm_solver_update_data(s.h, bi.ctypes.data_as(capi.c_i32p), bv.ctypes.data_as(capi.c_f64p), 2,
                                                ci.ctypes.data_as(capi.c_i32p), cv.ctypes.data_as(capi.c_f64p), 1, keep, 1.0)
        assert rc == CUADMM_EINVAL
        assert "init" in capi.lib.cuadmm_last_error().decode()
    with pytest.raises(cu.CuadmmError) as e:
        s.update_data(bi, bv, ci, cv)
    assert e.value.code == CUADMM_EINVAL
    # empty b and C, null pointers, and a null solver: still an error code, no crash
    assert capi.lib.cuadmm_solver_update_data(s.h, None, None, 0, None, None, 0, 0, 1.0) == CUADMM_EINVAL
    assert capi.lib.cuadmm_solver_update_data(None, None, None, 0, None, None, 0, 0, 1.0) == CUADMM_EINVAL
    s.close()


@pytest.mark.parametrize("args", [
    ([0, 1], [1.0], [0], [1.0]),                        # b lengths differ
    ([0], [1.0], [0, 2, 3], [1.0, 2.0]),                # C lengths differ
    ([[0, 1]], [[1.0, 2.0]], [0], [1.0]),               # 2-D b
    ([0], [1.0], [0], np.ones((1, 1))),                 # 2-D C values
    ([0.5], [1.0], [0], [1.0]),                         # non-integer indices
    ([0], [1.0], [2 ** 31], [1.0]),                     # index beyond int32
])
def test_wrapper_checks_shapes(args):
    s = cu.Solver(verbose=False)
    with pytest.raises(ValueError):
        s.update_data(*args)
    s.close()


def test_wrapper_passes_well_formed_arrays_to_the_library():
    # well-formed arguments of any integer dtype reach the C check, which rejects the uninitialised solver
    s = cu.Solver(verbose=False)
    with pytest.raises(cu.CuadmmError):
        s.update_data(np.array([0, 3], np.int64), [1.0, 2.0], [], [], keep_iterate=True, sig=2.0)
    s.close()

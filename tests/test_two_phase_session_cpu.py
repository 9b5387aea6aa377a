"""lpx_two_phase_session_open(_dev) without a device: the symbols are exported, every argument refusal happens before
any device work with the reason in lpx_last_error(), and a valid open fails loudly when there is no device."""
import ctypes as C

import numpy as np
import pytest

from linear_programming_solver_lpr381_b200 import _ffi as F

NEW = ("lpx_two_phase_session_open", "lpx_two_phase_session_open_dev", "lpx_session_two_phase_info")


def test_exported():
    L = F.lib()
    for name in NEW:
        assert name in F.EXPORTS and hasattr(L, name), name


@pytest.mark.parametrize("m,n,sense,rel,null", [
    (0, 2, 0, None, None), (2, 0, 0, None, None), (-1, 2, 0, None, None),
    (2, 2, 2, None, None), (2, 2, -1, None, None),
    (2, 2, 0, [0, 3], None), (2, 2, 0, [-1, 0], None),
    (2, 2, 0, None, "A"), (2, 2, 0, None, "b"), (2, 2, 0, None, "c"),
])
@pytest.mark.parametrize("dev", [False, True])
def test_refusals_before_any_device_work(m, n, sense, rel, null, dev):
    arr = dict(A=np.ones((2, 2)), b=np.ones(2), c=np.ones(2))
    if null:
        arr[null] = None
    rel = None if rel is None else np.array(rel, dtype=np.int32)
    L = F.lib()
    name = "lpx_two_phase_session_open_dev" if dev else "lpx_two_phase_session_open"
    opt = F.make_options()
    h = getattr(L, name)(m, n, sense, F.ptr(arr["A"]), F.ptr(rel), F.ptr(arr["b"]), F.ptr(arr["c"]),
                         C.cast(C.byref(opt), C.c_void_p))
    assert not h
    assert name + ": bad arguments" in F.last_error()


def test_info_on_a_null_session():
    ph, p1 = C.c_int(7), C.c_int(7)
    assert F.lib().lpx_session_two_phase_info(None, C.byref(ph), C.byref(p1)) == F.E_BAD_ARGS
    assert ph.value == 7 and p1.value == 7


def test_dual_and_two_phase_together_is_a_value_error():
    from linear_programming_solver_lpr381_b200 import api
    with pytest.raises(ValueError):
        api.Session(np.ones((1, 1)), np.ones(1), np.ones(1), [1], 1, dual=True, two_phase=True)


def test_fails_loudly_without_a_gpu():
    if F.lib().lpx_device_count() > 0:
        pytest.skip("a GPU is present")
    from linear_programming_solver_lpr381_b200 import api
    with pytest.raises(F.LpxError) as e:
        api.Session(np.ones((2, 2)), np.ones(2), np.ones(2), [1, 0], 1, two_phase=True)
    assert e.value.code == F.E_CUDA

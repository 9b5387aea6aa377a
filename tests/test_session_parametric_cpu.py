"""lpx_session_parametric without a device: the symbol is exported and its argument checks that need no session refuse
before any device work, with the reason in lpx_last_error()."""
import ctypes as C

import numpy as np
import pytest

from linear_programming_solver_lpr381_b200 import _ffi as F


def call(base, kind, pay, seg_cap, end):
    L = F.lib()
    return L.lpx_session_parametric(base, kind, F.ptr(pay), seg_cap, None, None if end is None else C.byref(end),
                                    *[None] * 7)


def test_exported():
    assert "lpx_session_parametric" in F.EXPORTS and hasattr(F.lib(), "lpx_session_parametric")


@pytest.mark.parametrize("kind,pay,seg_cap,with_end", [
    (1, np.array([1.0, 1.0]), 4, True),     # NULL base
    (1, None, 4, True),                     # NULL payload
    (1, np.array([1.0, 1.0]), 4, False),    # NULL end
    (0, np.array([1.0, 1.0]), 4, True),     # unknown kind
    (3, np.array([1.0, 1.0]), 4, True),
    (2, np.array([1.0, 1.0]), 0, True),     # seg_cap < 1
])
def test_refusals_before_any_device_work(kind, pay, seg_cap, with_end):
    end = C.c_int(99)
    assert call(None, kind, pay, seg_cap, end if with_end else None) == F.E_BAD_ARGS
    assert "lpx_session_parametric: bad arguments" in F.last_error()
    assert end.value == 99

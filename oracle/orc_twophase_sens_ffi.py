"""ctypes binding of oracle/orc_twophase_sens.cpp — TEST INFRASTRUCTURE ONLY.

The sensitivity report of a two-phase result (include/lpx.h) restated as sequential loops on the full-width tableau,
which it rebuilds by replaying orc_two_phase's pivot list.  Built into its own liborc_twophase_sens.so next to
liboracle.so.  Imported by tests/ and tools/, never by the product package.  two_phase / two_phase_batch (the solve
alone) are orc_twophase_ffi's, re-exported.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from orc_twophase_ffi import ITER_LIMIT, INFEASIBLE, OPTIMAL, UNBOUNDED, dims, two_phase, two_phase_batch  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
# orc_twophase_sens.cpp calls orc_two_phase and pivot; the rest is what those link against
_SRCS = ["orc_twophase_sens.cpp", "orc_twophase.cpp", "orc_parser.cpp", "orc_simplex.cpp", "orc_bnb.cpp",
         "orc_cutting.cpp", "orc_revised.cpp"]
_DEPS = _SRCS + ["orc_model.hpp", "orc_solvers.hpp", "orc_dotnet.hpp"]
_SO = os.path.join(_HERE, "liborc_twophase_sens.so")
_LIB = None


def build(force=False):
    newest = max(os.path.getmtime(os.path.join(_HERE, f)) for f in _DEPS)
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < newest:
        # -ffp-contract=off: separate multiply and add / subtract, as on the GPU
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-shared",
                               "-o", _SO] + [os.path.join(_HERE, f) for f in _SRCS])
    return _SO


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _i(a):
    return None if a is None else a.ctypes.data_as(_ip)


def two_phase_sensitivity_batch(A, b, c, rel=None, sense=0, max_iterations=10000, pivots_cap=None):
    """two_phase_batch's fields for `count` LPs of one shape, plus report (count, 4m + 3n): the two-phase sensitivity
    record of each LP, NaNs unless OPTIMAL."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    count, m, n = A.shape
    b = np.ascontiguousarray(b, dtype=np.float64).reshape(count, m)
    c = np.ascontiguousarray(c, dtype=np.float64).reshape(count, n)
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    cap = 4 * (m + n) if pivots_cap is None else pivots_cap
    rows, cols = dims(m, n, rel)
    out = dict(status=np.zeros(count, np.int32), phase1_pivots=np.zeros(count, np.int32),
               n_pivots=np.zeros(count, np.int32), pivots=np.zeros((count, cap, 2), np.int32),
               basis=np.zeros((count, m), np.int32), x=np.zeros((count, n)), z=np.zeros(count),
               tableau=np.zeros((count, rows, cols)), report=np.zeros((count, 4 * m + 3 * n)))
    lib().orc_two_phase_sensitivity(count, m, n, sense, _d(A), _i(rel), _d(b), _d(c), max_iterations, cap,
                                    *[_i(out[k]) for k in ("status", "phase1_pivots", "n_pivots", "pivots", "basis")],
                                    *[_d(out[k]) for k in ("x", "z", "tableau", "report")])
    return out


def two_phase_sensitivity(A, b, c, rel=None, sense=0, **kw):
    """One LP: the fields of two_phase_sensitivity_batch without the leading axis."""
    A = np.asarray(A, dtype=np.float64)
    r = two_phase_sensitivity_batch(A[None], np.asarray(b, np.float64)[None], np.asarray(c, np.float64)[None], rel,
                                    sense, **kw)
    return {k: v[0] for k, v in r.items()}

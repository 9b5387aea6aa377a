"""ctypes binding of oracle/orc_twophase.cpp — TEST INFRASTRUCTURE ONLY.

Two-phase Simplex (include/lpx.h) restated as sequential loops on the oracle's choose_leaving and pivot, built into its
own liborc_twophase.so next to liboracle.so.  Imported by tests/ and tools/, never by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# orc_twophase.cpp calls choose_leaving / pivot; the rest is what orc_simplex.cpp links against
_SRCS = ["orc_twophase.cpp", "orc_parser.cpp", "orc_simplex.cpp", "orc_bnb.cpp", "orc_cutting.cpp", "orc_revised.cpp"]
_DEPS = _SRCS + ["orc_model.hpp", "orc_solvers.hpp", "orc_dotnet.hpp"]
_SO = os.path.join(_HERE, "liborc_twophase.so")
_LIB = None

OPTIMAL, UNBOUNDED, INFEASIBLE, ITER_LIMIT = 0, 1, 2, -3


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


def dims(m, n, rel=None):
    """(rows, cols) of the output tableau: m + 1, n + s + 1 with s the non-EQ rows."""
    s = m if rel is None else int(np.sum(np.asarray(rel) != 2))
    return m + 1, n + s + 1


def two_phase_batch(A, b, c, rel=None, sense=0, max_iterations=10000, pivots_cap=None):
    """`count` LPs of one shape (A (count, m, n), b (count, m), c (count, n)).  Returns status, phase1_pivots,
    n_pivots (count), pivots (count, pivots_cap, 2), basis (count, m), x (count, n), z (count) and tableau
    (count, m + 1, n + s + 1)."""
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
               tableau=np.zeros((count, rows, cols)))
    lib().orc_two_phase(count, m, n, sense, _d(A), _i(rel), _d(b), _d(c), max_iterations, cap,
                        *[_i(out[k]) for k in ("status", "phase1_pivots", "n_pivots", "pivots", "basis")],
                        _d(out["x"]), _d(out["z"]), _d(out["tableau"]))
    return out


def two_phase(A, b, c, rel=None, sense=0, **kw):
    """One LP: the fields of two_phase_batch without the leading axis."""
    A = np.asarray(A, dtype=np.float64)
    r = two_phase_batch(A[None], np.asarray(b, np.float64)[None], np.asarray(c, np.float64)[None], rel, sense, **kw)
    return {k: v[0] for k, v in r.items()}

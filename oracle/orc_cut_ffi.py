"""ctypes binding of oracle/orc_cut.cpp — TEST INFRASTRUCTURE ONLY.

CuttingPlane.Solve's numbers for one IP in the layout of one instance of lpx_cutting_plane_batched (include/lpx.h),
restated on the oracle's primal_simplex and built into its own liborc_cut.so next to liboracle.so.  Imported by tests/
and tools/, never by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# orc_cut.cpp calls primal_simplex; the rest is what orc_simplex.cpp links against
_SRCS = ["orc_cut.cpp", "orc_parser.cpp", "orc_simplex.cpp", "orc_bnb.cpp", "orc_cutting.cpp", "orc_revised.cpp"]
_DEPS = _SRCS + ["orc_model.hpp", "orc_solvers.hpp", "orc_dotnet.hpp"]
_SO = os.path.join(_HERE, "liborc_cut.so")
_LIB = None


def build(force=False):
    newest = max(os.path.getmtime(os.path.join(_HERE, f)) for f in _DEPS)
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < newest:
        # -ffp-contract=off: separate multiply and subtract, as RyuJIT emits for the C# loops
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-shared",
                               "-o", _SO] + [os.path.join(_HERE, f) for f in _SRCS])
    return _SO


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def _d(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _i(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int))


def cutting_plane(A, b, c, rel=None, sense=0, max_iterations=10000):
    """orc_cut_solve: end, n_rounds, n_cuts, per round lp_status / lp_pivots (50, the round that threw included), per
    cut frac_var / cut_row / cut_a (50 x n) / cut_b (50), and the final LP's basis (m' + 49), x, z and tableau
    ((m' + 50) x (n + m' + 50) doubles, the final tableau compact at the start; zeros unless end is integral)."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    m, n = A.shape
    rel = np.zeros(m, dtype=np.int32) if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    b = np.ascontiguousarray(b, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    mm = m + int((rel == 2).sum())
    end, n_rounds, n_cuts, z = C.c_int(), C.c_int(), C.c_int(), C.c_double()
    lp_status, lp_pivots = np.zeros(50, np.int32), np.zeros(50, np.int32)
    frac_var, cut_row = np.zeros(50, np.int32), np.zeros(50, np.int32)
    cut_a, cut_b = np.zeros((50, n)), np.zeros(50)
    basis, x = np.zeros(mm + 49, np.int32), np.zeros(n)
    T = np.zeros((mm + 50) * (n + mm + 50))
    lib().orc_cut_solve(m, n, sense, _d(A), _i(rel), _d(b), _d(c), max_iterations, C.byref(end), C.byref(n_rounds),
                        C.byref(n_cuts), _i(lp_status), _i(lp_pivots), _i(frac_var), _i(cut_row), _d(cut_a), _d(cut_b),
                        _i(basis), _d(x), C.byref(z), _d(T))
    return dict(end=end.value, n_rounds=n_rounds.value, n_cuts=n_cuts.value, lp_status=lp_status, lp_pivots=lp_pivots,
                frac_var=frac_var, cut_row=cut_row, cut_a=cut_a, cut_b=cut_b, basis=basis, x=x, z=z.value, tableau=T)

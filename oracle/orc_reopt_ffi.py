"""ctypes binding of oracle/orc_reopt.cpp — TEST INFRASTRUCTURE ONLY.

Re-optimization of optimal Primal Simplex results (include/lpx.h) restated as sequential loops on top of the oracle's
primal_core and Mode B's dual_core, built into its own liborc_reopt.so next to liboracle.so.  Imported by tests/ and
tools/, never by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# orc_reopt.cpp includes orc_pooled.cpp; the rest is what orc_simplex.cpp links against
_SRCS = ["orc_reopt.cpp", "orc_parser.cpp", "orc_simplex.cpp", "orc_bnb.cpp", "orc_cutting.cpp", "orc_revised.cpp"]
_DEPS = _SRCS + ["orc_pooled.cpp", "orc_model.hpp", "orc_solvers.hpp", "orc_dotnet.hpp"]
_SO = os.path.join(_HERE, "liborc_reopt.so")
_LIB = None

RHS, COST, ROW, COL = 1, 2, 3, 4
KINDS = {"rhs": RHS, "cost": COST, "row": ROW, "col": COL}


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


def payload_stride(kind, m, n):
    return {RHS: m, COST: n, ROW: n + 2, COL: m + 1}[kind]


def dims(kind, m, n, rel=None):
    mm = m + (0 if rel is None else int(np.sum(np.asarray(rel) == 2)))
    return mm + 1 + (kind == ROW), n + mm + 1 + (kind in (ROW, COL))


def reopt(kind, m, n, base_status, base_basis, base_tableau, payload, rel=None, sense=0, src=None,
          max_iterations=10000, pivots_cap=64):
    """`count` = len(payload) queries of one kind against the bases (leading axis on base_status / base_basis /
    base_tableau); src (nullable) maps query -> base.  Returns status, n_pivots, pivots (count, cap, 2; -1 past the
    query's pivots), basis, x, z, tableau."""
    kind = KINDS.get(kind, kind)
    stride = payload_stride(kind, m, n)
    pay = np.ascontiguousarray(payload, dtype=np.float64).reshape(-1, stride)
    count = pay.shape[0]
    bst = np.ascontiguousarray(np.atleast_1d(base_status), dtype=np.int32)
    nb = bst.shape[0]
    bb = np.ascontiguousarray(base_basis, dtype=np.int32).reshape(nb, -1)
    bT = np.ascontiguousarray(base_tableau, dtype=np.float64).reshape(nb, -1)
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    src = None if src is None else np.ascontiguousarray(src, dtype=np.int32)
    rows, cols = dims(kind, m, n, rel)
    nx = n + 1 if kind == COL else n
    assert bT.shape[1] == (bb.shape[1] + 1) * (n + bb.shape[1] + 1)
    assert src is not None or nb >= count
    out = dict(status=np.zeros(count, np.int32), n_pivots=np.zeros(count, np.int32),
               pivots=np.full((count, max(pivots_cap, 1), 2), -1, np.int32), basis=np.zeros((count, rows - 1), np.int32),
               x=np.zeros((count, nx)), z=np.zeros(count), tableau=np.zeros((count, rows, cols)))
    lib().orc_reopt(kind, count, m, n, sense, _i(rel), _i(bst), _i(bb), _d(bT), _i(src), _d(pay), max_iterations,
                    _i(out["status"]), _i(out["n_pivots"]), _i(out["pivots"]), pivots_cap, _i(out["basis"]),
                    _d(out["x"]), _d(out["z"]), _d(out["tableau"]))
    return out


def extend_tableau(tableau, basis, var, side, val):
    """Mode B's child tableau (oracle/orc_pooled.cpp extend_tableau) of one parent tableau."""
    T = np.ascontiguousarray(tableau, dtype=np.float64)
    rows, cols = T.shape
    basis = np.ascontiguousarray(basis, dtype=np.int32)
    To = np.zeros((rows + 1, cols + 1))
    bo = np.zeros(rows, np.int32)
    lib().orc_extend_tableau(rows, cols, _d(T), _i(basis), var, side, C.c_double(val), _d(To), _i(bo))
    return To, bo


def dual_core(tableau, basis, pivots_cap=10000):
    """Mode B's Dual Simplex loop (dual_core) on a copy: status, pivots (k, 2), basis, tableau."""
    T = np.array(tableau, dtype=np.float64, order="C")
    rows, cols = T.shape
    b = np.array(basis, dtype=np.int32)
    npiv = C.c_int()
    piv = np.full((pivots_cap, 2), -1, np.int32)
    st = lib().orc_dual_core(rows, cols, _d(T), _i(b), C.byref(npiv), _i(piv), pivots_cap)
    return st, piv[: min(npiv.value, pivots_cap)], b, T

"""ctypes binding of oracle/orc_param.cpp — TEST INFRASTRUCTURE ONLY.

Parametric analysis of optimal Primal Simplex results (include/lpx.h) restated as sequential loops on the oracle's
choose_leaving and pivot, built into its own liborc_param.so next to liboracle.so.  Imported by tests/ and tools/,
never by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# orc_param.cpp calls choose_leaving / pivot; the rest is what orc_simplex.cpp links against
_SRCS = ["orc_param.cpp", "orc_parser.cpp", "orc_simplex.cpp", "orc_bnb.cpp", "orc_cutting.cpp", "orc_revised.cpp"]
_DEPS = _SRCS + ["orc_model.hpp", "orc_solvers.hpp", "orc_dotnet.hpp"]
_SO = os.path.join(_HERE, "liborc_param.so")
_LIB = None

RHS, COST = 1, 2
KINDS = {"rhs": RHS, "cost": COST}
REACHED, UNBOUNDED, INFEASIBLE, SEG_LIMIT, NO_BASE = 0, 1, 2, 3, 4


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
    return {RHS: m, COST: n}[kind] + 1


def dims(kind, m, n, rel=None):
    mm = m + (0 if rel is None else int(np.sum(np.asarray(rel) == 2)))
    return mm + 1 + (kind == COST), n + mm + 1 + (kind == RHS)


def parametric(kind, m, n, base_status, base_basis, base_tableau, payload, rel=None, sense=0, src=None, seg_cap=64):
    """`count` = len(payload) queries of one kind (payload rows: d, then theta_max) against the bases (leading axis
    on base_status / base_basis / base_tableau); src (nullable) maps query -> base.  Returns end, n_segments,
    n_pivots, segments (count, seg_cap, 4 + 2n), seg_pivots (count, seg_cap, 2), basis and tableau."""
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
    mm = bb.shape[1]
    assert bT.shape[1] == (mm + 1) * (n + mm + 1)
    assert src is not None or nb >= count
    out = dict(end=np.zeros(count, np.int32), n_segments=np.zeros(count, np.int32),
               n_pivots=np.zeros(count, np.int32), segments=np.zeros((count, seg_cap, 4 + 2 * n)),
               seg_pivots=np.zeros((count, seg_cap, 2), np.int32), basis=np.zeros((count, mm), np.int32),
               tableau=np.zeros((count, rows, cols)))
    lib().orc_param(kind, count, m, n, sense, _i(rel), _i(bst), _i(bb), _d(bT), _i(src), _d(pay), seg_cap,
                    *[_i(out[k]) for k in ("end", "n_segments", "n_pivots")], _d(out["segments"]),
                    _i(out["seg_pivots"]), _i(out["basis"]), _d(out["tableau"]))
    return out

"""ctypes binding of oracle/orc_sensitivity.cpp — TEST INFRASTRUCTURE ONLY.

The sensitivity report of include/lpx.h restated as sequential loops (strict < / > in index order), built into
its own liborc_sensitivity.so next to liboracle.so.  Imported by tests/ and tools/, never by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "orc_sensitivity.cpp")
_SO = os.path.join(_HERE, "liborc_sensitivity.so")
_LIB = None


def build(force=False):
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        # -ffp-contract=off: the report's divisions, subtractions and additions stay separate, as on the GPU
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra", "-shared",
                               "-o", _SO, _SRC])
    return _SO


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def sensitivity(b, c, status, basis, tableau, rel=None, sense=0):
    """The report of final Primal Simplex tableaux.  One LP (b[m], c[n], scalar status, basis[m'],
    tableau[rows][cols]) gives one record of 4m + 3n doubles; a batch (leading count axis on b, c, basis and
    tableau, status[count]) gives report[count][4m + 3n]."""
    b = np.ascontiguousarray(b, dtype=np.float64)
    single = b.ndim == 1
    b = b.reshape(-1, b.shape[-1])
    count, m = b.shape
    c = np.ascontiguousarray(c, dtype=np.float64).reshape(count, -1)
    n = c.shape[1]
    status = np.ascontiguousarray(np.atleast_1d(status), dtype=np.int32)
    basis = np.ascontiguousarray(basis, dtype=np.int32).reshape(count, -1)
    T = np.ascontiguousarray(tableau, dtype=np.float64).reshape(count, -1)
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    assert status.shape == (count,) and T.shape[1] == (basis.shape[1] + 1) * (n + basis.shape[1] + 1)
    rep = np.zeros((count, 4 * m + 3 * n))
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    lib().orc_sensitivity(count, m, n, sense, None if rel is None else rel.ctypes.data_as(ip), b.ctypes.data_as(dp),
                          c.ctypes.data_as(dp), status.ctypes.data_as(ip), basis.ctypes.data_as(ip),
                          T.ctypes.data_as(dp), rep.ctypes.data_as(dp))
    return rep[0] if single else rep

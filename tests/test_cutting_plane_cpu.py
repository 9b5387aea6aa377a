"""CPU suite for the cutting-plane entry points: the oracle's numbers-only CuttingPlane.Solve (oracle/orc_cut.cpp, the
reference lpx_cutting_plane_batched is checked against on the GPU) against the golden cases, the pure-Python
restatement and the oracle's text path; the argument checks and the missing-device failure of the C ABI."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_bits_equal, case_arrays, unhex
from cut_cases import random_ips

import orc_cut_ffi as cut
import pyref
from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

CUT_NAMES = ["cut_classic_incomplete", "cut_integral_root", "cut_from_z_row", "cut_three_vars", "cut_min_sense",
             "cut_eq_row", "cut_ge_error"]


def final_tableau(r, n):
    mm = r["basis"].shape[0] - 49
    rows, cols = mm + r["n_cuts"] + 1, n + mm + r["n_cuts"] + 1
    return r["tableau"][: rows * cols].reshape(rows, cols)


def check_unused(r, n):
    """The fill of what the run did not reach, and the final LP's zeros unless it ended integral."""
    R, k = 50, r["n_cuts"]
    assert r["n_cuts"] == (r["n_rounds"] if r["end"] == F.CUT_INCOMPLETE else r["n_rounds"] - 1)
    assert (r["lp_status"][r["n_rounds"]:] == F.RUNNING).all() and (r["lp_pivots"][r["n_rounds"]:] == 0).all()
    assert (r["frac_var"][k:] == -1).all() and (r["cut_row"][k:] == -1).all()
    assert_bits_equal(r["cut_a"][k:], np.zeros((R - k, n)), "unused cut_a")
    assert_bits_equal(r["cut_b"][k:], np.zeros(R - k), "unused cut_b")
    if r["end"] != F.CUT_INTEGER:
        assert not r["basis"].any() and not r["x"].any() and r["z"] == 0.0 and not r["tableau"].any()


@pytest.mark.parametrize("name", CUT_NAMES)
def test_oracle_entry_reproduces_golden(kat, name):
    case = kat["cut"][name]
    A, b, c, rel = case_arrays(case)
    n = A.shape[1]
    r = cut.cutting_plane(A, b, c, rel, case["sense"])
    assert r["end"] == case["end"]
    check_unused(r, n)
    cuts = case["cuts"]
    assert r["n_cuts"] == len(cuts)
    assert r["frac_var"][: len(cuts)].tolist() == [k["frac_var"] for k in cuts]
    assert r["cut_row"][: len(cuts)].tolist() == [k["row"] for k in cuts]
    assert_bits_equal(r["cut_a"][: len(cuts)], np.array([unhex(k["a"]) for k in cuts]).reshape(len(cuts), n), "cut a")
    assert_bits_equal(r["cut_b"][: len(cuts)], [unhex(k["b"]) for k in cuts], "cut b")
    rounds = [list(t) for t in zip(r["lp_pivots"].tolist(), r["lp_status"].tolist())][: r["n_rounds"]]
    if name == "cut_ge_error":
        # the golden rounds list only rounds that did not throw: the one round here threw before its first pivot
        assert case["rounds"] == [] and r["end"] == F.CUT_LP_ERROR and rounds == [[0, F.S_GE_ROW]]
        return
    assert rounds == case["rounds"]
    if case["end"] == F.CUT_INTEGER:
        assert r["basis"][: len(case["basis"])].tolist() == case["basis"]
        assert not r["basis"][len(case["basis"]):].any()
        assert_bits_equal(r["x"], unhex(case["x"]), "x")
        assert_bits_equal([r["z"]], [unhex(case["z"])], "z")
        T = final_tableau(r, n)
        assert_bits_equal(T, unhex(case["tableau"]), "tableau")
        assert not r["tableau"][T.size:].any()


def compare_with_pyref(r, p, n):
    assert r["end"] == p["end"]
    done = [(a, s) for a, s in zip(r["lp_pivots"].tolist(), r["lp_status"].tolist())][: r["n_rounds"]]
    if p["end"] == F.CUT_LP_ERROR:  # pyref lists the rounds that did not throw, the error code on its own
        assert done[:-1] == p["rounds"] and done[-1][1] == p["code"]
    else:
        assert done == p["rounds"]
    assert r["n_cuts"] == len(p["cuts"])
    for k, (fv, row, a, f0) in enumerate(p["cuts"]):
        assert (r["frac_var"][k], r["cut_row"][k]) == (fv, row)
        assert_bits_equal(r["cut_a"][k], a, "cut a")
        assert_bits_equal([r["cut_b"][k]], [f0], "cut b")
    if p["end"] == F.CUT_INTEGER:
        assert_bits_equal(r["x"], p["x"], "x")
        assert_bits_equal([r["z"]], [p["z"]], "z")
        assert r["basis"][: len(p["basis"])].tolist() == list(p["basis"])
        assert_bits_equal(final_tableau(r, n), p["tableau"], "tableau")


# (m, n, sense, rel, seed): EQ rows, Min, a GE row (an LP error in round 1) and unbounded directions among them
SHAPES = [(3, 3, 0, [0, 0, 0], 11), (4, 3, 1, [0, 2, 0, 0], 12), (2, 4, 0, [2, 0], 13), (5, 2, 0, [0, 0, 1, 0, 0], 14),
          (6, 5, 1, None, 15), (3, 6, 0, [0, 0, 2], 16)]


@pytest.mark.parametrize("m,n,sense,rel,seed", SHAPES)
def test_oracle_entry_matches_pyref_on_random_ips(m, n, sense, rel, seed):
    A, b, c = random_ips(5, m, n, seed)
    ends = set()
    for k in range(5):
        r = cut.cutting_plane(A[k], b[k], c[k], rel, sense)
        p = pyref.cutting_plane(A[k].tolist(), b[k].tolist(), c[k].tolist(), rel, sense)
        check_unused(r, n)
        compare_with_pyref(r, p, n)
        ends.add(r["end"])
    if rel is not None and 1 in rel:
        assert ends == {F.CUT_LP_ERROR}


def test_oracle_entry_iteration_limit():
    # pyref has no iteration limit (the GPU tests check this case against the kernel): max_iterations = 1 stops the
    # first round that needs a second pivot, which is recorded with LPX_S_ITER_LIMIT and 1 pivot
    A, b, c = random_ips(12, 4, 4, 21, box=0.0, unbounded=0.0)
    seen = 0
    for k in range(12):
        r = cut.cutting_plane(A[k], b[k], c[k], None, 0, max_iterations=1)
        check_unused(r, 4)
        full = cut.cutting_plane(A[k], b[k], c[k], None, 0)
        if r["end"] == F.CUT_LP_ERROR:
            seen += 1
            last = r["n_rounds"] - 1
            assert r["lp_status"][last] == F.S_ITER_LIMIT and r["lp_pivots"][last] == 1
            # every round before it is the full run's, pivot for pivot, cut for cut
            assert (r["lp_pivots"][:last] == full["lp_pivots"][:last]).all()
            assert_bits_equal(r["cut_b"][:last], full["cut_b"][:last], "cut b")
    assert seen > 0


@pytest.mark.parametrize("name", ["cut_classic_incomplete", "cut_three_vars", "cut_eq_row", "cut_min_sense"])
def test_oracle_entry_cuts_equal_text_path(orc, kat, name):
    case = kat["cut"][name]
    A, b, c, rel = case_arrays(case)
    r = cut.cutting_plane(A, b, c, rel, case["sense"])
    t = orc.solve_text(workloads.lp_to_text(A, b, c, rel, case["sense"]), "cutting plane")
    assert r["end"] == t["cut_end"] and r["n_cuts"] == len(t["cuts"])
    for k, g in enumerate(t["cuts"]):
        assert (r["frac_var"][k], r["cut_row"][k]) == (g["frac_var"], g["row"])
        assert_bits_equal(r["cut_a"][k], g["a"], "cut a")
        assert_bits_equal([r["cut_b"][k]], [g["b"]], "cut b")


def test_dims_without_a_device():
    from linear_programming_solver_lpr381_b200 import api
    assert api.cutting_plane_dims(3, 4) == (53, 57)
    assert api.cutting_plane_dims(3, 4, [0, 2, 0]) == (54, 58)
    rows, cols = C.c_int(), C.c_int()
    L = F.lib()
    assert L.lpx_cutting_plane_dims(0, 4, None, C.byref(rows), C.byref(cols)) == F.E_BAD_ARGS
    assert L.lpx_cutting_plane_dims(3, 0, None, C.byref(rows), C.byref(cols)) == F.E_BAD_ARGS
    bad = np.array([0, 3, 0], dtype=np.int32)
    assert L.lpx_cutting_plane_dims(3, 4, F.ptr(bad), C.byref(rows), C.byref(cols)) == F.E_BAD_ARGS


@pytest.mark.parametrize("count,m,n,sense,rel,kernel", [
    (0, 2, 2, 0, None, 0), (1, 0, 2, 0, None, 0), (1, 2, 0, 0, None, 0), (1, 2, 2, 2, None, 0),
    (1, 2, 2, 0, [0, 5], 0), (1, 2, 2, 0, [0, -1], 0), (1, 2, 2, 0, None, F.KERNEL_STREAM),
    (1, 2, 2, 0, None, F.KERNEL_CTA_REG), (1, 2, 2, 0, None, 99)])
def test_bad_arguments_before_any_device_work(count, m, n, sense, rel, kernel):
    A, b, c = np.ones((1, 2, 2)), np.ones((1, 2)), np.ones((1, 2))
    rel = None if rel is None else np.array(rel, dtype=np.int32)
    opt = F.make_options(kernel=kernel)
    end = np.zeros(1, np.int32)
    L = F.lib()
    head = [count, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt), F.ptr(end)] + [None] * 12
    assert L.lpx_cutting_plane_batched(*head, None) == F.E_BAD_ARGS
    if rel is None:  # the _dev call reads rel from the device, so only its other checks come first
        assert L.lpx_cutting_plane_batched_dev(*head, None, None) == F.E_BAD_ARGS


def test_fails_loudly_without_a_gpu():
    if F.lib().lpx_device_count() > 0:
        pytest.skip("a GPU is present")
    from linear_programming_solver_lpr381_b200 import api
    with pytest.raises(F.LpxError) as e:
        api.cutting_plane(np.ones((2, 2)), np.ones(2), np.ones(2))
    assert e.value.code == F.E_CUDA

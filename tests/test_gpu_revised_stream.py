"""GPU parity: the whole-GPU Revised Primal Simplex path of lpx_revised_solve (blocked Gauss-Jordan inversion
on the streaming look-ahead + pass kernels, grid-wide pricing) against the golden cases, the oracle and the
one-CTA kernel — status, iteration count, pivots, theta, the basis lists, x_B, x, every double of B^-1 and
every history record — and the routing of opt.kernel."""
import ctypes as C

import numpy as np
import pytest

import host_ffi as H
from conftest import assert_bits_equal, case_arrays, unhex

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

REV_NAMES = ["rev_wyndor", "rev_min_negative_costs", "rev_unbounded", "rev_degenerate_tie", "rev_three_vars",
             "rev_klee_minty3", "rev_needs_row_swaps", "rev_ge_row", "rev_neg_rhs", "rev_iter_limit"]
STREAM, CTA = F.KERNEL_STREAM, F.KERNEL_CTA_GLOBAL


def same_as_oracle(got, want, what, with_x=False):
    assert got["status"] == want["status"], what
    assert got["n_iters"] == want["n_iters"], what
    assert got["enter"].tolist() == want["enter"].tolist() and got["leave"].tolist() == want["leave"].tolist(), what
    assert_bits_equal(got["theta"], want["theta"], what + " theta")
    assert got["basis"].tolist() == want["basis"].tolist(), what
    assert_bits_equal(got["xB"], want["xB"], what + " xB")
    assert_bits_equal(got["Binv"], want["Binv"], what + " Binv")
    if want["status"] >= 0 or with_x:  # the oracle returns no solution for ITER_LIMIT
        assert_bits_equal(got["x"], want["x"], what + " x")


def same_as_cta(got, want, what):
    """Every output of lpx_revised_solve, history included."""
    assert got["status"] == want["status"] and got["n_iters"] == want["n_iters"], what
    if got["status"] != -11:
        same_as_oracle(got, want, what, with_x=True)
        assert got["nonbasic"].tolist() == want["nonbasic"].tolist(), what
    if "history" in want:
        assert_bits_equal(got["history"], want["history"], what + " history")


@pytest.mark.parametrize("name", REV_NAMES)
def test_stream_kat(lpx, kat, name):
    case = kat["rev"][name]
    A, b, c, rel = case_arrays(case)
    r = lpx.revised_solve(A, b, c, rel, case["sense"], max_iterations=case["max_iterations"], kernel=STREAM)
    assert r["status"] == case["status"]
    if case["status"] in (-10, -11):
        return
    assert [[int(e), int(l)] for e, l in zip(r["enter"], r["leave"])] == [p[:2] for p in case["pivots"]]
    assert_bits_equal(r["theta"], [unhex(p[2]) for p in case["pivots"]], "theta")
    assert r["basis"].tolist() == case["basis"]
    assert_bits_equal(r["xB"], unhex(case["xB"]), "xB")
    assert_bits_equal(r["Binv"], unhex(case["Binv"]), "Binv")
    if case["status"] >= 0:
        assert_bits_equal(r["x"], unhex(case["x"]), "x")


@pytest.mark.parametrize("pass_variant", [1, 2, 3])
@pytest.mark.parametrize("kblock", [1, 2, 7, 8, 16])
def test_stream_random_vs_oracle(lpx, orc, kblock, pass_variant):
    rng = np.random.default_rng(100 * kblock + pass_variant)
    seen = set()
    for t in range(16):
        m, n = int(rng.integers(1, 40)), int(rng.integers(1, 50))
        A = rng.integers(-2, 10, size=(m, n)).astype(float)
        b = rng.integers(0, 40, size=m).astype(float)
        c = rng.integers(-3, 10, size=n).astype(float)
        if t % 2:
            A = np.round(rng.random((m, n)) * 9 - 1, 3)
            b = np.round(rng.random(m) * 30, 3)
            c = np.round(rng.random(n) * 12 - 3, 3)
        sense = t % 2 if t % 4 < 2 else 1 - t % 2
        cap = 2 if t % 5 == 4 else 150
        if t == 3:  # a Max column that no row bounds: UNBOUNDED
            A[:, 0] = -np.abs(A[:, 0]) - 1
            c[0], sense = 100.0, 0
        if t == 4:  # positive data, Max, one iteration allowed: ITER_LIMIT
            A, b, c = workloads.lp_integer(m + 2, n + 2, t + kblock)
            sense, cap = 0, 1
        want = orc.revised_solve(A, b, c, None, sense, max_iterations=cap)
        got = lpx.revised_solve(A, b, c, None, sense, max_iterations=cap, kernel=STREAM, kblock=kblock,
                                pass_variant=pass_variant)
        what = f"case {t} {m}x{n} sense={sense} K={kblock} variant={pass_variant}"
        seen.add(want["status"])
        if want["status"] == -11:
            assert got["status"] == -11, what
            continue
        same_as_oracle(got, want, what)
    assert {0, 1, -3} <= seen


# B = [a_0 | a_1] after two iterations has d_1 = 5e-9 > 1e-9, but partial pivoting takes 100 first and leaves
# -5e-11 for the second column: "Singular basis encountered." inside iteration 2
SINGULAR = (np.array([[1.0, -1.0], [100.0, -99.999999995]]), np.array([1.0, 1000.0]), np.array([2.0, 1.0]))


@pytest.mark.parametrize("kblock", [1, 8])
def test_stream_singular(lpx, orc, kblock):
    A, b, c = SINGULAR
    assert orc.revised_solve(A, b, c)["status"] == -11
    want = lpx.revised_solve(A, b, c, kernel=CTA, history=8)
    got = lpx.revised_solve(A, b, c, kernel=STREAM, history=8, kblock=kblock)
    assert want["status"] == -11 and want["n_iters"] >= 1
    same_as_cta(got, want, "singular")


@pytest.mark.parametrize("val,row,col", [(-np.inf, 0, 2), (np.nan, 3, 1), (np.inf, 2, 7), (np.nan, 0, 7),
                                         (1e308, 1, 2)])
def test_stream_nonfinite(lpx, orc, val, row, col):
    A, b, c = workloads.lp_integer(6, 8, 5)
    A[row, col] = val
    want = orc.revised_solve(A, b, c)
    cta = lpx.revised_solve(A, b, c, kernel=CTA, history=16)
    got = lpx.revised_solve(A, b, c, kernel=STREAM, history=16, kblock=2)
    what = f"A[{row},{col}] = {val}"
    same_as_cta(got, cta, what)
    assert got["status"] == want["status"], what
    if want["status"] != -11:
        same_as_oracle(got, want, what)


def test_stream_history_vs_cta(lpx):
    rng = np.random.default_rng(77)
    for t in range(8):
        m, n = int(rng.integers(2, 48)), int(rng.integers(2, 70))
        A, b, c = workloads.lp_integer(m, n, 300 + t) if t % 2 else workloads.lp_decimal(m, n, 300 + t)
        sense = 0  # Max of positive costs: the slack basis is never optimal
        cap = 6 if t == 5 else 10000
        want = lpx.revised_solve(A, b, c, None, sense, max_iterations=cap, kernel=CTA, history=40)
        got = lpx.revised_solve(A, b, c, None, sense, max_iterations=cap, kernel=STREAM, history=40,
                                kblock=(1, 4, 8, 16)[t % 4])
        assert want["n_iters"] > 0
        same_as_cta(got, want, f"case {t} {m}x{n}")


def test_stream_history_buffer_refused(lpx):
    """A history the device cannot hold fails the call with a reason; nothing is written."""
    A, b, c = workloads.lp_integer(8, 12000, 1)
    m, n = A.shape
    L = F.lib()
    L.lpx_revised_history_stride.restype = C.c_size_t
    cap = (200 << 30) // (8 * L.lpx_revised_history_stride(m, n)) + 1  # > 200 GB of records
    hist = np.full(16, 7.0)
    status, n_iters = C.c_int(-99), C.c_int(-99)
    opt = F.make_options()
    rc = L.lpx_revised_solve(m, n, 0, F.ptr(A), None, F.ptr(b), F.ptr(c), C.byref(opt), C.byref(status),
                             C.byref(n_iters), None, None, 0, None, None, None, None, None, F.ptr(hist), cap)
    assert rc == -8 and "history" in F.last_error()
    assert (hist == 7.0).all()
    assert lpx.revised_solve(A, b, c)["status"] == 0  # the library is still usable


@pytest.mark.parametrize("m,n", [(8, 12000), (64, 11500)])
def test_past_cta_capacity(lpx, orc, m, n):
    A, b, c = workloads.lp_integer(m, n, 1)
    want = orc.revised_solve(A, b, c)
    got = lpx.revised_solve(A, b, c)
    assert want["status"] == 0
    same_as_oracle(got, want, f"{m}x{n}")
    with pytest.raises(F.LpxError) as e:
        lpx.revised_solve(A, b, c, kernel=CTA)
    assert e.value.code == -8


def test_past_cta_capacity_text(lpx, orc):
    A, b, c = workloads.lp_integer(8, 12000, 1)
    text = workloads.lp_to_text(A, b, c, np.zeros(8, dtype=np.int32), 0)
    want = orc.solve_text(text, "Revised Primal Simplex")
    got = H.solve_text(text, "Revised Primal Simplex")
    assert want["code"] == 0 and got["code"] == 0, (got["error"], want["error"])
    assert got["log"] == want["log"]
    assert got["report"] == want["report"]
    assert got["summary"] == want["summary"]
    assert got["chunks"] == want["chunks"]


def test_tall_square_optimal(lpx, orc):
    A, b, c = workloads.lp_integer(160, 160, 4)
    want = orc.revised_solve(A, b, c)
    got = lpx.revised_solve(A, b, c)
    assert want["status"] == 0 and want["n_iters"] > 20
    same_as_oracle(got, want, "160x160")


def test_tall_iteration_limit(lpx, orc):
    A, b, c = workloads.lp_decimal(512, 512, 6)
    want = orc.revised_solve(A, b, c, max_iterations=25)
    got = lpx.revised_solve(A, b, c, max_iterations=25)
    assert want["status"] == -3 and want["n_iters"] == 25
    same_as_oracle(got, want, "512x512")


def test_tall_1024_vs_cta(lpx):
    A, b, c = workloads.lp_decimal(1024, 1024, 7)
    want = lpx.revised_solve(A, b, c, max_iterations=1, kernel=CTA, history=2)
    got = lpx.revised_solve(A, b, c, max_iterations=1, kernel=STREAM, history=2)
    assert want["status"] == -3
    same_as_cta(got, want, "1024x1024")


def test_routing(lpx):
    L = F.lib()
    A, b, c = workloads.lp_integer(60, 90, 3)  # the existing mid-size shape: the one-CTA kernel, one launch
    L.lpx_reset_counters()
    lpx.revised_solve(A, b, c)
    assert L.lpx_kernel_launches() == 1
    L.lpx_reset_counters()
    lpx.revised_solve(A, b, c, kernel=STREAM)
    assert L.lpx_kernel_launches() > 1
    A, b, c = workloads.lp_integer(192, 96, 3)  # past the crossover
    L.lpx_reset_counters()
    lpx.revised_solve(A, b, c, max_iterations=2)
    assert L.lpx_kernel_launches() > 1
    L.lpx_reset_counters()
    lpx.revised_solve(A, b, c, max_iterations=2, kernel=CTA)
    assert L.lpx_kernel_launches() == 1

"""reg_variant 5, the condensed register kernel with 4 row warps x 16 rows and three register column slots,
against the oracle, bit for bit: status, pivot count, basis, x, z and every double of the tableau (incl. -0.0)."""
import numpy as np
import pytest

from conftest import assert_bits_equal

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu


def solve5(lpx, A, b, c, **kw):
    return lpx.primal_solve_batched(A, b, c, kernel=F.KERNEL_CTA_REG, reg_variant=5, **kw)


def check_batch(got, want, what):
    assert np.array_equal(got["status"], want["status"]), what
    assert np.array_equal(got["n_pivots"], want["n_pivots"]), what
    assert np.array_equal(got["basis"], want["basis"]), what
    assert_bits_equal(got["tableau"], want["tableau"], what + " tableau")
    assert_bits_equal(got["x"], want["x"], what + " x")
    assert_bits_equal(got["z"], want["z"], what + " z")


@pytest.mark.parametrize("kind", ["integer", "decimal"])
def test_c2_full_batch(lpx, orc, kind):
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=1, kind=kind)
    want = orc.primal_batch(A, b, c, threads=16, want_tableau=True)
    check_batch(solve5(lpx, A, b, c), want, f"C2 {kind}")


@pytest.mark.parametrize("m", [1, 31, 33, 63, 64])
def test_shapes(lpx, orc, m):
    for n in (1, 32, 33, 96, 127, 128):
        for sense in (0, 1):
            A, b, c = workloads.batch_c2(count=16, m=m, n=n, seed=7 + m + n, kind="decimal" if n % 2 else "integer")
            if sense == 1:
                c = -c
            want = orc.primal_batch(A, b, c if sense == 0 else -c, threads=8, want_tableau=True)
            check_batch(solve5(lpx, A, b, c, sense=sense), want, f"{m}x{n} sense={sense}")


def test_iteration_limit_unbounded_and_negative_rhs(lpx, orc):
    rng = np.random.default_rng(29)
    A = rng.integers(-3, 8, size=(60, 12, 15)).astype(float)
    b = rng.integers(-1, 30, size=(60, 12)).astype(float)
    c = rng.integers(-3, 9, size=(60, 15)).astype(float)
    A[50:, :, 0] = -1.0  # column 0 enters first and has no positive entry: unbounded
    b[50:] = np.abs(b[50:])
    c[50:, 0] = 9.0
    got = solve5(lpx, A, b, c, max_iterations=9)
    seen = set()
    for k in range(60):
        want = orc.primal_solve(A[k], b[k], c[k], None, 0, max_iterations=9)
        assert got["status"][k] == want["status"], k
        seen.add(want["status"])
        if want["status"] >= 0 or want["status"] == F.S_ITER_LIMIT:
            assert got["n_pivots"][k] == want["n_pivots"], k
        if want["status"] >= 0:
            assert_bits_equal(got["tableau"][k], want["tableau"], f"tableau {k}")
            assert_bits_equal(got["x"][k], want["x"], f"x {k}")
    assert {0, 1, -2, -3} <= seen


def test_near_ties_and_signed_zeros(lpx, orc):
    """The inputs of test_register_kernel_near_ties_and_signed_zeros: tied ratios, near-ties inside the 1e-9
    margin, zero ratios and -0.0 / +0.0 pairs."""
    rng = np.random.default_rng(5)
    count, m, n = 96, 16, 6
    A = rng.integers(1, 6, size=(count, m, n)).astype(np.float64)
    b = np.empty((count, m))
    c = rng.integers(1, 9, size=(count, n)).astype(np.float64)
    for k in range(count):
        base = float(rng.integers(2, 9))
        eps = rng.choice([0.0, 2e-10, 6e-10, 9.9e-10, 1.1e-9, 3e-9], size=m)
        b[k] = (base + eps) * A[k, :, 0]
        if k % 3 == 0:
            b[k, rng.integers(0, m, size=3)] = 0.0
        if k % 4 == 0:
            A[k, rng.integers(0, m), :] *= -1.0
        rng.shuffle(b[k])
    b = np.abs(b)
    want = orc.primal_batch(A, b, c, threads=8, want_tableau=True)
    check_batch(solve5(lpx, A, b, c), want, "near ties")


def test_wide_problems_are_refused(lpx):
    with pytest.raises(F.LpxError):
        solve5(lpx, *workloads.batch_c2(count=2, m=10, n=129, seed=1))


def test_sensitivity_report(lpx, orc):
    import orc_sens_ffi as sens
    sens.lib()
    A, b, c = workloads.batch_c2(count=512, m=64, n=128, seed=5, kind="decimal")
    want = orc.primal_batch(A, b, c, threads=16, want_tableau=True)
    report = sens.sensitivity(b, c, want["status"], want["basis"], want["tableau"])
    got = lpx.primal_solve_sensitivity_batched(A, b, c, kernel=F.KERNEL_CTA_REG, reg_variant=5)
    assert got["status"].tolist() == want["status"].tolist()
    assert got["n_pivots"].tolist() == want["n_pivots"].tolist()
    assert got["basis"].tolist() == want["basis"].tolist()
    assert_bits_equal(got["report"], report, "report")
    assert_bits_equal(got["x"], want["x"], "x")
    assert_bits_equal(got["z"], want["z"], "z")

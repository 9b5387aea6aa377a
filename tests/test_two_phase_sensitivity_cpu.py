"""CPU: the two-phase sensitivity oracle (oracle/orc_twophase_sens.cpp) pinned independently of
the GPU: the radiation-therapy LP's known duals, scipy's HiGHS marginals and re-solves inside and just past each range
on random mixed models of both senses, strong duality, bit-for-bit identity with the Primal Simplex report on all-'<='
models with b >= 0, the redundant-row rule, NaN records, and the C ABI's refusals and missing-device failure."""
import ctypes as C

import numpy as np
import pytest

from linear_programming_solver_lpr381_b200 import _ffi as F

OPTIMAL, UNBOUNDED, INFEASIBLE, ITER_LIMIT = 0, 1, 2, -3
LE, GE, EQ = 0, 1, 2
MAX, MIN = 0, 1
NAMES = ("shadow", "slack", "rhs_lo", "rhs_hi", "reduced", "cost_lo", "cost_hi")

RADIATION = ([[0.3, 0.1], [0.5, 0.5], [0.6, 0.4]], [2.7, 6, 6], [0.4, 0.5], [LE, EQ, GE], MIN)


@pytest.fixture(scope="module")
def tp():
    import orc_twophase_sens_ffi
    orc_twophase_sens_ffi.lib()
    return orc_twophase_sens_ffi


def split(rep, m, n):
    o = np.cumsum([0, m, m, m, m, n, n, n])
    return {k: rep[..., o[i]:o[i + 1]] for i, k in enumerate(NAMES)}


def as_written(z, sense):
    return -z if sense == MIN else z


def test_radiation_known_answer(tp):
    A, b, c, rel, sense = RADIATION
    r = tp.two_phase_sensitivity(A, b, c, rel, sense)
    assert r["status"] == OPTIMAL
    s = split(r["report"], 3, 2)
    np.testing.assert_allclose(s["shadow"], [-0.5, 1.1, 0.0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(s["slack"], [0.0, 0.0, 0.3], rtol=0, atol=1e-12)
    assert s["slack"][1] == 0.0 and not np.signbit(s["slack"][1])  # an '=' row: +0
    assert abs(float(np.dot(b, s["shadow"])) - 5.25) <= 1e-12
    assert abs(as_written(r["z"], sense) - 5.25) <= 1e-12
    # the '>=' row is slack by 0.3: its RHS can rise to 6.3 and fall without limit
    assert s["rhs_lo"][2] == -np.inf and abs(s["rhs_hi"][2] - 6.3) <= 1e-12


def feasible_mixed(seed, m, n):
    """A random mixed model with a known interior point x0 > 0, some rows negated (b < 0), continuous data."""
    r = np.random.default_rng(seed)
    A = r.normal(size=(m, n)).round(3)
    x0 = r.uniform(0.5, 2.0, size=n)
    rel = r.integers(0, 3, size=m).astype(np.int32)
    gap = r.uniform(0.2, 1.5, size=m)
    b = (A @ x0 + np.where(rel == LE, gap, np.where(rel == GE, -gap, 0.0))).round(4)
    c = r.normal(size=n).round(3)
    return A, b, c, rel


def highs(A, b, c, rel, sense):
    from scipy.optimize import linprog
    sg = 1.0 if sense == MIN else -1.0
    le, ge, eq = rel == LE, rel == GE, rel == EQ
    ub = np.vstack([A[le], -A[ge]])
    bub = np.concatenate([b[le], -b[ge]])
    h = linprog(sg * c, A_ub=ub if len(ub) else None, b_ub=bub if len(ub) else None,
                A_eq=A[eq] if eq.any() else None, b_eq=b[eq] if eq.any() else None,
                bounds=[(0, None)] * len(c), method="highs")
    return h, sg


def highs_duals(h, sg, rel):
    """d(objective as written)/d b_i from HiGHS's marginals: '>=' rows went in negated."""
    y = np.zeros(len(rel))
    nle = int((rel == LE).sum())
    y[rel == LE] = h.ineqlin.marginals[:nle]
    y[rel == GE] = -h.ineqlin.marginals[nle:]
    if (rel == EQ).any():
        y[rel == EQ] = h.eqlin.marginals
    return sg * y


def nondegenerate(r, m, n, rel):
    """Unique duals and ranges: every basic value clear of zero, no artificial basic, every non-basic reduced cost
    among the structural and slack columns clear of zero."""
    if r["status"] != OPTIMAL:
        return False
    T, ns = r["tableau"], n + int((rel != EQ).sum())
    if (r["basis"] >= ns).any() or (T[:m, -1] <= 1e-7).any():
        return False
    nonbasic = np.setdiff1d(np.arange(ns), r["basis"])
    return bool((T[m, nonbasic] > 1e-7).all())


def inner_points(lo, hi, v, scale):
    """Points strictly inside [lo, hi] around the model's value v."""
    if np.isfinite(lo) and np.isfinite(hi):
        return lo + 0.25 * (hi - lo), lo + 0.75 * (hi - lo)
    return tuple(p for p, ok in ((lo + 0.5 * scale, np.isfinite(lo)), (hi - 0.5 * scale, np.isfinite(hi)),
                                 (v - scale, not np.isfinite(lo)), (v + scale, not np.isfinite(hi))) if ok)


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_against_highs(tp, sense):
    checked = ranged = 0
    for t in range(300):
        m, n = 3 + t % 4, 3 + (t // 4) % 4
        A, b, c, rel = feasible_mixed(7000 + 1000 * sense + t, m, n)
        r = tp.two_phase_sensitivity(A, b, c, rel, sense)
        if not nondegenerate(r, m, n, rel):
            continue
        checked += 1
        s = split(r["report"], m, n)
        h, sg = highs(A, b, c, rel, sense)
        assert h.status == 0
        z0 = sg * h.fun
        assert abs(as_written(r["z"], sense) - z0) <= 1e-7 * max(1.0, abs(z0))
        np.testing.assert_allclose(s["shadow"], highs_duals(h, sg, rel), atol=1e-7, err_msg=str(t))
        np.testing.assert_allclose(s["reduced"], h.lower.marginals, atol=1e-7, err_msg=str(t))
        # strong duality: b.y is the objective as written
        assert abs(float(np.dot(b, s["shadow"])) - z0) <= 1e-7 * max(1.0, abs(z0))
        assert (s["slack"] >= 0).all() and not s["slack"][rel == EQ].any()
        if ranged >= 40:
            continue
        ranged += 1
        for i in range(m):
            lo, hi, y = s["rhs_lo"][i], s["rhs_hi"][i], s["shadow"][i]
            assert lo <= b[i] <= hi
            scale = max(1.0, abs(b[i]))
            for pt in inner_points(lo, hi, b[i], scale):
                bb = b.copy()
                bb[i] = pt
                h2, _ = highs(A, bb, c, rel, sense)
                assert h2.status == 0 and abs(sg * h2.fun - (z0 + y * (pt - b[i]))) < 1e-7 * max(1.0, abs(z0)), (t, i)
            for end, step in ((lo, -1e-4 * scale), (hi, 1e-4 * scale)):
                if not np.isfinite(end):
                    continue
                bb = b.copy()
                bb[i] = end + step
                h2, _ = highs(A, bb, c, rel, sense)
                assert h2.status != 0 or abs(sg * h2.fun - (z0 + y * (end + step - b[i]))) > 1e-9 * max(1.0, abs(z0)), \
                    (t, i, "past end")
        for j in range(n):
            lo, hi = s["cost_lo"][j], s["cost_hi"][j]
            assert lo <= c[j] <= hi
            scale = max(1.0, abs(c[j]))
            for pt in inner_points(lo, hi, c[j], scale):
                cc = c.copy()
                cc[j] = pt
                h2, _ = highs(A, b, cc, rel, sense)
                np.testing.assert_allclose(h2.x, h.x, atol=1e-7, err_msg=f"{t} {j}")
            for end, step in ((lo, -1e-4 * scale), (hi, 1e-4 * scale)):
                if not np.isfinite(end):
                    continue
                cc = c.copy()
                cc[j] = end + step
                h2, _ = highs(A, b, cc, rel, sense)
                assert h2.status != 0 or np.abs(h2.x - h.x).max() > 1e-7, (t, j, "past end")
    assert checked >= 60 and ranged == 40, (checked, ranged)


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_strong_duality_with_flipped_and_redundant_rows(tp, sense):
    seen_flip = seen_redundant = 0
    for t in range(200):
        m, n = 2 + t % 6, 2 + (t // 6) % 6
        A, b, c, rel = feasible_mixed(9000 + 1000 * sense + t, m, n)
        if t % 3 == 0 and m >= 2:  # row 1 repeats row 0 as an equality
            rel[0] = rel[1] = EQ
            A[1], b[1] = A[0], b[0]
        r = tp.two_phase_sensitivity(A, b, c, rel, sense)
        if r["status"] != OPTIMAL:
            assert np.isnan(r["report"]).all()
            continue
        s = split(r["report"], m, n)
        z = as_written(r["z"], sense)
        assert abs(float(np.dot(b, s["shadow"])) - z) <= 1e-8 * max(1.0, abs(z)), t
        tol = 1e-9 * np.maximum(1.0, np.abs(b))  # a redundant row's artificial sits at zero up to rounding
        assert (s["slack"] >= 0).all() and (s["rhs_lo"] <= b + tol).all() and (b - tol <= s["rhs_hi"]).all()
        seen_flip += int((b < 0).any())
        seen_redundant += int((r["basis"] >= n + int((rel != EQ).sum())).any())
    assert seen_flip > 20 and seen_redundant > 5


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_identity_with_primal_report_on_all_le(tp, orc, sense):
    import orc_sens_ffi
    for seed in range(60):
        r0 = np.random.default_rng(seed)
        m, n = int(r0.integers(1, 9)), int(r0.integers(1, 9))
        A = r0.integers(-3, 8, size=(m, n)).astype(float)
        b = r0.integers(0, 20, size=m).astype(float)
        c = r0.integers(-4, 9, size=n).astype(float)
        if seed % 5 == 0:
            b[0] = -0.0  # not flipped
        got = tp.two_phase_sensitivity(A, b, c, None, sense)
        p = orc.primal_solve(A, b, c, None, sense)
        want = orc_sens_ffi.sensitivity(b, c, p["status"], p["basis"], p["tableau"], None, sense)
        assert got["status"] == p["status"]
        assert got["report"].tobytes() == want.tobytes(), seed


def test_duplicated_equality_gives_a_single_point_range(tp):
    from scipy.optimize import linprog
    A, b, c, rel = [[1, 1, 0], [1, 1, 0], [0, 1, 1]], [2.0, 2.0, 3.0], [1, 2, 1], [EQ, EQ, LE]
    r = tp.two_phase_sensitivity(A, b, c, rel, MIN)
    assert r["status"] == OPTIMAL and r["basis"][1] >= 3 + 1  # the artificial of row 1 stayed basic
    s = split(r["report"], 3, 3)
    assert s["rhs_lo"][:2].tolist() == [2.0, 2.0] and s["rhs_hi"][:2].tolist() == [2.0, 2.0]
    for i in (0, 1):
        for d in (-1e-4, 1e-4):
            bb = np.array(b)
            bb[i] += d
            h = linprog(c, A_ub=[A[2]], b_ub=[bb[2]], A_eq=A[:2], b_eq=bb[:2], bounds=[(0, None)] * 3, method="highs")
            assert h.status == 2, (i, d)


def test_nan_records_unless_optimal(tp):
    cases = [([[1, 1], [1, 1]], [1, 3], [1, 1], [LE, GE], MAX, {}, INFEASIBLE),
             ([[1, -1], [1, 0]], [1, 0], [1, 1], [GE, GE], MAX, {}, UNBOUNDED)]
    from linear_programming_solver_lpr381_b200 import workloads
    A, b, c, rel, sense = workloads.batch_mixed(count=8, m=8, n=12, seed=2, sense=MIN)
    full = tp.two_phase_batch(A, b, c, rel, sense)
    k = int(np.argmax((full["status"] == OPTIMAL) & (full["n_pivots"] > full["phase1_pivots"] + 1)))
    A, b, c = A[k], b[k], c[k]
    p1, npv = int(full["phase1_pivots"][k]), int(full["n_pivots"][k])
    assert full["status"][k] == OPTIMAL and 0 < p1 < npv - 1
    # the limit in Phase I (0 and p1 - 1 pivots) and in Phase II (npv - 1)
    cases += [(A, b, c, rel, sense, dict(max_iterations=it), ITER_LIMIT) for it in (0, p1 - 1, npv - 1)]
    for A_, b_, c_, rel_, sense_, kw, status in cases:
        r = tp.two_phase_sensitivity(A_, b_, c_, rel_, sense_, **kw)
        assert r["status"] == status
        assert r["report"].shape == (4 * len(b_) + 3 * len(c_),) and np.isnan(r["report"]).all()
        plain = tp.two_phase(A_, b_, c_, rel_, sense_, **kw)
        for k in ("status", "phase1_pivots", "n_pivots", "pivots", "basis", "x", "z", "tableau"):
            assert np.asarray(plain[k]).tobytes() == np.asarray(r[k]).tobytes(), k


def test_new_exports():
    L = F.lib()
    for name in ("lpx_two_phase_solve_sensitivity_batched", "lpx_two_phase_solve_sensitivity_batched_dev",
                 "lpx_session_two_phase_sensitivity"):
        assert getattr(L, name).argtypes, name


@pytest.mark.parametrize("count,m,n,sense,rel,kernel,null", [
    (-1, 2, 2, 0, None, 0, None), (1, 0, 2, 0, None, 0, None), (1, 2, 0, 0, None, 0, None),
    (1, 2, 2, 2, None, 0, None), (1, 2, 2, 0, [0, 3], 0, None), (1, 2, 2, 0, [-1, 0], 0, None),
    (1, 2, 2, 0, None, F.KERNEL_STREAM, None), (1, 2, 2, 0, None, F.KERNEL_CTA_REG, None),
    (1, 2, 2, 0, None, 0, "A"), (1, 2, 2, 0, None, 0, "b"), (1, 2, 2, 0, None, 0, "c"),
    (1, 2, 2, 0, None, 0, "status"), (1, 2, 2, 0, None, 0, "report"),
])
def test_bad_arguments_before_any_device_work(count, m, n, sense, rel, kernel, null):
    arr = dict(A=np.ones((2, 2)), b=np.ones(2), c=np.ones(2), status=np.zeros(1, np.int32), report=np.zeros(14))
    if null:
        arr[null] = None
    rel = None if rel is None else np.array(rel, dtype=np.int32)
    opt = F.make_options(kernel=kernel)
    L = F.lib()
    total = C.c_longlong()
    assert L.lpx_two_phase_solve_sensitivity_batched(
        count, m, n, sense, F.ptr(arr["A"]), F.ptr(rel), F.ptr(arr["b"]), F.ptr(arr["c"]), C.byref(opt),
        F.ptr(arr["status"]), None, None, None, None, None, F.ptr(arr["report"]), C.byref(total)) == F.E_BAD_ARGS
    if rel is None:  # the _dev call reads rel from the device
        assert L.lpx_two_phase_solve_sensitivity_batched_dev(
            count, m, n, sense, F.ptr(arr["A"]), None, F.ptr(arr["b"]), F.ptr(arr["c"]), C.byref(opt),
            F.ptr(arr["status"]), None, None, None, None, None, F.ptr(arr["report"]), None, None) == F.E_BAD_ARGS


def test_session_call_refuses_a_null_session():
    assert F.lib().lpx_session_two_phase_sensitivity(None, F.ptr(np.zeros(4))) == F.E_BAD_ARGS


def test_fails_loudly_without_a_gpu():
    if F.lib().lpx_device_count() > 0:
        pytest.skip("a GPU is present")
    from linear_programming_solver_lpr381_b200 import api
    A, b, c, rel, sense = RADIATION
    with pytest.raises(F.LpxError) as e:
        api.two_phase_sensitivity(A, b, c, rel, sense)
    assert e.value.code == F.E_CUDA
    a, st, rep = np.ones(4), np.zeros(1, np.int32), np.zeros(14)
    with pytest.raises(F.LpxError) as e:
        api.two_phase_sensitivity_batched_dev(1, 2, 2, 0, a.ctypes.data, None, a.ctypes.data, a.ctypes.data,
                                              st.ctypes.data, None, None, None, None, None, rep.ctypes.data, None,
                                              None)
    assert e.value.code == F.E_CUDA

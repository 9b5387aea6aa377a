"""CPU: the two-phase Simplex oracle (oracle/orc_twophase.cpp) pinned independently of the GPU: known answers where
the reference-exact solvers fail, scipy's HiGHS on several hundred random mixed models, bit-for-bit identity with the
Primal Simplex oracle on all-'<=' models with b >= 0, and the C ABI's shape arithmetic, argument refusals and
missing-device failure."""
import ctypes as C

import numpy as np
import pytest

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

OPTIMAL, UNBOUNDED, INFEASIBLE, ITER_LIMIT = 0, 1, 2, -3
LE, GE, EQ = 0, 1, 2
MAX, MIN = 0, 1


@pytest.fixture(scope="module")
def tp():
    import orc_twophase_ffi
    orc_twophase_ffi.lib()
    return orc_twophase_ffi


def objective(c, x):
    return float(np.dot(c, x))


# (A, b, c, rel, sense, status, x, objective c.x as written)
KNOWN = {
    # Hillier & Lieberman's radiation-therapy LP
    "radiation": ([[0.3, 0.1], [0.5, 0.5], [0.6, 0.4]], [2.7, 6, 6], [0.4, 0.5], [LE, EQ, GE], MIN, OPTIMAL,
                  [7.5, 4.5], 5.25),
    "covering": ([[1, 1]], [2], [1, 1], [GE], MIN, OPTIMAL, [2, 0], 2.0),
    "equality": ([[1, 1]], [2], [1, 1], [EQ], MIN, OPTIMAL, [2, 0], 2.0),
    "infeasible_pair": ([[1, 1], [1, 1]], [1, 3], [1, 1], [LE, GE], MAX, INFEASIBLE, None, None),
    "unbounded_ge": ([[1, -1], [1, 0]], [1, 0], [1, 1], [GE, GE], MAX, UNBOUNDED, None, None),
    # -x1 - x2 <= -2 is x1 + x2 >= 2
    "negative_rhs_le": ([[-1, -1], [1, 0]], [-2, 3], [1, 2], [LE, LE], MIN, OPTIMAL, [2, 0], 2.0),
    # the second equality repeats the first: its artificial stays basic in a redundant row
    "duplicated_equality": ([[1, 1, 0], [1, 1, 0], [0, 1, 1]], [2, 2, 3], [1, 2, 1], [EQ, EQ, LE], MIN, OPTIMAL,
                            [2, 0, 0], 2.0),
}


@pytest.mark.parametrize("name", sorted(KNOWN))
def test_known_answers(tp, name):
    A, b, c, rel, sense, status, x, obj = KNOWN[name]
    r = tp.two_phase(A, b, c, rel, sense)
    assert r["status"] == status
    if status == OPTIMAL:
        assert np.allclose(r["x"], x, atol=1e-9, rtol=0)
        assert abs(objective(c, r["x"]) - obj) <= 1e-9
        assert abs(r["z"] - (-obj if sense == MIN else obj)) <= 1e-9  # z is the max form: -c.x for Min
    if name == "duplicated_equality":
        m, n, s = 3, 3, 1
        redundant = [i for i in range(m) if r["basis"][i] >= n + s]
        assert redundant == [1], r["basis"]
    if name == "radiation":
        assert r["phase1_pivots"] >= 1 and r["n_pivots"] >= r["phase1_pivots"]


def test_motivating_cases_against_the_reference_solvers(tp, orc):
    """'Min x1 + x2, x1 + x2 >= 2': the Dual Simplex oracle solves x1 + x2 <= 2 and reports 0.  'Min x1 + x2,
    x1 + x2 = 2': the Primal Simplex oracle reports OPTIMAL at x = 0.  The two-phase method gives 2 for both."""
    ge = tp.two_phase([[1, 1]], [2], [1, 1], [GE], MIN)
    d = orc.dual_solve(np.array([[1.0, 1.0]]), np.array([2.0]), np.array([1.0, 1.0]), np.array([GE], np.int32), MIN)
    assert ge["status"] == OPTIMAL and objective([1, 1], ge["x"]) == 2.0
    assert d["status"] == OPTIMAL and objective([1, 1], d["x"]) == 0.0
    eq = tp.two_phase([[1, 1]], [2], [1, 1], [EQ], MIN)
    p = orc.primal_solve(np.array([[1.0, 1.0]]), np.array([2.0]), np.array([1.0, 1.0]), np.array([EQ], np.int32), MIN)
    assert eq["status"] == OPTIMAL and objective([1, 1], eq["x"]) == 2.0
    assert p["status"] == OPTIMAL and not p["x"].any()


def random_mixed(seed, m, n):
    r = np.random.default_rng(seed)
    A = r.integers(-5, 6, size=(m, n)).astype(float)
    b = r.integers(-10, 11, size=m).astype(float)
    c = r.integers(-5, 6, size=n).astype(float)
    rel = r.integers(0, 3, size=m).astype(np.int32)
    return A, b, c, rel


def highs(A, b, c, rel, sense):
    from scipy.optimize import linprog
    sg = 1.0 if sense == MIN else -1.0
    ub = np.vstack([A[rel == LE], -A[rel == GE]])
    bub = np.concatenate([b[rel == LE], -b[rel == GE]])
    h = linprog(sg * c, A_ub=ub if len(ub) else None, b_ub=bub if len(ub) else None,
                A_eq=A[rel == EQ] if (rel == EQ).any() else None, b_eq=b[rel == EQ] if (rel == EQ).any() else None,
                bounds=[(0, None)] * len(c), method="highs")
    return {0: OPTIMAL, 2: INFEASIBLE, 3: UNBOUNDED}[h.status], (sg * h.fun if h.status == 0 else None)


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_highs_agreement(tp, sense):
    seen = set()
    for seed in range(200):
        m, n = 2 + seed % 6, 2 + (seed // 6) % 6
        A, b, c, rel = random_mixed(1000 * sense + seed, m, n)
        r = tp.two_phase(A, b, c, rel, sense)
        st, obj = highs(A, b, c, rel, sense)
        assert r["status"] == st, (seed, r["status"], st)
        seen.add(st)
        if st != OPTIMAL:
            continue
        got = objective(c, r["x"])
        assert abs(got - obj) <= 1e-7 * (1 + abs(got)), (seed, got, obj)
        assert abs(r["z"] - (-got if sense == MIN else got)) <= 1e-7 * (1 + abs(got))
        x = r["x"]
        assert (x >= -1e-9).all()
        ax = A @ x
        assert (ax[rel == LE] <= b[rel == LE] + 1e-7).all() and (ax[rel == GE] >= b[rel == GE] - 1e-7).all()
        assert np.allclose(ax[rel == EQ], b[rel == EQ], atol=1e-7, rtol=0)
    assert seen == {OPTIMAL, UNBOUNDED, INFEASIBLE}


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_mixed_workload_against_highs(tp, sense):
    A, b, c, rel, s = workloads.batch_mixed(count=24, m=16, n=24, seed=5, sense=sense, infeasible=0.25)
    assert (b < 0).any() and set(rel.tolist()) == {LE, GE, EQ}
    r = tp.two_phase_batch(A, b, c, rel, s)
    for k in range(len(A)):
        st, obj = highs(A[k], b[k], c[k], rel, s)
        assert r["status"][k] == st
        if st == OPTIMAL:
            got = objective(c[k], r["x"][k])
            assert abs(got - obj) <= 1e-7 * (1 + abs(got))
    assert set(r["status"].tolist()) == {OPTIMAL, INFEASIBLE}


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_identity_with_primal_oracle_on_all_le(tp, orc, sense):
    for seed in range(40):
        r0 = np.random.default_rng(seed)
        m, n = int(r0.integers(1, 9)), int(r0.integers(1, 9))
        A = r0.integers(-3, 8, size=(m, n)).astype(float)
        b = r0.integers(0, 20, size=m).astype(float)
        c = r0.integers(-4, 9, size=n).astype(float)
        if seed % 5 == 0:
            b[0] = -0.0  # not flipped
        got = tp.two_phase(A, b, c, None, sense, max_iterations=10000)
        want = orc.primal_solve(A, b, c, None, sense)
        assert got["status"] == want["status"] and got["phase1_pivots"] == 0
        assert got["n_pivots"] == want["n_pivots"]
        assert np.array_equal(got["pivots"][: got["n_pivots"]], want["pivots"])
        assert np.array_equal(got["basis"], want["basis"])
        for k in ("x", "z", "tableau"):
            assert np.asarray(got[k]).tobytes() == np.asarray(want[k]).tobytes(), (seed, k)


def test_iteration_limit_counts_both_phases(tp):
    """"iter > max_iterations" before each column choice, counting every pivot: a limit of k < N pivots stops after k
    pivots, in Phase I or in Phase II; N (the full count) still stops, before the optimality test; N + 1 finishes."""
    A, b, c, rel, s = workloads.batch_mixed(count=8, m=8, n=12, seed=2, sense=MIN)
    full = tp.two_phase_batch(A, b, c, rel, s)
    k = int(np.argmax((full["status"] == OPTIMAL) & (full["n_pivots"] > full["phase1_pivots"] + 1)))
    N, p1 = int(full["n_pivots"][k]), int(full["phase1_pivots"][k])
    assert full["status"][k] == OPTIMAL and 0 < p1 < N
    for it in range(N + 2):
        r = tp.two_phase(A[k], b[k], c[k], rel, s, max_iterations=it)
        assert r["status"] == (ITER_LIMIT if it <= N else OPTIMAL)
        assert r["n_pivots"] >= min(it, N) and r["phase1_pivots"] == min(r["n_pivots"], p1)
        n = int(r["n_pivots"])
        assert np.array_equal(r["pivots"][:n], full["pivots"][k][:n]) and (r["pivots"][n:] == -1).all()


def test_dims_without_a_device():
    from linear_programming_solver_lpr381_b200 import api
    assert api.two_phase_dims(3, 2) == (4, 6)
    assert api.two_phase_dims(3, 2, [EQ, GE, EQ]) == (4, 4)
    rows, cols = C.c_int(), C.c_int()
    L = F.lib()
    for args in ((0, 2, None), (3, 0, None), (3, 2, F.ptr(np.array([0, 3, 0], np.int32)))):
        assert L.lpx_two_phase_dims(*args, C.byref(rows), C.byref(cols)) == F.E_BAD_ARGS


@pytest.mark.parametrize("count,m,n,sense,rel,kernel,cap,null", [
    (-1, 2, 2, 0, None, 0, 4, None), (1, 0, 2, 0, None, 0, 4, None), (1, 2, 0, 0, None, 0, 4, None),
    (1, 2, 2, 2, None, 0, 4, None), (1, 2, 2, 0, [0, 3], 0, 4, None), (1, 2, 2, 0, [-1, 0], 0, 4, None),
    (1, 2, 2, 0, None, F.KERNEL_STREAM, 4, None), (1, 2, 2, 0, None, F.KERNEL_CTA_REG, 4, None),
    (1, 2, 2, 0, None, 0, -1, None), (1, 2, 2, 0, None, 0, 4, "A"), (1, 2, 2, 0, None, 0, 4, "b"),
    (1, 2, 2, 0, None, 0, 4, "c"), (1, 2, 2, 0, None, 0, 4, "status"),
])
def test_bad_arguments_before_any_device_work(count, m, n, sense, rel, kernel, cap, null):
    arr = dict(A=np.ones((2, 2)), b=np.ones(2), c=np.ones(2), status=np.zeros(1, np.int32))
    if null:
        arr[null] = None
    rel = None if rel is None else np.array(rel, dtype=np.int32)
    opt = F.make_options(kernel=kernel)
    L = F.lib()
    total = C.c_longlong()
    assert L.lpx_two_phase_solve_batched(count, m, n, sense, F.ptr(arr["A"]), F.ptr(rel), F.ptr(arr["b"]),
                                         F.ptr(arr["c"]), C.byref(opt), F.ptr(arr["status"]), None, None, None, cap,
                                         None, None, None, None, C.byref(total)) == F.E_BAD_ARGS
    if rel is None:  # the _dev call reads rel from the device
        assert L.lpx_two_phase_solve_batched_dev(count, m, n, sense, F.ptr(arr["A"]), None, F.ptr(arr["b"]),
                                                 F.ptr(arr["c"]), C.byref(opt), F.ptr(arr["status"]), None, None,
                                                 None, cap, None, None, None, None, None, None) == F.E_BAD_ARGS


def test_fails_loudly_without_a_gpu():
    if F.lib().lpx_device_count() > 0:
        pytest.skip("a GPU is present")
    from linear_programming_solver_lpr381_b200 import api
    with pytest.raises(F.LpxError) as e:
        api.two_phase_solve(np.ones((2, 2)), np.ones(2), np.ones(2), [GE, LE], MIN)
    assert e.value.code == F.E_CUDA
    a, st = np.ones(4), np.zeros(1, np.int32)
    with pytest.raises(F.LpxError) as e:
        api.two_phase_solve_batched_dev(1, 2, 2, 0, a.ctypes.data, None, a.ctypes.data, a.ctypes.data,
                                        st.ctypes.data, None, None, None, 0, None, None, None, None, None, None)
    assert e.value.code == F.E_CUDA

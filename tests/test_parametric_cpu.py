"""CPU: the parametric-analysis oracle (oracle/orc_param.cpp) pinned independently of the GPU: hand-derived Wyndor
breakpoints, scipy's HiGHS at the ends and midpoints of every segment and past every INFEASIBLE / UNBOUNDED end, the
definition's properties, bit-for-bit agreement with the sensitivity oracle's ranges, and the argument checks and the
missing-device failure of the C ABI."""
import ctypes as C

import numpy as np
import pytest

from test_reopt_cpu import random_lp

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

RHS, COST = 1, 2
REACHED, UNBOUNDED, INFEASIBLE, SEG_LIMIT, NO_BASE = 0, 1, 2, 3, 4
INF = np.inf


@pytest.fixture(scope="module")
def pm():
    import orc_param_ffi
    orc_param_ffi.lib()
    return orc_param_ffi


@pytest.fixture(scope="module")
def sens():
    import orc_sens_ffi
    orc_sens_ffi.lib()
    return orc_sens_ffi


def analyse(pm, base, kind, d, m, n, rel=None, sense=0, theta_max=INF, seg_cap=64):
    d = np.atleast_2d(np.asarray(d, dtype=float))
    pay = np.hstack([d, np.full((len(d), 1), theta_max)])
    return pm.parametric(kind, m, n, [base["status"]], [base["basis"]], [base["tableau"]], pay, rel, sense,
                         src=np.zeros(len(d), np.int32), seg_cap=seg_cap)


def segs(r, q=0):
    """(theta_lo, theta_hi, z0, dz) of query q's segments."""
    return [tuple(r["segments"][q, k, :4]) for k in range(r["n_segments"][q])]


@pytest.fixture(scope="module")
def wyndor(orc):
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    base = orc.primal_solve(p["A"], p["b"], p["c"], p["rel"], p["sense"])
    assert base["status"] == 0 and base["z"] == 36
    return p, base


def z_at(s, t):
    return s[2] + t * s[3]


@pytest.mark.parametrize("kind,d,end,want", [
    (RHS, [0, 0, 1], REACHED, [(0, 6, 36, 1), (6, INF, None, 0)]),          # b3 up: x1 reaches 4 at b3 = 24
    (RHS, [0, 0, -1], INFEASIBLE, [(0, 6, 36, -1), (6, 18, None, -2.5)]),   # b3 down: x2 hits 6 (b3 12), then 0
    (COST, [1, 0], REACHED, [(0, 4.5, 36, 2), (4.5, INF, None, 4)]),        # c1 up: past 7.5, x = (4, 3)
    (COST, [-1, 0], REACHED, [(0, 3, 36, -2), (3, INF, None, 0)]),          # c1 down: below 0, x = (0, 6)
])
def test_wyndor_hand_derived(pm, wyndor, kind, d, end, want):
    p, base = wyndor
    r = analyse(pm, base, kind, d, 3, 2, p["rel"], p["sense"])
    assert r["end"][0] == end and r["n_segments"][0] == len(want) and r["n_pivots"][0] == len(want) - 1
    got = segs(r)
    for g, w in zip(got, want):
        assert g[0] == w[0] and g[1] == w[1] and abs(g[3] - w[3]) < 1e-12
        if w[2] is not None:
            assert g[2] == w[2]
    for a, b in zip(got, got[1:]):  # continuous
        assert abs(z_at(a, a[1]) - z_at(b, b[0])) < 1e-12
    if kind == RHS and end == INFEASIBLE:
        assert abs(z_at(got[-1], 18)) < 1e-12 and abs(z_at(got[0], 6) - 30) < 1e-12
    if kind == RHS and end == REACHED:
        assert abs(z_at(got[0], 6) - 42) < 1e-12
    assert r["seg_pivots"][0, len(want) - 1].tolist() == [-1, -1]
    assert (r["seg_pivots"][0, :len(want) - 1] >= 0).all()


def test_wyndor_theta_max_and_seg_limit(pm, wyndor):
    p, base = wyndor
    r = analyse(pm, base, RHS, [0, 0, -1], 3, 2, p["rel"], p["sense"], theta_max=10)
    assert r["end"][0] == REACHED and [s[:2] for s in segs(r)] == [(0, 6), (6, 10)]
    r = analyse(pm, base, RHS, [0, 0, -1], 3, 2, p["rel"], p["sense"], theta_max=4)
    assert r["end"][0] == REACHED and [s[:2] for s in segs(r)] == [(0, 4)] and r["n_pivots"][0] == 0
    r = analyse(pm, base, COST, [1, 0], 3, 2, p["rel"], p["sense"], seg_cap=1)
    assert r["end"][0] == SEG_LIMIT and [s[:2] for s in segs(r)] == [(0, 4.5)]
    assert r["seg_pivots"][0, 0].tolist() == [-1, -1]
    # the final basis and tableau are the base's: no pivot was taken
    assert r["basis"][0].tolist() == base["basis"].tolist()
    assert r["tableau"][0][:-1].tobytes() == base["tableau"].tobytes()


def test_no_base(orc, pm):
    A, b, c = workloads.batch_c2(count=1, m=12, n=20, seed=1)
    base = orc.primal_solve(A[0], b[0], c[0], max_iterations=1)
    assert base["status"] == -3
    for kind, k in ((RHS, 12), (COST, 20)):
        r = analyse(pm, base, kind, np.ones(k), 12, 20)
        assert r["end"][0] == NO_BASE and r["n_segments"][0] == 0 and r["n_pivots"][0] == 0
        assert not r["segments"].any() and not r["basis"].any() and not r["tableau"].any()
        assert (r["seg_pivots"] == -1).all()


# ---- scipy HiGHS ----------------------------------------------------------------------------------------------------

def highs(A, b, c, rel, sense):
    from scipy.optimize import linprog
    A_ub, b_ub, A_eq, b_eq = [], [], [], []
    for i in range(len(b)):
        (A_eq if rel[i] == 2 else A_ub).append(A[i])
        (b_eq if rel[i] == 2 else b_ub).append(b[i])
    res = linprog(-c if sense == 0 else c, A_ub=np.array(A_ub) if A_ub else None, b_ub=b_ub or None,
                  A_eq=np.array(A_eq) if A_eq else None, b_eq=b_eq or None, bounds=[(0, None)] * len(c),
                  method="highs")
    status = {0: 0, 2: 2, 3: 1}[res.status]
    return status, (-res.fun if status == 0 else None)


def directions(kind, rng, m, n, count):
    k = m if kind == RHS else n
    out = []
    for q in range(count):
        d = np.zeros(k)
        if q % 2:
            d[rng.integers(k)] = float(rng.choice([-1.0, 1.0]) * rng.integers(1, 6))
        else:
            d = rng.integers(-5, 6, size=k).astype(float)
        out.append(d)
    return np.array(out)


def feasible(A, b, rel, x, tol=1e-7):
    ax = A @ x
    scale = 1.0 + np.abs(b)
    ok = np.where(rel == 2, np.abs(ax - b) <= tol * scale, ax <= b + tol * scale)
    return bool(ok.all() and (x >= -tol).all())


@pytest.mark.parametrize("kind", [RHS, COST])
@pytest.mark.parametrize("sense", [0, 1])
def test_highs_agreement(orc, pm, kind, sense):
    rng = np.random.default_rng(10 * kind + sense)
    ends = set()
    for seed in range(5):
        A, b, c, rel = random_lp(500 * kind + 10 * seed + sense, sense=sense)
        m, n = A.shape
        D = directions(kind, rng, m, n, 8)
        if kind == COST:  # a ray: x_{n-1} loosens every row and costs too much until its price rises along +-e_{n-1}
            A[:, n - 1] = np.where(rel == 2, 0.0, -rng.integers(0, 3, size=m))
            c[n - 1] = -1000.0 if sense == 0 else 1000.0
            D = np.vstack([D, np.eye(n)[n - 1] * (100.0 if sense == 0 else -100.0)])
        base = orc.primal_solve(A, b, c, rel, sense)
        assert base["status"] == 0
        r = analyse(pm, base, kind, D, m, n, rel, sense)
        for q in range(len(D)):
            ends.add(int(r["end"][q]))
            model = (lambda t: (b + t * D[q], c)) if kind == RHS else (lambda t: (b, c + t * D[q]))
            for k in range(r["n_segments"][q]):
                lo, hi, z0, dz = r["segments"][q, k, :4]
                x0, dx = r["segments"][q, k, 4:4 + n], r["segments"][q, k, 4 + n:]
                pts = [lo, (lo + hi) / 2, hi] if np.isfinite(hi) else [lo, lo + 1.0, lo + 10.0]
                for t in pts:
                    bt, ct = model(t)
                    st, want = highs(A, bt, ct, rel, sense)
                    assert st == 0, (seed, q, k, t)
                    z = z0 + t * dz
                    assert abs(z - want) <= 1e-9 * max(1.0, abs(want)), (seed, q, k, t, z, want)
                    assert feasible(A, bt, rel, x0 + t * dx), (seed, q, k, t)
            last = r["segments"][q, r["n_segments"][q] - 1, 1]
            if r["end"][q] in (INFEASIBLE, UNBOUNDED):
                bt, ct = model(last + max(1.0, 0.1 * last))
                assert highs(A, bt, ct, rel, sense)[0] == {INFEASIBLE: 2, UNBOUNDED: 1}[int(r["end"][q])]
    assert REACHED in ends and {RHS: INFEASIBLE, COST: UNBOUNDED}[kind] in ends


# ---- properties -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", [RHS, COST])
def test_continuity_and_convexity(orc, pm, kind):
    rng = np.random.default_rng(3 + kind)
    for seed in range(6):
        for sense in (0, 1):
            A, b, c, rel = random_lp(70 + seed, sense=sense)
            base = orc.primal_solve(A, b, c, rel, sense)
            m, n = A.shape
            D = directions(kind, rng, m, n, 6)
            r = analyse(pm, base, kind, D, m, n, rel, sense)
            for q in range(len(D)):
                s = segs(r, q)
                assert s[0][0] == 0 and s[0][2] == base["z"]
                for a, bb in zip(s, s[1:]):
                    assert a[1] == bb[0]
                    za, zb = z_at(a, a[1]), z_at(bb, bb[0])
                    assert abs(za - zb) <= 1e-9 * max(1.0, abs(za))
                    tol = 1e-9 * max(1.0, abs(a[3]))
                    assert (bb[3] <= a[3] + tol) if kind == RHS else (bb[3] >= a[3] - tol)
                assert r["n_pivots"][q] == r["n_segments"][q] - 1


def test_zero_direction(orc, pm):
    A, b, c, rel = random_lp(5)
    base = orc.primal_solve(A, b, c, rel)
    m, n = A.shape
    for kind, k in ((RHS, m), (COST, n)):
        for tmax in (0.0, 2.5, INF):
            r = analyse(pm, base, kind, np.array([0.0, -0.0] * k)[:k], m, n, rel, theta_max=tmax)
            assert r["end"][0] == REACHED and segs(r) == [(0.0, tmax, base["z"], 0.0)]
            assert r["segments"][0, 0, 4:4 + n].tobytes() == base["x"].tobytes()


# ---- agreement with the sensitivity oracle --------------------------------------------------------------------------

def test_sensitivity_agreement(orc, pm, sens):
    checked = 0
    for seed in range(8):
        for sense in (0, 1):
            A, b, c, rel = random_lp(300 + seed, sense=sense)
            base = orc.primal_solve(A, b, c, rel, sense)
            m, n = A.shape
            rep = sens.sensitivity(b, c, 0, base["basis"], base["tableau"], rel, sense)
            lo, hi = rep[2 * m:3 * m], rep[3 * m:4 * m]
            chi = rep[4 * m + 2 * n:]
            E = np.eye(m)
            for sgn, edge in ((1.0, hi), (-1.0, lo)):
                r = analyse(pm, base, RHS, sgn * E, m, n, rel, sense)
                for i in range(m):
                    t = r["segments"][i, 0, 1]
                    if t > 0:
                        assert (b[i] + t if sgn > 0 else b[i] - t) == edge[i], (seed, sense, i, sgn)
                        checked += 1
            r = analyse(pm, base, COST, np.eye(n), m, n, rel, sense)
            for j in range(n):
                t = r["segments"][j, 0, 1]
                if t > 0:
                    assert c[j] + t == chi[j], (seed, sense, j)
                    checked += 1
    assert checked > 200


# ---- the C ABI without a device ---------------------------------------------------------------------------------------

def test_strides_and_dims_without_a_device():
    from linear_programming_solver_lpr381_b200 import api
    L = F.lib()
    assert api.param_payload_stride("rhs", 3, 5) == 4 and api.param_payload_stride("cost", 3, 5) == 6
    assert L.lpx_param_payload_stride(7, 3, 5) == 0 and L.lpx_param_segment_stride(5) == 14
    assert api.parametric_dims("rhs", 3, 2) == (4, 7) and api.parametric_dims("cost", 3, 2) == (5, 6)
    assert api.parametric_dims("rhs", 3, 2, [0, 2, 0]) == (5, 8)
    rows, cols = C.c_int(), C.c_int()
    for args in ((0, 3, 2, None), (1, 0, 2, None), (2, 3, 0, None), (1, 3, 2, F.ptr(np.array([0, 3, 0], np.int32)))):
        assert L.lpx_parametric_dims(*args, C.byref(rows), C.byref(cols)) == F.E_BAD_ARGS


@pytest.mark.parametrize("kind,count,m,n,sense,seg_cap,rel,kernel,tmax", [
    (0, 1, 2, 2, 0, 4, None, 0, 1.0), (3, 1, 2, 2, 0, 4, None, 0, 1.0), (1, -1, 2, 2, 0, 4, None, 0, 1.0),
    (1, 1, 0, 2, 0, 4, None, 0, 1.0), (2, 1, 2, 0, 0, 4, None, 0, 1.0), (1, 1, 2, 2, 2, 4, None, 0, 1.0),
    (1, 1, 2, 2, 0, 0, None, 0, 1.0), (2, 1, 2, 2, 0, 4, [0, 5], 0, 1.0), (1, 1, 2, 2, 0, 4, None, F.KERNEL_STREAM, 1.0),
    (1, 1, 2, 2, 0, 4, None, 99, 1.0), (1, 1, 2, 2, 0, 4, None, 0, -1.0), (2, 1, 2, 2, 0, 4, None, 0, np.nan),
    (1, 1, 2, 2, 0, 4, None, 0, -np.inf)])
def test_bad_arguments_before_any_device_work(kind, count, m, n, sense, seg_cap, rel, kernel, tmax):
    A, b, c = np.ones((2, 2)), np.ones(2), np.ones(2)
    rel = None if rel is None else np.array(rel, dtype=np.int32)
    pay = np.array([1.0, 1.0, tmax])
    opt = F.make_options(kernel=kernel)
    end = np.zeros(1, np.int32)
    L = F.lib()
    assert L.lpx_parametric(kind, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt), count,
                            F.ptr(pay), seg_cap, None, F.ptr(end), *[None] * 6) == F.E_BAD_ARGS
    if rel is None and np.isfinite(tmax) and tmax >= 0:  # the _dev call reads rel and theta_max from the device
        assert L.lpx_parametric_batched_dev(kind, count, m, n, sense, None, F.ptr(end), F.ptr(end), F.ptr(A), None,
                                            F.ptr(pay), seg_cap, C.byref(opt), F.ptr(end), *[None] * 8) == F.E_BAD_ARGS


def test_fails_loudly_without_a_gpu():
    if F.lib().lpx_device_count() > 0:
        pytest.skip("a GPU is present")
    from linear_programming_solver_lpr381_b200 import api
    with pytest.raises(F.LpxError) as e:
        api.parametric("rhs", np.ones((2, 2)), np.ones(2), np.ones(2), [[1.0, 0.0]])
    assert e.value.code == F.E_CUDA
    pay, st = np.array([1.0, 0.0, 1.0]), np.zeros(1, np.int32)
    with pytest.raises(F.LpxError) as e:
        api.parametric_batched_dev("rhs", 1, 2, 2, 0, None, st.ctypes.data, st.ctypes.data, pay.ctypes.data, None,
                                   pay.ctypes.data, 4, st.ctypes.data, None, None, None, None, None, None, None, None)
    assert e.value.code == F.E_CUDA
    with pytest.raises(F.LpxError) as e:  # a direction of the wrong length is refused before the library is called
        api.parametric("cost", np.ones((2, 2)), np.ones(2), np.ones(2), [[1.0, 0.0, 0.0]])
    assert e.value.code == F.E_BAD_ARGS

"""CPU: the re-optimization oracle (oracle/orc_reopt.cpp) pinned independently of the GPU: hand-derived Wyndor
answers, scipy's HiGHS on every modified model from scratch, and the definition's properties (identity, agreement
with Mode B's bound row, agreement with the sensitivity report)."""
import numpy as np
import pytest

from linear_programming_solver_lpr381_b200 import workloads

RHS, COST, ROW, COL = 1, 2, 3, 4


@pytest.fixture(scope="module")
def ro():
    import orc_reopt_ffi
    orc_reopt_ffi.lib()
    return orc_reopt_ffi


@pytest.fixture(scope="module")
def sens():
    import orc_sens_ffi
    orc_sens_ffi.lib()
    return orc_sens_ffi


def base_of(orc, A, b, c, rel=None, sense=0, max_iterations=10000):
    return orc.primal_solve(A, b, c, rel, sense, max_iterations=max_iterations)


def query(ro, base, kind, payload, m, n, rel=None, sense=0, **kw):
    return ro.reopt(kind, m, n, [base["status"]], [base["basis"]], [base["tableau"]], np.atleast_2d(payload), rel,
                    sense, src=np.zeros(len(np.atleast_2d(payload)), np.int32), **kw)


@pytest.fixture(scope="module")
def wyndor(orc):
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    base = base_of(orc, p["A"], p["b"], p["c"], p["rel"], p["sense"])
    assert base["status"] == 0 and base["z"] == 36 and base["x"].tolist() == [2, 6]
    return p, base


@pytest.mark.parametrize("kind,payload,status,z,x,min_piv,max_piv", [
    (RHS, [0, 0, 12], 0, 42, [4, 6], 1, 99),        # b3 18 -> 30
    (RHS, [0, 0, 2], 0, 38, None, 0, 0),            # b3 18 -> 20, inside [12, 24]
    (ROW, [1, 1, 0, 7], 0, 33, [1, 6], 1, 99),      # x1 + x2 <= 7
    (ROW, [1, 0, 1, 3], 0, 31.5, [3, 4.5], 1, 99),  # x1 >= 3
    (ROW, [1, 0, 1, 5], 2, None, None, 0, 99),      # x1 >= 5: infeasible
    (COST, [5, 0], 0, 47, [4, 3], 1, 99),           # c1 3 -> 8, past 7.5
    (COL, [0, 0, 1, 4], 0, 72, [0, 0, 18], 1, 99),  # x3 in row 3 only, c3 = 4 > its shadow price 1
])
def test_wyndor_hand_derived(ro, wyndor, kind, payload, status, z, x, min_piv, max_piv):
    # the new activity uses row 3 alone and earns 4 per unit of it, x1 1 and x2 2.5: x3 = 18 takes all of row 3
    p, base = wyndor
    r = query(ro, base, kind, payload, 3, 2, p["rel"], p["sense"])
    assert r["status"][0] == status
    assert min_piv <= r["n_pivots"][0] <= max_piv
    if z is not None:
        assert abs(r["z"][0] - z) < 1e-12
    if x is not None:
        np.testing.assert_allclose(r["x"][0], x, rtol=0, atol=1e-12)


# ---- scipy HiGHS on the modified model ----------------------------------------------------------------------------

def random_lp(seed, m=7, n=9, sense=0, n_eq=2):
    rng = np.random.default_rng(seed)
    A = rng.integers(1, 9, size=(m, n)).astype(float)
    b = rng.integers(10, 60, size=m).astype(float)
    rel = np.zeros(m, np.int32)
    for i in rng.choice(m, n_eq, replace=False):  # EQ rows at b = 0 keep x = 0 feasible for the Primal Simplex
        rel[i] = 2
        b[i] = 0.0
        A[i] = rng.integers(-4, 5, size=n)
    c = rng.integers(1, 12, size=n).astype(float)
    if sense == 1:
        c = -c  # Min with costs that pay
    return A, b, c, rel


def highs(A, b, c, rel, sense, extra_row=None):
    from scipy.optimize import linprog
    A_ub, b_ub, A_eq, b_eq = [], [], [], []
    for i in range(len(b)):
        (A_eq if rel[i] == 2 else A_ub).append(A[i] if rel[i] != 1 else -A[i])
        (b_eq if rel[i] == 2 else b_ub).append(b[i] if rel[i] != 1 else -b[i])
    if extra_row is not None:
        a, r, beta = extra_row
        A_ub.append(a if r == 0 else -a)
        b_ub.append(beta if r == 0 else -beta)
    obj = -c if sense == 0 else c
    res = linprog(obj, A_ub=np.array(A_ub) if A_ub else None, b_ub=b_ub or None, A_eq=np.array(A_eq) if A_eq else None,
                  b_eq=b_eq or None, bounds=[(0, None)] * len(c), method="highs")
    status = {0: 0, 2: 2, 3: 1}[res.status]
    return status, (-res.fun if status == 0 else None)  # the engine's z is the max-form value


def payloads(kind, rng, A, b, c, rel, sense, base, rep, count):
    m, n = A.shape
    out = []
    for k in range(count):
        if kind == RHS:
            d = np.zeros(m)
            i = rng.integers(m)
            if rel[i] == 2:
                d[i] = rng.choice([-1.0, 1.0]) * rng.integers(1, 4)
            else:
                lo, hi = rep["rhs_lo"][i], rep["rhs_hi"][i]
                span = 10.0 if not np.isfinite(hi - lo) else max(hi - lo, 1.0)
                d[i] = float(np.round(rng.uniform(-1.5, 1.5) * span - b[i] * (k % 5 == 0), 3))
            d[i] = max(d[i], -b[i]) if rel[i] != 2 and k % 7 else d[i]
            out.append(d)
        elif kind == COST:
            d = np.zeros(n)
            j = rng.integers(n)
            d[j] = float(np.round(rng.uniform(-2, 2) * (abs(c[j]) + 1), 3))
            out.append(d)
        elif kind == ROW:
            a = rng.integers(0, 5, size=n).astype(float)
            r = int(rng.integers(2))
            ax = float(a @ base["x"])
            beta = float(np.round(ax * rng.uniform(0.3, 1.6) + (50 * (k % 6 == 0) if r else 0), 3))
            out.append(np.concatenate([a, [r, beta]]))
        else:
            a = rng.integers(-2, 6, size=m).astype(float)
            a[rel == 2] = np.where(rng.random(int(np.sum(rel == 2))) < 0.5, 0.0, a[rel == 2])
            if k % 5 == 0:
                a = -np.abs(a)  # a column that only loosens: unbounded when it pays
                a[rel == 2] = 0.0
            cn = float(rng.integers(1, 15))
            out.append(np.concatenate([a, [cn if sense == 0 else -cn]]))
    return np.array(out)


@pytest.mark.parametrize("kind", [RHS, COST, ROW, COL])
@pytest.mark.parametrize("sense", [0, 1])
def test_highs_agreement(orc, ro, sens, kind, sense):
    rng = np.random.default_rng(100 * kind + sense)
    seen = set()
    for seed in range(6):
        A, b, c, rel = random_lp(1000 * kind + 10 * seed + sense, sense=sense)
        base = base_of(orc, A, b, c, rel, sense)
        assert base["status"] == 0
        m, n = A.shape
        rep = dict(zip(("shadow", "slack", "rhs_lo", "rhs_hi", "reduced", "cost_lo", "cost_hi"),
                       np.split(sens.sensitivity(b, c, 0, base["basis"], base["tableau"], rel, sense),
                                np.cumsum([m, m, m, m, n, n])[:])))
        pay = payloads(kind, rng, A, b, c, rel, sense, base, rep, 12)
        r = query(ro, base, kind, pay, m, n, rel, sense)
        for q in range(len(pay)):
            if kind == RHS:
                want = highs(A, b + pay[q], c, rel, sense)
            elif kind == COST:
                want = highs(A, b, c + pay[q], rel, sense)
            elif kind == ROW:
                want = highs(A, b, c, rel, sense, (pay[q][:n], int(pay[q][n]), pay[q][n + 1]))
            else:
                want = highs(np.hstack([pay[q][:m, None], A]), b, np.concatenate([[pay[q][m]], c]), rel, sense)
            assert r["status"][q] == want[0], (seed, q, pay[q])
            seen.add(int(r["status"][q]))
            if want[0] == 0:
                assert abs(r["z"][q] - want[1]) <= 1e-7 * max(1.0, abs(want[1])), (seed, q)
    assert 0 in seen
    if kind != COST:
        assert {RHS: 2, ROW: 2, COL: 1}[kind] in seen  # the infeasible / unbounded outcome is reached too


# ---- properties --------------------------------------------------------------------------------------------------

def test_identity(orc, ro):
    for sense in (0, 1):
        A, b, c, rel = random_lp(7 + sense, sense=sense)
        base = base_of(orc, A, b, c, rel, sense)
        m, n = A.shape
        for kind, pay in ((RHS, np.array([0.0, -0.0] * 4)[:m]), (COST, np.array([-0.0, 0.0] * 5)[:n])):
            r = query(ro, base, kind, pay, m, n, rel, sense)
            assert r["status"][0] == base["status"] and r["n_pivots"][0] == 0
            assert r["tableau"][0].tobytes() == base["tableau"].tobytes()
            assert r["basis"][0].tolist() == base["basis"].tolist()
            assert r["x"][0].tobytes() == base["x"].tobytes() and r["z"][0] == base["z"]
        # a column that does not pay: the base with one inserted column, nothing else
        pay = np.concatenate([np.zeros(m), [-1.0 if sense == 0 else 1.0]])
        r = query(ro, base, COL, pay, m, n, rel, sense)
        T = base["tableau"]
        assert r["n_pivots"][0] == 0 and r["status"][0] == 0
        want = np.hstack([T[:, :n], np.zeros((T.shape[0], 1)), T[:, n:]])
        want[-1, n] = 1.0
        assert r["tableau"][0].tobytes() == want.tobytes()
        assert r["basis"][0].tolist() == [v + 1 if v >= n else v for v in base["basis"]]
        assert r["z"][0] == base["z"] and r["x"][0][n:].tolist() == [0.0] and r["x"][0][:n].tobytes() == base["x"].tobytes()


def test_mode_b_agreement(orc, ro):
    """A ROW query with a = e_k on a basic x_k builds Mode B's bound row bit for bit, with the same pivots."""
    checked = 0
    for seed in range(12):
        A, b, c = workloads.ip_c4(m=8, n=12, seed=seed)
        base = base_of(orc, A, b, c)
        m, n = A.shape
        for k in [int(v) for v in base["basis"] if v < n]:
            xk = base["x"][k]
            for side, val in ((0, np.floor(xk)), (1, np.ceil(xk)), (0, xk), (1, 0.0)):
                To, bo = ro.extend_tableau(base["tableau"], base["basis"], k, side, val)
                pay = np.zeros(n + 2)
                pay[k], pay[n], pay[n + 1] = 1.0, side, val
                r = query(ro, base, ROW, pay, m, n)
                st, piv, bf, Tf = ro.dual_core(To, bo)
                assert r["status"][0] == (0 if st == 0 else st)
                assert r["n_pivots"][0] == len(piv)
                assert r["pivots"][0][:len(piv)].tolist() == piv.tolist()
                assert r["basis"][0].tolist() == bf.tolist()
                assert r["tableau"][0].tobytes() == Tf.tobytes()
                checked += 1
    assert checked > 50


def test_mode_b_build_bits(orc, ro):
    """The ROW build equals extend_tableau's child bit for bit, signed zeros included, on both sides: a bound the base
    already satisfies takes no pivot, so the query's result is its build."""
    A, b, c = workloads.ip_c4(m=8, n=12, seed=3)
    base = base_of(orc, A, b, c)
    m, n = A.shape
    T = base["tableau"].copy()
    T[:-1, :n] = np.where(T[:-1, :n] == 0, -0.0, T[:-1, :n])  # negative zeros in the rows the bound row reads
    base = dict(base, tableau=T)
    for k in [int(v) for v in base["basis"] if v < n]:
        for side, val in ((0, np.ceil(base["x"][k]) + 1), (1, 0.0)):
            To, bo = ro.extend_tableau(T, base["basis"], k, side, val)
            pay = np.zeros(n + 2)
            pay[k], pay[n], pay[n + 1] = 1.0, side, val
            r = query(ro, base, ROW, pay, m, n)
            assert r["n_pivots"][0] == 0
            assert r["tableau"][0].tobytes() == To.tobytes() and r["basis"][0].tolist() == bo.tolist()


def test_sensitivity_agreement(orc, ro, sens):
    for seed in range(8):
        A, b, c = workloads.batch_c2(count=1, m=12, n=20, seed=seed)
        A, b, c = A[0], b[0], c[0]
        base = base_of(orc, A, b, c)
        m, n = A.shape
        rep = sens.sensitivity(b, c, 0, base["basis"], base["tableau"])
        shadow, lo, hi = rep[:m], rep[2 * m:3 * m], rep[3 * m:4 * m]
        clo, chi = rep[4 * m + n:4 * m + 2 * n], rep[4 * m + 2 * n:]
        for i in range(m):
            for t in (0.25, 0.75):
                if not (np.isfinite(lo[i]) and np.isfinite(hi[i])) or hi[i] - lo[i] < 1e-6:
                    continue
                d = np.zeros(m)
                d[i] = (lo[i] + t * (hi[i] - lo[i])) - b[i]
                if d[i] == 0:
                    continue
                r = query(ro, base, RHS, d, m, n)
                assert r["n_pivots"][0] == 0 and r["status"][0] == 0
                assert r["z"][0] == base["z"] + d[i] * shadow[i]  # Max, LE row: bit for bit
            for edge, sgn in ((hi[i], 1), (lo[i], -1)):
                if np.isfinite(edge):
                    d = np.zeros(m)
                    d[i] = edge - b[i] + sgn * (1.0 + 0.1 * abs(edge))
                    r = query(ro, base, RHS, d, m, n)
                    assert r["n_pivots"][0] >= 1 or r["status"][0] == 2
        for j in range(n):
            for t in (0.25, 0.75):
                if not (np.isfinite(clo[j]) and np.isfinite(chi[j])) or chi[j] - clo[j] < 1e-6:
                    continue
                d = np.zeros(n)
                d[j] = clo[j] + t * (chi[j] - clo[j]) - c[j]
                r = query(ro, base, COST, d, m, n)
                assert r["n_pivots"][0] == 0 and r["basis"][0].tolist() == base["basis"].tolist()
                assert r["x"][0].tobytes() == base["x"].tobytes()
            if np.isfinite(chi[j]):
                d = np.zeros(n)
                d[j] = chi[j] - c[j] + 1.0 + 0.1 * abs(chi[j])
                r = query(ro, base, COST, d, m, n)
                assert r["n_pivots"][0] >= 1 or r["status"][0] == 1


def test_status_follows_base(orc, ro):
    A, b, c = workloads.batch_c2(count=1, m=12, n=20, seed=1)
    A, b, c = A[0], b[0], c[0]
    base = base_of(orc, A, b, c, max_iterations=1)
    assert base["status"] == -3
    m, n = A.shape
    for kind, stride in ((RHS, m), (COST, n), (ROW, n + 2), (COL, m + 1)):
        r = query(ro, base, kind, np.ones(stride) * (kind != ROW), m, n)
        assert r["status"][0] == -3 and r["n_pivots"][0] == 0
        assert not r["tableau"].any() and not r["x"].any() and not r["basis"].any() and r["z"][0] == 0


def test_iteration_limit(orc, ro):
    A, b, c = workloads.batch_c2(count=1, m=12, n=20, seed=2)
    A, b, c = A[0], b[0], c[0]
    base = base_of(orc, A, b, c)
    m, n = A.shape
    r = query(ro, base, COST, np.full(n, 50.0), m, n, max_iterations=1)
    assert r["status"][0] == -3 and r["n_pivots"][0] == 1

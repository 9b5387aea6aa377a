"""CPU: the sensitivity oracle (oracle/orc_sensitivity.cpp) pinned independently of the tableau it reads:
textbook values, a basis-matrix restatement in numpy, and scipy's HiGHS."""
import numpy as np
import pytest

from linear_programming_solver_lpr381_b200 import workloads


@pytest.fixture(scope="module")
def sens():
    import orc_sens_ffi
    orc_sens_ffi.lib()
    return orc_sens_ffi


def solve_report(orc, sens, A, b, c, rel=None, sense=0):
    r = orc.primal_solve(A, b, c, rel, sense)
    m, n = A.shape
    rep = sens.sensitivity(b, c, r["status"], r["basis"], r["tableau"], rel, sense)
    o = np.cumsum([0, m, m, m, m, n, n, n])
    names = ("shadow", "slack", "rhs_lo", "rhs_hi", "reduced", "cost_lo", "cost_hi")
    return r, {k: rep[o[i]:o[i + 1]] for i, k in enumerate(names)}


def test_wyndor_textbook(orc, sens):
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    _, s = solve_report(orc, sens, p["A"], p["b"], p["c"], p["rel"], p["sense"])
    close = dict(rtol=0, atol=1e-12)
    np.testing.assert_allclose(s["shadow"], [0, 1.5, 1], **close)
    np.testing.assert_allclose(s["reduced"], [0, 0], **close)
    np.testing.assert_allclose(s["rhs_lo"], [2, 6, 12], **close)
    np.testing.assert_allclose(s["rhs_hi"], [np.inf, 18, 24], **close)
    np.testing.assert_allclose(s["cost_lo"], [0, 2], **close)
    np.testing.assert_allclose(s["cost_hi"], [7.5, np.inf], **close)
    np.testing.assert_allclose(s["slack"], [2, 0, 0], **close)
    _, s = solve_report(orc, sens, p["A"], p["b"], -p["c"], p["rel"], 1)
    np.testing.assert_allclose(s["shadow"], [0, -1.5, -1], **close)
    np.testing.assert_allclose(s["cost_lo"], [-7.5, -np.inf], **close)
    np.testing.assert_allclose(s["cost_hi"], [0, -2], **close)


def test_non_optimal_status_gives_nan_record(sens):
    rep = sens.sensitivity(np.ones(2), np.ones(3), 1, np.array([3, 4]), np.zeros((3, 6)))
    assert rep.shape == (17,) and np.isnan(rep).all()


def basis_restatement(A, b, c, rel, sense, basis):
    """The report from B = [A' | I][:, basis] without reading the tableau."""
    m, n = A.shape
    rows, bb, row1 = [], [], []
    for i in range(m):
        row1.append(len(rows))
        rows.append(A[i])
        bb.append(b[i])
        if rel[i] == 2:
            rows.append(-A[i])
            bb.append(-b[i])
    Ap, bp = np.array(rows), np.array(bb)
    mm = len(rows)
    M = np.hstack([Ap, np.eye(mm)])
    cp = np.concatenate([c if sense == 0 else -c, np.zeros(mm)])
    B = M[:, basis]
    y = np.linalg.solve(B.T, cp[basis])
    beta = np.linalg.solve(B, bp)
    BinvM = np.linalg.solve(B, M)
    d = y @ M - cp
    basic = np.zeros(n + mm, dtype=bool)
    basic[basis] = True
    rowof = {int(k): r for r, k in enumerate(basis)}
    eps = 1e-9
    out = dict(shadow=[], slack=[], rhs_lo=[], rhs_hi=[], reduced=list(d[:n]), cost_lo=[], cost_hi=[])
    for i in range(m):
        k1 = n + row1[i]
        u = y[row1[i]] - (y[row1[i] + 1] if rel[i] == 2 else 0.0)
        g = BinvM[:, k1] - (BinvM[:, k1 + 1] if rel[i] == 2 else 0.0)
        out["shadow"].append(-u if sense == 1 else u)
        out["slack"].append(beta[rowof[k1]] if k1 in rowof else 0.0)
        lo = [-(beta[r] / g[r]) for r in range(mm) if g[r] > eps]
        hi = [-(beta[r] / g[r]) for r in range(mm) if g[r] < -eps]
        out["rhs_lo"].append(b[i] + max(lo) if lo else -np.inf)
        out["rhs_hi"].append(b[i] + min(hi) if hi else np.inf)
    for j in range(n):
        if not basic[j]:
            lo, hi = (-np.inf, c[j] + d[j]) if sense == 0 else (c[j] - d[j], np.inf)
        else:
            r = rowof[j]
            ks = [k for k in range(n + mm) if not basic[k]]
            dl = [-(d[k] / BinvM[r, k]) for k in ks if BinvM[r, k] > eps]
            dh = [-(d[k] / BinvM[r, k]) for k in ks if BinvM[r, k] < -eps]
            dl = max(dl) if dl else -np.inf
            dh = min(dh) if dh else np.inf
            lo, hi = (c[j] + dl, c[j] + dh) if sense == 0 else (c[j] - dh, c[j] - dl)
        out["cost_lo"].append(lo)
        out["cost_hi"].append(hi)
    return {k: np.array(v, dtype=float) for k, v in out.items()}


def random_lps(count, seed):
    rng = np.random.default_rng(seed)
    for t in range(count):
        m, n = int(rng.integers(2, 10)), int(rng.integers(2, 12))
        gen = workloads.lp_decimal if t % 2 else workloads.lp_integer
        A, b, c = gen(m, n, seed * 1000 + t)
        sense = int(rng.integers(0, 2))
        if sense == 1:
            c = -c  # a Min whose optimum is not x = 0
        rel = np.zeros(m, dtype=np.int32)
        if t % 3 == 0:
            rel[rng.choice(m, size=max(1, m // 3), replace=False)] = 2
            b = b.copy()
            b[rel == 2] = 0.0
        yield t, A, b, c, rel, sense


def test_oracle_matches_basis_restatement(orc, sens):
    checked = 0
    for t, A, b, c, rel, sense in random_lps(60, 17):
        r, s = solve_report(orc, sens, A, b, c, rel, sense)
        if r["status"] != 0:
            continue
        checked += 1
        want = basis_restatement(A, b, c, rel, sense, r["basis"])
        for k, v in want.items():
            np.testing.assert_allclose(s[k], v, rtol=1e-9, atol=1e-9, err_msg=f"LP {t} {k}")
    assert checked >= 45


def test_against_highs(orc, sens):
    linprog = pytest.importorskip("scipy.optimize").linprog
    checked = 0
    for t in range(40):
        m, n = 5, 7
        A, b, c = workloads.lp_decimal(m, n, 500 + t)
        sense = t % 2
        if sense == 1:
            c = -c
        r, s = solve_report(orc, sens, A, b, c, None, sense)
        T = r["tableau"]
        nonbasic = np.setdiff1d(np.arange(n + m), r["basis"])
        if r["status"] != 0 or (T[:m, -1] <= 1e-7).any() or (T[m, nonbasic] <= 1e-7).any():
            continue  # degenerate: duals or ranges are not unique
        checked += 1
        obj = -c if sense == 0 else c

        def solve(bb=b, cc=obj):
            h = linprog(cc, A_ub=A, b_ub=bb, bounds=[(0, None)] * n, method="highs")
            assert h.status == 0
            return h

        h = solve()
        sign = -1.0 if sense == 0 else 1.0
        np.testing.assert_allclose(s["shadow"], sign * h.ineqlin.marginals, atol=1e-7)
        np.testing.assert_allclose(s["reduced"], h.lower.marginals, atol=1e-7)
        user = lambda v: -v if sense == 0 else v  # noqa: E731  objective as written
        z0 = user(h.fun)
        for i in range(m):
            lo, hi, y = s["rhs_lo"][i], s["rhs_hi"][i], s["shadow"][i]
            scale = max(1.0, abs(b[i]))
            for pt in (lo + 0.25 * (hi - lo), lo + 0.75 * (hi - lo)) if np.isfinite(hi) else (lo + 0.5 * scale,):
                bb = b.copy()
                bb[i] = pt
                assert abs(user(solve(bb).fun) - (z0 + y * (pt - b[i]))) < 1e-7 * max(1.0, abs(z0)), (t, i)
            for end, step in ((lo, -1e-4 * scale), (hi, 1e-4 * scale)):
                if not np.isfinite(end) or end + step < 0:
                    continue
                bb = b.copy()
                bb[i] = end + step
                h2 = linprog(obj, A_ub=A, b_ub=bb, bounds=[(0, None)] * n, method="highs")
                assert h2.status != 0 or abs(user(h2.fun) - (z0 + y * (end + step - b[i]))) > 1e-9 * max(1.0, abs(z0)), \
                    (t, i, "past end")
        for j in range(n):
            lo, hi = s["cost_lo"][j], s["cost_hi"][j]
            scale = max(1.0, abs(c[j]))
            inner = [lo + 0.5 * (hi - lo)] if np.isfinite(lo) and np.isfinite(hi) else \
                [(lo if np.isfinite(lo) else hi) + (scale if np.isfinite(lo) else -scale) * 0.5]
            for pt in inner:
                cc = c.copy()
                cc[j] = pt
                np.testing.assert_allclose(solve(cc=-cc if sense == 0 else cc).x, h.x, atol=1e-7)
            for end, step in ((lo, -1e-4 * scale), (hi, 1e-4 * scale)):
                if not np.isfinite(end):
                    continue
                cc = c.copy()
                cc[j] = end + step
                assert np.abs(solve(cc=-cc if sense == 0 else cc).x - h.x).max() > 1e-7, (t, j, "past end")
    assert checked >= 5

"""GPU: what-if queries on an optimal streaming session (lpx_session_reoptimize) must equal oracle/orc_reopt.cpp run on
the base session's tableau and basis, bit for bit (status, pivot list, basis, x, z, every tableau double), and the
batched route (lpx_reoptimize_batched_dev) on the same base."""
import numpy as np
import pytest

from conftest import assert_bits_equal
from test_gpu_reopt import CAP, run_dev
from test_reopt_cpu import payloads, random_lp

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

RHS, COST, ROW, COL = 1, 2, 3, 4
CHUNKS = [1, 5, 11]


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


def to_optimum(s):
    st, tot = F.RUNNING, 0
    while st == F.RUNNING:
        st, tot = s.step(512)
    return st, tot


def run_query(q):
    """Step a query session to a terminal status in uneven chunks (1, 5, 11, then 512s); all its outputs."""
    st, tot, k = F.RUNNING, 0, 0
    while st == F.RUNNING:
        st, tot = q.step(CHUNKS[k] if k < len(CHUNKS) else 512)
        k += 1
    basis, x, z = q.solution()
    return dict(status=st, n_pivots=tot, pivots=q.pivots(CAP), basis=basis, x=x, z=z, tableau=q.tableau())


def check_one(got, want, q, what):
    assert got["status"] == want["status"][q], what
    assert got["n_pivots"] == want["n_pivots"][q], what
    assert np.array_equal(got["pivots"], want["pivots"][q]), what + " pivots"
    assert np.array_equal(got["basis"], want["basis"][q]), what + " basis"
    assert_bits_equal(got["x"], want["x"][q], what + " x")
    assert_bits_equal([got["z"]], [want["z"][q]], what + " z")
    assert_bits_equal(got["tableau"], want["tableau"][q], what + " tableau")


def base_state(s):
    basis, x, z = s.solution()
    return dict(basis=basis, x=x, z=z, tableau=s.tableau())


def oracle(ro, kind, base, pay, m, n, rel=None, sense=0, max_iterations=10000):
    pay = np.atleast_2d(pay)
    return ro.reopt(kind, m, n, [0], [base["basis"]], [base["tableau"]], pay, rel, sense,
                    np.zeros(len(pay), np.int32), max_iterations, CAP)


def batched(kind, base, pay, m, n, rel=None, sense=0, **opt):
    """The batched route on the session's final tableau, uploaded as a base."""
    import torch
    dev = torch.device("cuda:0")
    bases = dict(rel=None if rel is None else torch.from_numpy(np.ascontiguousarray(rel, np.int32)).to(dev),
                 status=torch.zeros(1, dtype=torch.int32, device=dev),
                 basis=torch.from_numpy(np.ascontiguousarray(base["basis"][None], np.int32)).to(dev),
                 tableau=torch.from_numpy(np.ascontiguousarray(base["tableau"][None])).to(dev))
    pay = np.atleast_2d(pay)
    return run_dev(kind, bases, pay, m, n, sense, np.zeros(len(pay), np.int32), **opt)


def sens_dict(rep, m, n):
    keys = ("shadow", "slack", "rhs_lo", "rhs_hi", "reduced", "cost_lo", "cost_hi")
    return dict(zip(keys, np.split(rep, np.cumsum([m, m, m, m, n, n]))))


@pytest.mark.parametrize("protocol", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("sense", [0, 1])
@pytest.mark.parametrize("shape", [(64, 128), (150, 300)], ids=["64x128", "150x300"])
def test_each_kind_against_oracle_and_batched_route(lpx, sens, ro, shape, sense, protocol):
    m, n = shape
    A, b, c, rel = random_lp(1000 * protocol + 10 * sense + m, m=m, n=n, sense=sense, n_eq=3)
    s = lpx.Session(A, b, c, rel=rel, sense=sense, single_cta_select=protocol)
    st, tot = to_optimum(s)
    assert st == F.OPTIMAL
    base = base_state(s)
    rep = sens_dict(s.sensitivity()["report"], m, n)
    rng = np.random.default_rng(protocol + 7 * sense + m)
    moved = 0
    for kind in (RHS, COST, ROW, COL):
        pay = np.array(payloads(kind, rng, A, b, c, rel, sense, base, rep, 4))
        want = oracle(ro, kind, base, pay, m, n, rel, sense)
        check_batched = batched(kind, base, pay, m, n, rel, sense)
        for f in ("status", "n_pivots", "pivots", "basis"):
            assert np.array_equal(check_batched[f], want[f]), f"batched route {f}, kind {kind}"
        for f in ("x", "z", "tableau"):
            assert_bits_equal(check_batched[f], want[f], f"batched route {f}, kind {kind}")
        for q in range(len(pay)):
            qs = s.reoptimize(kind, pay[q])
            assert (qs.rows, qs.cols) == want["tableau"].shape[1:]
            check_one(run_query(qs), want, q, f"{shape} sense {sense} protocol {protocol} kind {kind} query {q}")
            qs.close()
        moved += int((want["n_pivots"] > 0).sum())
    assert moved > 0
    # the base is where it was
    assert s.sync() == (F.OPTIMAL, tot)
    after = base_state(s)
    assert np.array_equal(after["basis"], base["basis"])
    assert_bits_equal(after["tableau"], base["tableau"], "base tableau after the queries")
    s.close()


@pytest.fixture(scope="module")
def small_base(lpx):
    A, b, c, rel = random_lp(4242, m=64, n=128, n_eq=3)
    s = lpx.Session(A, b, c, rel=rel)
    st, tot = to_optimum(s)
    assert st == F.OPTIMAL
    yield A, b, c, rel, s, tot
    s.close()


def test_outcomes(lpx, ro, small_base):
    """RHS / ROW queries that end INFEASIBLE, a COL query that ends UNBOUNDED, COST queries that hit a small
    max_iterations, and a zero payload of each kind (OPTIMAL, 0 pivots, the base's bits)."""
    A, b, c, rel, s, _ = small_base
    m, n = A.shape
    base = base_state(s)
    le = int(np.flatnonzero(rel == 0)[0])
    cases = []
    d = np.zeros(m)
    d[le] = -b[le] - 1000.0  # a.x <= -1000 with a >= 1
    cases.append((RHS, d, {}, F.INFEASIBLE))
    # an added row the feasible set cannot meet (x_j >= 1e4 against a.x <= b with a >= 1, or sum x <= -5), and a
    # column that only loosens the rows and pays: the first candidate the oracle ends as expected is used
    rows = [np.concatenate([np.eye(n)[j], [1.0, 1e4]]) for j in range(8)] + [np.concatenate([np.ones(n), [0.0, -5.0]])]
    cols = [np.concatenate([np.where(rel == 2, 0.0, -1.0), [10.0]])]
    cols += [np.concatenate([-np.eye(m)[i] * (rel[i] != 2), [10.0]]) for i in range(8)]
    for kind, cand, expect in ((ROW, rows, F.INFEASIBLE), (COL, cols, F.UNBOUNDED)):
        hit = [p for p in cand if oracle(ro, kind, base, p, m, n, rel)["status"][0] == expect]
        assert hit, (kind, expect)
        cases.append((kind, hit[0], {}, expect))
    for kind in (RHS, COST, ROW, COL):
        cases.append((kind, np.zeros(lpx.reopt_payload_stride(kind, m, n)), {}, F.OPTIMAL))
    limited = 0
    for j in range(n):
        dc = np.zeros(n)
        dc[j] = 50.0 * (abs(c[j]) + 1)
        want = oracle(ro, COST, base, dc, m, n, rel, 0, max_iterations=1)
        if want["status"][0] == F.S_ITER_LIMIT:
            cases.append((COST, dc, dict(max_iterations=1), F.S_ITER_LIMIT))
            limited += 1
            if limited == 3:
                break
    assert limited > 0
    for kind, pay, opts, expect in cases:
        want = oracle(ro, kind, base, pay, m, n, rel, 0, opts.get("max_iterations", 10000))
        assert want["status"][0] == expect, (kind, expect)
        q = s.reoptimize(kind, pay, **opts)
        got = run_query(q)
        check_one(got, want, 0, f"outcome kind {kind} expect {expect}")
        if expect == F.OPTIMAL and not pay.any():
            assert got["n_pivots"] == 0
            T = got["tableau"]
            if kind in (RHS, COST):
                assert_bits_equal(T, base["tableau"], f"zero payload kind {kind}")
            else:
                assert T.shape == (base["tableau"].shape[0] + (kind == ROW), base["tableau"].shape[1] + 1)
        q.close()


def test_base_isolation(lpx, ro, small_base):
    A, b, c, rel, s, tot = small_base
    m, n = A.shape
    base = base_state(s)
    piv0 = s.pivots(tot)
    rng = np.random.default_rng(3)
    rep = sens_dict(s.sensitivity()["report"], m, n)
    pays = [(kind, np.array(payloads(kind, rng, A, b, c, rel, 0, base, rep, 1))[0]) for kind in (RHS, ROW, COL)]
    qs = [s.reoptimize(kind, pay) for kind, pay in pays]
    states = [[F.RUNNING, 0] for _ in qs]
    for rnd in range(200):
        for k in (rnd % 3, (rnd + 2) % 3, (rnd + 1) % 3):
            if states[k][0] == F.RUNNING:
                states[k] = list(qs[k].step(1 + rnd % 4))
        if all(st != F.RUNNING for st, _ in states):
            break
    outs = []
    for q in qs:
        basis, x, z = q.solution()
        outs.append(dict(status=q.sync()[0], n_pivots=q.sync()[1], pivots=q.pivots(CAP), basis=basis, x=x, z=z,
                         tableau=q.tableau()))
    for k in (1, 2, 0):
        qs[k].close()
    for (kind, pay), got in zip(pays, outs):
        check_one(got, oracle(ro, kind, base, pay, m, n, rel), 0, f"interleaved kind {kind}")
    assert s.sync() == (F.OPTIMAL, tot)
    assert np.array_equal(s.pivots(tot), piv0)
    after = base_state(s)
    assert np.array_equal(after["basis"], base["basis"])
    assert_bits_equal(after["x"], base["x"], "base x")
    assert_bits_equal(after["tableau"], base["tableau"], "base tableau")
    kind, pay = pays[0]
    again = s.reoptimize(kind, pay)
    check_one(run_query(again), oracle(ro, kind, base, pay, m, n, rel), 0, "re-query")
    again.close()


def test_refusals(lpx):
    A, b, c = workloads.lp_integer(64, 128, 2)
    pay = np.zeros(64)
    running = lpx.Session(A, b, c)
    st, _ = running.step(1)
    assert st == F.RUNNING
    with pytest.raises(F.LpxError, match="not LPX_OPTIMAL"):
        running.reoptimize(RHS, pay)
    st, _ = to_optimum(running)
    assert st == F.OPTIMAL
    for kind in (0, 5):
        with pytest.raises(F.LpxError):
            running.reoptimize(kind, pay)
    row = np.zeros(130)
    row[128] = 2.0
    with pytest.raises(F.LpxError, match="rel"):
        running.reoptimize(ROW, row)
    assert not F.lib().lpx_session_reoptimize(running._h, RHS, None, None)
    assert not F.lib().lpx_session_reoptimize(None, RHS, F.ptr(pay), None)
    rep = np.zeros(lpx.sensitivity_stride(65, 128))
    for kind, p in ((ROW, np.concatenate([np.ones(128), [0.0, 1e9]])), (COL, np.concatenate([np.ones(64), [1.0]]))):
        q = running.reoptimize(kind, p)
        assert F.lib().lpx_session_sensitivity(q._h, F.ptr(rep)) == F.E_BAD_ARGS
        q.close()
    running.close()
    Au = np.array([[1.0, -1.0], [-1.0, 1.0]])
    unb = lpx.Session(Au, np.array([1.0, 2.0]), np.array([1.0, 1.0]))
    st, _ = unb.step(10)
    assert st == F.UNBOUNDED
    with pytest.raises(F.LpxError, match="not LPX_OPTIMAL"):
        unb.reoptimize(COST, np.zeros(2))
    unb.close()


@pytest.mark.parametrize("sense", [0, 1])
def test_chaining_into_sensitivity(lpx, ro, sens, sense):
    A, b, c, rel = random_lp(77 + sense, m=64, n=128, sense=sense, n_eq=3)
    m, n = A.shape
    s = lpx.Session(A, b, c, rel=rel, sense=sense)
    assert to_optimum(s)[0] == F.OPTIMAL
    base = base_state(s)
    rep = sens_dict(s.sensitivity()["report"], m, n)
    rng = np.random.default_rng(5 + sense)
    checked = 0
    for kind in (RHS, COST):
        for pay in payloads(kind, rng, A, b, c, rel, sense, base, rep, 6):
            q = s.reoptimize(kind, pay)
            got = run_query(q)
            check_one(got, oracle(ro, kind, base, pay, m, n, rel, sense), 0, f"chained kind {kind}")
            if got["status"] != F.OPTIMAL:
                q.close()
                continue
            b2, c2 = (b + pay, c) if kind == RHS else (b, c + pay)
            want = sens.sensitivity(b2, c2, 0, got["basis"], got["tableau"], rel, sense)
            assert_bits_equal(q.sensitivity()["report"], want, f"chained report kind {kind}")
            checked += 1
            q.close()
    assert checked >= 4
    s.close()


def test_c3_full_size(lpx, ro):
    """One C3 base (4096 x 8192) at OPTIMAL and one short query of each kind, bit for bit against the oracle."""
    A, b, c = workloads.large_c3()
    m, n = A.shape
    s = lpx.Session(A, b, c)
    st, tot = to_optimum(s)
    assert st == F.OPTIMAL
    base = base_state(s)
    rep = sens_dict(s.sensitivity()["report"], m, n)
    T = base["tableau"]
    # RHS: the binding constraint with the narrowest finite upper range, moved just past it
    hi_gap = np.where((rep["shadow"] > 0) & np.isfinite(rep["rhs_hi"]), rep["rhs_hi"] - b, np.inf)
    i = int(np.argmin(hi_gap))
    d = np.zeros(m)
    d[i] = hi_gap[i] * 1.001 + 1e-3
    # COST: a non-basic column made just attractive enough to enter
    nb = np.setdiff1d(np.arange(n), base["basis"])
    j = int(nb[np.argmin(rep["reduced"][nb] + 1e9 * (rep["reduced"][nb] <= 1e-6))])
    dc = np.zeros(n)
    dc[j] = rep["reduced"][j] * 1.001 + 1e-6
    # ROW: cap one positive basic variable a little below its value
    bj = int(np.flatnonzero(base["x"] > 1e-6)[0])
    row = np.zeros(n + 2)
    row[bj] = 1.0
    row[n + 1] = float(np.round(base["x"][bj] * 0.99, 6))
    # COL: a new activity using three binding rows, priced just above what they are worth
    rows3 = np.argsort(-rep["shadow"])[:3]
    col = np.zeros(m + 1)
    col[rows3] = 1.0
    col[m] = float(rep["shadow"][rows3].sum()) * 1.01 + 1e-6
    for kind, pay in ((RHS, d), (COST, dc), (ROW, row), (COL, col)):
        want = oracle(ro, kind, base, pay, m, n)
        q = s.reoptimize(kind, pay)
        got = run_query(q)
        print(f"C3 base ({tot} pivots), kind {kind}: status {got['status']}, {got['n_pivots']} warm pivots")
        check_one(got, want, 0, f"C3 kind {kind}")
        q.close()
        del want, got
    after = s.tableau()
    assert_bits_equal(after, T, "C3 base tableau after the queries")
    s.close()

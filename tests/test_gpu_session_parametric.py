"""GPU: parametric analysis of an optimal streaming session (lpx_session_parametric) must equal oracle/orc_param.cpp run
on the base session's tableau and basis bit for bit (end, segment and pivot counts, every segment double, the pivot
pairs, the final basis and the final working tableau), and the batched route (lpx_parametric_batched_dev) on the same
base."""
import numpy as np
import pytest

from conftest import assert_bits_equal
from test_gpu_parametric import run_dev, with_tmax
from test_parametric_cpu import directions
from test_reopt_cpu import random_lp

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

RHS, COST = 1, 2
REACHED, UNBOUNDED, INFEASIBLE, SEG_LIMIT, NO_BASE = 0, 1, 2, 3, 4
CAP = 24
FIELDS = ("end", "n_segments", "n_pivots", "seg_pivots", "basis")


@pytest.fixture(scope="module")
def pm():
    import orc_param_ffi
    orc_param_ffi.lib()
    return orc_param_ffi


def to_optimum(s):
    st, tot = F.RUNNING, 0
    while st == F.RUNNING:
        st, tot = s.step(512)
    return st, tot


def base_state(s):
    basis, _, _ = s.solution()
    return dict(basis=basis, tableau=s.tableau())


def oracle(pm, kind, base, D, tmax, m, n, rel=None, sense=0, seg_cap=CAP, status=0):
    pay = with_tmax(np.atleast_2d(D), tmax)
    return pm.parametric(kind, m, n, [status], [base["basis"]], [base["tableau"]], pay, rel, sense,
                         np.zeros(len(pay), np.int32), seg_cap)


def check(got, want, q, what):
    for k in FIELDS:
        assert np.array_equal(got[k], want[k][q]), f"{what}: {k}"
    assert_bits_equal(got["segments"], want["segments"][q], what + " segments")
    assert_bits_equal(got["tableau"], want["tableau"][q], what + " tableau")


def batched(kind, base, D, tmax, m, n, rel=None, sense=0, seg_cap=CAP):
    """The batched route on the session's tableau, uploaded as a base."""
    import torch
    dev = torch.device("cuda:0")
    bases = dict(rel=None if rel is None else torch.from_numpy(np.ascontiguousarray(rel, np.int32)).to(dev),
                 status=torch.zeros(1, dtype=torch.int32, device=dev),
                 basis=torch.from_numpy(np.ascontiguousarray(base["basis"][None], np.int32)).to(dev),
                 tableau=torch.from_numpy(np.ascontiguousarray(base["tableau"][None])).to(dev))
    pay = with_tmax(np.atleast_2d(D), tmax)
    return run_dev(kind, bases, pay, m, n, sense, np.zeros(len(pay), np.int32), seg_cap=seg_cap)


def run_all(s, pm, kind, base, D, tmax, m, n, rel=None, sense=0, seg_cap=CAP, what="", **opts):
    """Every direction through the session call, against the oracle; returns the oracle's results."""
    want = oracle(pm, kind, base, D, tmax, m, n, rel, sense, seg_cap)
    tm = np.broadcast_to(np.asarray(tmax, float), (len(D),))
    for q in range(len(D)):
        got = s.parametric(kind, D[q], tm[q], seg_cap=seg_cap, **opts)
        check(got, want, q, f"{what} kind {kind} direction {q} {opts}")
    return want


@pytest.mark.parametrize("protocol", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("sense", [0, 1])
@pytest.mark.parametrize("shape", [(64, 128), (150, 300)], ids=["64x128", "150x300"])
def test_kinds_options_and_protocols(lpx, pm, shape, sense, protocol):
    m, n = shape
    A, b, c, rel = random_lp(2000 * protocol + 10 * sense + m, m=m, n=n, sense=sense, n_eq=3)
    s = lpx.Session(A, b, c, rel=rel, sense=sense, single_cta_select=protocol)
    st, tot = to_optimum(s)
    assert st == F.OPTIMAL
    base = base_state(s)
    rng = np.random.default_rng(protocol + 7 * sense + m)
    pivoted = 0
    for kind in (RHS, COST):
        D = directions(kind, rng, m, n, 6)
        tmax = np.where(np.arange(len(D)) % 3 == 2, 4.0, np.inf)
        want = oracle(pm, kind, base, D, tmax, m, n, rel, sense)
        b_got = batched(kind, base, D, tmax, m, n, rel, sense)
        for q in range(len(D)):
            check({k: v[q] for k, v in b_got.items()}, want, q, f"batched route kind {kind} direction {q}")
        for kb in (1, 8, 16):
            for variant in (1, 3):
                for q in range(len(D)):
                    got = s.parametric(kind, D[q], tmax[q], seg_cap=CAP, kblock=kb, pass_variant=variant)
                    check(got, want, q, f"{shape} sense {sense} protocol {protocol} kind {kind} K {kb} v {variant}")
        pivoted += int((want["n_pivots"] > 0).sum())
    assert pivoted > 0
    # the base is where it was, and can still be stepped
    assert s.sync() == (F.OPTIMAL, tot)
    after = base_state(s)
    assert np.array_equal(after["basis"], base["basis"])
    assert_bits_equal(after["tableau"], base["tableau"], "base tableau after the analyses")
    assert s.step(5) == (F.OPTIMAL, tot)
    s.close()


@pytest.mark.parametrize("kind", [RHS, COST])
@pytest.mark.parametrize("sense", [0, 1])
def test_every_end(lpx, pm, kind, sense):
    A, b, c, rel = random_lp(500 + 2 * kind + sense, m=40, n=70, sense=sense, n_eq=3)
    m, n = A.shape
    rng = np.random.default_rng(60 + 2 * kind + sense)
    if kind == COST:  # a costly ray (a zero column stays zero in every tableau), so that UNBOUNDED ends occur
        A[:, n - 1] = 0.0
        c[n - 1] = -1000.0 if sense == 0 else 1000.0
    s = lpx.Session(A, b, c, rel=rel, sense=sense)
    assert to_optimum(s)[0] == F.OPTIMAL
    base = base_state(s)
    k = m if kind == RHS else n
    D = np.vstack([directions(kind, rng, m, n, 40), np.zeros(k)])
    if kind == COST:
        D[:40:7] = np.eye(n)[n - 1] * (100.0 if sense == 0 else -100.0)
    tmax = rng.choice([np.inf, 0.0, 1.5, 40.0], size=len(D))
    tmax[-1] = np.inf
    if kind == COST:
        tmax[:40:7] = np.inf
    ends = set()
    for seg_cap in (CAP, 2):
        want = run_all(s, pm, kind, base, D, tmax, m, n, rel, sense, seg_cap, "every end", kblock=4)
        reached = want["end"] == REACHED
        ends |= set(want["end"].tolist())
        ends |= {"inf"} if np.isinf(want["segments"][reached, :, 1]).any() else set()
        ends |= {"finite"} if (np.isfinite(tmax[reached]) & (tmax[reached] > 0)).any() else set()
        # the zero direction: one segment [0, theta_max] with slope +0
        assert want["n_segments"][-1] == 1 and want["end"][-1] == REACHED
        assert want["segments"][-1, 0, 3] == 0.0 and not np.signbit(want["segments"][-1, 0, 3])
    assert {REACHED, SEG_LIMIT, "inf", "finite", {RHS: INFEASIBLE, COST: UNBOUNDED}[kind]} <= ends
    s.close()
    # NO_BASE: a base stepped only part way
    part = lpx.Session(A, b, c, rel=rel, sense=sense)
    st, _ = part.step(1)
    assert st == F.RUNNING
    got = part.parametric(kind, D[0], np.inf, seg_cap=4)
    assert got["end"] == NO_BASE and got["n_segments"] == 0 and got["n_pivots"] == 0
    assert not got["segments"].any() and (got["seg_pivots"] == -1).all()
    assert not got["basis"].any() and not got["tableau"].any()
    part.close()


@pytest.mark.parametrize("kind", [RHS, COST])
@pytest.mark.parametrize("shape", [(64, 111), (64, 110), (64, 14000), (64, 30000)],
                         ids=["W%16=0", "W%16=15", "some-vectors-global", "all-row-vectors-global"])
def test_shapes_and_placement(lpx, pm, kind, shape):
    """W = n + m + 1 a multiple of 16 (the RHS leading dimension must grow for g) and one below; and widths where the
    look-ahead's row-length vectors no longer all fit in shared memory (14000: the last one placed goes to global
    memory; 30000: none of them fits)."""
    m, n = shape
    A, b, c = workloads.lp_integer(m, n, 5)
    s = lpx.Session(A, b, c)
    assert to_optimum(s)[0] == F.OPTIMAL
    base = base_state(s)
    rng = np.random.default_rng(n + kind)
    D = directions(kind, rng, m, n, 4)
    if kind == RHS:
        D[0] = -b  # towards b = 0: every breakpoint down to the origin
    want = run_all(s, pm, kind, base, D, np.inf, m, n, what=f"shape {shape}", kblock=8)
    assert (want["n_pivots"] > 0).any()
    if n <= 111:
        b_got = batched(kind, base, D, np.inf, m, n)
        for q in range(len(D)):
            check({k: v[q] for k, v in b_got.items()}, want, q, f"batched route shape {shape}")
    s.close()


def test_chaining_and_refusals(lpx, pm):
    A, b, c, rel = random_lp(91, m=64, n=128, n_eq=3)
    m, n = A.shape
    s = lpx.Session(A, b, c, rel=rel)
    assert to_optimum(s)[0] == F.OPTIMAL
    base = base_state(s)
    rng = np.random.default_rng(4)
    # RHS / COST query sessions are bases, analysed on their modified model
    for qkind, pay in ((1, np.where(rel == 2, 0.0, 3.0)), (2, np.round(rng.uniform(-2, 2, size=n), 3))):
        q = s.reoptimize(qkind, pay)
        assert to_optimum(q)[0] == F.OPTIMAL
        qbase = base_state(q)
        for kind in (RHS, COST):
            run_all(q, pm, kind, qbase, directions(kind, rng, m, n, 4), np.inf, m, n, rel, what=f"query {qkind} base")
        q.close()
    # ROW / COL query sessions and Dual Simplex sessions are refused, as is every bad argument
    row = s.reoptimize(3, np.concatenate([np.ones(n), [0.0, 1e9]]))
    col = s.reoptimize(4, np.concatenate([np.where(rel == 2, 0.0, 1.0), [1.0]]))
    dual = lpx.Session(A, b, c, rel=rel, dual=True)
    L = F.lib()
    end = np.full(1, 99, np.int32)
    d = np.append(np.zeros(m), np.inf)
    for sess, what in ((row, "added row"), (col, "added row or column"), (dual, "Dual Simplex")):
        assert L.lpx_session_parametric(sess._h, RHS, F.ptr(d), 4, None, F.ptr(end), *[None] * 7) == F.E_BAD_ARGS
        assert what in F.last_error()
    for kind, tm, seg_cap in ((RHS, np.nan, 4), (RHS, -1.0, 4), (COST, -np.inf, 4), (5, 1.0, 4), (RHS, 1.0, 0)):
        pay = np.append(np.zeros(m if kind == RHS else n), tm)
        assert L.lpx_session_parametric(s._h, kind, F.ptr(pay), seg_cap, None, F.ptr(end), *[None] * 7) == F.E_BAD_ARGS
    assert L.lpx_session_parametric(s._h, RHS, None, 4, None, F.ptr(end), *[None] * 7) == F.E_BAD_ARGS
    assert L.lpx_session_parametric(s._h, RHS, F.ptr(d), 4, None, None, *[None] * 7) == F.E_BAD_ARGS
    assert end[0] == 99
    # NULL outputs: end is still written, and the full call still gives the oracle's bits
    D = directions(RHS, rng, m, n, 2)
    want = oracle(pm, RHS, base, D, np.inf, m, n, rel)
    ns = np.zeros(1, np.int32)
    for q in range(2):
        pay = np.append(D[q], np.inf)
        assert L.lpx_session_parametric(s._h, RHS, F.ptr(pay), CAP, None, F.ptr(end), *[None] * 7) == 0
        assert end[0] == want["end"][q]
        assert L.lpx_session_parametric(s._h, RHS, F.ptr(pay), CAP, None, F.ptr(end), F.ptr(ns),
                                        *[None] * 6) == 0
        assert ns[0] == want["n_segments"][q]
        check(s.parametric(RHS, D[q], seg_cap=CAP), want, q, "after NULL outputs")
    for sess in (row, col, dual, s):
        sess.close()


def test_c3_full_size(lpx, pm):
    """One C3 base (4096 x 8192) at OPTIMAL: an RHS direction towards b = 0 and a dense integer COST direction,
    bit for bit against the oracle."""
    A, b, c = workloads.large_c3()
    m, n = A.shape
    s = lpx.Session(A, b, c)
    st, tot = to_optimum(s)
    assert st == F.OPTIMAL
    base = base_state(s)
    rng = np.random.default_rng(3)
    for kind, d in ((RHS, -b), (COST, rng.integers(-5, 6, size=n).astype(float))):
        want = oracle(pm, kind, base, d[None], np.inf, m, n, seg_cap=20)
        got = s.parametric(kind, d, seg_cap=20)
        print(f"C3 base ({tot} pivots), kind {kind}: end {got['end']}, {got['n_segments']} segments")
        check(got, want, 0, f"C3 kind {kind}")
        del want, got
    assert_bits_equal(s.tableau(), base["tableau"], "C3 base tableau after the analyses")
    s.close()

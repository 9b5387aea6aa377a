"""GPU: the two-phase session (lpx_two_phase_session_open, include/lpx.h "Two-phase Simplex") must equal
oracle/orc_twophase.cpp and lpx_two_phase_solve_batched bit for bit (status, both pivot counts, the pivot list, basis, x,
z and every tableau double) at every K, pass variant and split of the work into steps; equal lpx_session_open on
all-'<=' models with b >= 0, full C3 included; and solve the C3-sized mixed model the batched call refuses."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_bits_equal
from test_two_phase_cpu import KNOWN, highs, random_mixed

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import api, workloads

pytestmark = pytest.mark.gpu

OPTIMAL, UNBOUNDED, INFEASIBLE, ITER_LIMIT, RUNNING = 0, 1, 2, -3, F.RUNNING
LE, GE, EQ = 0, 1, 2
MAX, MIN = 0, 1
UNEVEN = (1, 5, 11, 48)


@pytest.fixture(scope="module")
def tp():
    import orc_twophase_ffi
    orc_twophase_ffi.lib()
    return orc_twophase_ffi


def check(got, want, what):
    """NaNs compare as NaNs whatever their sign and payload bits, as in test_gpu_two_phase.py; every other double bit
    for bit."""
    for k in ("status", "phase1_pivots", "n_pivots", "pivots", "basis"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k}: {got[k]} vs {want[k]}"
    for k in ("x", "z", "tableau"):
        g, w = np.asarray(got[k], np.float64), np.asarray(want[k], np.float64)
        assert np.array_equal(np.isnan(g), np.isnan(w)), f"{what} {k}: NaN positions"
        assert_bits_equal(np.where(np.isnan(g), np.nan, g), np.where(np.isnan(w), np.nan, w), f"{what} {k}")


def outputs(s, cap, status, total):
    basis, x, z = s.solution()
    _, p1 = s.two_phase_info()
    return dict(status=status, phase1_pivots=p1, n_pivots=total, pivots=s.pivots(cap), basis=basis, x=x,
                z=np.float64(z), tableau=s.tableau())


def run(A, b, c, rel, sense, K=0, variant=0, chunks=None, max_iterations=10000, cap=None):
    """One two-phase session stepped to its end.  chunks: the step sizes before the 512s (None: one large step)."""
    m, n = np.shape(A)
    cap = 4 * (m + n) if cap is None else cap
    s = api.Session(A, b, c, rel, sense, max_iterations=max_iterations, kblock=K, pass_variant=variant, two_phase=True)
    try:
        if chunks is None:
            st, tot = s.step(max_iterations + m + 1)
        else:
            st = RUNNING
            for k in chunks:
                st, tot = s.step(k)
                if st != RUNNING:
                    break
            while st == RUNNING:
                st, tot = s.step(512)
        return outputs(s, cap, st, tot)
    finally:
        s.close()


def oracle(tp, A, b, c, rel, sense, max_iterations=10000, cap=None):
    m, n = np.shape(A)
    r = tp.two_phase(A, b, c, rel, sense, max_iterations=max_iterations, pivots_cap=4 * (m + n) if cap is None else cap)
    r["z"] = np.float64(r["z"])
    return r


def models():
    """The known answers (both senses), random mixed models and a batch_mixed instance that together reach OPTIMAL,
    UNBOUNDED and INFEASIBLE."""
    out = []
    for name in sorted(KNOWN):
        A, b, c, rel, sense = KNOWN[name][:5]
        for sn in (sense, 1 - sense):
            out.append((f"{name}/{sn}", np.asarray(A, float), np.asarray(b, float), np.asarray(c, float),
                        np.asarray(rel, np.int32), sn))
    for seed in range(6):
        A, b, c, rel = random_mixed(seed, 6, 5)
        for sn in (MAX, MIN):
            out.append((f"random{seed}/{sn}", A, b, c, rel, sn))
    for sn in (MAX, MIN):
        A, b, c, rel, _ = workloads.batch_mixed(count=1, m=24, n=40, seed=3, sense=sn)
        out.append((f"mixed/{sn}", A[0], b[0], c[0], rel, sn))
    return out


# ---- 1. against the oracle, stepped -----------------------------------------------------------------------------

@pytest.mark.parametrize("variant", [1, 2, 3])
@pytest.mark.parametrize("K", [1, 2, 7, 8, 16])
def test_against_the_oracle_stepped(tp, K, variant):
    seen = set()
    for name, A, b, c, rel, sense in models():
        want = oracle(tp, A, b, c, rel, sense)
        seen.add(int(want["status"]))
        for chunks in (UNEVEN, None):
            got = run(A, b, c, rel, sense, K, variant, chunks)
            check(got, want, f"{name} K={K} variant={variant} chunks={chunks}")
    assert {OPTIMAL, UNBOUNDED, INFEASIBLE} <= seen


# ---- 2. each path -----------------------------------------------------------------------------------------------

def initial_tableau(A, b, c, rel, sense):
    """The definition's initial tableau ((m + 2) x W) in numpy, and n + s."""
    m, n = A.shape
    flip = b < 0.0
    ns = n + int((rel != EQ).sum())
    slk, art, sk, a = [-1] * m, [-1] * m, n, 0
    for i in range(m):
        rn = 1 - rel[i] if (flip[i] and rel[i] != EQ) else rel[i]
        if rel[i] != EQ:
            slk[i], sk = sk, sk + 1
        if rn != 0:
            art[i], a = ns + a, a + 1
    W = ns + a + 1
    T = np.zeros((m + 2, W))
    for i in range(m):
        T[i, :n] = -A[i] if flip[i] else A[i]
        T[i, W - 1] = -b[i] if flip[i] else b[i]
        if slk[i] >= 0:
            T[i, slk[i]] = -1.0 if art[i] >= 0 else 1.0
        if art[i] >= 0:
            T[i, art[i]] = 1.0
    T[m, :n] = -(-c if sense == MIN else c)
    for j in list(range(ns)) + [W - 1]:
        w = 0.0
        for i in range(m):
            if art[i] >= 0:
                w = w - T[i, j]
        T[m + 1, j] = w
    return T, ns


def pivot_elements(A, b, c, rel, sense, r):
    """Replays the oracle's pivots (PrimalSimplex.Pivot, rows 0..m+1 in Phase I and the drive-out, 0..m after) on
    the initial tableau in numpy; returns the pivot element of each.  The replay must reproduce the oracle's tableau."""
    m = A.shape[0]
    T, ns = initial_tableau(A, b, c, rel, sense)
    els = []
    for k, (e, l) in enumerate(r["pivots"][: r["n_pivots"]]):
        piv = T[l, e]
        els.append(piv)
        T[l] = T[l] / piv
        for i in range(m + 2 if k < r["phase1_pivots"] else m + 1):
            if i != l:
                T[i] = T[i] - T[i, e] * T[l]
    assert np.hstack([T[: m + 1, :ns], T[: m + 1, -1:]]).tobytes() == r["tableau"].tobytes()
    return els


def phase1_simplex_pivots(tp, A, b, c, rel, sense, p1):
    """Pivots of Phase I before the drive-out: the least limit k at which the drive-out still pivots past it."""
    for k in range(p1 + 1):
        if tp.two_phase(A, b, c, rel, sense, max_iterations=k)["n_pivots"] > k:
            return k
    return p1


def test_redundant_equality_keeps_its_artificial(tp):
    A, b, c, rel, sense = KNOWN["duplicated_equality"][:5]
    A, b, c, rel = np.asarray(A, float), np.asarray(b, float), np.asarray(c, float), np.asarray(rel, np.int32)
    want = oracle(tp, A, b, c, rel, sense)
    for K in (1, 16):
        got = run(A, b, c, rel, sense, K)
        check(got, want, f"K={K}")
        assert got["basis"][1] >= 3 + 1  # n + s: the artificial of row 1 stays basic


def test_drive_out_pivot_on_a_negative_element(tp):
    """A model whose drive-out pivots on a negative element, found by replaying the oracle's pivots: Phase I's own
    pivots have an element > 1e-9, so a negative element among the first phase1_pivots is a drive-out pivot."""
    for seed in range(2000):
        m, n = 2 + seed % 7, 2 + (seed // 7) % 6
        A, b, c, rel = random_mixed(seed, m, n)
        want = oracle(tp, A, b, c, rel, MAX)
        if any(e < 0 for e in pivot_elements(A, b, c, rel, MAX, want)[: want["phase1_pivots"]]):
            break
    else:
        pytest.fail("no model with a negative drive-out pivot")
    for K in (1, 8):
        for variant in (1, 3):
            check(run(A, b, c, rel, MAX, K, variant, UNEVEN), want, f"seed {seed} K={K} variant={variant}")


def three_kinds(tp):
    """A batch_mixed instance with Phase I, drive-out and Phase II pivots, 16 or fewer in all."""
    A, b, c, rel, sense = workloads.batch_mixed(count=1, m=5, n=4, seed=1, sense=MAX)
    A, b, c = A[0], b[0], c[0]
    want = oracle(tp, A, b, c, rel, sense)
    ps = phase1_simplex_pivots(tp, A, b, c, rel, sense, want["phase1_pivots"])
    assert want["status"] == OPTIMAL and 1 <= ps < want["phase1_pivots"] < want["n_pivots"] <= 16
    return A, b, c, rel, sense, want, ps


def test_all_three_kinds_inside_one_block(tp):
    A, b, c, rel, sense, want, _ = three_kinds(tp)
    for variant in (1, 2, 3):
        s = api.Session(A, b, c, rel, sense, kblock=16, pass_variant=variant, two_phase=True)
        st, tot = s.step(16)  # one look-ahead and one pass
        assert st == OPTIMAL and tot == want["n_pivots"]
        check(outputs(s, 4 * 9, st, tot), want, f"variant={variant}")
        s.close()


def test_iteration_limit_in_each_phase_and_through_the_drive_out(tp):
    A, b, c, rel, sense, full, ps = three_kinds(tp)
    p1, N = full["phase1_pivots"], full["n_pivots"]
    kinds = set()
    for it in range(N + 2):
        want = oracle(tp, A, b, c, rel, sense, max_iterations=it)
        for K in (1, 16):
            got = run(A, b, c, rel, sense, K, max_iterations=it, chunks=(1,))
            check(got, want, f"max_iterations={it} K={K}")
        if it == 0:
            assert want["status"] == ITER_LIMIT and want["n_pivots"] == 0
        if want["status"] == ITER_LIMIT:
            kinds.add("phase1" if it < ps else ("drive-out" if want["n_pivots"] > it else "phase2"))
    assert kinds == {"phase1", "drive-out", "phase2"}, kinds


def test_phase_boundary_and_steps_after_the_end(tp):
    A, b, c, rel, sense, want, _ = three_kinds(tp)
    p1 = int(want["phase1_pivots"])
    for K in (1, 4, 16):
        s = api.Session(A, b, c, rel, sense, kblock=K, two_phase=True)
        assert s.two_phase_info() == (1, 0)
        st, tot = s.step(p1)
        assert (st, tot) == (RUNNING, p1) and s.two_phase_info() == (2, p1)
        assert s.sync() == (RUNNING, p1)
        st, tot = s.step(1000)
        ref = outputs(s, 36, st, tot)
        check(ref, want, f"K={K}")
        for _ in range(2):
            assert s.step(7) == (st, tot) and s.sync() == (st, tot)
        check(outputs(s, 36, st, tot), want, f"K={K} after the end")
        s.close()


def test_infeasible_leaves_phase_one(tp):
    A, b, c, rel, sense = KNOWN["infeasible_pair"][:5]
    s = api.Session(np.asarray(A, float), np.asarray(b, float), np.asarray(c, float), rel, sense, two_phase=True)
    st, tot = s.step(100)
    assert st == INFEASIBLE and s.two_phase_info()[0] == 1
    s.close()


# ---- 3. medium shapes: oracle, the batched call, HiGHS ------------------------------------------------------------

@pytest.mark.parametrize("sense", [MAX, MIN])
@pytest.mark.parametrize("shape", [(300, 600), (512, 1024)])
def test_medium_against_oracle_batched_and_highs(lpx, tp, shape, sense):
    A, b, c, rel, _ = workloads.large_mixed(*shape, seed=11, sense=sense)
    cap, it = 4 * sum(shape), 60000  # these models take up to ~17 000 pivots
    want = oracle(tp, A, b, c, rel, sense, max_iterations=it)
    got = run(A, b, c, rel, sense, chunks=UNEVEN, max_iterations=it)
    check(got, want, f"{shape} session")
    bat = lpx.two_phase_solve_batched(A[None], b[None], c[None], rel, sense, pivots_cap=cap, max_iterations=it)
    check({k: v[0] for k, v in bat.items() if k != "total_pivots"}, want, f"{shape} batched")
    hs, hz = highs(A, b, c, rel, sense)
    assert got["status"] == hs
    if hs == OPTIMAL:
        zc = -got["z"] if sense == MIN else got["z"]  # z is the max form
        assert abs(zc - hz) <= 1e-6 * (1 + abs(hz))


# ---- 4. global-memory vectors ------------------------------------------------------------------------------------

def test_objective_row_in_global_memory(tp):
    A, b, c, rel, sense = workloads.large_mixed(48, 40000, seed=2, sense=MIN)
    assert (A.shape[1] + 48) * 8 > 227 * 1024  # the objective row alone exceeds one CTA's shared memory
    want = oracle(tp, A, b, c, rel, sense)
    for K in (1, 8):
        check(run(A, b, c, rel, sense, K, chunks=UNEVEN), want, f"K={K}")


# ---- 5. identity with the primal session ------------------------------------------------------------------------

def primal_outputs(A, b, c, sense, cap, **kw):
    s = api.Session(A, b, c, None, sense, **kw)
    st = RUNNING
    while st == RUNNING:
        st, tot = s.step(512)
    basis, x, z = s.solution()
    out = dict(status=st, n_pivots=tot, pivots=s.pivots(cap), basis=basis, x=x, z=np.float64(z), tableau=s.tableau())
    s.close()
    return out


def same_as_primal(got, want, what):
    for k in ("status", "n_pivots", "pivots", "basis"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k}"
    for k in ("x", "z", "tableau"):
        assert_bits_equal(got[k], want[k], f"{what} {k}")


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_identity_with_the_primal_session(sense):
    A, b, c = workloads.batch_c2(count=3, m=64, n=128, seed=5)
    for k in range(3):
        want = primal_outputs(A[k], b[k], c[k], sense, 800)
        got = run(A[k], b[k], c[k], None, sense, chunks=UNEVEN, cap=800)
        assert got["phase1_pivots"] == 0
        same_as_primal(got, want, f"LP {k}")


def test_identity_with_the_primal_session_on_c3():
    A, b, c = workloads.large_c3()
    m, n = A.shape
    want = primal_outputs(A, b, c, 0, 10000)
    got = run(A, b, c, None, 0, cap=10000)
    assert got["status"] == OPTIMAL and got["phase1_pivots"] == 0
    same_as_primal(got, want, "C3")


# ---- 6. the full-size mixed model -------------------------------------------------------------------------------

def test_full_size_mixed_model(lpx):
    """The pivot count of this family grows faster than m (6 000 at 300 x 600, 17 000 at 512 x 1024; the full model
    takes 54 415 Phase I and 1 080 234 Phase II pivots, about a minute, see tools/two_phase_session_probe.py), so it
    is run to a raised limit of 30 000 pivots, inside Phase I, and the status reached is asserted."""
    A, b, c, rel, sense = workloads.large_mixed(4096, 8192)
    m, n = A.shape
    with pytest.raises(F.LpxError) as e:
        lpx.two_phase_solve_batched(A[None], b[None], c[None], rel, sense, pivots_cap=1, want_tableau=False)
    assert e.value.code == F.E_CAPACITY
    ref = None
    for K, variant in ((8, 3), (1, 1), (1, 3), (8, 1), (16, 1), (16, 3)):
        got = run(A, b, c, rel, sense, K, variant, max_iterations=30000, cap=30000 + m)
        if ref is None:
            ref = got
            assert got["status"] in (OPTIMAL, ITER_LIMIT), got["status"]
            assert 0 < got["phase1_pivots"] <= got["n_pivots"]
            if got["status"] == ITER_LIMIT:
                assert got["n_pivots"] == 30000
                continue
            x = got["x"]
            ax = A @ x
            tol = 1e-6 * (1 + np.abs(b))
            assert (x >= 0).all()
            assert (ax[rel == LE] <= b[rel == LE] + tol[rel == LE]).all()
            assert (ax[rel == GE] >= b[rel == GE] - tol[rel == GE]).all()
            assert (np.abs(ax[rel == EQ] - b[rel == EQ]) <= tol[rel == EQ]).all()
            assert abs(got["z"] - (-c @ x)) <= 1e-9 * abs(got["z"])
        else:
            check(got, ref, f"K={K} variant={variant}")


# ---- 7. interface ------------------------------------------------------------------------------------------------

def test_device_pointer_open_equals_host_open(tp):
    import torch
    A, b, c, rel, sense = workloads.large_mixed(64, 96, seed=4, sense=MIN)
    m, n = A.shape
    dev = torch.device("cuda:0")
    dA, db, dc = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (A, b, c))
    torch.cuda.synchronize()
    s = api.Session(dA.data_ptr(), db.data_ptr(), dc.data_ptr(), rel=rel, sense=sense, device_ptrs=True, m=m, n=n,
                    two_phase=True)
    st = RUNNING
    while st == RUNNING:
        st, tot = s.step(512)
    got = outputs(s, 4 * (m + n), st, tot)
    s.close()
    check(got, run(A, b, c, rel, sense), "_dev")
    check(got, oracle(tp, A, b, c, rel, sense), "_dev vs oracle")


def test_session_calls_and_refusals():
    A, b, c, rel, sense = workloads.large_mixed(40, 70, seed=6, sense=MIN)
    m, n = A.shape
    s = api.Session(A, b, c, rel, sense, two_phase=True)
    assert (s.rows, s.cols) == api.two_phase_dims(m, n, rel)
    r, cc, sil = C.c_int(), C.c_int(), C.c_int(5)
    L = F.lib()
    F.check(L.lpx_session_dims(s._h, C.byref(r), C.byref(cc)))
    assert (r.value, cc.value) == (m + 1, n + int((rel != EQ).sum()) + 1)
    F.check(L.lpx_session_silent_pivots(s._h, C.byref(sil)))
    assert sil.value == 0 and s.silent == 0
    L.lpx_session_profile.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    us = (C.c_double * 3)()
    F.check(L.lpx_session_profile(s._h, 2, us))
    assert all(v > 0 for v in us)
    st, tot = s.step(5000)
    assert st == OPTIMAL and tot > 3
    full = s.pivots(tot)
    small = np.full((3, 2), -7, np.int32)
    F.check(L.lpx_session_read_pivots(s._h, F.ptr(small), 2))
    assert np.array_equal(small[:2], full[:2]) and (small[2] == -7).all()
    with pytest.raises(F.LpxError) as e:
        s.sensitivity()
    assert e.value.code == F.E_BAD_ARGS and "two-phase" in F.last_error()
    with pytest.raises(F.LpxError) as e:
        s.parametric("rhs", np.ones(m))
    assert e.value.code == F.E_BAD_ARGS and "two-phase" in F.last_error()
    with pytest.raises(F.LpxError) as e:
        s.reoptimize("rhs", np.zeros(m))
    assert "two-phase" in F.last_error()
    ph, p1 = C.c_int(), C.c_int()
    q = api.Session(A[:, :], np.abs(b), c, None, sense)  # a primal session reports phase 0
    F.check(L.lpx_session_two_phase_info(q._h, C.byref(ph), C.byref(p1)))
    assert (ph.value, p1.value) == (0, 0)
    q.close()
    s.close()

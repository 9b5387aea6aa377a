"""GPU: the two-phase sensitivity report (include/lpx.h, "Sensitivity analysis of a two-phase result") must equal
oracle/orc_twophase_sens.cpp's orc_two_phase_sensitivity bit for bit, through the batched call (the solve kernel's
epilogue), its device entry and the two-phase session's HBM kernels; the solve outputs must equal
lpx_two_phase_solve_batched's, and on all-'<=' models with b >= 0 the report must equal the Primal Simplex one."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, assert_bits_equal
from test_gpu_kernel_builds import cta_carve_total, smem_optin
from test_gpu_two_phase import random_batch
from test_two_phase_cpu import KNOWN, highs

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import api, workloads

pytestmark = pytest.mark.gpu

OPTIMAL, UNBOUNDED, INFEASIBLE, ITER_LIMIT, RUNNING = 0, 1, 2, -3, F.RUNNING
LE, GE, EQ = 0, 1, 2
MAX, MIN = 0, 1
SOLVE = ("status", "phase1_pivots", "n_pivots", "basis", "x", "z")


@pytest.fixture(scope="module")
def tp():
    import orc_twophase_sens_ffi
    orc_twophase_sens_ffi.lib()
    return orc_twophase_sens_ffi


def check(got, want, what):
    for k in ("status", "phase1_pivots", "n_pivots", "basis"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k}"
    for k in ("x", "z", "report"):
        assert_bits_equal(got[k], want[k], f"{what} {k}")


def both(lpx, tp, A, b, c, rel, sense, max_iterations=10000, **opt):
    got = lpx.two_phase_sensitivity_batched(A, b, c, rel, sense, max_iterations=max_iterations, **opt)
    want = tp.two_phase_sensitivity_batch(A, b, c, rel, sense, max_iterations=max_iterations, pivots_cap=0)
    assert got["total_pivots"] == int(want["n_pivots"].sum())
    return got, want


@pytest.mark.parametrize("name", sorted(KNOWN))
def test_known_answers(lpx, tp, name):
    A, b, c, rel, sense = KNOWN[name][:5]
    A, b, c = np.asarray(A, float), np.asarray(b, float), np.asarray(c, float)
    for sn in (sense, 1 - sense):
        got, want = both(lpx, tp, A[None], b[None], c[None], rel, sn)
        check(got, want, f"{name}/{sn}")
        one = lpx.two_phase_sensitivity(A, b, c, rel, sn)
        assert_bits_equal(one["report"], want["report"][0], name)


def test_radiation_duals(lpx):
    A, b, c, rel, sense = KNOWN["radiation"][:5]
    r = lpx.two_phase_sensitivity(A, b, c, rel, sense)
    np.testing.assert_allclose(r["shadow"], [-0.5, 1.1, 0.0], rtol=0, atol=1e-12)
    assert abs(r["slack"][2] - 0.3) <= 1e-12 and abs(float(np.dot(b, r["shadow"])) - 5.25) <= 1e-12


@pytest.mark.parametrize("sense", [MAX, MIN])
@pytest.mark.parametrize("shape", [(3, 4), (6, 5), (9, 12)])
def test_random_batches_reach_every_status(lpx, tp, sense, shape):
    m, n = shape
    seen, redundant, flipped = set(), 0, 0
    for seed in range(6):
        A, b, c, rel = random_batch(100 * m + seed, 96, m, n, dup_eq=seed % 2 == 1)
        got, want = both(lpx, tp, A, b, c, rel, sense)
        check(got, want, f"{shape} seed {seed}")
        seen |= set(got["status"].tolist())
        ok = got["status"] == OPTIMAL
        redundant += int((got["basis"][ok] >= n + int((rel != EQ).sum())).sum())
        flipped += int((b[ok] < 0).sum())
    # and one with an iteration limit in each phase
    A, b, c, rel = random_batch(7 * m, 96, m, n)
    got, want = both(lpx, tp, A, b, c, rel, sense, max_iterations=2)
    check(got, want, f"{shape} limit")
    seen |= set(got["status"].tolist())
    assert {OPTIMAL, INFEASIBLE, UNBOUNDED, ITER_LIMIT} <= seen and redundant > 0 and flipped > 0


@pytest.mark.parametrize("sense", [MIN, MAX])
def test_full_c2_sized_mixed_batch_and_unchanged_solve_outputs(lpx, tp, sense):
    A, b, c, rel, s = workloads.batch_mixed(count=4096, seed=1, sense=sense, infeasible=0.05)
    got, want = both(lpx, tp, A, b, c, rel, s)
    check(got, want, f"C2 mixed sense {sense}")
    assert {OPTIMAL, INFEASIBLE} <= set(got["status"].tolist())
    plain = lpx.two_phase_solve_batched(A, b, c, rel, s, pivots_cap=0, want_tableau=False)
    for k in SOLVE:
        assert_bits_equal(got[k], plain[k], k)
    assert got["total_pivots"] == plain["total_pivots"]


@pytest.mark.parametrize("kernel", [F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL])
@pytest.mark.parametrize("threads", [128, 256, 512])
def test_kernels_and_cta_sizes(lpx, tp, kernel, threads):
    A, b, c, rel, s = workloads.batch_mixed(count=64, m=24, n=40, seed=3, sense=MIN, infeasible=0.2)
    got, want = both(lpx, tp, A, b, c, rel, s, kernel=kernel, threads=threads)
    check(got, want, f"kernel {kernel} threads {threads}")


def test_shared_memory_edge(lpx, tp):
    """The report builds take the solve's fit decision: the widest shape that fits runs in shared memory, one more
    column is refused when shared memory is forced and runs in global memory under AUTO."""
    m = 24
    rel = np.array([GE] * 8 + [EQ] * 8 + [LE] * 8, np.int32)
    s = int((rel != EQ).sum())
    ne = 1
    while cta_carve_total(m + 2, ne + 1 + s + m + 1) <= smem_optin():
        ne += 1
    for n in (ne, ne + 1):
        A, b, c, _, _ = workloads.batch_mixed(count=8, m=m, n=n, seed=n, sense=MIN)
        for k in range(8):
            ax = A[k] @ np.where(np.arange(n) % 5 == 0, 1.0, 0.0)
            b[k] = np.where(rel == LE, ax + 2, np.where(rel == GE, ax - 2, ax))
        c = np.abs(c) + 1
        got, want = both(lpx, tp, A, b, c, rel, MIN)
        check(got, want, f"edge n {n}")
        if n == ne:
            check(lpx.two_phase_sensitivity_batched(A, b, c, rel, MIN, kernel=F.KERNEL_CTA_SMEM), want, f"smem n {n}")
        else:
            with pytest.raises(F.LpxError) as e:
                lpx.two_phase_sensitivity_batched(A, b, c, rel, MIN, kernel=F.KERNEL_CTA_SMEM)
            assert e.value.code == F.E_CAPACITY


def test_null_optional_outputs(lpx, tp):
    import ctypes as C
    A, b, c, rel, s = workloads.batch_mixed(count=32, m=16, n=24, seed=6, sense=MIN, infeasible=0.2)
    want = tp.two_phase_sensitivity_batch(A, b, c, rel, s, pivots_cap=0)
    st, rep = np.zeros(32, np.int32), np.zeros((32, 4 * 16 + 3 * 24))
    opt = F.make_options()
    A_, b_, c_ = (np.ascontiguousarray(v) for v in (A, b, c))
    F.check(F.lib().lpx_two_phase_solve_sensitivity_batched(32, 16, 24, s, F.ptr(A_), F.ptr(rel), F.ptr(b_), F.ptr(c_),
                                                            C.byref(opt), F.ptr(st), None, None, None, None, None,
                                                            F.ptr(rep), None))
    assert np.array_equal(st, want["status"])
    assert_bits_equal(rep, want["report"], "NULL outputs")


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_identity_with_the_primal_report_on_all_le(lpx, sense):
    A, b, c = workloads.batch_c2(count=256, m=64, n=128, seed=4)
    if sense == MIN:
        c = c - 5.0  # some negative costs, so Min has pivots to make
    got = lpx.two_phase_sensitivity_batched(A, b, c, None, sense)
    want = lpx.primal_solve_sensitivity_batched(A, b, c, None, sense)
    for k in ("status", "n_pivots", "basis"):
        assert np.array_equal(got[k], want[k]), k
    for k in ("x", "z", "report"):
        assert_bits_equal(got[k], want[k], k)


def test_dev_call_on_a_side_stream(lpx, tp):
    import torch
    dev = torch.device("cuda:0")
    A, b, c, rel, s = workloads.batch_mixed(count=128, m=32, n=48, seed=12, sense=MIN, infeasible=0.1)
    want = tp.two_phase_sensitivity_batch(A, b, c, rel, s, pivots_cap=0)
    count, m, n = A.shape
    stride = api.sensitivity_stride(m, n)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in dict(A=A, b=b, c=c, rel=rel).items()}
    o = dict(status=torch.full((count,), 99, dtype=torch.int32, device=dev),
             phase1_pivots=torch.full((count,), 99, dtype=torch.int32, device=dev),
             n_pivots=torch.full((count,), 99, dtype=torch.int32, device=dev),
             basis=torch.full((count, m), 7, dtype=torch.int32, device=dev),
             x=torch.full((count, n), 7.0, dtype=torch.float64, device=dev),
             z=torch.full((count,), 7.0, dtype=torch.float64, device=dev),
             report=torch.full((count, stride), 7.0, dtype=torch.float64, device=dev))
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        lpx.two_phase_sensitivity_batched_dev(count, m, n, s, t["A"].data_ptr(), t["rel"].data_ptr(), t["b"].data_ptr(),
                                              t["c"].data_ptr(), *[o[k].data_ptr() for k in SOLVE],
                                              o["report"].data_ptr(), total.data_ptr(), side.cuda_stream)
    torch.cuda.synchronize()
    check({k: v.cpu().numpy() for k, v in o.items()}, want, "dev side stream")
    assert int(total.item()) == int(want["n_pivots"].sum())
    # every optional output NULL
    st = torch.full((count,), 99, dtype=torch.int32, device=dev)
    rep = torch.full((count, stride), 7.0, dtype=torch.float64, device=dev)
    lpx.two_phase_sensitivity_batched_dev(count, m, n, s, t["A"].data_ptr(), t["rel"].data_ptr(), t["b"].data_ptr(),
                                          t["c"].data_ptr(), st.data_ptr(), None, None, None, None, None,
                                          rep.data_ptr(), None, 0)
    torch.cuda.synchronize()
    assert np.array_equal(st.cpu().numpy(), want["status"])
    assert_bits_equal(rep.cpu().numpy(), want["report"], "dev NULL outputs")


# ---- sessions ----------------------------------------------------------------------------------------------------

def session_report(A, b, c, rel, sense, K=0, chunks=None, max_iterations=60000):
    """A two-phase session stepped to its end (chunks: the step sizes first, then 512s); its status, solution and
    report."""
    m = np.shape(A)[0]
    s = api.Session(A, b, c, rel, sense, max_iterations=max_iterations, kblock=K, two_phase=True)
    try:
        if chunks is None:
            st, _ = s.step(max_iterations + m + 1)
        else:
            st = RUNNING
            for k in list(chunks) + [512] * 100000:
                st, _ = s.step(k)
                if st != RUNNING:
                    break
        basis, x, z = s.solution()
        rep = s.two_phase_sensitivity()
        again = s.two_phase_sensitivity()  # the tableau is only read
        assert_bits_equal(again["report"], rep["report"], "second call")
        return dict(status=st, basis=basis, x=x, z=np.float64(z), report=rep["report"])
    finally:
        s.close()


UNEVEN = (1, 3, 2, 7, 13, 5, 64, 1, 200)


@pytest.mark.parametrize("sense", [MAX, MIN])
@pytest.mark.parametrize("shape", [(300, 600), (512, 1024)])
def test_session_against_oracle_and_batched(lpx, tp, shape, sense):
    A, b, c, rel, _ = workloads.large_mixed(*shape, seed=11, sense=sense)
    it = 60000
    want = tp.two_phase_sensitivity(A, b, c, rel, sense, max_iterations=it, pivots_cap=0)
    bat = lpx.two_phase_sensitivity(A, b, c, rel, sense, max_iterations=it)
    assert_bits_equal(bat["report"], want["report"], f"{shape} batched")
    for K, chunks in ((1, UNEVEN), (8, None), (16, UNEVEN)):
        got = session_report(A, b, c, rel, sense, K, chunks, max_iterations=it)
        assert got["status"] == want["status"] and np.array_equal(got["basis"], want["basis"])
        assert_bits_equal(got["report"], want["report"], f"{shape} session K={K}")
    if want["status"] == OPTIMAL:
        z = -want["z"] if sense == MIN else want["z"]
        assert abs(float(np.dot(b, want["report"][:shape[0]])) - z) <= 1e-6 * (1 + abs(z))


def test_session_small_models_against_the_oracle(tp):
    for name in sorted(KNOWN):
        A, b, c, rel, sense = KNOWN[name][:5]
        A, b, c, rel = np.asarray(A, float), np.asarray(b, float), np.asarray(c, float), np.asarray(rel, np.int32)
        for sn in (sense, 1 - sense):
            want = tp.two_phase_sensitivity(A, b, c, rel, sn, pivots_cap=0)
            for K in (1, 8):
                got = session_report(A, b, c, rel, sn, K, chunks=(1,))
                assert got["status"] == want["status"], name
                assert_bits_equal(got["report"], want["report"], f"{name}/{sn} K={K}")
                if want["status"] != OPTIMAL:
                    assert np.isnan(got["report"]).all()


def test_session_refusals(lpx):
    A, b, c, rel, sense = workloads.large_mixed(40, 70, seed=6, sense=MIN)
    rep = np.zeros(api.sensitivity_stride(40, 70))
    L = F.lib()
    tps = api.Session(A, b, c, rel, sense, two_phase=True)
    try:
        tps.step(100000)
        with pytest.raises(F.LpxError) as e:  # the Primal Simplex report keeps refusing a two-phase session
            tps.sensitivity()
        assert e.value.code == F.E_BAD_ARGS
    finally:
        tps.close()
    Al, bl, cl = workloads.batch_c2(count=1, m=24, n=40, seed=2)
    for kw in (dict(), dict(dual=True)):
        s = api.Session(Al[0], bl[0], cl[0], None, MAX, **kw)
        try:
            s.step(100000)
            assert L.lpx_session_two_phase_sensitivity(s._h, F.ptr(rep)) == F.E_BAD_ARGS
            assert "two-phase" in F.last_error()
            if not kw:
                q = s.reoptimize("rhs", bl[0] + 1.0)
                try:
                    assert L.lpx_session_two_phase_sensitivity(q._h, F.ptr(rep)) == F.E_BAD_ARGS
                finally:
                    q.close()
        finally:
            s.close()


def test_session_at_a_size_the_batched_call_refuses(lpx, tp):
    A, b, c, rel, sense = workloads.large_mixed(48, 40000, seed=2, sense=MIN)
    m, n = A.shape
    with pytest.raises(F.LpxError) as e:
        lpx.two_phase_sensitivity(A, b, c, rel, sense)
    assert e.value.code == F.E_CAPACITY
    want = tp.two_phase_sensitivity(A, b, c, rel, sense, pivots_cap=0)
    got = session_report(A, b, c, rel, sense, 8)
    assert got["status"] == want["status"] == OPTIMAL
    assert_bits_equal(got["report"], want["report"], "48 x 40000 session")
    y, red = got["report"][:m], got["report"][4 * m:4 * m + n]
    # HiGHS's optimum, strong duality b.y, and y a dual-feasible certificate of it (Min: A^T y <= c, y <= 0 on '<='
    # rows, y >= 0 on '>=' rows)
    hs, hz = highs(A, b, c, rel, sense)
    assert hs == OPTIMAL
    assert abs(float(np.dot(b, y)) - hz) <= 1e-6 * (1 + abs(hz))
    assert (A.T @ y <= c + 1e-7).all() and (y[rel == LE] <= 1e-12).all() and (y[rel == GE] >= -1e-12).all()
    np.testing.assert_allclose(red, c - A.T @ y, atol=1e-6)


def test_cli_two_phase_sensitivity_block(lpx, tp, tmp_path):
    exe = os.path.join(ROOT, "linear_programming_solver_lpr381_b200", "lpr381")
    import orc_ffi
    for name in ("radiation", "duplicated_equality", "infeasible_pair"):
        A, b, c, rel, sense = KNOWN[name][:5]
        model = tmp_path / f"{name}.txt"
        model.write_text(workloads.lp_to_text(np.asarray(A, float), np.asarray(b, float), np.asarray(c, float), rel,
                                              sense))
        out = subprocess.run([exe, "--two-phase-sensitivity", str(model)], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr
        plain = subprocess.run([exe, "--two-phase", str(model)], capture_output=True, text=True, timeout=120)
        p = orc_ffi.parse_text(model.read_text())
        r = tp.two_phase_sensitivity(p["A"], p["b"], p["c"], p["rel"], p["sense"])
        m, n = len(p["b"]), len(p["c"])
        want = plain.stdout + "\nTwo-Phase Sensitivity Analysis:\n"
        if r["status"] != OPTIMAL:
            assert out.stdout.startswith(want) and len(out.stdout.splitlines()) == len(want.splitlines()) + 1
            continue

        def num(v):
            return ("-inf" if v < 0 else "inf") if np.isinf(v) else orc_ffi.fmt_custom(v)
        s = api.split_sensitivity(r["report"], m, n)
        for j in range(n):
            want += (f"x{j + 1}: reduced cost {num(s['reduced'][j])}, cost range [{num(s['cost_lo'][j])}, "
                     f"{num(s['cost_hi'][j])}]\n")
        for i in range(m):
            want += (f"Constraint {i + 1}: shadow price {num(s['shadow'][i])}, slack {num(s['slack'][i])}, "
                     f"RHS range [{num(s['rhs_lo'][i])}, {num(s['rhs_hi'][i])}]\n")
        by = 0.0
        for i in range(m):
            by += float(p["b"][i]) * float(s["shadow"][i])
        want += f"Dual objective b.y = {num(by)}\n"
        want += f"Objective as written = {num(-r['z'] if p['sense'] == MIN else r['z'])}\n"
        assert out.stdout == want, name
    model = tmp_path / "radiation.txt"
    for extra in (["--sensitivity"], ["--two-phase"], ["--parametric", "rhs 1 0 0"], ["--what-if", "rhs 1 3"],
                  ["--export"]):
        bad = subprocess.run([exe, "--two-phase-sensitivity"] + extra + [str(model)], capture_output=True, text=True,
                             timeout=120)
        assert bad.returncode == 2, extra
    bad = subprocess.run([exe, "--two-phase-sensitivity", "Primal Simplex", str(model)], capture_output=True,
                         text=True, timeout=120)
    assert bad.returncode == 2
    bad = subprocess.run([exe, "--two-phase", "--sensitivity", str(model)], capture_output=True, text=True, timeout=120)
    assert bad.returncode == 2

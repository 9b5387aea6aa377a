"""GPU: the two-phase Simplex (include/lpx.h, "Two-phase Simplex") must equal oracle/orc_twophase.cpp bit for bit:
status, both pivot counts, the pivot list, basis, x, z and every tableau double (-0.0 included), through the host-buffer
call and the device entry; and lpx_primal_solve_batched on all-'<=' batches with b >= 0."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, assert_bits_equal
from test_gpu_kernel_builds import cta_carve_total, smem_optin
from test_two_phase_cpu import KNOWN, random_mixed

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

OPTIMAL, UNBOUNDED, INFEASIBLE, ITER_LIMIT = 0, 1, 2, -3
LE, GE, EQ = 0, 1, 2
MAX, MIN = 0, 1


@pytest.fixture(scope="module")
def tp():
    import orc_twophase_ffi
    orc_twophase_ffi.lib()
    return orc_twophase_ffi


def check(got, want, what, nan_payloads=False):
    """nan_payloads: NaNs compare as NaNs, whatever their sign and payload bits (the definition does not fix them,
    and the host's and the device's invalid operations produce different ones); every other double bit for bit."""
    for k in ("status", "phase1_pivots", "n_pivots", "pivots", "basis"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k}"
    for k in ("x", "z", "tableau"):
        g, w = np.asarray(got[k], np.float64), np.asarray(want[k], np.float64)
        if nan_payloads:
            assert np.array_equal(np.isnan(g), np.isnan(w)), f"{what} {k}: NaN positions"
            g, w = np.where(np.isnan(g), np.nan, g), np.where(np.isnan(w), np.nan, w)
        assert_bits_equal(g, w, f"{what} {k}")


def solve_both(lpx, tp, A, b, c, rel, sense, cap=None, max_iterations=10000, **opt):
    got = lpx.two_phase_solve_batched(A, b, c, rel, sense, max_iterations=max_iterations, pivots_cap=cap, **opt)
    want = tp.two_phase_batch(A, b, c, rel, sense, max_iterations=max_iterations, pivots_cap=cap)
    assert got["total_pivots"] == int(want["n_pivots"].sum())
    return got, want


def random_batch(seed, count, m, n, dup_eq=False):
    """`count` LPs sharing one rel pattern, b of both signs; dup_eq: row 1 repeats row 0 as an equality (a redundant
    row whose artificial stays basic after the drive-out)."""
    rng = np.random.default_rng(seed)
    rel = rng.integers(0, 3, size=m).astype(np.int32)
    A = np.empty((count, m, n))
    b = np.empty((count, m))
    c = np.empty((count, n))
    for k in range(count):
        A[k], b[k], c[k], _ = random_mixed(seed * 1000 + k, m, n)
    if dup_eq:
        rel[0] = rel[1] = EQ
        A[:, 1], b[:, 1] = A[:, 0], b[:, 0]
    return A, b, c, rel


@pytest.mark.parametrize("name", sorted(KNOWN))
def test_known_answers(lpx, tp, name):
    A, b, c, rel, sense = KNOWN[name][:5]
    A, b, c = np.asarray(A, float), np.asarray(b, float), np.asarray(c, float)
    got, want = solve_both(lpx, tp, A[None], b[None], c[None], rel, sense)
    check(got, want, name)
    one = lpx.two_phase_solve(A, b, c, rel, sense)
    assert one["status"] == KNOWN[name][5] and np.array_equal(one["pivots"], want["pivots"][0][: want["n_pivots"][0]])


@pytest.mark.parametrize("sense", [MAX, MIN])
@pytest.mark.parametrize("shape", [(3, 4), (6, 5), (9, 12)])
def test_random_batches_reach_every_status(lpx, tp, sense, shape):
    m, n = shape
    seen, drive = set(), 0
    for seed in range(6):
        A, b, c, rel = random_batch(100 * m + seed, 96, m, n, dup_eq=seed % 2 == 1)
        got, want = solve_both(lpx, tp, A, b, c, rel, sense)
        check(got, want, f"{shape} seed {seed}")
        seen |= set(got["status"].tolist())
        s = int((rel != EQ).sum())
        drive += int((got["basis"] >= n + s).sum())  # artificials left basic in redundant rows
    assert {OPTIMAL, INFEASIBLE, UNBOUNDED} <= seen and drive > 0


@pytest.mark.parametrize("sense", [MIN, MAX])
def test_full_c2_sized_mixed_batch(lpx, tp, sense):
    A, b, c, rel, s = workloads.batch_mixed(count=4096 if sense == MIN else 512, seed=1, sense=sense, infeasible=0.05)
    got, want = solve_both(lpx, tp, A, b, c, rel, s, cap=512)
    check(got, want, f"C2 mixed sense {sense}")
    assert {OPTIMAL, INFEASIBLE} <= set(got["status"].tolist())
    assert (got["phase1_pivots"] > 0).all()


@pytest.mark.parametrize("sense", [MAX, MIN])
def test_identity_with_primal_on_all_le(lpx, sense):
    A, b, c = workloads.batch_c2(count=256, m=64, n=128, seed=4)
    if sense == MIN:
        c = c - 5.0  # some negative costs, so Min has pivots to make
    got = lpx.two_phase_solve_batched(A, b, c, None, sense, pivots_cap=0)
    want = lpx.primal_solve_batched(A, b, c, None, sense)
    for k in ("status", "n_pivots", "basis"):
        assert np.array_equal(got[k], want[k]), k
    assert not got["phase1_pivots"].any()
    for k in ("x", "z", "tableau"):
        assert_bits_equal(got[k], want[k], k)
    # the pivot list against the single-LP Primal Simplex entry point
    for k in range(4):
        one = lpx.primal_solve(A[k], b[k], c[k], None, sense)
        mine = lpx.two_phase_solve(A[k], b[k], c[k], None, sense)
        assert np.array_equal(one["pivots"], mine["pivots"])


@pytest.mark.parametrize("kernel", [F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL])
@pytest.mark.parametrize("threads", [128, 256, 512])
def test_kernels_and_cta_sizes(lpx, tp, kernel, threads):
    A, b, c, rel, s = workloads.batch_mixed(count=64, m=24, n=40, seed=3, sense=MIN, infeasible=0.2)
    got, want = solve_both(lpx, tp, A, b, c, rel, s, kernel=kernel, threads=threads)
    check(got, want, f"kernel {kernel} threads {threads}")


def edge_n(m, s):
    """The widest n whose tableau, (m + 2) x (n + s + m + 1), still fits in shared memory."""
    n = 1
    while cta_carve_total(m + 2, n + 1 + s + m + 1) <= smem_optin():
        n += 1
    return n


def test_shared_memory_edge(lpx, tp):
    m = 24
    rel = np.array([GE] * 8 + [EQ] * 8 + [LE] * 8, np.int32)
    s = int((rel != EQ).sum())
    ne = edge_n(m, s)
    for n in (ne - 1, ne, ne + 1):
        A, b, c, _, _ = workloads.batch_mixed(count=8, m=m, n=n, seed=n, sense=MIN)
        for k in range(8):
            ax = A[k] @ np.where(np.arange(n) % 5 == 0, 1.0, 0.0)
            b[k] = np.where(rel == LE, ax + 2, np.where(rel == GE, ax - 2, ax))
        c = np.abs(c) + 1
        got, want = solve_both(lpx, tp, A, b, c, rel, MIN)
        check(got, want, f"edge n {n}")
        if n <= ne:
            check(lpx.two_phase_solve_batched(A, b, c, rel, MIN, kernel=F.KERNEL_CTA_SMEM), want, f"smem n {n}")
        else:
            with pytest.raises(F.LpxError) as e:
                lpx.two_phase_solve_batched(A, b, c, rel, MIN, kernel=F.KERNEL_CTA_SMEM)
            assert e.value.code == F.E_CAPACITY


def test_iteration_limit_in_both_phases(lpx, tp):
    A, b, c, rel, s = workloads.batch_mixed(count=64, m=16, n=24, seed=8, sense=MIN)
    full = tp.two_phase_batch(A, b, c, rel, s)
    p1 = full["phase1_pivots"]
    for it in (1, int(np.median(p1)), int(p1.max()) + 2, int(full["n_pivots"].max()) - 1):
        got, want = solve_both(lpx, tp, A, b, c, rel, s, max_iterations=it)
        check(got, want, f"max_iterations {it}")
        assert (got["status"] == ITER_LIMIT).any()
    # reached in Phase I for some LPs and in Phase II for others
    got, _ = solve_both(lpx, tp, A, b, c, rel, s, max_iterations=int(np.median(p1)))
    lim = got["status"] == ITER_LIMIT
    assert (got["n_pivots"][lim] == got["phase1_pivots"][lim]).any()
    got, _ = solve_both(lpx, tp, A, b, c, rel, s, max_iterations=int(p1.max()) + 2)
    lim = got["status"] == ITER_LIMIT
    assert lim.any() and (got["n_pivots"][lim] > got["phase1_pivots"][lim]).all()


def test_small_pivot_cap_and_null_outputs(lpx, tp):
    A, b, c, rel, s = workloads.batch_mixed(count=32, m=16, n=24, seed=6, sense=MIN)
    got, want = solve_both(lpx, tp, A, b, c, rel, s, cap=5)
    check(got, want, "pivots_cap 5")
    assert (got["n_pivots"] > 5).all()
    import ctypes as C
    L = F.lib()
    st = np.zeros(32, np.int32)
    opt = F.make_options()
    A_, b_, c_ = (np.ascontiguousarray(v) for v in (A, b, c))
    F.check(L.lpx_two_phase_solve_batched(32, 16, 24, s, F.ptr(A_), F.ptr(rel), F.ptr(b_), F.ptr(c_), C.byref(opt),
                                          F.ptr(st), None, None, None, 0, None, None, None, None, None))
    assert np.array_equal(st, want["status"])


def test_inf_and_nan_entries(lpx, tp):
    A, b, c, rel = random_batch(77, 64, 5, 6)
    A[1, 0, 0] = np.inf
    A[2, 1, 1] = np.nan
    b[3, 2] = -np.inf
    b[4, 0] = np.nan
    c[5, 3] = np.nan
    c[6, 0] = -np.inf
    b[7, 1] = -0.0
    A[8, 2] = -0.0
    for sense in (MAX, MIN):
        got, want = solve_both(lpx, tp, A, b, c, rel, sense)
        check(got, want, f"inf / nan sense {sense}", nan_payloads=True)


def test_dev_call_on_a_side_stream(lpx, tp):
    import torch
    dev = torch.device("cuda:0")
    A, b, c, rel, s = workloads.batch_mixed(count=128, m=32, n=48, seed=12, sense=MIN, infeasible=0.1)
    want = tp.two_phase_batch(A, b, c, rel, s, pivots_cap=64)
    count, m, n = A.shape
    rows, cols = lpx.two_phase_dims(m, n, rel)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in dict(A=A, b=b, c=c, rel=rel).items()}
    o = dict(status=torch.full((count,), 99, dtype=torch.int32, device=dev),
             phase1_pivots=torch.full((count,), 99, dtype=torch.int32, device=dev),
             n_pivots=torch.full((count,), 99, dtype=torch.int32, device=dev),
             pivots=torch.full((count, 64, 2), 7, dtype=torch.int32, device=dev),
             basis=torch.full((count, m), 7, dtype=torch.int32, device=dev),
             x=torch.full((count, n), 7.0, dtype=torch.float64, device=dev),
             z=torch.full((count,), 7.0, dtype=torch.float64, device=dev),
             tableau=torch.full((count, rows, cols), 7.0, dtype=torch.float64, device=dev))
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        lpx.two_phase_solve_batched_dev(count, m, n, s, t["A"].data_ptr(), t["rel"].data_ptr(), t["b"].data_ptr(),
                                        t["c"].data_ptr(), o["status"].data_ptr(), o["phase1_pivots"].data_ptr(),
                                        o["n_pivots"].data_ptr(), o["pivots"].data_ptr(), 64, o["basis"].data_ptr(),
                                        o["x"].data_ptr(), o["z"].data_ptr(), o["tableau"].data_ptr(),
                                        total.data_ptr(), side.cuda_stream)
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy() for k, v in o.items()}
    check(got, want, "dev side stream")
    assert int(total.item()) == int(want["n_pivots"].sum())
    # NULL outputs except status, and rel == NULL (all LE)
    st = torch.full((count,), 99, dtype=torch.int32, device=dev)
    lpx.two_phase_solve_batched_dev(count, m, n, s, t["A"].data_ptr(), None, t["b"].data_ptr(), t["c"].data_ptr(),
                                    st.data_ptr(), None, None, None, 0, None, None, None, None, None, 0)
    torch.cuda.synchronize()
    assert np.array_equal(st.cpu().numpy(), tp.two_phase_batch(A, b, c, None, s)["status"])


def test_cli_two_phase_block(lpx, tp, tmp_path):
    exe = os.path.join(ROOT, "linear_programming_solver_lpr381_b200", "lpr381")
    A, b, c, rel, sense = KNOWN["radiation"][:5]
    model = tmp_path / "radiation.txt"
    model.write_text(workloads.lp_to_text(np.asarray(A, float), np.asarray(b, float), np.asarray(c, float), rel, sense))
    out = subprocess.run([exe, "--two-phase", str(model)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    import orc_ffi
    p = orc_ffi.parse_text(model.read_text())
    r = tp.two_phase(p["A"], p["b"], p["c"], p["rel"], p["sense"])
    names = ["x1", "x2", "s1", "s3", "a2", "a3"]
    want = "Two-Phase Simplex:\nStatus: OPTIMAL\n"
    want += f"z* = {orc_ffi.fmt_custom(r['z'])}\n"
    want += "x* = [" + ", ".join(orc_ffi.fmt_custom(v) for v in r["x"]) + "]\n"
    p1, npv = int(r["phase1_pivots"]), int(r["n_pivots"])
    for title, lo, hi in (("Phase I", 0, p1), ("Phase II", p1, npv)):
        want += f"{title}: {hi - lo} pivots\n"
        for k in range(lo, hi):
            e, l = r["pivots"][k]
            want += f"  {names[e]} enters in row {l + 1}\n"
    assert out.stdout == want
    assert "z* = -5.25\nx* = [7.5, 4.5]\n" in want
    for extra in (["--sensitivity"], ["--parametric", "rhs 1 0 0"], ["--what-if", "rhs 1 3"]):
        bad = subprocess.run([exe, "--two-phase"] + extra + [str(model)], capture_output=True, text=True, timeout=120)
        assert bad.returncode == 2

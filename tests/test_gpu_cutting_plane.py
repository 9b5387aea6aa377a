"""GPU suite for lpx_cutting_plane_batched(_dev): CuttingPlane.Solve with every round on the device, one CTA per IP,
bit for bit against the oracle's numbers-only entry (oracle/orc_cut.cpp) — every round's status and pivots, every cut,
and the final LP of the integral ends."""
import ctypes as C

import numpy as np
import pytest

import host_ffi as H
import orc_cut_ffi as cut
from conftest import assert_bits_equal, case_arrays
from cut_cases import random_ips
from test_gpu_kernel_builds import cta_carve_total, smem_optin

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

CUT_NAMES = ["cut_classic_incomplete", "cut_integral_root", "cut_from_z_row", "cut_three_vars", "cut_min_sense",
             "cut_eq_row", "cut_ge_error"]
FIELDS_I = ("end", "n_rounds", "n_cuts", "lp_status", "lp_pivots", "frac_var", "cut_row", "basis")
FIELDS_D = ("cut_a", "cut_b", "x", "z", "tableau")


def oracle_batch(A, b, c, rel, sense, max_iterations=10000):
    rs = [cut.cutting_plane(A[k], b[k], c[k], rel, sense, max_iterations=max_iterations) for k in range(len(A))]
    return {f: np.stack([np.asarray(r[f]) for r in rs]) for f in FIELDS_I + FIELDS_D}


def assert_same(got, want, fields=FIELDS_I + FIELDS_D):
    for f in fields:
        if f in FIELDS_I:
            g, w = np.asarray(got[f]), np.asarray(want[f])
            assert np.array_equal(g, w), f"{f}: first difference at {np.argwhere(g != w)[0]}"
        else:
            assert_bits_equal(np.asarray(got[f]).reshape(np.shape(want[f])), want[f], f)


def run(lpx, A, b, c, rel=None, sense=0, **kw):
    got = lpx.cutting_plane_batched(A, b, c, rel, sense, **kw)
    assert got["total_pivots"] == int(got["lp_pivots"].sum())
    return got


@pytest.mark.parametrize("name", CUT_NAMES)
def test_golden_cases(lpx, kat, name):
    case = kat["cut"][name]
    A, b, c, rel = case_arrays(case)
    got = run(lpx, A[None], b[None], c[None], rel, case["sense"])
    want = oracle_batch(A[None], b[None], c[None], rel, case["sense"])
    assert got["end"][0] == case["end"]
    assert_same(got, want)


@pytest.mark.parametrize("name", CUT_NAMES)
def test_single_ip_against_the_host_route(lpx, kat, name):
    # the host layer's CuttingPlane (one lpx_primal_solve per round, the text included): same cuts, same final LP
    case = kat["cut"][name]
    A, b, c, rel = case_arrays(case)
    got = lpx.cutting_plane(A, b, c, rel, case["sense"])
    host = H.solve_text(workloads.lp_to_text(A, b, c, rel, case["sense"]), "cutting plane")
    assert got["n_cuts"] == len(host["cuts"])
    for k, h in enumerate(host["cuts"]):
        assert_bits_equal(got["cut_a"][k], h["a"], "cut a")
        assert_bits_equal([got["cut_b"][k]], [h["b"]], "cut b")
    if got["end"] == F.CUT_INTEGER:
        assert_bits_equal(got["tableau"], host["tableau"], "final tableau")
        assert_bits_equal(got["x"], host["x"], "x")
    else:
        assert got["tableau"] is None and host["tableau"] is None


# (m, n, sense, rel, max_iterations, seed): 256 IPs each; with max_iterations 3 some instances throw the iteration
# limit in some round, next to integral roots and 50-round runs in the same launch
RANDOM = [(2, 3, 0, None, 10000, 31), (5, 6, 1, [0, 2, 0, 0, 0], 10000, 32), (8, 8, 0, None, 3, 33),
          (6, 4, 0, [0, 0, 2, 0, 0, 0], 4, 34)]


@pytest.mark.parametrize("m,n,sense,rel,max_iterations,seed", RANDOM)
def test_random_batch(lpx, m, n, sense, rel, max_iterations, seed):
    A, b, c = random_ips(256, m, n, seed)
    if sense == 1:
        c = -c  # Min of positive costs stops at x = 0
    got = run(lpx, A, b, c, rel, sense, max_iterations=max_iterations)
    want = oracle_batch(A, b, c, rel, sense, max_iterations)
    assert_same(got, want)
    ends = set(got["end"].tolist())
    assert {F.CUT_INTEGER, F.CUT_INCOMPLETE} <= ends
    assert (got["lp_status"] == F.UNBOUNDED).any()
    if max_iterations < 10:
        assert F.CUT_LP_ERROR in ends and (got["lp_status"] == F.S_ITER_LIMIT).any()
        assert len(set(got["n_rounds"].tolist())) > 2  # instances end in different rounds of one launch


@pytest.mark.parametrize("rel,negate", [([0, 1, 0], False), ([0, 0, 0], True), ([2, 0, 1], False)])
def test_lp_error_in_round_one(lpx, rel, negate):
    A, b, c = random_ips(64, 3, 4, 41)
    if negate:
        b[:, 1] = -b[:, 1]
    got = run(lpx, A, b, c, rel, 0)
    assert_same(got, oracle_batch(A, b, c, rel, 0))
    assert (got["end"] == F.CUT_LP_ERROR).all() and (got["n_rounds"] == 1).all() and (got["lp_pivots"] == 0).all()
    assert (got["lp_status"][:, 0] == (F.S_NEG_RHS if negate else F.S_GE_ROW)).all()


def test_c4_shape_fifty_rounds_in_shared_memory(lpx):
    Ak, bk, ck = zip(*[workloads.ip_c4(m=60, n=120, seed=100 + k) for k in range(32)])
    A, b, c = np.stack(Ak), np.stack(bk), np.stack(ck)
    assert cta_carve_total(60 + 50, 120 + 60 + 50) == 208912 <= smem_optin()
    got = run(lpx, A, b, c, kernel=F.KERNEL_CTA_SMEM)
    want = oracle_batch(A, b, c, None, 0)
    assert_same(got, want)
    assert (got["end"] == F.CUT_INCOMPLETE).all() and (got["n_cuts"] == 50).all()
    assert_same(run(lpx, A, b, c), want)  # AUTO takes the same path


def test_kernels_and_cta_sizes_agree(lpx):
    A, b, c = random_ips(96, 6, 7, 51)
    c = -c  # Min
    rel = [0, 2, 0, 0, 0, 0]
    want = oracle_batch(A, b, c, rel, 1, 6)
    for kernel in (F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL):
        for threads in (128, 256, 512):
            assert_same(run(lpx, A, b, c, rel, 1, max_iterations=6, kernel=kernel, threads=threads), want)
        # the global-memory build without an output tableau works in library scratch
        got = run(lpx, A, b, c, rel, 1, max_iterations=6, kernel=kernel, want_tableau=False)
        assert_same(got, want, [f for f in FIELDS_I + FIELDS_D if f != "tableau"])


def test_capacity_edge(lpx):
    # the last n whose 50-round tableau fits one CTA's shared memory for m = 40 (two '=' rows: m' = 42), and n + 1
    m, rel = 40, [2, 2] + [0] * 38
    mm = m + 2
    n = 1
    while cta_carve_total(mm + 50, n + 1 + mm + 50) <= smem_optin():
        n += 1
    for nn, fits in ((n, True), (n + 1, False)):
        Ak, bk, ck = zip(*[workloads.ip_c4(m=m, n=nn, seed=200 + k) for k in range(3)])
        A, b, c = np.stack(Ak), np.stack(bk), np.stack(ck)
        want = oracle_batch(A, b, c, rel, 0, 40)
        assert_same(run(lpx, A, b, c, rel, max_iterations=40), want)
        if fits:
            assert_same(run(lpx, A, b, c, rel, max_iterations=40, kernel=F.KERNEL_CTA_SMEM), want)
        else:
            with pytest.raises(F.LpxError) as e:
                run(lpx, A, b, c, rel, max_iterations=40, kernel=F.KERNEL_CTA_SMEM)
            assert e.value.code == F.E_CAPACITY


def test_dev_call_on_a_side_stream(lpx):
    import torch
    dev = torch.device("cuda:0")
    count, m, n, sense, rel = 128, 5, 6, 0, [0, 0, 2, 0, 0]
    A, b, c = random_ips(count, m, n, 61)
    want = oracle_batch(A, b, c, rel, sense, 5)
    max_rows, max_cols = lpx.cutting_plane_dims(m, n, rel)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in (("A", A), ("b", b), ("c", c))}
    t["rel"] = torch.tensor(rel, dtype=torch.int32, device=dev)
    shapes = dict(end=(count,), n_rounds=(count,), n_cuts=(count,), lp_status=(count, 50), lp_pivots=(count, 50),
                  frac_var=(count, 50), cut_row=(count, 50), basis=(count, max_rows - 1))
    o = {k: torch.full(s, 7, dtype=torch.int32, device=dev) for k, s in shapes.items()}
    o.update(cut_a=torch.full((count, 50, n), 7.0, dtype=torch.float64, device=dev),
             cut_b=torch.full((count, 50), 7.0, dtype=torch.float64, device=dev),
             x=torch.full((count, n), 7.0, dtype=torch.float64, device=dev),
             z=torch.full((count,), 7.0, dtype=torch.float64, device=dev),
             tableau=torch.full((count, max_rows * max_cols), 7.0, dtype=torch.float64, device=dev))
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        lpx.cutting_plane_batched_dev(count, m, n, sense, t["A"].data_ptr(), t["rel"].data_ptr(), t["b"].data_ptr(),
                                      t["c"].data_ptr(), *[o[k].data_ptr() for k in FIELDS_I[:7]],
                                      o["cut_a"].data_ptr(), o["cut_b"].data_ptr(), o["basis"].data_ptr(),
                                      o["x"].data_ptr(), o["z"].data_ptr(), o["tableau"].data_ptr(),
                                      total.data_ptr(), side.cuda_stream, max_iterations=5)
    side.synchronize()
    got = {k: v.cpu().numpy() for k, v in o.items()}
    assert_same(got, want)
    assert int(total.item()) == int(want["lp_pivots"].sum())


def test_null_outputs(lpx):
    A, b, c = random_ips(64, 4, 5, 71)
    want = oracle_batch(A, b, c, None, 0, 5)
    opt = F.make_options(5)
    for kernel in (F.KERNEL_AUTO, F.KERNEL_CTA_GLOBAL):
        opt.kernel = kernel
        end = np.zeros(64, np.int32)
        rc = F.lib().lpx_cutting_plane_batched(64, 4, 5, 0, F.ptr(A), None, F.ptr(b), F.ptr(c), C.byref(opt),
                                               F.ptr(end), *([None] * 12), None)
        F.check(rc)
        assert np.array_equal(end, want["end"])
        cut_b = np.zeros((64, 50))  # one output alone: the cut store of cut_a is library scratch
        F.check(F.lib().lpx_cutting_plane_batched(64, 4, 5, 0, F.ptr(A), None, F.ptr(b), F.ptr(c), C.byref(opt),
                                                  F.ptr(end), *([None] * 7), F.ptr(cut_b), *([None] * 4), None))
        assert_bits_equal(cut_b, want["cut_b"], "cut_b")

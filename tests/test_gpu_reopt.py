"""GPU: re-optimization (include/lpx.h, "Re-optimization") must equal oracle/orc_reopt.cpp bit for bit: status,
pivot list, basis, x, z and every tableau double, through the device entry and the host-buffer call."""
import numpy as np
import pytest

from conftest import assert_bits_equal
from test_reopt_cpu import payloads, random_lp

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

RHS, COST, ROW, COL = 1, 2, 3, 4
CAP = 48


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


def check(got, want, what):
    assert got["status"].tolist() == want["status"].tolist(), what
    assert got["n_pivots"].tolist() == want["n_pivots"].tolist(), what
    assert np.array_equal(got["pivots"], want["pivots"]), what + " pivots"
    assert np.array_equal(got["basis"], want["basis"]), what + " basis"
    assert_bits_equal(got["x"], want["x"], what + " x")
    assert_bits_equal(got["z"], want["z"], what + " z")
    assert_bits_equal(got["tableau"], want["tableau"], what + " tableau")


def device_bases(A, b, c, rel=None, sense=0, max_iterations=10000):
    """Bases on the device from lpx_primal_solve_batched_dev: dict of torch tensors."""
    import torch
    from linear_programming_solver_lpr381_b200 import api
    dev = torch.device("cuda:0")
    count, m, n = A.shape
    mm = m + (0 if rel is None else int(np.sum(rel == 2)))
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in (("A", A), ("b", b), ("c", c))}
    t["rel"] = None if rel is None else torch.from_numpy(np.ascontiguousarray(rel, np.int32)).to(dev)
    t["status"] = torch.zeros(count, dtype=torch.int32, device=dev)
    t["basis"] = torch.zeros((count, mm), dtype=torch.int32, device=dev)
    t["tableau"] = torch.zeros((count, mm + 1, n + mm + 1), dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    api.primal_solve_batched_dev(count, m, n, sense, t["A"].data_ptr(), t["rel"].data_ptr() if t["rel"] is not None
                                 else None, t["b"].data_ptr(), t["c"].data_ptr(), t["status"].data_ptr(), None,
                                 t["basis"].data_ptr(), None, None, t["tableau"].data_ptr(), None, stream,
                                 max_iterations=max_iterations)
    torch.cuda.synchronize()
    return t


def run_dev(kind, bases, payload, m, n, sense=0, src=None, **opt):
    import torch
    from linear_programming_solver_lpr381_b200 import api
    dev = torch.device("cuda:0")
    rel = bases["rel"]
    relh = None if rel is None else rel.cpu().numpy()
    rows, cols = api.reopt_dims(kind, m, n, relh)
    count = payload.shape[0]
    nx = n + 1 if kind == COL else n
    pay = torch.from_numpy(np.ascontiguousarray(payload, np.float64)).to(dev)
    srct = None if src is None else torch.from_numpy(np.ascontiguousarray(src, np.int32)).to(dev)
    o = dict(status=torch.full((count,), 99, dtype=torch.int32, device=dev),
             n_pivots=torch.full((count,), 99, dtype=torch.int32, device=dev),
             pivots=torch.full((count, CAP, 2), -1, dtype=torch.int32, device=dev),
             basis=torch.full((count, rows - 1), 7, dtype=torch.int32, device=dev),
             x=torch.full((count, nx), 7.0, dtype=torch.float64, device=dev),
             z=torch.full((count,), 7.0, dtype=torch.float64, device=dev),
             tableau=torch.full((count, rows, cols), 7.0, dtype=torch.float64, device=dev))
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    api.reoptimize_batched_dev(kind, count, m, n, sense, None if rel is None else rel.data_ptr(),
                               bases["status"].data_ptr(), bases["basis"].data_ptr(), bases["tableau"].data_ptr(),
                               None if srct is None else srct.data_ptr(), pay.data_ptr(), o["status"].data_ptr(),
                               o["n_pivots"].data_ptr(), o["pivots"].data_ptr(), CAP, o["basis"].data_ptr(),
                               o["x"].data_ptr(), o["z"].data_ptr(), o["tableau"].data_ptr(), total.data_ptr(),
                               torch.cuda.current_stream().cuda_stream, **opt)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in o.items()}
    assert int(total.item()) == int(out["n_pivots"].sum())
    return out


def run_oracle(ro, kind, bases, payload, m, n, sense=0, src=None, max_iterations=10000):
    rel = None if bases["rel"] is None else bases["rel"].cpu().numpy()
    return ro.reopt(kind, m, n, bases["status"].cpu().numpy(), bases["basis"].cpu().numpy(),
                    bases["tableau"].cpu().numpy(), payload, rel, sense, src, max_iterations, CAP)


def c2_payload(kind, rng, count, m, n, x=None):
    if kind == RHS:
        d = np.zeros((count, m))
        d[np.arange(count), rng.integers(m, size=count)] = np.round(rng.uniform(-300, 300, count), 2)
        return d
    if kind == COST:
        d = np.zeros((count, n))
        d[np.arange(count), rng.integers(n, size=count)] = np.round(rng.uniform(-9, 9, count), 2)
        return d
    if kind == ROW:
        a = np.where(rng.random((count, n)) < 0.1, rng.integers(1, 9, (count, n)), 0).astype(float)
        rel = rng.integers(2, size=count).astype(float)
        beta = np.round(rng.uniform(0.0, 1.5, count) * ((a * x).sum(1) if x is not None else 50.0), 2)
        return np.hstack([a, rel[:, None], beta[:, None]])
    a = rng.integers(0, 9, (count, m)).astype(float)
    a[rng.random((count, m)) < 0.7] = 0.0
    return np.hstack([a, rng.integers(1, 20, (count, 1)).astype(float)])


@pytest.fixture(scope="module")
def c2_bases():
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=11)
    return A, b, c, device_bases(A, b, c)


@pytest.mark.parametrize("kind", [RHS, COST, ROW, COL])
def test_c2_batch_each_kind(ro, orc, c2_bases, kind):
    A, b, c, bases = c2_bases
    ref = orc.primal_batch(A[:64], b[:64], c[:64], want_tableau=True)
    assert_bits_equal(bases["tableau"][:64].cpu().numpy(), ref["tableau"], "base tableaux")
    rng = np.random.default_rng(kind)
    pay = c2_payload(kind, rng, 4096, 64, 128)
    got = run_dev(kind, bases, pay, 64, 128)
    want = run_oracle(ro, kind, bases, pay, 64, 128)
    check(got, want, f"C2 kind {kind}")
    assert (got["n_pivots"] > 0).any()


def test_one_base_many_queries(lpx, orc, ro, sens):
    A, b, c = workloads.batch_c2(count=1, m=64, n=128, seed=3)
    A, b, c = A[0], b[0], c[0]
    base = orc.primal_solve(A, b, c)
    rep = sens.sensitivity(b, c, 0, base["basis"], base["tableau"])
    lo, hi = rep[128:192], rep[192:256]
    rng = np.random.default_rng(1)
    i = rng.integers(64, size=4096)
    span = np.where(np.isfinite(hi - lo), hi - lo, 100.0)[i]
    d = np.zeros((4096, 64))
    d[np.arange(4096), i] = np.where(np.isfinite(lo[i]), lo[i], b[i] - 100.0) - b[i] + rng.uniform(-0.5, 1.5, 4096) * span
    for kind, pay in ((RHS, d), (COST, c2_payload(COST, rng, 1024, 64, 128)), (ROW, c2_payload(ROW, rng, 1024, 64, 128,
                                                                                                 base["x"])),
                      (COL, c2_payload(COL, rng, 1024, 64, 128))):
        got = lpx.reoptimize(kind, A, b, c, pay, pivots_cap=CAP)
        want = ro.reopt(kind, 64, 128, [0], [base["basis"]], [base["tableau"]], pay, src=np.zeros(len(pay), np.int32),
                        pivots_cap=CAP)
        assert got["base_status"] == 0
        check(got, want, f"one base, kind {kind}")
        if kind == RHS:
            assert (got["n_pivots"] == 0).any() and (got["n_pivots"] > 0).any()


@pytest.mark.parametrize("sense", [0, 1])
@pytest.mark.parametrize("kind", [RHS, COST, ROW, COL])
def test_mixed_models(lpx, orc, ro, sens, kind, sense):
    """Min, EQ rows at b = 0, GE cut rows, infeasible and unbounded outcomes, through the host-buffer call."""
    rng = np.random.default_rng(7 * kind + sense)
    statuses = set()
    for seed in range(4):
        A, b, c, rel = random_lp(500 + 10 * seed + kind, sense=sense)
        m, n = A.shape
        base = orc.primal_solve(A, b, c, rel, sense)
        rep = dict(zip(("shadow", "slack", "rhs_lo", "rhs_hi", "reduced", "cost_lo", "cost_hi"),
                       np.split(sens.sensitivity(b, c, 0, base["basis"], base["tableau"], rel, sense),
                                np.cumsum([m, m, m, m, n, n]))))
        assert base["status"] == 0
        pay = payloads(kind, rng, A, b, c, rel, sense, base, rep, 40)
        got = lpx.reoptimize(kind, A, b, c, pay, rel, sense, pivots_cap=CAP)
        want = ro.reopt(kind, m, n, [0], [base["basis"]], [base["tableau"]], pay, rel, sense,
                        np.zeros(len(pay), np.int32), pivots_cap=CAP)
        check(got, want, f"kind {kind} sense {sense} seed {seed}")
        statuses |= set(got["status"].tolist())
        if kind in (COST, COL):  # a small iteration limit on the queries (the base solved in full)
            bases = device_bases(A[None], b[None], c[None], rel, sense)
            src = np.zeros(len(pay), np.int32)
            got = run_dev(kind, bases, pay, m, n, sense, src, max_iterations=1)
            check(got, run_oracle(ro, kind, bases, pay, m, n, sense, src, 1), f"kind {kind} max_iterations 1")
            statuses |= set(got["status"].tolist())
    assert 0 in statuses
    assert (2 if kind in (RHS, ROW) else 1) in statuses or kind == COST
    if kind in (COST, COL):
        assert -3 in statuses


def test_src_map_with_repeated_bases(ro):
    A, b, c, rel = random_lp(77, m=9, n=14)
    A, b, c = (np.stack([v] * 8) for v in (A, b, c))
    rng = np.random.default_rng(4)
    A = A + rng.integers(0, 3, A.shape)  # EQ rows stay at b = 0
    bases = device_bases(A, b, c, rel)
    src = rng.integers(8, size=600).astype(np.int32)
    for kind in (RHS, COST, ROW, COL):
        stride = {RHS: 9, COST: 14, ROW: 16, COL: 10}[kind]
        pay = np.round(rng.uniform(-3, 6, (600, stride)), 1)
        pay[rng.random(pay.shape) < 0.6] = 0.0
        if kind == ROW:
            pay[:, 14] = rng.integers(2, size=600)
            pay[:, 15] = np.abs(pay[:, 15]) * 5
        got = run_dev(kind, bases, pay, 9, 14, src=src)
        want = run_oracle(ro, kind, bases, pay, 9, 14, src=src)
        check(got, want, f"src map kind {kind}")


@pytest.mark.parametrize("threads", [128, 256, 512])
@pytest.mark.parametrize("kernel", [F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL])
def test_forced_kernels_and_threads(ro, c2_bases, kernel, threads):
    A, b, c, full = c2_bases
    bases = dict(full, status=full["status"][:256], basis=full["basis"][:256], tableau=full["tableau"][:256])
    rng = np.random.default_rng(threads + kernel)
    for kind in (RHS, COST, ROW, COL):
        pay = c2_payload(kind, rng, 256, 64, 128)
        got = run_dev(kind, bases, pay, 64, 128, kernel=kernel, threads=threads)
        check(got, run_oracle(ro, kind, bases, pay, 64, 128), f"kernel {kernel} threads {threads} kind {kind}")


def test_shared_memory_edge(lpx, ro):
    """m = 63, n = 372 is the last shared-memory shape (DESIGN §2): RHS / COST queries stay there, ROW / COL queries
    outgrow it and take the global-memory build under AUTO, and are refused when shared memory is forced."""
    m, n = 63, 372
    A, b, c = workloads.batch_c2(count=16, m=m, n=n, seed=9)
    bases = device_bases(A, b, c)
    rng = np.random.default_rng(5)
    for kind in (RHS, COST, ROW, COL):
        pay = c2_payload(kind, rng, 16, m, n)
        check(run_dev(kind, bases, pay, m, n), run_oracle(ro, kind, bases, pay, m, n), f"edge kind {kind}")
        if kind in (ROW, COL):
            with pytest.raises(F.LpxError) as e:
                run_dev(kind, bases, pay, m, n, kernel=F.KERNEL_CTA_SMEM)
            assert e.value.code == -8
        else:
            check(run_dev(kind, bases, pay, m, n, kernel=F.KERNEL_CTA_SMEM), run_oracle(ro, kind, bases, pay, m, n),
                  f"edge kind {kind} forced shared memory")


def test_non_optimal_bases_and_refusals(lpx, ro):
    A, b, c = workloads.batch_c2(count=32, m=12, n=20, seed=6)
    bases = device_bases(A, b, c, max_iterations=6)
    st = bases["status"].cpu().numpy()
    assert (st == -3).any() and (st == 0).any()
    rng = np.random.default_rng(2)
    for kind in (RHS, COST, ROW, COL):
        pay = c2_payload(kind, rng, 32, 12, 20)
        got = run_dev(kind, bases, pay, 12, 20)
        check(got, run_oracle(ro, kind, bases, pay, 12, 20), f"non-optimal kind {kind}")
        assert (got["status"][st == -3] == -3).all() and (got["n_pivots"][st == -3] == 0).all()
    pay = c2_payload(RHS, rng, 32, 12, 20)
    for kernel in (F.KERNEL_STREAM, F.KERNEL_CTA_REG, F.KERNEL_CTA_CLUSTER):
        with pytest.raises(F.LpxError) as e:
            run_dev(RHS, bases, pay, 12, 20, kernel=kernel)
        assert e.value.code == -4
    for kind in (0, 5):
        with pytest.raises(F.LpxError) as e:
            run_dev(kind, bases, pay, 12, 20)
        assert e.value.code == -4
    bad = c2_payload(ROW, rng, 32, 12, 20)
    bad[5, 20] = 2.0
    with pytest.raises(F.LpxError) as e:
        run_dev(ROW, bases, bad, 12, 20)
    assert e.value.code == -4
    with pytest.raises(F.LpxError) as e:
        lpx.reoptimize(ROW, A[0], b[0], c[0], bad)
    assert e.value.code == -4
    got = lpx.reoptimize(RHS, A[0], b[0], c[0], pay, max_iterations=1)
    assert got["base_status"] == -3 and (got["status"] == -3).all() and not got["tableau"].any()


def test_chaining_into_sensitivity(lpx, ro, sens, c2_bases):
    """RHS / COST result tableaux are final Primal-Simplex-shaped tableaux: their sensitivity report, with the
    modified b / c, equals the oracle's report of the oracle's result."""
    import torch
    A, b, c, bases = c2_bases
    rng = np.random.default_rng(8)
    for kind in (RHS, COST):
        pay = c2_payload(kind, rng, 4096, 64, 128)
        got = run_dev(kind, bases, pay, 64, 128)
        want = run_oracle(ro, kind, bases, pay, 64, 128)
        b2, c2 = (b + pay, c) if kind == RHS else (b, c + pay)
        dev = torch.device("cuda:0")
        tb, tc = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (b2, c2))
        tst, tbas, tT = (torch.from_numpy(np.ascontiguousarray(got[k])).to(dev) for k in ("status", "basis", "tableau"))
        rep = torch.zeros((4096, lpx.sensitivity_stride(64, 128)), dtype=torch.float64, device=dev)
        lpx.sensitivity_batched_dev(4096, 64, 128, 0, None, tb.data_ptr(), tc.data_ptr(), tst.data_ptr(),
                                    tbas.data_ptr(), tT.data_ptr(), rep.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        wrep = sens.sensitivity(b2, c2, want["status"], want["basis"], want["tableau"])
        assert_bits_equal(rep.cpu().numpy(), wrep, f"chained report kind {kind}")


def test_cli_what_if_block(lpx, orc, ro, tmp_path):
    import os
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "linear_programming_solver_lpr381_b200", "lpr381")
    model = tmp_path / "wyndor.txt"
    model.write_text(workloads.WYNDOR_TEXT)
    specs = [("rhs 3 30", RHS, [0, 0, 12]), ("cost 1 8", COST, [5, 0]), ("row 1x1 + 1x2 <= 7", ROW, [1, 1, 0, 7]),
             ("row 1x1 + 0x2 >= 5", ROW, [1, 0, 1, 5]), ("col 4 0 0 1", COL, [0, 0, 1, 4]), ("rhs 3 20", RHS, [0, 0, 2])]
    args = [exe]
    for s, _, _ in specs:
        args += ["--what-if", s]
    out = subprocess.run(args + ["Primal Simplex", str(model)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    base = orc.primal_solve(p["A"], p["b"], p["c"], p["rel"], p["sense"])
    want = "What-if:\n"
    for s, kind, pay in specs:
        r = ro.reopt(kind, 3, 2, [0], [base["basis"]], [base["tableau"]], [pay], p["rel"], p["sense"], [0])
        st = int(r["status"][0])
        want += f"{s}: {dict([(0, 'OPTIMAL'), (1, 'UNBOUNDED'), (2, 'INFEASIBLE')])[st]}, {r['n_pivots'][0]} pivots"
        if st == 0:
            want += f", z {orc.fmt_custom(r['z'][0])}, x ({', '.join(orc.fmt_custom(v) for v in r['x'][0])})"
        want += "\n"
    assert "Final Report:" in out.stdout and out.stdout.endswith("\n\n" + want)
    assert "rhs 3 30: OPTIMAL, 1 pivots, z 42, x (4, 6)\n" in want
    ge = tmp_path / "ge.txt"
    ge.write_text("Max: 3x1 + 5x2\n1x1 + 0x2 >= 4\n0x1 + 2x2 <= 12\n")
    out = subprocess.run([exe, "--what-if", "rhs 2 10", "Primal Simplex", str(ge)], capture_output=True, text=True,
                         timeout=120)
    assert out.stdout == "What-if:\n" + F.status_message(F.S_GE_ROW) + "\n"

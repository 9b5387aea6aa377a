"""GPU: parametric analysis (include/lpx.h, "Parametric analysis") must equal oracle/orc_param.cpp bit for bit: end,
segment and pivot counts, every segment double, the segments' pivots, the final basis and the final working tableau,
through the device entry and the host-buffer call."""
import numpy as np
import pytest

from conftest import assert_bits_equal, case_arrays
from test_gpu_reopt import device_bases
from test_parametric_cpu import directions
from test_reopt_cpu import random_lp

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

RHS, COST = 1, 2
REACHED, UNBOUNDED, INFEASIBLE, SEG_LIMIT, NO_BASE = 0, 1, 2, 3, 4
CAP = 24
FIELDS = ("end", "n_segments", "n_pivots", "segments", "seg_pivots", "basis", "tableau")


@pytest.fixture(scope="module")
def pm():
    import orc_param_ffi
    orc_param_ffi.lib()
    return orc_param_ffi


def check(got, want, what):
    for k in ("end", "n_segments", "n_pivots", "seg_pivots", "basis"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k}"
    assert_bits_equal(got["segments"], want["segments"], what + " segments")
    assert_bits_equal(got["tableau"], want["tableau"], what + " tableau")


def run_dev(kind, bases, payload, m, n, sense=0, src=None, seg_cap=CAP, nulls=(), stream=None, **opt):
    import torch
    from linear_programming_solver_lpr381_b200 import api
    dev = torch.device("cuda:0")
    rel = bases["rel"]
    rows, cols = api.parametric_dims(kind, m, n, None if rel is None else rel.cpu().numpy())
    count = payload.shape[0]
    mm = bases["basis"].shape[1]
    pay = torch.from_numpy(np.ascontiguousarray(payload, np.float64)).to(dev)
    srct = None if src is None else torch.from_numpy(np.ascontiguousarray(src, np.int32)).to(dev)
    o = dict(end=torch.full((count,), 99, dtype=torch.int32, device=dev),
             n_segments=torch.full((count,), 99, dtype=torch.int32, device=dev),
             n_pivots=torch.full((count,), 99, dtype=torch.int32, device=dev),
             segments=torch.full((count, seg_cap, 4 + 2 * n), 7.0, dtype=torch.float64, device=dev),
             seg_pivots=torch.full((count, seg_cap, 2), 7, dtype=torch.int32, device=dev),
             basis=torch.full((count, mm), 7, dtype=torch.int32, device=dev),
             tableau=torch.full((count, rows, cols), 7.0, dtype=torch.float64, device=dev))
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    ptrs = {k: (None if k in nulls else v.data_ptr()) for k, v in o.items()}
    side = stream or torch.cuda.current_stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        api.parametric_batched_dev(kind, count, m, n, sense, None if rel is None else rel.data_ptr(),
                                   bases["status"].data_ptr(), bases["basis"].data_ptr(), bases["tableau"].data_ptr(),
                                   None if srct is None else srct.data_ptr(), pay.data_ptr(), seg_cap,
                                   *[ptrs[k] for k in FIELDS], total.data_ptr(), side.cuda_stream, **opt)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in o.items()}
    if "n_pivots" not in nulls:
        assert int(total.item()) == int(out["n_pivots"].sum())
    return out


def run_oracle(pm, kind, bases, payload, m, n, sense=0, src=None, seg_cap=CAP):
    rel = None if bases["rel"] is None else bases["rel"].cpu().numpy()
    return pm.parametric(kind, m, n, bases["status"].cpu().numpy(), bases["basis"].cpu().numpy(),
                         bases["tableau"].cpu().numpy(), payload, rel, sense, src, seg_cap)


def with_tmax(D, tmax):
    return np.hstack([D, np.broadcast_to(np.asarray(tmax, float), (len(D),))[:, None]])


def test_exports(lpx):
    L = F.lib()
    for name in ("lpx_param_payload_stride", "lpx_param_segment_stride", "lpx_parametric_dims",
                 "lpx_parametric_batched_dev", "lpx_parametric"):
        assert hasattr(L, name) and name in F.EXPORTS


def test_wyndor_and_golden_cases(lpx, orc, pm, kat):
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    cases = [("wyndor", p["A"], p["b"], p["c"], p["rel"], p["sense"], 10000)]
    for name, case in sorted(kat["lp"].items()):
        A, b, c, rel = case_arrays(case)
        cases.append((name, A, b, c, rel, case["sense"], case["max_iterations"]))
    seen = 0
    for name, A, b, c, rel, sense, it in cases:
        want_base = orc.primal_solve(A, b, c, rel, sense, max_iterations=it)
        if want_base["status"] != 0:
            continue
        seen += 1
        m, n = A.shape
        for kind, k in ((RHS, m), (COST, n)):
            D = np.vstack([np.eye(k), -np.eye(k), np.ones(k), directions(kind, np.random.default_rng(seen), m, n, 4)])
            tmax = np.where(np.arange(len(D)) % 3 == 2, 5.0, np.inf)
            got = lpx.parametric(kind, A, b, c, D, tmax, rel, sense, seg_cap=CAP, max_iterations=it)
            assert got["base_status"] == 0
            want = pm.parametric(kind, m, n, [0], [want_base["basis"]], [want_base["tableau"]], with_tmax(D, tmax),
                                 rel, sense, np.zeros(len(D), np.int32), CAP)
            check(got, want, f"{name} kind {kind}")
    assert seen >= 5
    got = lpx.parametric("rhs", p["A"], p["b"], p["c"], [[0, 0, -1]], rel=p["rel"], sense=p["sense"])
    assert got["end"][0] == INFEASIBLE and got["theta_hi"][0, :2].tolist() == [6.0, 18.0]
    assert got["dz"][0, :2].tolist() == [-1.0, -2.5]


@pytest.mark.parametrize("kind", [RHS, COST])
@pytest.mark.parametrize("sense", [0, 1])
def test_random_batches_with_mixed_ends(lpx, pm, kind, sense):
    rng = np.random.default_rng(40 + 2 * kind + sense)
    ends = set()
    for seed in range(4):
        A, b, c, rel = random_lp(900 + 10 * seed + sense, m=9, n=12, sense=sense)
        m, n = A.shape
        if kind == COST:  # a costly ray, so that UNBOUNDED ends occur
            A[:, n - 1] = np.where(rel == 2, 0.0, -rng.integers(0, 3, size=m))
            c[n - 1] = -1000.0 if sense == 0 else 1000.0
        # 5 OPTIMAL bases and 1 cut off by the iteration limit
        bases = device_bases(np.stack([A] * 6), np.stack([b] * 6), np.stack([c] * 6), rel, sense,
                             max_iterations=10000)
        nob = device_bases(A[None], b[None], c[None], rel, sense, max_iterations=1)
        for key in ("status", "basis", "tableau"):
            bases[key][5] = nob[key][0]
        D = directions(kind, rng, m, n, 60)
        if kind == COST:
            D[::7] = np.eye(n)[n - 1] * (100.0 if sense == 0 else -100.0)
        tmax = rng.choice([np.inf, 0.0, 1.5, 40.0], size=len(D))
        pay = with_tmax(D, tmax)
        src = rng.integers(0, 6, size=len(D)).astype(np.int32)
        seg_cap = 2 if seed == 3 else CAP
        got = run_dev(kind, bases, pay, m, n, sense, src, seg_cap=seg_cap)
        check(got, run_oracle(pm, kind, bases, pay, m, n, sense, src, seg_cap), f"kind {kind} seed {seed}")
        ends |= set(got["end"].tolist())
        reached = got["end"] == REACHED
        ends |= {"inf"} if np.isinf(got["segments"][reached, :, 1]).any() else set()
        ends |= {"finite"} if (np.isfinite(tmax[reached]) & (tmax[reached] > 0)).any() else set()
    assert {REACHED, NO_BASE, SEG_LIMIT, "inf", "finite", {RHS: INFEASIBLE, COST: UNBOUNDED}[kind]} <= ends


@pytest.fixture(scope="module")
def c2_bases():
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=11)
    return A, b, c, device_bases(A, b, c)


@pytest.mark.parametrize("kind", [RHS, COST])
def test_c2_one_query_per_base(pm, c2_bases, kind):
    A, b, c, bases = c2_bases
    rng = np.random.default_rng(kind)
    D = directions(kind, rng, 64, 128, 4096)
    pay = with_tmax(D, np.inf)
    check(run_dev(kind, bases, pay, 64, 128), run_oracle(pm, kind, bases, pay, 64, 128), f"C2 kind {kind}")


@pytest.mark.parametrize("kind", [RHS, COST])
def test_one_base_many_queries(pm, c2_bases, kind):
    _, _, _, bases = c2_bases
    rng = np.random.default_rng(10 + kind)
    D = directions(kind, rng, 64, 128, 2048)
    pay = with_tmax(D, rng.choice([np.inf, 3.0], size=len(D)))
    src = np.full(len(D), 17, np.int32)
    check(run_dev(kind, bases, pay, 64, 128, src=src), run_oracle(pm, kind, bases, pay, 64, 128, src=src),
          f"one base kind {kind}")


@pytest.mark.parametrize("kernel", [F.KERNEL_AUTO, F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL])
@pytest.mark.parametrize("threads", [128, 256, 512])
def test_forced_kernels_and_threads(pm, c2_bases, kernel, threads):
    _, _, _, bases = c2_bases
    rng = np.random.default_rng(threads + kernel)
    for kind in (RHS, COST):
        D = directions(kind, rng, 64, 128, 256)
        pay = with_tmax(D, np.inf)
        src = rng.integers(0, 4096, size=256).astype(np.int32)
        check(run_dev(kind, bases, pay, 64, 128, src=src, kernel=kernel, threads=threads),
              run_oracle(pm, kind, bases, pay, 64, 128, src=src), f"kind {kind} kernel {kernel} threads {threads}")


def test_shared_memory_edge(lpx, pm):
    """m = 63, n = 372 is the last shared-memory shape of the base (DESIGN §2): the direction column or row makes the
    working tableau outgrow it, so AUTO takes the global-memory build and a forced shared-memory build is refused."""
    m, n = 63, 372
    A, b, c = workloads.batch_c2(count=16, m=m, n=n, seed=9)
    bases = device_bases(A, b, c)
    rng = np.random.default_rng(5)
    for kind in (RHS, COST):
        pay = with_tmax(directions(kind, rng, m, n, 16), np.inf)
        check(run_dev(kind, bases, pay, m, n), run_oracle(pm, kind, bases, pay, m, n), f"edge kind {kind}")
        with pytest.raises(F.LpxError) as e:
            run_dev(kind, bases, pay, m, n, kernel=F.KERNEL_CTA_SMEM)
        assert e.value.code == F.E_CAPACITY
    # one size down the working tableau fits again
    A, b, c = workloads.batch_c2(count=16, m=62, n=372, seed=9)
    bases = device_bases(A, b, c)
    for kind in (RHS, COST):
        pay = with_tmax(directions(kind, rng, 62, 372, 16), np.inf)
        check(run_dev(kind, bases, pay, 62, 372, kernel=F.KERNEL_CTA_SMEM), run_oracle(pm, kind, bases, pay, 62, 372),
              f"edge - 1 kind {kind}")


def test_dev_call_on_a_side_stream_with_null_outputs(pm, c2_bases):
    import torch
    _, _, _, bases = c2_bases
    rng = np.random.default_rng(77)
    pay = with_tmax(directions(RHS, rng, 64, 128, 512), 2.0)
    want = run_oracle(pm, RHS, bases, pay, 64, 128)
    got = run_dev(RHS, bases, pay, 64, 128, stream=torch.cuda.Stream())
    check(got, want, "side stream")
    got = run_dev(RHS, bases, pay, 64, 128, nulls=("n_segments", "n_pivots", "segments", "seg_pivots", "basis",
                                                   "tableau"))
    assert np.array_equal(got["end"], want["end"])
    assert (got["n_segments"] == 99).all() and (got["segments"] == 7.0).all() and (got["tableau"] == 7.0).all()


def test_inf_and_nan_directions(lpx, pm):
    A, b, c, rel = random_lp(31, m=6, n=8)
    bases = device_bases(A[None], b[None], c[None], rel)
    for kind, k in ((RHS, 6), (COST, 8)):
        D = np.zeros((4, k))
        D[0, 1], D[1, 2], D[2, 0], D[2, 3] = np.inf, np.nan, -np.inf, 1.0
        D[3, :] = np.nan
        pay = with_tmax(D, np.inf)
        src = np.zeros(4, np.int32)
        check(run_dev(kind, bases, pay, 6, 8, src=src), run_oracle(pm, kind, bases, pay, 6, 8, src=src),
              f"inf / nan kind {kind}")


def test_refusals(lpx, c2_bases):
    _, _, _, bases = c2_bases
    pay = with_tmax(np.ones((4, 64)), np.inf)
    for bad in (-1.0, np.nan, -np.inf):
        p = pay.copy()
        p[2, -1] = bad
        with pytest.raises(F.LpxError) as e:
            run_dev(RHS, bases, p, 64, 128)
        assert e.value.code == F.E_BAD_ARGS
    for kernel in (F.KERNEL_STREAM, F.KERNEL_CTA_REG, F.KERNEL_CTA_CLUSTER):
        with pytest.raises(F.LpxError) as e:
            run_dev(RHS, bases, pay, 64, 128, kernel=kernel)
        assert e.value.code == F.E_BAD_ARGS
    A, b, c = workloads.batch_c2(count=1, m=12, n=20, seed=1)
    got = lpx.parametric("cost", A[0], b[0], c[0], np.ones((3, 20)), max_iterations=1)
    assert got["base_status"] == -3 and (got["end"] == NO_BASE).all() and not got["tableau"].any()


def test_cli_parametric_block(lpx, orc, pm, tmp_path):
    import os
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "linear_programming_solver_lpr381_b200", "lpr381")
    model = tmp_path / "wyndor.txt"
    model.write_text(workloads.WYNDOR_TEXT)
    specs = [("rhs 0 0 1", RHS, [0, 0, 1], np.inf), ("rhs 0 0 -1", RHS, [0, 0, -1], np.inf),
             ("cost 1 0 to 3", COST, [1, 0], 3.0), ("cost -1 0.5", COST, [-1, 0.5], np.inf),
             ("rhs 1 1 1 to 0", RHS, [1, 1, 1], 0.0)]
    args = [exe]
    for s, _, _, _ in specs:
        args += ["--parametric", s]
    out = subprocess.run(args + ["Primal Simplex", str(model)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    base = orc.primal_solve(p["A"], p["b"], p["c"], p["rel"], p["sense"])
    names = ["x1", "x2", "c1", "c2", "c3"]
    ends = {REACHED: "theta_max reached", UNBOUNDED: "unbounded beyond the last breakpoint",
            INFEASIBLE: "infeasible beyond the last breakpoint", SEG_LIMIT: "segment limit reached"}

    def num(v):
        return ("inf" if v > 0 else "-inf") if np.isinf(v) else orc.fmt_custom(v)

    want = "Parametric:\n"
    for s, kind, d, tmax in specs:
        r = pm.parametric(kind, 3, 2, [0], [base["basis"]], [base["tableau"]], [list(d) + [tmax]], p["rel"],
                          p["sense"], [0], 256)
        want += f"{s}: {r['n_segments'][0]} segments\n"
        for k in range(r["n_segments"][0]):
            lo, hi, z0, dz = r["segments"][0, k, :4]
            zhi = z0 if dz == 0 else z0 + hi * dz
            want += f"  theta [{num(lo)}, {num(hi)}]: z {num(z0 + lo * dz)} -> {num(zhi)}, slope {num(dz)}"
            row, col = r["seg_pivots"][0, k]
            if row >= 0:
                want += f", then {names[col]} enters in row {row + 1}"
            want += "\n"
        want += f"  end: {ends[int(r['end'][0])]}\n"
    assert "Final Report:" in out.stdout and out.stdout.endswith("\n\n" + want)
    assert "rhs 0 0 -1: 2 segments\n  theta [0, 6]: z 36 -> 30, slope -1, then" in want
    bad = subprocess.run([exe, "--parametric", "rhs 1 2", "Primal Simplex", str(model)], capture_output=True,
                         text=True, timeout=120)
    assert bad.returncode == 1 and "Parametric spec incorrect: rhs 1 2" in bad.stderr

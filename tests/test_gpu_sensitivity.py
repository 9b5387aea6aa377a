"""GPU: the sensitivity report (include/lpx.h) computed next to the final tableaux must equal, bit for bit and NaN
records included, the sequential restatement oracle/orc_sensitivity.cpp applied to the oracle's tableaux."""
import os

import numpy as np
import pytest

from conftest import ROOT, assert_bits_equal, case_arrays

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sens():
    import orc_sens_ffi
    orc_sens_ffi.lib()
    return orc_sens_ffi


def oracle_batch(orc, sens, A, b, c, rel=None, sense=0, max_iterations=10000):
    """Oracle solve of every instance, then orc_sensitivity on the oracle's tableaux."""
    out = dict(status=[], n_pivots=[], basis=[], x=[], z=[], report=[])
    for k in range(A.shape[0]):
        r = orc.primal_solve(A[k], b[k], c[k], rel, sense, max_iterations=max_iterations, pivots_cap=1)
        out["status"].append(r["status"])
        out["report"].append(sens.sensitivity(b[k], c[k], r["status"], r["basis"], r["tableau"], rel, sense))
        for key in ("n_pivots", "basis", "x", "z"):
            out[key].append(r[key])
    return {k: np.array(v) for k, v in out.items()}


def check_against_oracle(got, want, what, full=True):
    assert got["status"].tolist() == want["status"].tolist(), what
    assert_bits_equal(got["report"], want["report"], what + " report")
    if full:
        ok = want["status"] == 0
        assert got["n_pivots"][ok].tolist() == want["n_pivots"][ok].tolist(), what
        assert got["basis"][ok].tolist() == want["basis"][ok].tolist(), what
        assert_bits_equal(got["x"][ok], want["x"][ok], what + " x")
        assert_bits_equal(got["z"][ok], want["z"][ok], what + " z")


def test_new_symbols_are_exported():
    L = F.lib()
    for name in ("lpx_sensitivity_stride", "lpx_sensitivity_batched_dev", "lpx_primal_solve_sensitivity_batched",
                 "lpx_session_sensitivity"):
        assert hasattr(L, name), name
        assert name in F.EXPORTS
    assert L.lpx_sensitivity_stride(64, 128) == 640


def test_kat_primal_optimal_and_wyndor(lpx, orc, sens, kat):
    seen = 0
    for name, case in sorted(kat["lp"].items()):
        A, b, c, rel = case_arrays(case)
        want = orc.primal_solve(A, b, c, rel, case["sense"], max_iterations=case["max_iterations"])
        if want["status"] != 0:
            continue
        seen += 1
        got = lpx.primal_solve_sensitivity_batched(A[None], b[None], c[None], rel, case["sense"],
                                                   max_iterations=case["max_iterations"])
        rep = sens.sensitivity(b, c, 0, want["basis"], want["tableau"], rel, case["sense"])
        assert got["status"][0] == 0, name
        assert_bits_equal(got["report"][0], rep, name)
    assert seen >= 5
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    got = lpx.primal_solve_sensitivity_batched(p["A"][None], p["b"][None], p["c"][None], p["rel"], p["sense"])
    assert got["shadow"][0].tolist() == [0.0, 1.5, 1.0]
    assert got["rhs_lo"][0].tolist() == [2.0, 6.0, 12.0] and got["rhs_hi"][0].tolist() == [np.inf, 18.0, 24.0]
    assert got["cost_lo"][0].tolist() == [0.0, 2.0] and got["cost_hi"][0].tolist() == [7.5, np.inf]


@pytest.fixture(scope="module", params=["integer", "decimal"])
def c2(request, orc, sens):
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=5, kind=request.param)
    ref = orc.primal_batch(A, b, c, threads=16, want_tableau=True)
    ref["report"] = sens.sensitivity(b, c, ref["status"], ref["basis"], ref["tableau"])
    return request.param, A, b, c, ref


@pytest.mark.parametrize("cfg", [dict(), dict(reg_variant=2), dict(kernel=F.KERNEL_CTA_SMEM),
                                 dict(kernel=F.KERNEL_CTA_GLOBAL)], ids=["default", "reg2", "smem", "global"])
def test_c2_full_batch(lpx, c2, cfg):
    kind, A, b, c, ref = c2
    got = lpx.primal_solve_sensitivity_batched(A, b, c, **cfg)
    plain = lpx.primal_solve_batched(A, b, c, want_tableau=False, **cfg)
    for key in ("status", "n_pivots", "basis"):
        assert got[key].tolist() == plain[key].tolist(), (kind, cfg, key)
    assert_bits_equal(got["x"], plain["x"], f"{kind} {cfg} x")
    assert_bits_equal(got["z"], plain["z"], f"{kind} {cfg} z")
    assert (ref["status"] == 0).all()
    check_against_oracle(got, ref, f"C2 {kind} {cfg}")


def test_dev_entry_on_torch_tensors(lpx, orc, sens):
    import torch
    A, b, c = workloads.batch_c2(count=256, m=64, n=128, seed=9)
    count, m, n = A.shape
    dev = torch.device("cuda:0")
    tA, tb, tc = (torch.from_numpy(v).to(dev) for v in (A, b, c))
    st = torch.zeros(count, dtype=torch.int32, device=dev)
    npv = torch.zeros(count, dtype=torch.int32, device=dev)
    bas = torch.zeros((count, m), dtype=torch.int32, device=dev)
    x = torch.zeros((count, n), dtype=torch.float64, device=dev)
    z = torch.zeros(count, dtype=torch.float64, device=dev)
    T = torch.zeros((count, m + 1, n + m + 1), dtype=torch.float64, device=dev)
    rep = torch.full((count, lpx.sensitivity_stride(m, n)), 7.0, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    lpx.primal_solve_batched_dev(count, m, n, 0, tA.data_ptr(), None, tb.data_ptr(), tc.data_ptr(), st.data_ptr(),
                                 npv.data_ptr(), bas.data_ptr(), x.data_ptr(), z.data_ptr(), T.data_ptr(), None, stream)
    lpx.sensitivity_batched_dev(count, m, n, 0, None, tb.data_ptr(), tc.data_ptr(), st.data_ptr(), bas.data_ptr(),
                                T.data_ptr(), rep.data_ptr(), stream)
    torch.cuda.synchronize()
    want = oracle_batch(orc, sens, A, b, c)
    got = dict(status=st.cpu().numpy(), n_pivots=npv.cpu().numpy(), basis=bas.cpu().numpy(), x=x.cpu().numpy(),
               z=z.cpu().numpy(), report=rep.cpu().numpy())
    check_against_oracle(got, want, "_dev")


def mixed_batch(seed, count, m, n, sense, eq_rows=0, unbounded_every=5):
    rng = np.random.default_rng(seed)
    A = rng.integers(-2, 8, size=(count, m, n)).astype(float)
    b = rng.integers(0, 30, size=(count, m)).astype(float)
    c = rng.integers(-3, 9, size=(count, n)).astype(float)
    rel = np.zeros(m, dtype=np.int32)
    rel[rng.choice(m, size=eq_rows, replace=False)] = 2
    b[:, rel == 2] = 0.0  # EQ rows with b = 0: degenerate, RHS ranges with +-0 ratios
    A[::unbounded_every, :, 0] = -np.abs(A[::unbounded_every, :, 0])  # a column with no positive entry
    A[::unbounded_every, rel == 2, 0] = 0.0  # (the negated copy of an EQ row would bound it)
    c[::unbounded_every, 0] = 5.0
    if sense == 1:
        c = -c  # Min: attractive columns are the negative ones, and the unbounded column stays attractive
    return A, b, c, rel


@pytest.mark.parametrize("sense", [0, 1])
@pytest.mark.parametrize("shape", [(12, 20), (30, 45), (150, 300)], ids=["12x20", "30x45", "150x300_global"])
def test_mixed_batches(lpx, orc, sens, sense, shape):
    m, n = shape
    count = 64 if m < 100 else 12
    A, b, c, rel = mixed_batch(1000 * m + sense, count, m, n, sense, eq_rows=max(1, m // 6))
    want = oracle_batch(orc, sens, A, b, c, rel, sense)
    got = lpx.primal_solve_sensitivity_batched(A, b, c, rel, sense)
    check_against_oracle(got, want, f"mixed {shape} sense={sense}")
    assert set(want["status"].tolist()) >= {0, 1}, want["status"]
    # iteration limit: the instances that need more pivots get NaN records, their neighbours stay exact
    lim = int(np.median(want["n_pivots"][want["status"] == 0]))
    want = oracle_batch(orc, sens, A, b, c, rel, sense, max_iterations=lim)
    got = lpx.primal_solve_sensitivity_batched(A, b, c, rel, sense, max_iterations=lim)
    assert (want["status"] == F.S_ITER_LIMIT).any() and (want["status"] == 0).any()
    check_against_oracle(got, want, f"mixed {shape} sense={sense} limit={lim}", full=False)


def test_ge_row_batch_gives_nan_records(lpx):
    A, b, c = workloads.batch_c2(count=8, m=6, n=9, seed=2)
    rel = np.array([0, 0, 1, 0, 0, 0], dtype=np.int32)
    got = lpx.primal_solve_sensitivity_batched(A, b, c, rel)
    assert (got["status"] == F.S_GE_ROW).all()
    assert np.isnan(got["report"]).all()


def test_tie_rule_sweep(lpx, orc, sens):
    """Entries at and just beside +-1e-9, equal ratios and b = 0 rows (ratios of +-0.0)."""
    rng = np.random.default_rng(4242)
    tiny = np.array([1e-9, -1e-9, 1.0000001e-9, -1.0000001e-9, 0.9999999e-9, 2e-9, 0.0, -0.0])
    for t in range(12):
        m, n = int(rng.integers(3, 14)), int(rng.integers(3, 18))
        count = 32
        A = rng.choice([1.0, 2.0, 4.0, 0.5, -1.0, 0.0], size=(count, m, n))
        mask = rng.random((count, m, n)) < 0.25
        A[mask] = rng.choice(tiny, size=int(mask.sum()))
        b = rng.choice([0.0, 0.0, 4.0, 8.0, 2.0], size=(count, m))
        c = rng.choice([1.0, 2.0, 4.0, 0.0, -1.0, 1e-9], size=(count, n))
        rel = rng.choice([0, 0, 0, 2], size=m).astype(np.int32)
        sense = int(rng.integers(0, 2))
        want = oracle_batch(orc, sens, A, b, c, rel, sense, max_iterations=500)
        got = lpx.primal_solve_sensitivity_batched(A, b, c, rel, sense, max_iterations=500)
        check_against_oracle(got, want, f"tie sweep {t}", full=False)


def _session_to_optimum(lpx, A, b, c, cap=10000):
    s = lpx.Session(A, b, c)
    st, tot = F.RUNNING, 0
    while st == F.RUNNING and tot < cap:
        st, tot = s.step(min(512, cap - tot))
    return s, st, tot


@pytest.mark.parametrize("shape", [(1024, 2048), (4096, 8192)], ids=["1024x2048", "C3"])
def test_session(lpx, sens, shape):
    m, n = shape
    A, b, c = workloads.large_c3(m, n) if shape == (4096, 8192) else workloads.lp_integer(m, n, 31)
    s, st, tot = _session_to_optimum(lpx, A, b, c)
    print(f"session {m}x{n}: status {st} after {tot} pivots")
    got = s.sensitivity()
    basis, _, _ = s.solution()
    want = sens.sensitivity(b, c, st, basis, s.tableau())
    assert_bits_equal(got["report"], want, f"session {m}x{n}")
    if st != F.OPTIMAL:
        assert np.isnan(got["report"]).all()
        if shape == (1024, 2048):
            pytest.fail(f"mid-size session did not reach OPTIMAL within 10000 pivots (status {st})")
    s.close()


def test_cli_sensitivity_block(lpx, orc, tmp_path):
    import subprocess
    exe = os.path.join(ROOT, "linear_programming_solver_lpr381_b200", "lpr381")
    model = tmp_path / "wyndor.txt"
    model.write_text(workloads.WYNDOR_TEXT)
    out = subprocess.run([exe, "--sensitivity", "Primal Simplex", str(model)], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 0, out.stderr
    p = orc.parse_text(workloads.WYNDOR_TEXT)
    s = lpx.primal_solve_sensitivity_batched(p["A"][None], p["b"][None], p["c"][None], p["rel"], p["sense"])

    def num(v):
        return ("-inf" if v < 0 else "inf") if np.isinf(v) else orc.fmt_custom(v)

    want = "Sensitivity Analysis:\n"
    for j in range(2):
        want += (f"x{j + 1}: reduced cost {num(s['reduced'][0][j])}, cost range [{num(s['cost_lo'][0][j])}, "
                 f"{num(s['cost_hi'][0][j])}]\n")
    for i in range(3):
        want += (f"Constraint {i + 1}: shadow price {num(s['shadow'][0][i])}, slack {num(s['slack'][0][i])}, "
                 f"RHS range [{num(s['rhs_lo'][0][i])}, {num(s['rhs_hi'][0][i])}]\n")
    assert "Final Report:" in out.stdout and out.stdout.endswith("\n\n" + want)
    assert "Constraint 2: shadow price 1.5, slack 0, RHS range [6, 18]" in want
    ge = tmp_path / "ge.txt"
    ge.write_text("Max: 3x1 + 5x2\n1x1 + 0x2 >= 4\n0x1 + 2x2 <= 12\n")
    out = subprocess.run([exe, "--sensitivity", "Primal Simplex", str(ge)], capture_output=True, text=True, timeout=120)
    assert out.stdout == "Sensitivity Analysis:\n" + F.status_message(F.S_GE_ROW) + "\n"

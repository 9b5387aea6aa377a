"""GPU: Dual Simplex on a large LP whose tableau lives in HBM (lpx_dual_session_open, lpx_dual_solve with the streaming
kernel) must equal the oracle's DualSimplex.Solve (oracle/orc_simplex.cpp dual_simplex) bit for bit: status, pivot
count, silent pivots, pivot list, basis, x, z and every tableau double, -0.0 included, under the per-pivot protocols
(1, 2) and the blocked dual look-ahead (0, 3, 4)."""
import numpy as np
import pytest

from conftest import assert_bits_equal

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

CHUNKS = [1, 5, 11, 48]
CAP = 10200


def mixed_lp(seed, m, n):
    """'<=', '>=' and '=' rows around a feasible point x0 >= 0; about 30 % of the rows have mostly negative
    coefficients, so every relation appears with b > 0 and with b < 0."""
    r = np.random.default_rng(seed)
    A = r.integers(-2, 10, size=(m, n)).astype(float)
    A[r.random(m) < 0.3] *= -1
    rel = r.choice([0, 1, 2], size=m, p=[0.5, 0.3, 0.2]).astype(np.int32)
    x0 = np.zeros(n)
    k = max(1, n // 8)
    x0[r.choice(n, size=k, replace=False)] = r.integers(1, 6, size=k)
    s = A @ x0
    slack = r.integers(0, n, size=m).astype(float)
    b = np.where(rel == 0, s + slack, np.where(rel == 1, s - slack, s))
    c = r.integers(1, 10, size=n).astype(float)
    return A, b, c, rel


def problem(name):
    kind, m, n = name.split(":")
    m, n = int(m), int(n)
    if kind == "mixed":
        return mixed_lp(7 * m + n, m, n)
    if kind == "large_dual":
        return workloads.large_dual(m, n, seed=3)[:4]
    A, b, c = workloads.lp_integer(m, n, 5)
    return A, b, c, None


_oracle_cache = {}


def oracle(orc, name, sense):
    key = (name, sense)
    if key not in _oracle_cache:
        A, b, c, rel = problem(name)
        _oracle_cache[key] = orc.dual_solve(A, b, c, rel, sense)
    return _oracle_cache[key]


def run(s, chunks=CHUNKS):
    """Step a session to a terminal status in uneven chunks (then 512s); all its outputs."""
    st, tot, k = F.RUNNING, 0, 0
    while st == F.RUNNING:
        st, tot = s.step(chunks[k] if k < len(chunks) else 512)
        k += 1
    basis, x, z = s.solution()
    return dict(status=st, n_pivots=tot, silent=s.silent, pivots=s.pivots(CAP)[: min(tot, CAP)], basis=basis, x=x, z=z,
                tableau=s.tableau())


def check(got, want, what):
    assert got["status"] == want["status"], what
    assert got["n_pivots"] == want["n_pivots"], what
    assert got["silent"] == want["silent"], what
    if want["status"] == F.S_ITER_LIMIT:
        return  # the oracle exports nothing else after the iteration-limit exception (test_iteration_limit)
    assert np.array_equal(got["pivots"], want["pivots"]), what + " pivots"
    assert np.array_equal(got["basis"], want["basis"]), what + " basis"
    assert_bits_equal(got["x"], want["x"], what + " x")
    assert_bits_equal([got["z"]], [want["z"]], what + " z")
    assert_bits_equal(got["tableau"], want["tableau"], what + " tableau")


def session(lpx, name, sense, **opts):
    A, b, c, rel = problem(name)
    return lpx.Session(A, b, c, rel=rel, sense=sense, dual=True, **opts)


# ---- 1. stepped sessions under every protocol --------------------------------------------------------------------
@pytest.mark.parametrize("protocol", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("sense", [0, 1])
@pytest.mark.parametrize("name", ["mixed:64:128", "mixed:150:300", "large_dual:96:384"])
def test_stepped_session_against_oracle(lpx, orc, name, sense, protocol):
    want = oracle(orc, name, sense)
    s = session(lpx, name, sense, single_cta_select=protocol)
    assert (s.rows, s.cols) == (want["rows"], want["cols"])
    check(run(s), want, f"{name} sense {sense} protocol {protocol}")
    s.close()


@pytest.mark.parametrize("protocol", [0, 1])
@pytest.mark.parametrize("name,sense", [("large_dual:512:1024", 1), ("mixed:300:600", 1)])
def test_larger_shapes(lpx, orc, name, sense, protocol):
    want = oracle(orc, name, sense)
    assert want["status"] in (F.OPTIMAL, F.INFEASIBLE) and want["n_pivots"] > 200
    s = session(lpx, name, sense, single_cta_select=protocol)
    check(run(s), want, f"{name} protocol {protocol}")
    s.close()


# ---- 2. each way the silent phase ends ---------------------------------------------------------------------------
def test_silent_phase_endings(lpx, orc):
    """Zero silent pivots (no entering column) is test_stepped_session_against_oracle's large_dual Min case."""
    # no leaving row: the most negative z_j (c_0 = 50, Max) belongs to a column with no entry above 1e-9 (zero in the
    # '=' rows, so their negated copies have none either).  The Dual Simplex loop then runs from a tableau that is not
    # dual feasible: with '=' rows it cycles to the 10000-pivot limit; with '<=' rows of b < 0 over a <= 0 (flipped to
    # b > 0 by the preparation) it is OPTIMAL at once.
    cases = []
    for eq in (True, False):
        r = np.random.default_rng(11)
        m, n = 40, 90
        A = r.integers(1, 10, size=(m, n)).astype(float)
        b = r.integers(n, 4 * n, size=m).astype(float)
        zero0 = np.arange(m) % 4 == 0 if eq else np.arange(m) % 8 == 0
        rel = np.where(zero0, 2, 0).astype(np.int32) if eq else np.zeros(m, np.int32)
        if not eq:
            b[zero0] = -r.integers(1, 20, size=int(zero0.sum()))
            A[zero0] *= -1
        A[:, 0] = np.where(zero0, 0.0, -r.integers(0, 3, size=m))
        c = r.integers(1, 10, size=n).astype(float)
        c[0] = 50.0
        cases.append(("no leaving row" + (" (cycles)" if eq else ""), A, b, c, rel, 0))
    # the 100-pivot guard: an all-'<=' Max LP whose Primal Simplex needs more than 100 pivots; after the guard its RHS
    # is non-negative, so the reference reports OPTIMAL at once
    Ag, bg, cg = workloads.lp_integer(1024, 2048, 5)
    cases.append(("guard", Ag, bg, cg, None, 0))
    # zero silent pivots: Min with c >= 0 starts dual feasible
    want = oracle(orc, "large_dual:96:384", 1)
    assert want["silent"] == 0 and want["n_pivots"] > 0
    for what, A, b, c, rel, sense in cases:
        w = orc.dual_solve(A, b, c, rel, sense)
        for protocol in (0, 1):
            s = lpx.Session(A, b, c, rel=rel, sense=sense, dual=True, single_cta_select=protocol)
            got = run(s)
            check(got, w, f"{what} protocol {protocol}")
            s.close()
        if what == "no leaving row (cycles)":
            assert w["silent"] == 0 and w["status"] == F.S_ITER_LIMIT and w["n_pivots"] == 10000
        elif what == "no leaving row":
            assert w["silent"] == 0 and w["status"] == F.OPTIMAL and w["tableau"][-1].min() == -50.0
        else:
            assert w["silent"] == 100 and w["n_pivots"] == 100 and w["status"] == F.OPTIMAL
            assert w["tableau"][-1, :-1].min() < -1e-9  # not optimal for the Primal Simplex: the reference's verdict


# ---- 3. INFEASIBLE and ITER_LIMIT --------------------------------------------------------------------------------
def test_infeasible_and_iteration_limit(lpx, orc):
    r = np.random.default_rng(5)
    m, n = 30, 60
    A = r.integers(1, 10, size=(m, n)).astype(float)
    b = r.integers(n, 4 * n, size=m).astype(float)
    rel = np.zeros(m, np.int32)
    rel[7] = 2
    b[7] = -1000.0  # an '=' row with a >= 0 and b < 0: its first copy leaves and has no negative entry
    c = r.integers(0, 10, size=n).astype(float)
    w = orc.dual_solve(A, b, c, rel, 1)
    assert w["status"] == F.INFEASIBLE
    for protocol in (0, 1):
        s = lpx.Session(A, b, c, rel=rel, sense=1, dual=True, single_cta_select=protocol)
        check(run(s), w, f"infeasible protocol {protocol}")
        s.close()
    # a mixed Max LP that cycles to the 10000-pivot limit (100 silent + 10000 Dual Simplex pivots).  The oracle exports
    # no pivots or tableau after the iteration-limit exception: the blocked protocols are held to the per-pivot one
    w = oracle(orc, "mixed:64:128", 0)
    assert w["status"] == F.S_ITER_LIMIT and w["n_pivots"] == 10100 and w["silent"] == 100
    ref = None
    for opts in (dict(single_cta_select=1), dict(single_cta_select=0), dict(single_cta_select=4, kblock=16)):
        s = session(lpx, "mixed:64:128", 0, max_iterations=5, **opts)  # opt.max_iterations does not apply
        got = run(s)
        s.close()
        check(got, w, f"iteration limit {opts}")
        if ref is None:
            ref = got
            continue
        assert np.array_equal(got["pivots"], ref["pivots"]) and np.array_equal(got["basis"], ref["basis"])
        assert_bits_equal(got["tableau"], ref["tableau"], f"iteration limit {opts} tableau")


# ---- 4. block sizes and pass variants ----------------------------------------------------------------------------
@pytest.mark.parametrize("kblock", [1, 2, 7, 16])
def test_block_sizes_and_pass_variants(lpx, orc, kblock):
    name = "mixed:150:300"
    want = oracle(orc, name, 1)
    assert want["n_pivots"] > 100
    for variant in (1, 2, 3):
        s = session(lpx, name, 1, single_cta_select=4, kblock=kblock, pass_variant=variant)
        check(run(s, [3, 17, 29]), want, f"K {kblock} pass variant {variant}")
        s.close()


# ---- 5. lpx_dual_solve routing -----------------------------------------------------------------------------------
def compare_solve(got, want, what):
    got = dict(got)
    check(got, want, what)


def test_dual_solve_stream_and_routing(lpx, orc):
    lib = F.lib()
    for name, sense in (("mixed:64:128", 1), ("large_dual:96:384", 1), ("large_dual:96:384", 0)):
        A, b, c, rel = problem(name)
        want = oracle(orc, name, sense)
        compare_solve(lpx.dual_solve(A, b, c, rel, sense, kernel=F.KERNEL_STREAM), want, f"{name} {sense} stream")
        for kernel in (F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL):
            try:
                got = lpx.dual_solve(A, b, c, rel, sense, kernel=kernel)
            except F.LpxError as e:
                assert e.code == F.E_CAPACITY and kernel == F.KERNEL_CTA_SMEM
                continue
            compare_solve(got, want, f"{name} {sense} kernel {kernel}")
    # past the single-solve rule (no shared-memory fit, more than 96 K elements): AUTO streams
    A, b, c, rel, sense = workloads.large_dual(100, 300, seed=4)
    rows, cols = lpx.tableau_dims(100, 300, rel)
    assert rows * cols > 96 * 1024
    want = orc.dual_solve(A, b, c, rel, sense, history=True)
    lib.lpx_reset_counters()
    compare_solve(lpx.dual_solve(A, b, c, rel, sense), want, "auto past the rule")
    assert lib.lpx_kernel_launches() > 1
    # ... unless the history is requested: the per-CTA global-memory kernel, one launch, history as before
    lib.lpx_reset_counters()
    got = lpx.dual_solve(A, b, c, rel, sense, history=len(want["history"]))
    assert lib.lpx_kernel_launches() == 1
    compare_solve(got, want, "auto with history")
    assert_bits_equal(got["history"], want["history"], "history")
    with pytest.raises(F.LpxError) as ei:
        lpx.dual_solve(A, b, c, rel, sense, kernel=F.KERNEL_STREAM, history=4)
    assert ei.value.code == F.E_CAPACITY and "history" in str(ei.value)


# ---- 6. device-pointer open, refusals ----------------------------------------------------------------------------
def test_dev_open_and_refusals(lpx, orc):
    import torch
    name, sense = "mixed:64:128", 1
    A, b, c, rel = problem(name)
    m, n = A.shape
    dev = torch.device("cuda:0")
    dA, db, dc = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (A, b, c))
    torch.cuda.synchronize()
    s = lpx.Session(dA.data_ptr(), db.data_ptr(), dc.data_ptr(), rel=rel, sense=sense, device_ptrs=True, m=m, n=n,
                    dual=True)
    check(run(s), oracle(orc, name, sense), "dev open")
    # refusals: no sensitivity report, no re-optimization base
    with pytest.raises(F.LpxError) as ei:
        s.sensitivity()
    assert ei.value.code == F.E_BAD_ARGS and "Dual Simplex" in str(ei.value)
    with pytest.raises(F.LpxError, match="Dual Simplex"):
        s.reoptimize(1, np.zeros(m))
    s.close()
    # a primal session reports no silent pivots
    Ap, bp, cp = workloads.lp_integer(16, 32, 1)
    p = lpx.Session(Ap, bp, cp)
    assert p.silent == 0 and not p.dual
    p.close()
    # bad arguments
    lib = F.lib()
    opt = None
    A1 = np.ones((2, 2))
    b1 = np.ones(2)
    assert not lib.lpx_dual_session_open(0, 2, 0, F.ptr(A1), None, F.ptr(b1), F.ptr(b1), opt)
    assert not lib.lpx_dual_session_open(2, 2, 2, F.ptr(A1), None, F.ptr(b1), F.ptr(b1), opt)
    assert not lib.lpx_dual_session_open(2, 2, 0, None, None, F.ptr(b1), F.ptr(b1), opt)
    assert "bad arguments" in F.last_error()
    bad_rel = np.array([0, 5], np.int32)
    assert not lib.lpx_dual_session_open(2, 2, 0, F.ptr(A1), F.ptr(bad_rel), F.ptr(b1), F.ptr(b1), opt)
    assert lib.lpx_session_silent_pivots(None, None) == F.E_BAD_ARGS


# ---- 7. full size: blocked against per pivot ---------------------------------------------------------------------
def test_full_size_blocked_against_per_pivot(lpx):
    """large_dual(2048, 8192) (4097 x 12289, C3's shape): the blocked dual look-ahead (K = 8 and 16) and the per-pivot
    protocol stepped to the same pivot count in uneven chunks agree on every tableau double, the pivot list and the
    basis.  (The oracle would need about 50 M multiply-subtracts per pivot.)"""
    A, b, c, rel, sense = workloads.large_dual()
    ref = lpx.Session(A, b, c, rel=rel, sense=sense, dual=True, single_cta_select=1)
    assert (ref.rows, ref.cols) == (4097, 12289) and ref.silent == 0
    chunks = [3, 13, 24, 37]  # 77 pivots: more than 5 blocks of 8 or 16, none aligned
    st, tot = F.RUNNING, 0
    for k in chunks:
        st, tot = ref.step(k)
    assert st == F.RUNNING and tot == sum(chunks)
    T = ref.tableau()
    basis, x, z = ref.solution()
    piv = ref.pivots(tot)
    ref.close()
    for kblock in (8, 16):
        s = lpx.Session(A, b, c, rel=rel, sense=sense, dual=True, single_cta_select=4, kblock=kblock)
        for k in chunks:
            got = s.step(k)
        assert got == (st, tot)
        assert np.array_equal(s.pivots(tot), piv), kblock
        gb, gx, gz = s.solution()
        assert np.array_equal(gb, basis)
        assert_bits_equal(gx, x, f"K {kblock} x")
        assert_bits_equal([gz], [z], f"K {kblock} z")
        assert_bits_equal(s.tableau(), T, f"K {kblock} tableau")
        s.close()


# ---- 8. randomized slice: the streaming kernel next to the per-CTA kernels ---------------------------------------
def test_fuzz_slice_stream_against_per_cta(lpx, orc):
    """The dual family of tests/fuzz_parity.py's single solves (tie-provoking integer, tie and decimal data, random
    '<=' / '>=' / '=' rows, both senses), with LPX_KERNEL_STREAM against the oracle and against the per-CTA kernel."""
    import fuzz_parity
    rng = np.random.default_rng(20261021)
    for t in range(24):
        m, n = int(rng.integers(1, 70)), int(rng.integers(1, 90))
        kind = ("int", "tie", "dec")[t % 3]
        A, b, c = fuzz_parity.gen(rng, m, n, kind)
        rel = rng.choice([0, 1, 2], size=m).astype(np.int32)
        sense = int(rng.integers(0, 2))
        want = orc.dual_solve(A, b, c, rel, sense)
        got = lpx.dual_solve(A, b, c, rel, sense, kernel=F.KERNEL_STREAM)
        what = f"fuzz {t} {kind} {m}x{n} sense {sense}"
        check(dict(got), want, what)
        if want["status"] == F.S_ITER_LIMIT:
            cta = lpx.dual_solve(A, b, c, rel, sense, kernel=F.KERNEL_CTA_GLOBAL)
            assert cta["status"] == got["status"] and np.array_equal(cta["pivots"], got["pivots"]), what
            assert_bits_equal(got["tableau"], cta["tableau"], what + " tableau against the per-CTA kernel")

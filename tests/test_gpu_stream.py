"""GPU parity for the whole-GPU streaming kernels (BASELINE config 3) through lpx_session_*."""
import numpy as np
import pytest

from conftest import assert_bits_equal

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu


def build_tableau(A, b, c):
    m, n = A.shape
    T = np.zeros((m + 1, n + m + 1))
    T[:m, :n] = A
    T[:m, n:n + m] = np.eye(m)
    T[:m, -1] = b
    T[m, :n] = -c
    return T


_C3 = {}


def _c3_oracle(orc, npiv):
    """The oracle's tableau after `npiv` pivots of the C3 instance (≈ 6 s on one core; computed once)."""
    if npiv not in _C3:
        A, b, c = workloads.large_c3()
        T = build_tableau(A, b, c)
        basis = np.arange(8192, 8192 + 4096, dtype=np.int32)
        ost, onp, opiv = orc.primal_core(T, basis, npiv)
        assert onp == npiv
        _C3[npiv] = (A, b, c, T, basis, opiv)
    return _C3[npiv]


PROTOCOLS = [(0, 0), (0, 1), (0, 3), (0, 5), (0, 16), (0, 11), (4, 0), (4, 3), (3, 0), (3, 5), (1, 0), (2, 0)]  # (protocol, pivots per HBM pass)


@pytest.mark.parametrize("protocol,kblock", PROTOCOLS)
def test_medium_full_solve(lpx, orc, protocol, kblock):
    A, b, c = workloads.lp_integer(256, 512, 7)
    want = orc.primal_solve(A, b, c)
    s = lpx.Session(A, b, c, single_cta_select=protocol, kblock=kblock)
    st, tot = F.RUNNING, 0
    while st == F.RUNNING:
        st, tot = s.step(64)
    assert st == want["status"] and tot == want["n_pivots"]
    assert s.pivots(tot)[:tot].tolist() == want["pivots"].tolist()
    basis, x, z = s.solution()
    assert basis.tolist() == want["basis"].tolist()
    assert_bits_equal(x, want["x"], "x")
    assert_bits_equal([z], [want["z"]], "z")
    assert_bits_equal(s.tableau(), want["tableau"], "tableau")
    s.close()


@pytest.mark.parametrize("protocol,kblock", PROTOCOLS)
def test_degenerate_and_repeated_rows_inside_a_block(lpx, orc, protocol, kblock):
    """Small dense LPs where the same row leaves several times within one look-ahead block and
    ties are frequent; plus EQ rows (negative RHS rows) and a Min objective."""
    rng = np.random.default_rng(23)
    for t in range(8):
        m, n = int(rng.integers(3, 12)), int(rng.integers(3, 14))
        A = rng.integers(-2, 7, size=(m, n)).astype(float)
        b = rng.integers(0, 12, size=m).astype(float)
        c = rng.integers(-2, 9, size=n).astype(float)
        rel = rng.choice([0, 0, 0, 2], size=m).astype(np.int32)
        sense = t % 2
        want = orc.primal_solve(A, b, c, rel, sense, max_iterations=60)
        s = lpx.Session(A, b, c, rel=rel, sense=sense, max_iterations=60, single_cta_select=protocol, kblock=kblock)
        st, tot = F.RUNNING, 0
        while st == F.RUNNING:
            st, tot = s.step(7)
        assert st == want["status"] and tot == want["n_pivots"], t
        assert s.pivots(max(tot, 1))[:tot].tolist() == want["pivots"].tolist(), t
        if st >= 0:
            assert_bits_equal(s.tableau(), want["tableau"], f"tableau {t}")
        s.close()


def test_step_granularity_is_invisible(lpx):
    A, b, c = workloads.lp_decimal(96, 200, 3)
    s1 = lpx.Session(A, b, c)
    s2 = lpx.Session(A, b, c, single_cta_select=2)
    s1.step(3)
    s1.step(5)
    st1, t1 = s1.step(4)
    st2, t2 = s2.step(12)
    assert (st1, t1) == (st2, t2)
    assert_bits_equal(s1.tableau(), s2.tableau(), "tableau")
    s1.close()
    s2.close()


def test_iteration_limit_and_unbounded(lpx, orc):
    A, b, c = workloads.lp_integer(64, 128, 2)
    want = orc.primal_solve(A, b, c, max_iterations=5)
    s = lpx.Session(A, b, c, max_iterations=5)
    st, tot = s.step(100)
    assert st == F.S_ITER_LIMIT == want["status"] and tot == 5
    assert s.pivots(5)[:5].tolist() == want["pivots"].tolist()
    s.close()
    A = np.array([[1.0, -1.0], [-1.0, 1.0]])
    s = lpx.Session(A, np.array([1.0, 2.0]), np.array([1.0, 1.0]))
    st, tot = s.step(10)
    w = orc.primal_solve(A, np.array([1.0, 2.0]), np.array([1.0, 1.0]))
    assert st == w["status"] == F.UNBOUNDED and tot == w["n_pivots"]
    assert_bits_equal(s.tableau(), w["tableau"], "unbounded tableau")
    s.close()


def test_c3_full_size_first_pivots(lpx, orc):
    """4096 x 8192: the first pivots against the oracle's arithmetic loop, every tableau bit."""
    A, b, c = workloads.large_c3()
    npiv = 6
    s = lpx.Session(A, b, c)
    assert (s.rows, s.cols) == (4097, 12289)
    st, tot = s.step(npiv)
    assert st == F.RUNNING and tot == npiv
    T = build_tableau(A, b, c)
    basis = np.arange(8192, 8192 + 4096, dtype=np.int32)
    ost, onp, opiv = orc.primal_core(T, basis, npiv)
    assert onp == npiv
    assert s.pivots(npiv)[:npiv].tolist() == opiv.tolist()
    got = s.tableau()
    assert_bits_equal(got, T, "C3 tableau after %d pivots" % npiv)
    gb, gx, gz = s.solution()
    assert gb.tolist() == basis.tolist()
    assert_bits_equal([gz], [T[-1, -1]], "z")
    # size-independent property over a longer window: basic columns stay exact unit vectors
    st, tot = s.step(40)
    got = s.tableau()
    gb, gx, gz = s.solution()
    for i in (0, 17, 4095):
        col = got[:, gb[i]]
        unit = np.zeros(4097)
        unit[i] = 1.0
        assert np.array_equal(np.abs(col), unit)
    s.close()


# pass variants 1 and 2 are the LDG/STG block passes, stream_update_block_kernel<8, 2, 4>, <8, 1, 4>, <16, 2, 2> and
# <16, 1, 4> (lpx_stream.cu:581-587); protocol 0 with kblock <= 8 takes the pipelined kernel whatever the variant
@pytest.mark.parametrize("protocol,kblock,pass_variant", [(0, 0, 0), (0, 0, 3), (0, 16, 0), (4, 0, 3), (4, 3, 1),
                                                          (4, 8, 2), (0, 16, 1), (4, 11, 2)])
def test_c3_full_size_pipelined_blocks(lpx, orc, protocol, kblock, pass_variant):
    """4096 x 8192 through the production protocols over >= 8 look-ahead blocks, stepped in uneven
    chunks (so blocks are cut short and the Fbuf/Pbuf/Lbuf halves and the ping-pong tableau buffers
    flip at odd places): pivot list and every tableau bit against the oracle's arithmetic loop
    (R/Models/PrimalSimplex.cs:205-257)."""
    chunks = (5, 11, 48, 8, 1)
    npiv = sum(chunks)
    A, b, c, T, basis, opiv = _c3_oracle(orc, npiv)
    s = lpx.Session(A, b, c, single_cta_select=protocol, kblock=kblock, pass_variant=pass_variant)
    tot = 0
    for k in chunks:
        st, tot = s.step(k)
        assert st == F.RUNNING
    assert tot == npiv
    assert s.pivots(npiv)[:npiv].tolist() == opiv.tolist()
    assert_bits_equal(s.tableau(), T, "C3 tableau after %d pivots" % npiv)
    gb, gx, gz = s.solution()
    assert gb.tolist() == basis.tolist()
    assert_bits_equal([gz], [T[-1, -1]], "z")
    s.close()


# (kblock, pass_variant, protocol); the ids of the TMA-staged cases stay the kblock alone
BLOCK_PASSES = [pytest.param(k, 3, 0, id=str(k)) for k in (0, 3, 16)] + \
    [pytest.param(k, v, 4 if k <= 8 else 0, id=f"{k}-ldg{v}") for v in (1, 2) for k in (0, 3, 16)]


@pytest.mark.parametrize("kblock,pass_variant,protocol", BLOCK_PASSES)
def test_tma_staged_pass(lpx, orc, kblock, pass_variant, protocol):
    """The blocked HBM pass: pass_variant 3 stages it through shared memory by cp.async.bulk, 1 and 2 are the
    LDG/STG passes with two / one doubles per thread.  The small LPs give a row chunk of one row per CTA."""
    for (m, n, seed) in [(256, 512, 7), (100, 37, 3), (9, 700, 5)]:
        A, b, c = workloads.lp_integer(m, n, seed)
        want = orc.primal_solve(A, b, c)
        s = lpx.Session(A, b, c, kblock=kblock, pass_variant=pass_variant, single_cta_select=protocol)
        st, tot = F.RUNNING, 0
        while st == F.RUNNING:
            st, tot = s.step(50)
        assert st == want["status"] and tot == want["n_pivots"], (m, n)
        assert s.pivots(tot)[:tot].tolist() == want["pivots"].tolist()
        assert_bits_equal(s.tableau(), want["tableau"], f"tableau {m}x{n}")
        s.close()
    rng = np.random.default_rng(5)
    for t in range(6):
        m, n = int(rng.integers(3, 12)), int(rng.integers(3, 14))
        A = rng.integers(-2, 7, size=(m, n)).astype(float)
        b = rng.integers(0, 12, size=m).astype(float)
        c = rng.integers(-2, 9, size=n).astype(float)
        rel = rng.choice([0, 0, 0, 2], size=m).astype(np.int32)
        want = orc.primal_solve(A, b, c, rel, 0, max_iterations=60)
        s = lpx.Session(A, b, c, rel=rel, max_iterations=60, kblock=kblock, pass_variant=pass_variant,
                        single_cta_select=protocol)
        st, tot = F.RUNNING, 0
        while st == F.RUNNING:
            st, tot = s.step(7)
        assert st == want["status"] and tot == want["n_pivots"], t
        if st >= 0:
            assert_bits_equal(s.tableau(), want["tableau"], f"tableau {t}")
        s.close()

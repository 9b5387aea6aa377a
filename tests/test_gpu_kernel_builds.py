"""GPU parity for the kernel builds and loop regimes that only the tableau shape and the options select.

Every GPU result is compared bit for bit with the oracle, but that only checks the code that runs.  These tests
pick shapes and options so that each build and each regime of the per-tableau kernels runs at least once:

- the second and later trips of the column-pair update loops: `cta_update` (primal, THREADS-32 update threads),
  `cta_pivot` (dual, THREADS) and both update loops of `cta_cluster_simplex_kernel`, which take more than one
  trip only when the tableau has more column pairs than update threads;
- every CTA size of `cta_simplex_kernel` (`lpx_options.threads` 128 / 256 / 512, shared or global tableau),
  also inside Branch & Bound and the pooled tree (Mode B);
- both sides of each capacity edge between the shared-memory kernel, the 2- and 4-CTA clusters, the
  global-memory tableau and streaming, from a restatement of the shared-memory carve;
- the builds that only an environment switch selects (DESIGN §7a), in a subprocess each.

Data come from the integer / decimal generators of `workloads.py`, so a mismatch points at the code path.
Run as a script (`python tests/test_gpu_kernel_builds.py <switch>`), the file is the subprocess body.
"""
import os
import subprocess
import sys
from functools import lru_cache

import numpy as np
import pytest

from conftest import assert_bits_equal

from linear_programming_solver_lpr381_b200 import _ffi as F
from linear_programming_solver_lpr381_b200 import workloads

pytestmark = pytest.mark.gpu

PRIMAL_KERNELS = [F.KERNEL_AUTO, F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL, F.KERNEL_CTA_CLUSTER]
DUAL_KERNELS = [F.KERNEL_AUTO, F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL, F.KERNEL_CTA_CLUSTER]
KNAME = {F.KERNEL_AUTO: "auto", F.KERNEL_CTA_SMEM: "smem", F.KERNEL_CTA_GLOBAL: "global",
         F.KERNEL_STREAM: "stream", F.KERNEL_CTA_CLUSTER: "cluster"}


# ---- the shared-memory carve, restated --------------------------------------------------------------------------
# cta_carve (lpx_cta.cuh:83-107) and cta_cluster_carve (lpx_cta_cluster.cuh:28-58), in bytes, for a tableau of
# R rows (constraints after '=' expansion + the objective row) and W columns (n + R; the last one is the RHS).

def cta_carve_total(R, W, smem_T=True):
    off = ((W + 2) & ~1) * 8 + R * 8 + W * 8 + 34 * 16 + 3 * R * 4 + 16 * 4  # prow fcol zc red rsrc rsgn basis ctl
    off = (off + 15) & ~15
    if smem_T:
        off += R * ((W + 1) & ~1) * 8  # rows padded to an even length
    return off


def cluster_carve_total(R, W, cl):
    H = (R + cl - 1) // cl  # rows per CTA
    off = ((W + 2) & ~1) * 8 + max(R, W) * 8 + H * 8 + W * 8 + 34 * 16 + 8 * 16 + 3 * R * 4 + 16 * 4
    off = (off + 15) & ~15
    return off + H * ((W + 1) & ~1) * 8


@lru_cache(maxsize=None)
def smem_optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def fits_smem(R, W):
    return cta_carve_total(R, W) <= smem_optin()


def fits_cluster(R, W, cl):
    return cluster_carve_total(R, W, cl) <= smem_optin()


def cluster_size(R, W):
    """cta_cluster_size_for (lpx_cta.cu:36-44) without LPX_CLUSTER4."""
    return 2 if fits_cluster(R, W, 2) else (4 if fits_cluster(R, W, 4) else 0)


SINGLE_CTA_ELEMS = 96 * 1024  # lpx_primal_solve (lpx_cta.cu:446-455): past this, AUTO streams a single solve


def auto_route(R, W):
    """Which kernel family lpx_primal_solve picks under AUTO for an all-'<=' LP without history."""
    if fits_smem(R, W):
        return "smem"
    if R * W > SINGLE_CTA_ELEMS:
        return "stream"
    return "cluster" if cluster_size(R, W) else "global"


def last_n(m, pred):
    """Largest n >= 1 with pred(R, W) for an all-'<=' LP of m rows (0: none); pred is monotone in n."""
    R = m + 1
    if not pred(R, R + 1):
        return 0
    lo, hi = 1, 1
    while pred(R, R + hi):
        lo, hi = hi, hi * 2
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if pred(R, R + mid) else (lo, mid)
    return lo


def edges(m):
    """The capacity edges of an all-'<=' LP with m rows, as the last n on the lower side of each."""
    return {
        "smem": last_n(m, fits_smem),
        "cluster2": last_n(m, lambda R, W: fits_cluster(R, W, 2)),
        "cluster4": last_n(m, lambda R, W: fits_cluster(R, W, 4)),
        "single96k": last_n(m, lambda R, W: R * W <= SINGLE_CTA_ELEMS),
    }


def accepts(kernel, R, W):
    if kernel == F.KERNEL_CTA_SMEM:
        return fits_smem(R, W)
    if kernel == F.KERNEL_CTA_CLUSTER:
        return fits_cluster(R, W, 4)
    return True


# ---- problems and comparisons ---------------------------------------------------------------------------------

def dual_rel(mm):
    """A '>=' / '<=' / '=' row pattern that expands to exactly mm tableau rows (the dual's '>=' rows flip)."""
    rel, k, pat = [], 0, (1, 0, 2, 1, 0)
    while k < mm:
        r = pat[len(rel) % len(pat)]
        if r == 2 and k + 2 > mm:
            r = 1
        rel.append(r)
        k += 2 if r == 2 else 1
    return np.array(rel, dtype=np.int32)


@lru_cache(maxsize=None)
def primal_lp(R, W, kind="integer"):
    m, n = R - 1, W - R
    if kind == "decimal":
        return workloads.lp_decimal(m, n, 1000 + R + W)
    return workloads.lp_integer(m, n, 1000 + R + W)


@lru_cache(maxsize=None)
def dual_lp(R, W):
    """Tie-free decimal data: the integer generator's dual problems often cycle to the iteration limit."""
    rel = dual_rel(R - 1)
    A, b, c = workloads.lp_decimal(len(rel), W - R, 2000 + R + W)
    return A, b, c, rel


@lru_cache(maxsize=None)
def primal_want(orc, R, W, kind="integer", max_iterations=10000):
    A, b, c = primal_lp(R, W, kind)
    return orc.primal_solve(A, b, c, max_iterations=max_iterations)


@lru_cache(maxsize=None)
def dual_want(orc, R, W):
    A, b, c, rel = dual_lp(R, W)
    return orc.dual_solve(A, b, c, rel, 1)


def compare(got, want, what):
    assert got["status"] == want["status"], what
    if "silent" in want:
        assert got["silent"] == want["silent"], what
    if want["status"] < 0 and want["status"] != F.S_ITER_LIMIT:
        return
    assert got["n_pivots"] == want["n_pivots"], what
    if want["status"] == F.S_ITER_LIMIT and "silent" in want:
        return  # the oracle's Dual Simplex exports nothing after the iteration-limit exception
    assert got["pivots"].tolist() == want["pivots"].tolist(), what
    if want["status"] == F.S_ITER_LIMIT:
        return
    assert got["basis"].tolist() == want["basis"].tolist(), what
    assert_bits_equal(got["x"], want["x"], what + " x")
    assert_bits_equal([got["z"]], [want["z"]], what + " z")
    assert_bits_equal(got["tableau"], want["tableau"], what + " tableau")


def refused(call):
    with pytest.raises(F.LpxError) as ei:
        call()
    assert ei.value.code == F.E_CAPACITY, str(ei.value)


def run_primal(lpx, orc, R, W, kernel, threads=0, kind="integer"):
    A, b, c = primal_lp(R, W, kind)
    assert lpx.tableau_dims(*A.shape) == (R, W)
    what = f"primal {R}x{W} {KNAME[kernel]} threads={threads}"
    if not accepts(kernel, R, W):
        refused(lambda: lpx.primal_solve(A, b, c, kernel=kernel, threads=threads))
        return None
    got = lpx.primal_solve(A, b, c, kernel=kernel, threads=threads)
    compare(got, primal_want(orc, R, W, kind), what)
    return got


def run_dual(lpx, orc, R, W, kernel, threads=0):
    A, b, c, rel = dual_lp(R, W)
    assert lpx.tableau_dims(A.shape[0], A.shape[1], rel) == (R, W)
    what = f"dual {R}x{W} {KNAME[kernel]} threads={threads}"
    if not accepts(kernel, R, W):
        refused(lambda: lpx.dual_solve(A, b, c, rel, 1, kernel=kernel, threads=threads))
        return None
    got = lpx.dual_solve(A, b, c, rel, 1, kernel=kernel, threads=threads)
    compare(got, dual_want(orc, R, W), what)
    return got


# ---- 1. trip regimes of the column-pair update loops ----------------------------------------------------------
# A tableau of W columns has (W + 1) / 2 column pairs; the update loops take ceil(pairs / U) trips once the pairs
# reach U (rounded up to whole warps).  Under AUTO the per-CTA kernels run 256 threads while rows x width < 8192
# and 512 beyond (lpx_cta.cu:101-107); clusters always run 512.  Shapes as (rows, width):
PRIMAL_TRIP_SHAPES = [
    # U = 224 (256 threads): just below, at and above 2U = 448 columns; 228 pairs (not a multiple of U); the
    # last 256-thread shape (18 x 455 = 8190 elements: m = 17, n = 437) and the first 512-thread one
    (18, 447), (18, 448), (18, 449), (18, 455), (18, 456),
    # U = 480 (512 threads): around 2U = 960; m = 17, n = 943; m = 27, n = 933 / 934 (the last width that fits)
    (28, 959), (28, 960), (18, 961), (28, 961), (28, 962),
    # one row, m = 1, n = 4093 / 4094: 2047 / 2048 pairs, five trips
    (2, 4095), (2, 4096),
    # 4-CTA clusters under AUTO: m = 63, n = 1000 and n = 1454 (the last that fits four CTAs), 532 / 759 pairs
    (64, 1064), (64, 1518),
]
DUAL_TRIP_SHAPES = [
    # U = 256 (256 threads): around 2U = 512 (rows 9: m = 8 incl. one '=' row, n = 504 at width 513)
    (9, 511), (9, 512), (9, 513), (9, 515),
    # U = 512 (512 threads and the cluster's dual pivot): around 2U = 1024
    (16, 1023), (16, 1024), (16, 1025), (16, 1101),
    # a 4-CTA cluster with 550 pairs
    (64, 1100),
]
# U = 96 / 128: the 128-thread build (threads = 128 only)
PRIMAL_T128_SHAPES = [(9, 191), (9, 192), (9, 193), (9, 481)]
DUAL_T128_SHAPES = [(9, 255), (9, 256), (9, 257), (9, 301)]


def shape_id(s):
    return f"{s[0]}x{s[1]}"


@pytest.mark.parametrize("shape", PRIMAL_TRIP_SHAPES, ids=shape_id)
@pytest.mark.parametrize("kernel", PRIMAL_KERNELS, ids=lambda k: KNAME[k])
def test_primal_update_trips(lpx, orc, shape, kernel):
    run_primal(lpx, orc, *shape, kernel)


@pytest.mark.parametrize("shape", DUAL_TRIP_SHAPES, ids=shape_id)
@pytest.mark.parametrize("kernel", DUAL_KERNELS, ids=lambda k: KNAME[k])
def test_dual_pivot_trips(lpx, orc, shape, kernel):
    run_dual(lpx, orc, *shape, kernel)


def test_decimal_data_on_wide_rows(lpx, orc):
    """Tie-free decimal data on the two-trip shapes of every family."""
    for R, W, kernels in ((18, 455, PRIMAL_KERNELS), (28, 962, PRIMAL_KERNELS), (64, 1064, [F.KERNEL_CTA_CLUSTER])):
        for kernel in kernels:
            run_primal(lpx, orc, R, W, kernel, kind="decimal")


@pytest.mark.parametrize("kernel,shape", [(F.KERNEL_CTA_SMEM, (18, 455)), (F.KERNEL_CTA_GLOBAL, (18, 455)),
                                          (F.KERNEL_CTA_SMEM, (28, 962)), (F.KERNEL_CTA_CLUSTER, (28, 962)),
                                          (F.KERNEL_CTA_CLUSTER, (64, 1064))],
                         ids=lambda v: KNAME[v] if isinstance(v, int) else shape_id(v))
def test_history_on_wide_rows(lpx, orc, kernel, shape):
    """The iteration history (every intermediate tableau) on a multi-trip shape of each family, primal and dual."""
    R, W = shape
    A, b, c = primal_lp(R, W)
    want = orc.primal_solve(A, b, c, history=True)
    got = lpx.primal_solve(A, b, c, kernel=kernel, history=want["n_pivots"] + 1)
    assert len(got["history"]) == want["n_pivots"] + 1
    assert_bits_equal(got["history"], want["history"], f"primal history {R}x{W} {KNAME[kernel]}")
    if R * W < 30000:
        Ad, bd, cd, rel = dual_lp(R, W)
        want = orc.dual_solve(Ad, bd, cd, rel, 1, history=True)
        got = lpx.dual_solve(Ad, bd, cd, rel, 1, kernel=kernel, history=len(want["history"]))
        assert_bits_equal(got["history"], want["history"], f"dual history {R}x{W} {KNAME[kernel]}")


# ---- 2. CTA sizes -----------------------------------------------------------------------------------------------

def random_small_primal(t_count=60):
    """The generator of test_random_small_vs_oracle."""
    rng = np.random.default_rng(101)
    for _ in range(t_count):
        m, n = int(rng.integers(1, 24)), int(rng.integers(1, 40))
        A = rng.integers(-3, 10, size=(m, n)).astype(float)
        b = rng.integers(0, 40, size=m).astype(float)
        c = rng.integers(-4, 10, size=n).astype(float)
        rel = rng.choice([0, 0, 0, 0, 2], size=m).astype(np.int32)
        yield A, b, c, rel, int(rng.integers(0, 2))


def random_small_dual(t_count=60):
    """The generator of test_random_dual_vs_oracle."""
    rng = np.random.default_rng(77)
    for _ in range(t_count):
        m, n = int(rng.integers(1, 16)), int(rng.integers(1, 24))
        A = rng.integers(0, 9, size=(m, n)).astype(float)
        b = rng.integers(1, 25, size=m).astype(float)
        c = rng.integers(1, 9, size=n).astype(float)
        rel = rng.choice([0, 1, 2], size=m).astype(np.int32)
        yield A, b, c, rel, int(rng.integers(0, 2))


@lru_cache(maxsize=None)
def random_small_wants(orc):
    p = [orc.primal_solve(A, b, c, rel, s, max_iterations=300) for A, b, c, rel, s in random_small_primal()]
    d = [orc.dual_solve(A, b, c, rel, s) for A, b, c, rel, s in random_small_dual()]
    return p, d


def run_random_small(lpx, orc, kernel, threads):
    wp, wd = random_small_wants(orc)
    for t, (A, b, c, rel, s) in enumerate(random_small_primal()):
        got = lpx.primal_solve(A, b, c, rel, s, max_iterations=300, kernel=kernel, threads=threads)
        compare(got, wp[t], f"random primal {t} {KNAME[kernel]} threads={threads}")
    for t, (A, b, c, rel, s) in enumerate(random_small_dual()):
        got = lpx.dual_solve(A, b, c, rel, s, kernel=kernel, threads=threads)
        compare(got, wd[t], f"random dual {t} {KNAME[kernel]} threads={threads}")


def bnb_batch():
    return zip(*[workloads.ip_c4(m=20, n=30, seed=600 + k) for k in range(8)])


@lru_cache(maxsize=None)
def bnb_wants(orc):
    As, bs, cs = bnb_batch()
    return [orc.bnb_simplex(As[k], bs[k], cs[k], node_cap=1 << 16) for k in range(len(As))]


def check_bnb_batch(got, wants, what):
    for k, want in enumerate(wants):
        assert bool(got["found"][k]) == want["found"], (what, k)
        assert got["n_nodes"][k] == want["n_nodes"], (what, k)
        assert got["lp_pivots"][k] == want["total_pivots"], (what, k)
        if want["found"]:
            assert_bits_equal([got["best_z"][k]], [want["best_z"]], f"{what} best_z {k}")
            assert_bits_equal(got["best_x"][k], want["best_x"], f"{what} best_x {k}")


@pytest.mark.parametrize("threads", [128, 256, 512])
@pytest.mark.parametrize("kernel", [F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL], ids=lambda k: KNAME[k])
def test_cta_size_builds(lpx, orc, monkeypatch, kernel, threads):
    """lpx_options.threads selects cta_simplex_kernel<threads, kernel == SMEM>: the trip shapes, the small random
    primal / dual sets, a Branch & Bound batch on the full-tableau node kernels and one pooled-tree instance."""
    for R, W in PRIMAL_TRIP_SHAPES[:12] + PRIMAL_T128_SHAPES:
        run_primal(lpx, orc, R, W, kernel, threads)
    for R, W in DUAL_TRIP_SHAPES[:8] + DUAL_T128_SHAPES:
        run_dual(lpx, orc, R, W, kernel, threads)
    run_random_small(lpx, orc, kernel, threads)
    # Branch & Bound: the full-tableau node launches (lpx_bnb.cu:293, :550) take the option too
    As, bs, cs = (np.stack(v) for v in bnb_batch())
    monkeypatch.setenv("LPX_BNB_FULL_TABLEAU", "1")
    bk = F.KERNEL_CTA_GLOBAL if kernel == F.KERNEL_CTA_GLOBAL else F.KERNEL_AUTO
    check_bnb_batch(lpx.bnb_simplex_batched(As, bs, cs, kernel=bk, threads=threads), bnb_wants(orc),
                    f"bnb {KNAME[kernel]} threads={threads}")
    monkeypatch.delenv("LPX_BNB_FULL_TABLEAU")
    # a traced tree takes the other driver (node records in the reference's order, lpx_bnb.cu:293)
    want = bnb_wants(orc)[0]
    got = lpx.bnb_simplex(As[0], bs[0], cs[0], trace=True, kernel=bk, threads=threads)
    assert got["n_nodes"] == want["n_nodes"] and got["lp_pivots"] == want["total_pivots"]
    assert [nd["n_pivots"] for nd in got["nodes"]] == want["pivots"].tolist()
    assert [nd["outcome"] for nd in got["nodes"]] == want["outcome"].tolist()
    assert got["found"] == want["found"]
    if want["found"]:
        assert_bits_equal(got["best_x"], want["best_x"], f"traced bnb best_x {KNAME[kernel]} threads={threads}")
    if kernel == F.KERNEL_CTA_SMEM:  # Mode B picks shared or global memory itself (lpx_pooled.cu:307, :400)
        A, b, c = workloads.ip_c4(m=8, n=12, seed=5)
        want = orc.bnb_pooled(A, b, c, batch=16)
        got = lpx.bnb_pooled(A, b, c, batch=16, threads=threads)
        assert want["rc"] == 0 and got["found"] == want["found"] and got["n_nodes"] == want["n_nodes"]
        assert got["node_id"].tolist() == want["node_id"].tolist()
        assert got["pivots"].tolist() == want["pivots"].tolist()
        assert_bits_equal(got["z"], want["z"], f"pooled node z threads={threads}")
        if want["found"]:
            assert_bits_equal(got["best_x"], want["best_x"], f"pooled best_x threads={threads}")


@pytest.mark.parametrize("threads", [0, 64, 384, 1024])
def test_unsupported_cta_sizes_fall_back_to_auto(lpx, orc, threads):
    """A threads value outside {128, 256, 512} is the automatic choice: the same bits as threads = 0."""
    for R, W in ((18, 455), (18, 456), (28, 962), (9, 481)):
        A, b, c = primal_lp(R, W)
        for kernel in (F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL):
            auto = lpx.primal_solve(A, b, c, kernel=kernel)
            got = run_primal(lpx, orc, R, W, kernel, threads)
            assert_bits_equal(got["tableau"], auto["tableau"], f"{R}x{W} threads={threads} vs auto")
    for R, W in ((9, 513), (16, 1025)):
        run_dual(lpx, orc, R, W, F.KERNEL_CTA_SMEM, threads)
    run_random_small(lpx, orc, F.KERNEL_AUTO, threads)


# ---- 3. capacity edges ------------------------------------------------------------------------------------------
EDGE_ROWS = [63, 127, 200]


def test_carve_restatement_matches_the_library(lpx):
    """Forced shared-memory and forced cluster solves are accepted at the last n the carve allows and refused one
    column later; max_iterations = 1 keeps the probes cheap."""
    for m in EDGE_ROWS:
        e = edges(m)
        for kernel, last in ((F.KERNEL_CTA_SMEM, e["smem"]), (F.KERNEL_CTA_CLUSTER, e["cluster4"])):
            if last:
                A, b, c = workloads.lp_integer(m, last, 3)
                r = lpx.primal_solve(A, b, c, max_iterations=1, kernel=kernel)
                assert r["status"] in (F.OPTIMAL, F.S_ITER_LIMIT), (m, last, KNAME[kernel])
            A, b, c = workloads.lp_integer(m, last + 1, 3)
            refused(lambda: lpx.primal_solve(A, b, c, max_iterations=1, kernel=kernel))
        # the dual takes the same carve: a tableau of the same shape from '>=' and '=' rows
        rel = dual_rel(m)
        for kernel, last in ((F.KERNEL_CTA_SMEM, e["smem"]), (F.KERNEL_CTA_CLUSTER, e["cluster4"])):
            A, b, c = workloads.lp_integer(len(rel), last + 1, 3)
            refused(lambda: lpx.dual_solve(A, b, c, rel, 1, kernel=kernel))


def test_edges_at_232448_bytes():
    """The edges the carve gives on a B200 (232 448 bytes of opt-in shared memory per block); the tests below
    compute them from the device's own limit."""
    if smem_optin() != 232448:
        pytest.skip(f"opt-in shared memory is {smem_optin()} bytes")
    assert edges(63) == dict(smem=372, cluster2=758, cluster4=1454, single96k=1472)
    assert edges(127) == dict(smem=92, cluster2=300, cluster4=692, single96k=640)
    assert edges(200) == dict(smem=0, cluster2=73, cluster4=327, single96k=288)


def edge_cases():
    out = []
    for m in EDGE_ROWS:
        for name in ("smem", "cluster2", "cluster4", "single96k"):
            out.append((m, name))
    return out


@pytest.mark.parametrize("m,edge", edge_cases(), ids=lambda v: str(v))
def test_solves_across_capacity_edges(lpx, orc, m, edge):
    """n_edge - 1, n_edge and n_edge + 1 under AUTO and each forced kernel that takes the shape (primal), the same
    for the dual with '>=' rows; a single AUTO solve is one launch unless it streams."""
    last = edges(m)[edge]
    R = m + 1
    lib = F.lib()
    for n in (last - 1, last, last + 1):
        if n < 1:
            continue
        W = n + R
        A, b, c = workloads.lp_integer(m, n, 7 + n)
        want = orc.primal_solve(A, b, c)
        lib.lpx_reset_counters()
        compare(lpx.primal_solve(A, b, c), want, f"primal m={m} n={n} auto")
        launches = lib.lpx_kernel_launches()
        route = auto_route(R, W)
        if route == "stream":
            assert launches > 1, (m, n, route, launches)
        else:
            assert launches == 1, (m, n, route, launches)
        for kernel in (F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL, F.KERNEL_CTA_CLUSTER) + \
                ((F.KERNEL_STREAM,) if edge == "single96k" else ()):
            what = f"primal m={m} n={n} {KNAME[kernel]}"
            if not accepts(kernel, R, W):
                refused(lambda: lpx.primal_solve(A, b, c, kernel=kernel))
                continue
            compare(lpx.primal_solve(A, b, c, kernel=kernel), want, what)
        if m == 200 and edge != "single96k":  # the same tableau shape: '>=' and '=' rows, 200 after expansion
            rel = dual_rel(m)
            Ad, bd, cd = workloads.lp_decimal(len(rel), n, 7 + n)
            assert lpx.tableau_dims(len(rel), n, rel) == (R, W)
            wd = orc.dual_solve(Ad, bd, cd, rel, 1)
            for kernel in DUAL_KERNELS:
                if not accepts(kernel, R, W):
                    refused(lambda: lpx.dual_solve(Ad, bd, cd, rel, 1, kernel=kernel))
                    continue
                compare(lpx.dual_solve(Ad, bd, cd, rel, 1, kernel=kernel), wd, f"dual m={m} n={n} {KNAME[kernel]}")


def test_history_past_the_single_solve_limit(lpx, orc):
    """A history request where AUTO would stream goes to the global-memory per-CTA kernel (lpx_cta.cu:454)."""
    m = 63
    n = edges(m)["single96k"] + 1
    assert auto_route(m + 1, n + m + 1) == "stream"
    A, b, c = workloads.lp_integer(m, n, 5)
    want = orc.primal_solve(A, b, c, history=4)
    F.lib().lpx_reset_counters()
    got = lpx.primal_solve(A, b, c, history=4)
    assert F.lib().lpx_kernel_launches() == 1
    compare(got, want, "history past 96K")
    assert_bits_equal(got["history"], want["history"], "history past 96K")


@pytest.mark.parametrize("m,edge", edge_cases(), ids=lambda v: str(v))
def test_batched_across_capacity_edges(lpx, orc, m, edge):
    """A small batch on each side of each edge under AUTO: far past the register kernel's n + m <= 192, so the
    batch lands in cta_launch (shared memory, cluster or global memory; batches never stream)."""
    last = edges(m)[edge]
    for n in (last, last + 1):
        if n < 1:
            continue
        A, b, c = workloads.batch_c2(count=3, m=m, n=n, seed=n)
        want = orc.primal_batch(A, b, c, threads=3, want_tableau=True)
        got = lpx.primal_solve_batched(A, b, c)
        what = f"batched m={m} n={n}"
        assert np.array_equal(got["status"], want["status"]), what
        assert np.array_equal(got["n_pivots"], want["n_pivots"]), what
        assert np.array_equal(got["basis"], want["basis"]), what
        assert_bits_equal(got["x"], want["x"], what + " x")
        assert_bits_equal(got["z"], want["z"], what + " z")
        assert_bits_equal(got["tableau"], want["tableau"], what + " tableau")


# ---- 4. builds behind environment switches (read once per process: one subprocess each) -----------------------

def _switch_cluster4(lpx, orc):
    """LPX_CLUSTER4=1: 4-CTA clusters first.  With 2, 3, 5, 6 or 9 tableau rows one CTA owns no rows."""
    for R in (2, 3, 5, 6, 9):
        for W in (R + 7, R + 40):
            for kind in ("integer", "decimal"):
                run_primal(lpx, orc, R, W, F.KERNEL_CTA_CLUSTER, kind=kind)
            run_dual(lpx, orc, R, W, F.KERNEL_CTA_CLUSTER)
            A, b, c = primal_lp(R, W)
            want = orc.primal_solve(A, b, c, history=True)
            got = lpx.primal_solve(A, b, c, kernel=F.KERNEL_CTA_CLUSTER, history=want["n_pivots"] + 1)
            assert_bits_equal(got["history"], want["history"], f"cluster4 history {R}x{W}")
            Ad, bd, cd, rel = dual_lp(R, W)
            want = orc.dual_solve(Ad, bd, cd, rel, 1, history=True)
            got = lpx.dual_solve(Ad, bd, cd, rel, 1, kernel=F.KERNEL_CTA_CLUSTER, history=len(want["history"]))
            assert_bits_equal(got["history"], want["history"], f"cluster4 dual history {R}x{W}")
    for R, W in ((64, 364), (28, 962)):  # mid-size, and two trips per update
        for kernel in (F.KERNEL_CTA_CLUSTER, F.KERNEL_AUTO):
            run_primal(lpx, orc, R, W, kernel)
            run_dual(lpx, orc, R, W, kernel)


def _switch_bnb_trace(lpx, orc):
    """LPX_BNB_TRACE=1: the pipelined Branch & Bound driver runs cta_condensed_kernel<512, true>."""
    As, bs, cs = (np.stack(v) for v in bnb_batch())
    check_bnb_batch(lpx.bnb_simplex_batched(As, bs, cs), bnb_wants(orc), "bnb trace")


def _switch_cta_prof(lpx, orc):
    """LPX_CTA_PROF=1: the profiling path of cta_simplex_kernel, single solves of every build."""
    for kernel in (F.KERNEL_CTA_SMEM, F.KERNEL_CTA_GLOBAL):
        for threads in (128, 256, 512):
            for R, W in ((18, 455), (9, 193)):
                run_primal(lpx, orc, R, W, kernel, threads)
            run_dual(lpx, orc, 9, 513, kernel, threads)
    run_primal(lpx, orc, 5, 60, F.KERNEL_AUTO, kind="decimal")


SWITCHES = {"LPX_CLUSTER4": _switch_cluster4, "LPX_BNB_TRACE": _switch_bnb_trace, "LPX_CTA_PROF": _switch_cta_prof}


@pytest.mark.parametrize("switch", sorted(SWITCHES))
def test_environment_switch_builds(switch):
    env = dict(os.environ, **{switch: "1"})
    env["PYTHONPATH"] = os.pathsep.join(p for p in sys.path if p)
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), switch], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, f"{switch}: exit {r.returncode}\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    assert f"{switch} ok" in r.stdout
    if switch == "LPX_CTA_PROF":
        assert "[cta prof]" in r.stderr


if __name__ == "__main__":
    import orc_ffi
    from linear_programming_solver_lpr381_b200 import api

    orc_ffi.lib()
    F.check(F.lib().lpx_init(0))
    SWITCHES[sys.argv[1]](api, orc_ffi)
    print(f"{sys.argv[1]} ok")

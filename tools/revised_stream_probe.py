"""Revised Primal Simplex on the whole GPU -> <out>/r08_revised_stream.json (default out: profiles/).

Per-iteration time: lpx_revised_solve returns after a device synchronise, so a host clock around the call times
the GPU work.  With T(k) the time of a call capped at k iterations (initial inversion, then k iterations of
pricing, ratio test and re-inversion), iteration = (T(k) - T(0)) / k: the calls' fixed costs cancel.
Split of an iteration (whole-GPU path): one more call capped at k iterations under torch.profiler with CUDA
activities; the kernels' GPU timestamps are summed by phase: look-ahead (rev_lookahead_kernel), pass (the blocked
pass kernels), rest of the inversion ([B | I] build, B^-1 extraction, x_B, history record) and pricing / ratio
(pi, r_N, entering arg-min, d and ratios, leaving row + list update).  Per inversion = over the k + 1 inversions,
per pricing = over the k iterations.  Kernel time excludes launch gaps, so the phases can sum to less than the
host-clock iteration.  The one-CTA kernel is one launch, so it has no such split: its first call T(0) - T1(0)
(T1(0): the same call on a 1 x 1 model) is one A | I build + one inversion, and pricing = iteration - that.
1. The crossover sweep: the one-CTA kernel (LPX_KERNEL_CTA_GLOBAL) and the stream (LPX_KERNEL_STREAM, K = 8) at
   m in {64, 96, 128, 256, 512, 1024}, square (n = m) and wide (n = 8m), lp_decimal data.  The one-CTA kernel is
   skipped where the m^3 extrapolation of its previous inversion exceeds --cta-budget seconds.
2. K in {1, 4, 8, 16} at m = 1024 and 2048 (square), with whether [B | I] fits the 126 MB L2.
3. Full solves past the one-CTA capacity under AUTO: lp_integer(64, 20000), lp_integer(32, 100000), checked
   against the oracle bit for bit when --oracle is given, with the kernel launches of the call and how many of them
   were enqueued after the solve had ended (the rest of the last chunk; they return at once).
4. A tall solve: lp_decimal(1024, 1024) to OPTIMAL or --tall-cap iterations.
The card name, power limit and max SM clock are read in the same call.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402
from session_reopt_probe import card  # noqa: E402

L2_BYTES = 126 << 20


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def fixed_cost(rounds, **kw):
    """T(0) of a 1 x 1 model: the call's copies, launches and synchronisations."""
    one = np.ones((1, 1)), np.ones(1), np.ones(1)
    api.revised_solve(*one, max_iterations=0, **kw)
    return float(np.median([timed(lambda: api.revised_solve(*one, max_iterations=0, **kw))[0] for _ in range(rounds)]))


def split(A, b, c, k, rounds, **kw):
    """(first call ms, iteration ms) from T(0) and T(k), medians over `rounds`."""
    api.revised_solve(A, b, c, max_iterations=0, **kw)  # warm-up: modules, workspaces
    t0 = float(np.median([timed(lambda: api.revised_solve(A, b, c, max_iterations=0, **kw))[0]
                          for _ in range(rounds)]))
    tk, r = [], None
    for _ in range(rounds):
        t, r = timed(lambda: api.revised_solve(A, b, c, max_iterations=k, **kw))
        tk.append(t)
    it = (float(np.median(tk)) - t0) / max(r["n_iters"], 1)
    out = dict(first_call_ms=round(max(t0 - fixed_cost(rounds, **kw), 0.0), 3), iteration_ms=round(it, 3),
               iterations=r["n_iters"], status=r["status"])
    if kw.get("kernel") == F.KERNEL_CTA_GLOBAL:
        out["pricing_ms"] = round(it - out["first_call_ms"], 3)
    else:
        out.update(kernel_split(A, b, c, k, **kw))
    return out


PHASES = (("lookahead", ("rev_lookahead_kernel",)), ("pass", ("stream_update_block",)),
          ("inversion_rest", ("rev_build_kernel", "rev_extract_kernel", "rev_xb_kernel", "rev_record_kernel")),
          ("pricing", ("rev_pi_kernel", "rev_rn_kernel", "rev_enter_kernel", "rev_dir_kernel", "rev_leave_kernel")))


def kernel_split(A, b, c, k, **kw):
    import tempfile
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = api.revised_solve(A, b, c, max_iterations=k, **kw)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    us = {p: 0.0 for p, _ in PHASES}
    kernels = 0
    for e in events:
        if e.get("cat") != "kernel":
            continue
        kernels += 1
        for p, keys in PHASES:
            if any(key in e.get("name", "") for key in keys):
                us[p] += float(e.get("dur", 0.0))
    if kernels == 0:
        return dict(kernel_split="not measured (no kernel events in the profiler trace)")
    it = max(r["n_iters"], 1)
    inv = (us["lookahead"] + us["pass"] + us["inversion_rest"]) / (it + 1)
    return dict(kernel_us_per_inversion=round(inv, 1), lookahead_us_per_inversion=round(us["lookahead"] / (it + 1), 1),
                pass_us_per_inversion=round(us["pass"] / (it + 1), 1),
                kernel_us_per_pricing=round(us["pricing"] / it, 1), profiled_kernels=kernels)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory for r08_revised_stream.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cta-budget", type=float, default=30.0, help="seconds one one-CTA inversion may take")
    ap.add_argument("--tall-cap", type=int, default=3000)
    ap.add_argument("--oracle", action="store_true", help="check the full solves against the oracle")
    args = ap.parse_args()
    F.check(F.lib().lpx_init(0))
    res = dict(card=card(), rounds=args.rounds, method=__doc__.split("\n\n")[1])

    # 1. crossover sweep
    sweep = []
    for shape in ("square", "wide"):
        cta_inv_s, cta_m = None, None
        for m in (64, 96, 128, 256, 512, 1024):
            n = m if shape == "square" else 8 * m
            A, b, c = workloads.lp_decimal(m, n, 11)
            k = 8 if m <= 256 else 3
            row = dict(shape=shape, m=m, n=n, k=k)
            row["stream_k8"] = split(A, b, c, k, args.rounds, kernel=F.KERNEL_STREAM, kblock=8)
            predicted = None if cta_inv_s is None else cta_inv_s * (m / cta_m) ** 3
            if predicted is not None and predicted > args.cta_budget:
                row["cta"] = "not measured (predicted %.0f s per inversion)" % predicted
            else:
                try:
                    row["cta"] = split(A, b, c, min(k, 2), 1 if m >= 512 else args.rounds, kernel=F.KERNEL_CTA_GLOBAL)
                    cta_inv_s, cta_m = row["cta"]["first_call_ms"] / 1e3, m
                except F.LpxError as e:
                    row["cta"] = "refused: %s" % e
            sweep.append(row)
            print(json.dumps(row), flush=True)
    res["crossover_sweep"] = sweep

    # 2. block size
    ks = []
    for m in (1024, 2048):
        A, b, c = workloads.lp_decimal(m, m, 12)
        ld = (2 * m + 15) // 16 * 16
        row = dict(m=m, aug_mb=round(m * ld * 8 / 2**20, 1), aug_l2_resident=m * ld * 8 < L2_BYTES)
        for K in (1, 4, 8, 16):
            row["k%d" % K] = split(A, b, c, 2, args.rounds, kernel=F.KERNEL_STREAM, kblock=K)
        ks.append(row)
        print(json.dumps(row), flush=True)
    res["block_size"] = ks

    # 3. full solves past the one-CTA capacity, 4. the tall solve
    full = []
    for m, n, cap, gen in ((64, 20000, 10000, workloads.lp_integer), (32, 100000, 10000, workloads.lp_integer),
                           (1024, 1024, args.tall_cap, workloads.lp_decimal)):
        A, b, c = gen(m, n, 1)
        api.revised_solve(A, b, c, max_iterations=1)
        F.lib().lpx_reset_counters()
        t, r = timed(lambda: api.revised_solve(A, b, c, max_iterations=cap))
        launches = int(F.lib().lpx_kernel_launches())
        # set-up, then (n_iters + 1) x (5 pricing kernels + build + ceil(m / 8) x (look-ahead + pass) + extract + x_B)
        needed = 1 + (r["n_iters"] + 1) * (8 + 2 * ((m + 7) // 8))
        row = dict(m=m, n=n, generator=gen.__name__, max_iterations=cap, status=r["status"], iterations=r["n_iters"],
                   solve_ms=round(t, 1), ms_per_iteration=round(t / max(r["n_iters"], 1), 3), launches=launches,
                   launches_after_the_end=launches - needed)
        if args.oracle:
            import orc_ffi
            w = orc_ffi.revised_solve(A, b, c, max_iterations=cap)
            row["bit_exact_vs_oracle"] = bool(
                w["status"] == r["status"] and w["n_iters"] == r["n_iters"] and
                np.array_equal(w["enter"], r["enter"]) and np.array_equal(w["leave"], r["leave"]) and
                w["theta"].tobytes() == r["theta"].tobytes() and np.array_equal(w["basis"], r["basis"]) and
                w["Binv"].tobytes() == r["Binv"].tobytes() and w["xB"].tobytes() == r["xB"].tobytes() and
                (w["status"] < 0 or w["x"].tobytes() == r["x"].tobytes()))  # no oracle x for ITER_LIMIT
        full.append(row)
        print(json.dumps(row), flush=True)
    res["full_solves"] = full

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r08_revised_stream.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()

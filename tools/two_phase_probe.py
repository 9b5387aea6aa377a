"""Two-phase Simplex timings on one GPU -> <out>/r12_two_phase.json (default out: profiles/).

Workloads:
  mixed     4096 LPs of workloads.batch_mixed (64 x 128, Min, '<=' / '>=' / '=' rows, some b < 0, 5 % infeasible)
  all_le    4096 LPs of workloads.batch_c2 (64 x 128, Max, all '<=', b >= 0): no artificial, Phase I empty
Per workload:
  kernel    lpx_two_phase_solve_batched_dev on device buffers (status, both pivot counts, basis, x, z and the tableau;
            no pivot list), CUDA events around the call, warmed up, median of the timed repeats
  host      lpx_two_phase_solve_batched (host buffers in and out, wall clock around the call, which ends in a stream
            synchronise), median
  pivots    Phase I (drive-out included) and Phase II pivots per LP
  mixed: the oracle (oracle/orc_twophase.cpp) on one host thread and on all of them (ctypes releases the GIL), and
         the bit-equality of every output with it; HiGHS (scipy.optimize.linprog, method "highs") per LP on a sample,
         for context only: a different algorithm (dual simplex / IPM with presolve), not the same pivots
  all_le: lpx_primal_solve_batched_dev (AUTO: the register-resident kernel) timed the same way, alternated with the
          two-phase call, and the ratio; outputs checked bit-equal
The card name, power limit and max SM clock are read in the same call.
"""
import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--count", type=int, default=4096)
    args = ap.parse_args()
    import torch
    import orc_twophase_ffi as tp

    F.check(F.lib().lpx_init(0))
    dev = torch.device("cuda:0")
    res = dict(gpu=gpu_info(), reps=args.reps, count=args.count, workloads={})

    def events(fn, reps):
        fn()
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts)), ts

    def wall(fn, reps):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ts)), ts

    def device_call(A, b, c, rel, sense):
        count, m, n = A.shape
        rows, cols = api.two_phase_dims(m, n, rel)
        t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in dict(A=A, b=b, c=c).items()}
        trel = None if rel is None else torch.from_numpy(np.ascontiguousarray(rel, np.int32)).to(dev)
        o = dict(status=torch.zeros(count, dtype=torch.int32, device=dev),
                 phase1_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
                 n_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
                 basis=torch.zeros((count, m), dtype=torch.int32, device=dev),
                 x=torch.zeros((count, n), dtype=torch.float64, device=dev),
                 z=torch.zeros(count, dtype=torch.float64, device=dev),
                 tableau=torch.zeros((count, rows, cols), dtype=torch.float64, device=dev))
        s = torch.cuda.current_stream().cuda_stream

        def run():
            api.two_phase_solve_batched_dev(count, m, n, sense, t["A"].data_ptr(),
                                            None if trel is None else trel.data_ptr(), t["b"].data_ptr(),
                                            t["c"].data_ptr(), o["status"].data_ptr(), o["phase1_pivots"].data_ptr(),
                                            o["n_pivots"].data_ptr(), None, 0, o["basis"].data_ptr(),
                                            o["x"].data_ptr(), o["z"].data_ptr(), o["tableau"].data_ptr(), None, s)
        return run, t, o

    # ---- mixed ----------------------------------------------------------------------------------------------------
    A, b, c, rel, sense = workloads.batch_mixed(count=args.count, seed=1, sense=1, infeasible=0.05)
    run, _, o = device_call(A, b, c, rel, sense)
    k_ms, k_all = events(run, args.reps)
    h_ms, h_all = wall(lambda: api.two_phase_solve_batched(A, b, c, rel, sense, pivots_cap=0), max(3, args.reps // 3))
    got = {k: v.cpu().numpy() for k, v in o.items()}
    p1 = got["phase1_pivots"].astype(float)
    p2 = (got["n_pivots"] - got["phase1_pivots"]).astype(float)
    t0 = time.perf_counter()
    want = tp.two_phase_batch(A, b, c, rel, sense, pivots_cap=0)
    orc1 = time.perf_counter() - t0
    threads = os.cpu_count() or 1
    chunks = np.array_split(np.arange(args.count), threads)
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda ix: tp.two_phase_batch(A[ix], b[ix], c[ix], rel, sense, pivots_cap=0), chunks))
    orcN = time.perf_counter() - t0
    same = all(np.array_equal(got[k], want[k]) for k in ("status", "phase1_pivots", "n_pivots", "basis")) and all(
        got[k].tobytes() == want[k].tobytes() for k in ("x", "z", "tableau"))
    from scipy.optimize import linprog
    sample = range(0, args.count, max(1, args.count // 64))
    t0 = time.perf_counter()
    for k in sample:
        linprog(c[k], A_ub=np.vstack([A[k][rel == 0], -A[k][rel == 1]]),
                b_ub=np.concatenate([b[k][rel == 0], -b[k][rel == 1]]), A_eq=A[k][rel == 2], b_eq=b[k][rel == 2],
                method="highs")
    highs_ms = (time.perf_counter() - t0) * 1e3 / len(sample)
    res["workloads"]["mixed"] = dict(
        shape=[64, 128], sense="Min", rel_counts=[int((rel == r).sum()) for r in range(3)],
        negative_b_share=float((b < 0).mean()),
        status_counts={str(s): int((got["status"] == s).sum()) for s in np.unique(got["status"])},
        kernel_ms=k_ms, kernel_ms_all=k_all, host_call_ms=h_ms, host_call_ms_all=h_all,
        phase1_pivots_per_lp=float(p1.mean()), phase2_pivots_per_lp=float(p2.mean()),
        pivots_per_s_kernel=float(got["n_pivots"].sum() / (k_ms * 1e-3)),
        oracle_one_thread_s=orc1, oracle_threads=threads, oracle_all_threads_s=orcN, bit_equal_to_oracle=bool(same),
        highs_ms_per_lp=highs_ms, highs_sample=len(sample),
        highs_note="context only: HiGHS is a different algorithm (presolve, dual simplex / IPM), one LP at a time")
    print("mixed", json.dumps({k: v for k, v in res["workloads"]["mixed"].items() if not k.endswith("_all")}),
          flush=True)

    # ---- all <= : two-phase against the Primal Simplex batch (register kernel) ------------------------------------
    A, b, c = workloads.batch_c2(count=args.count, m=64, n=128, seed=1)
    run2, t2, o2 = device_call(A, b, c, None, 0)
    count, m, n = A.shape
    p = dict(status=torch.zeros(count, dtype=torch.int32, device=dev),
             n_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
             basis=torch.zeros((count, m), dtype=torch.int32, device=dev),
             x=torch.zeros((count, n), dtype=torch.float64, device=dev),
             z=torch.zeros(count, dtype=torch.float64, device=dev),
             tableau=torch.zeros((count, m + 1, n + m + 1), dtype=torch.float64, device=dev))
    s = torch.cuda.current_stream().cuda_stream

    def primal():
        api.primal_solve_batched_dev(count, m, n, 0, t2["A"].data_ptr(), None, t2["b"].data_ptr(), t2["c"].data_ptr(),
                                     p["status"].data_ptr(), p["n_pivots"].data_ptr(), p["basis"].data_ptr(),
                                     p["x"].data_ptr(), p["z"].data_ptr(), p["tableau"].data_ptr(), None, s)
    tw, pr = [], []
    for _ in range(max(3, args.reps // 3)):  # alternated
        tw.append(events(run2, 3)[0])
        pr.append(events(primal, 3)[0])
    eq = all(torch.equal(o2[k], p[k]) for k in ("status", "n_pivots", "basis")) and all(
        o2[k].cpu().numpy().tobytes() == p[k].cpu().numpy().tobytes() for k in ("x", "z", "tableau"))
    res["workloads"]["all_le"] = dict(
        shape=[64, 128], sense="Max", two_phase_kernel_ms=float(np.median(tw)), two_phase_kernel_ms_all=tw,
        primal_kernel_ms=float(np.median(pr)), primal_kernel_ms_all=pr,
        two_phase_over_primal=float(np.median(tw) / np.median(pr)), pivots_per_lp=float(p["n_pivots"].float().mean()),
        bit_equal_to_primal=bool(eq and not o2["phase1_pivots"].any()))
    print("all_le", json.dumps({k: v for k, v in res["workloads"]["all_le"].items() if not k.endswith("_all")}),
          flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r12_two_phase.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

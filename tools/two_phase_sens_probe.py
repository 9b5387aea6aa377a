"""Two-phase sensitivity report timings on one GPU -> <out>/r14_two_phase_sensitivity.json (default out: profiles/).

Batched: 4096 LPs of workloads.batch_mixed (64 x 128, Min, '<=' / '>=' / '=' rows, some b < 0, 5 % infeasible).
  kernel   lpx_two_phase_solve_sensitivity_batched_dev (status, both pivot counts, basis, x, z, report) against
           lpx_two_phase_solve_batched_dev with the same outputs and no report (no tableau, no pivot list), on device
           buffers.  CUDA events around `inner` back-to-back launches of one build, the two builds alternated per
           repeat; medians and their ratio.
  host     lpx_two_phase_solve_sensitivity_batched (host buffers in and out, the call ends in a stream synchronise)
           against lpx_two_phase_solve_batched without the tableau, wall clock, alternated, medians.
  outputs  the report and the solve outputs bit-equal to oracle/orc_twophase_sens.cpp.
Session: workloads.large_mixed at 1024 x 2048 and 4096 x 8192 (Min), solved once at K = 8 (solve time and pivots
  recorded), then lpx_session_two_phase_sensitivity against lpx_session_read_tableau (both synchronous, host
  buffers), wall clock, alternated, medians; and the strong-duality residual |b.y - objective| of the report.
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
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unavailable"


def median(ts):
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--inner", type=int, default=5)
    ap.add_argument("--count", type=int, default=4096)
    ap.add_argument("--sessions", default="1024x2048,4096x8192")
    args = ap.parse_args()
    import torch
    import orc_twophase_sens_ffi as tp

    F.check(F.lib().lpx_init(0))
    dev = torch.device("cuda:0")
    res = dict(gpu=gpu_info(), reps=args.reps, inner=args.inner, count=args.count)

    # ---- batched ---------------------------------------------------------------------------------------------------
    A, b, c, rel, sense = workloads.batch_mixed(count=args.count, seed=1, sense=1, infeasible=0.05)
    count, m, n = A.shape
    stride = api.sensitivity_stride(m, n)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in dict(A=A, b=b, c=c, rel=rel).items()}
    o = dict(status=torch.zeros(count, dtype=torch.int32, device=dev),
             phase1_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
             n_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
             basis=torch.zeros((count, m), dtype=torch.int32, device=dev),
             x=torch.zeros((count, n), dtype=torch.float64, device=dev),
             z=torch.zeros(count, dtype=torch.float64, device=dev),
             report=torch.zeros((count, stride), dtype=torch.float64, device=dev))
    s = torch.cuda.current_stream().cuda_stream
    ins = [t[k].data_ptr() for k in ("A", "rel", "b", "c")]
    outs = [o[k].data_ptr() for k in ("status", "phase1_pivots", "n_pivots")]

    def plain():
        api.two_phase_solve_batched_dev(count, m, n, sense, *ins, *outs, None, 0, o["basis"].data_ptr(),
                                        o["x"].data_ptr(), o["z"].data_ptr(), None, None, s)

    def report():
        api.two_phase_sensitivity_batched_dev(count, m, n, sense, *ins, *outs, o["basis"].data_ptr(),
                                              o["x"].data_ptr(), o["z"].data_ptr(), o["report"].data_ptr(), None, s)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.inner):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.inner

    for fn in (plain, report, plain, report):  # warm-up: module load, attributes, workspace
        fn()
    torch.cuda.synchronize()
    tk = dict(plain=[], report=[])
    for _ in range(args.reps):
        tk["plain"].append(timed(plain))
        tk["report"].append(timed(report))
    got = {k: v.cpu().numpy() for k, v in o.items()}

    def wall(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    hplain = lambda: api.two_phase_solve_batched(A, b, c, rel, sense, pivots_cap=0, want_tableau=False)  # noqa: E731
    hrep = lambda: api.two_phase_sensitivity_batched(A, b, c, rel, sense)  # noqa: E731
    hplain(), hrep()
    th = dict(plain=[], report=[])
    for _ in range(max(3, args.reps // 2)):
        th["plain"].append(wall(hplain))
        th["report"].append(wall(hrep))
    host = hrep()

    threads = os.cpu_count() or 1
    chunks = np.array_split(np.arange(count), threads)
    with cf.ThreadPoolExecutor(threads) as ex:
        parts = list(ex.map(lambda ix: tp.two_phase_sensitivity_batch(A[ix], b[ix], c[ix], rel, sense, pivots_cap=0),
                            chunks))
    want = {k: np.concatenate([p[k] for p in parts]) for k in ("status", "phase1_pivots", "n_pivots", "basis", "x", "z",
                                                                "report")}
    same = all(np.array_equal(got[k], want[k]) and np.array_equal(host[k], want[k])
               for k in ("status", "phase1_pivots", "n_pivots", "basis")) and all(
        got[k].tobytes() == want[k].tobytes() and host[k].tobytes() == want[k].tobytes() for k in ("x", "z", "report"))
    p1 = got["phase1_pivots"].astype(float)
    res["batched"] = dict(
        workload="batch_mixed(count=%d, m=64, n=128, seed=1, sense=Min, infeasible=0.05)" % count,
        kernel_ms=dict(plain=median(tk["plain"]), report=median(tk["report"]),
                       ratio=median(tk["report"]) / median(tk["plain"]), all=tk),
        host_ms=dict(plain=median(th["plain"]), report=median(th["report"]), all=th),
        phase1_pivots_mean=float(p1.mean()), phase2_pivots_mean=float((got["n_pivots"] - p1).mean()),
        optimal=int((got["status"] == 0).sum()), bit_equal_to_oracle=bool(same))

    # ---- sessions -------------------------------------------------------------------------------------------------
    res["session"] = []
    for shape in args.sessions.split(","):
        sm, sn = (int(v) for v in shape.split("x"))
        A1, b1, c1, rel1, sense1 = workloads.large_mixed(sm, sn)
        ses = api.Session(A1, b1, c1, rel1, sense1, max_iterations=10 ** 7, kblock=8, two_phase=True)
        try:
            t0 = time.perf_counter()
            st, piv = ses.step(10 ** 7)
            solve_s = time.perf_counter() - t0
            _, p1s = ses.two_phase_info()
            first = ses.two_phase_sensitivity()["report"]
            T = np.zeros((ses.rows, ses.cols))
            rep = np.zeros(api.sensitivity_stride(sm, sn))
            L = F.lib()
            ts = dict(report=[], read_tableau=[])
            for _ in range(args.reps):
                ts["report"].append(wall(lambda: F.check(L.lpx_session_two_phase_sensitivity(ses._h, F.ptr(rep)))))
                ts["read_tableau"].append(wall(lambda: F.check(L.lpx_session_read_tableau(ses._h, F.ptr(T)))))
            _, _, z = ses.solution()
            obj = -z if sense1 == 1 else z
            res["session"].append(dict(
                workload="large_mixed(%d, %d), K = 8" % (sm, sn), status=st, pivots=piv, phase1_pivots=p1s,
                solve_s=solve_s, report_ms=median(ts["report"]), read_tableau_ms=median(ts["read_tableau"]), all=ts,
                repeat_bit_equal=bool(rep.tobytes() == first.tobytes()),
                strong_duality_residual=float(abs(np.dot(b1, rep[:sm]) - obj)), objective=float(obj)))
        finally:
            ses.close()

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r14_two_phase_sensitivity.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "session"} | dict(
        session=[{k: v for k, v in d.items() if k != "all"} for d in res["session"]]), default=str)[:3000])


if __name__ == "__main__":
    main()

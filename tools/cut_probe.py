"""Gomory cutting-plane timings on one GPU -> <out>/r09_cutting_plane.json (default out: profiles/).

Workloads: C4-shaped IPs (workloads.ip_c4, 60 x 120) x 148 and x 592, and 8 x 12 x 4096 — integer data with a
fractional root, so every IP runs all 50 rounds (the reference's cut never removes the current vertex).
  new     lpx_cutting_plane_batched (host buffers, tableau not requested; wall clock around the call, which ends in a
          stream synchronise) and lpx_cutting_plane_batched_dev (CUDA events around the launch on device tensors)
  driver  the baseline: a Python round driver over api.primal_solve_batched — round k solves every instance still
          running as one batched call of shape m + k - 1 and makes the cuts in numpy; checked bit-equal to the new call
          (ends, rounds, pivots, cuts, final LPs) and timed in the same rounds, alternated with it
  host    the per-IP host route (host_ffi.solve_text, "cutting plane": one lpx_primal_solve per round, text included)
  oracle  oracle/orc_cut.cpp (CuttingPlane.Solve's numbers, no text) on one host thread
The card name, power limit and max SM clock are read in the same call.
"""
import argparse
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

R = F.CUT_MAX_ROUNDS


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unavailable"


def batch(count, m, n, seed):
    Ak, bk, ck = zip(*[workloads.ip_c4(m=m, n=n, seed=seed + k) for k in range(count)])
    return np.stack(Ak), np.stack(bk), np.stack(ck)


def round_driver(A, b, c, max_iterations=10000):
    """CuttingPlane.Solve for a batch (all rows '<=', Max) from one primal_solve_batched call per round."""
    count, m, n = A.shape
    end = np.full(count, F.CUT_INCOMPLETE, np.int32)
    n_rounds = np.zeros(count, np.int32)
    lp_status, lp_pivots = np.full((count, R), F.RUNNING, np.int32), np.zeros((count, R), np.int32)
    cut_a, cut_b = np.zeros((count, R, n)), np.zeros((count, R))
    final = {}
    active = np.arange(count)
    for r in range(R):
        if len(active) == 0:
            break
        Ak = np.concatenate([A[active], cut_a[active, :r]], axis=1)
        bk = np.concatenate([b[active], cut_b[active, :r]], axis=1)
        res = api.primal_solve_batched(Ak, bk, c[active], max_iterations=max_iterations)
        lp_status[active, r], lp_pivots[active, r] = res["status"], res["n_pivots"]
        n_rounds[active] = r + 1
        keep = []
        for q, k in enumerate(active):
            if res["status"][q] < 0:
                end[k] = F.CUT_LP_ERROR
                continue
            x = res["x"][q]
            f = x - np.floor(x)
            frac = np.nonzero((f > 1e-9) & (f < 1 - 1e-9))[0]
            if len(frac) == 0:
                end[k] = F.CUT_INTEGER
                final[k] = (res["basis"][q], x, res["z"][q], res["tableau"][q])
                continue
            row = int(np.nonzero(res["basis"][q] == frac[0])[0][0]) + 1
            trow = res["tableau"][q][row]
            fa = trow[:n] - np.floor(trow[:n])
            cut_a[k, r] = np.where(fa > 1e-9, fa, 0.0)
            cut_b[k, r] = trow[-1] - np.floor(trow[-1])
            keep.append(k)
        active = np.array(keep, dtype=np.int64)
    return dict(end=end, n_rounds=n_rounds, lp_status=lp_status, lp_pivots=lp_pivots, cut_a=cut_a, cut_b=cut_b,
                final=final)


def same(new, drv):
    ok = (np.array_equal(new["end"], drv["end"]) and np.array_equal(new["n_rounds"], drv["n_rounds"])
          and np.array_equal(new["lp_status"], drv["lp_status"]) and np.array_equal(new["lp_pivots"], drv["lp_pivots"])
          and new["cut_a"].tobytes() == drv["cut_a"].tobytes() and new["cut_b"].tobytes() == drv["cut_b"].tobytes())
    for k, (basis, x, z, T) in drv["final"].items():
        rows = len(basis) + 1
        ok = ok and np.array_equal(new["basis"][k][: len(basis)], basis) and new["x"][k].tobytes() == x.tobytes()
        ok = ok and new["z"][k] == z and new["tableau"][k].reshape(-1)[: T.size].tobytes() == T.tobytes() and rows > 0
    return bool(ok)


def dev_timing(A, b, c, reps):
    import torch
    dev = torch.device("cuda:0")
    count, m, n = A.shape
    max_rows, max_cols = api.cutting_plane_dims(m, n)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in (("A", A), ("b", b), ("c", c))}
    i32 = dict(dtype=torch.int32, device=dev)
    o = dict(end=torch.zeros(count, **i32), n_rounds=torch.zeros(count, **i32), lp_pivots=torch.zeros((count, R), **i32),
             cut_a=torch.zeros((count, R, n), dtype=torch.float64, device=dev),
             cut_b=torch.zeros((count, R), dtype=torch.float64, device=dev))
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        api.cutting_plane_batched_dev(count, m, n, 0, t["A"].data_ptr(), None, t["b"].data_ptr(), t["c"].data_ptr(),
                                      o["end"].data_ptr(), o["n_rounds"].data_ptr(), None, None,
                                      o["lp_pivots"].data_ptr(), None, None, o["cut_a"].data_ptr(),
                                      o["cut_b"].data_ptr(), None, None, None, None, total.data_ptr(), stream)
    launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps, int(o["n_rounds"].sum().item()), int(o["lp_pivots"].sum().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory for r09_cutting_plane.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import host_ffi
    import orc_cut_ffi

    F.check(F.lib().lpx_init(0))
    res = dict(gpu=gpu_info(), workloads=[])
    for count, m, n, seed in ((148, 60, 120, 1000), (592, 60, 120, 1000), (4096, 8, 12, 5000)):
        A, b, c = batch(count, m, n, seed)
        new = api.cutting_plane_batched(A, b, c)  # warm-up of the shape, and the results the driver must equal
        drv = round_driver(A, b, c)
        w = dict(shape=[m, n], count=count, ends={str(e): int((new["end"] == e).sum()) for e in range(3)},
                 rounds=int(new["n_rounds"].sum()), lp_pivots=int(new["lp_pivots"].sum()), bit_equal=same(new, drv))
        t_new, t_drv = [], []
        for _ in range(args.rounds):  # alternated in the same rounds
            t0 = time.perf_counter()
            api.cutting_plane_batched(A, b, c, want_tableau=False)
            t_new.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            round_driver(A, b, c)
            t_drv.append(time.perf_counter() - t0)
        tn, td = float(np.median(t_new)), float(np.median(t_drv))
        t_dev, rounds, piv = dev_timing(A, b, c, args.reps)
        assert rounds == w["rounds"] and piv == w["lp_pivots"]

        def rates(t):
            return dict(seconds=t, ips_per_s=count / t, rounds_per_s=rounds / t, lp_pivots_per_s=piv / t)
        w["new_host_buffers"] = rates(tn)
        w["new_dev_kernel"] = rates(t_dev)
        w["driver_primal_batched"] = rates(td)
        w["speedup_host_vs_driver"] = td / tn
        # the per-IP host route and the oracle, on a few instances
        few = 2 if m >= 60 else 8
        t0 = time.perf_counter()
        for k in range(few):
            h = host_ffi.solve_text(workloads.lp_to_text(A[k], b[k], c[k]), "cutting plane")
            assert len(h["cuts"]) == new["n_cuts"][k]
        w["host_route_seconds_per_ip"] = (time.perf_counter() - t0) / few
        t0 = time.perf_counter()
        for k in range(few):
            o = orc_cut_ffi.cutting_plane(A[k], b[k], c[k])
            assert o["cut_b"].tobytes() == new["cut_b"][k].tobytes()
        w["oracle_seconds_per_ip"] = (time.perf_counter() - t0) / few
        res["workloads"].append(w)
        print(json.dumps(w), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r09_cutting_plane.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()

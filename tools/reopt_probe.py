"""Re-optimization timings on one GPU -> <out>/r05_reopt.json (default out: profiles/).

One C2-shaped base (64 x 128, workloads.batch_c2) and 4096 queries of each kind through lpx_reoptimize_batched_dev,
CUDA events around `reps` launches per round.  For the RHS scenarios with b + db >= 0 a cold re-solve of all 4096
modified LPs with lpx_primal_solve_batched_dev is timed in the same rounds, alternated with the warm run, and its z is
compared with the warm z.  The oracle (oracle/orc_reopt.cpp, one host thread) is timed on the same queries.  The card
name, power limit and max SM clock are read in the same call.
"""
import argparse
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

RHS, COST, ROW, COL = 1, 2, 3, 4


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory for r05_reopt.json")
    ap.add_argument("--count", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    import orc_ffi
    import orc_reopt_ffi

    F.check(F.lib().lpx_init(0))
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    m, n, count = 64, 128, args.count
    A, b, c = workloads.batch_c2(count=1, m=m, n=n, seed=3)
    A, b, c = A[0], b[0], c[0]
    base = orc_ffi.primal_solve(A, b, c)
    tb = {"status": torch.tensor([base["status"]], dtype=torch.int32, device=dev),
          "basis": torch.from_numpy(base["basis"]).to(dev), "tableau": torch.from_numpy(base["tableau"]).to(dev)}
    rng = np.random.default_rng(0)
    # RHS: one entry per query, across and beyond its range, b + db >= 0 (so the cold re-solve is a Primal Simplex LP)
    d = np.zeros((count, m))
    i = rng.integers(m, size=count)
    d[np.arange(count), i] = np.maximum(np.round(rng.uniform(-0.9, 1.5, count) * b[i], 2), -b[i])
    row_a = np.where(rng.random((count, n)) < 0.1, rng.integers(1, 9, (count, n)), 0).astype(float)
    row = np.hstack([row_a, np.zeros((count, 1)), np.round(rng.uniform(0.3, 1.2, count) * (row_a @ base["x"]), 2)[:, None]])
    col_a = rng.integers(0, 9, (count, m)).astype(float)
    col_a[rng.random((count, m)) < 0.7] = 0.0
    col = np.hstack([col_a, rng.integers(1, 30, (count, 1)).astype(float)])
    queries = {"rhs": (RHS, d), "row": (ROW, row), "col": (COL, col)}
    src = torch.zeros(count, dtype=torch.int32, device=dev)

    def outputs(kind):
        rows, cols = api.reopt_dims(kind, m, n)
        nx = n + 1 if kind == COL else n
        return dict(status=torch.zeros(count, dtype=torch.int32, device=dev),
                    n_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
                    basis=torch.zeros((count, rows - 1), dtype=torch.int32, device=dev),
                    x=torch.zeros((count, nx), dtype=torch.float64, device=dev),
                    z=torch.zeros(count, dtype=torch.float64, device=dev))

    def warm_launch(kind, pay, o):
        api.reoptimize_batched_dev(kind, count, m, n, 0, None, tb["status"].data_ptr(), tb["basis"].data_ptr(),
                                   tb["tableau"].data_ptr(), src.data_ptr(), pay.data_ptr(), o["status"].data_ptr(),
                                   o["n_pivots"].data_ptr(), None, 0, o["basis"].data_ptr(), o["x"].data_ptr(),
                                   o["z"].data_ptr(), None, None, stream)

    cold_A = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(A, (count, m, n)))).to(dev)
    cold_b = torch.from_numpy(b[None, :] + d).to(dev)
    cold_c = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(c, (count, n)))).to(dev)
    cold = dict(status=torch.zeros(count, dtype=torch.int32, device=dev),
                n_pivots=torch.zeros(count, dtype=torch.int32, device=dev),
                basis=torch.zeros((count, m), dtype=torch.int32, device=dev),
                x=torch.zeros((count, n), dtype=torch.float64, device=dev),
                z=torch.zeros(count, dtype=torch.float64, device=dev))

    def cold_launch():
        api.primal_solve_batched_dev(count, m, n, 0, cold_A.data_ptr(), None, cold_b.data_ptr(), cold_c.data_ptr(),
                                     cold["status"].data_ptr(), cold["n_pivots"].data_ptr(), cold["basis"].data_ptr(),
                                     cold["x"].data_ptr(), cold["z"].data_ptr(), None, None, stream)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.reps

    pays = {k: torch.from_numpy(np.ascontiguousarray(p)).to(dev) for k, (_, p) in queries.items()}
    outs = {k: outputs(kind) for k, (kind, _) in queries.items()}
    times = {k: [] for k in list(queries) + ["cold_rhs"]}
    for _ in range(args.rounds):
        for k, (kind, _) in queries.items():
            times[k].append(timed(lambda: warm_launch(kind, pays[k], outs[k])))
        times["cold_rhs"].append(timed(cold_launch))
    result = {"gpu": gpu_info(), "base": {"m": m, "n": n, "base_pivots": int(base["n_pivots"]), "z": base["z"]},
              "queries": count, "rounds": args.rounds, "launches_per_round": args.reps}
    for k, (kind, pay) in queries.items():
        o = {f: v.cpu().numpy() for f, v in outs[k].items()}
        t0 = time.perf_counter()
        ref = orc_reopt_ffi.reopt(kind, m, n, [base["status"]], [base["basis"]], [base["tableau"]], pay,
                                  src=np.zeros(count, np.int32), pivots_cap=0)
        t_orc = time.perf_counter() - t0
        ms = float(np.median(times[k]))
        result[k] = {"ms_per_batch_median": ms, "ms_per_batch_all": times[k], "queries_per_s": count / ms * 1e3,
                     "warm_pivots_per_query": float(o["n_pivots"].mean()),
                     "status_counts": {str(s): int((o["status"] == s).sum()) for s in np.unique(o["status"])},
                     "oracle_host_s": t_orc, "oracle_queries_per_s": count / t_orc,
                     "bit_equal_to_oracle": bool(np.array_equal(o["status"], ref["status"]) and
                                                 o["z"].tobytes() == ref["z"].tobytes() and
                                                 o["x"].tobytes() == ref["x"].tobytes())}
    cz = cold["z"].cpu().numpy()
    cs = cold["status"].cpu().numpy()
    wz = outs["rhs"]["z"].cpu().numpy()
    ws = outs["rhs"]["status"].cpu().numpy()
    both = (cs == 0) & (ws == 0)
    ms = float(np.median(times["cold_rhs"]))
    result["cold_rhs"] = {"ms_per_batch_median": ms, "ms_per_batch_all": times["cold_rhs"],
                          "lps_per_s": count / ms * 1e3, "pivots_per_lp": float(cold["n_pivots"].cpu().numpy().mean()),
                          "status_equal": bool(np.array_equal(cs, ws)),
                          "z_max_rel_diff": float(np.max(np.abs(cz[both] - wz[both]) / np.maximum(1.0, np.abs(cz[both]))))}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r05_reopt.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {a: b for a, b in v.items() if "all" not in a})
                      for k, v in result.items()}, indent=1))


if __name__ == "__main__":
    main()

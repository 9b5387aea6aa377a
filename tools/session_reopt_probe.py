"""What-if queries on one large optimal session -> <out>/r06_session_reopt.json (default out: profiles/).

One C3 base (4096 x 8192, workloads.large_c3) solved to OPTIMAL in a streaming session.  The sensitivity report picks
the queries: an RHS change just past its range and one well past it, a cost change that lets one column enter, a cap
on one basic variable (ROW) and a new activity priced just above its rows' shadow prices (COL).  Per query, in
`rounds` alternating rounds: the warm route (lpx_session_reoptimize, then steps to a terminal status; host clock
around work that ends in a device synchronise) and the same modified model solved cold by a fresh session
(lpx_session_open + steps).  Medians are reported with the pivot counts and both objective values.  The per-pivot
times of the Dual Simplex pair (stream_dual_select_kernel / stream_update_kernel<4>) come from lpx_session_profile on
a fresh query session.  The card name, power limit and max SM clock are read in the same call.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402

RHS, COST, ROW, COL = 1, 2, 3, 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def to_end(s):
    st, tot = F.RUNNING, 0
    while st == F.RUNNING:
        st, tot = s.step(512)
    return st, tot


def queries(A, b, c, base_x, basis, rep):
    m, n = A.shape
    shadow, rhs_hi, reduced = rep["shadow"], rep["rhs_hi"], rep["reduced"]
    gap = np.where((shadow > 0) & np.isfinite(rhs_hi), rhs_hi - b, np.inf)
    i = int(np.argmin(gap))
    near, far = np.zeros(m), np.zeros(m)
    near[i] = gap[i] * 1.001 + 1e-3
    far[i] = gap[i] + 0.5 * b[i]
    nb = np.setdiff1d(np.arange(n), basis)
    j = int(nb[np.argmin(reduced[nb] + 1e9 * (reduced[nb] <= 1e-6))])
    dc = np.zeros(n)
    dc[j] = reduced[j] * 1.001 + 1e-6
    bj = int(np.flatnonzero(base_x > 1e-6)[0])
    row = np.zeros(n + 2)
    row[bj] = 1.0
    row[n + 1] = float(np.round(base_x[bj] * 0.99, 6))
    rows3 = np.argsort(-shadow)[:3]
    col = np.zeros(m + 1)
    col[rows3] = 1.0
    col[m] = float(shadow[rows3].sum()) * 1.01 + 1e-6
    # name -> (kind, payload, cold model (A, b, c), what the query is)
    return {
        "rhs_just_past": (RHS, near, (A, b + near, c), f"b_{i} to {rhs_hi[i]:.6g} + 0.1 % of the gap (range hi)"),
        "rhs_well_past": (RHS, far, (A, b + far, c), f"b_{i} to its range hi + 0.5 b_{i}"),
        "cost": (COST, dc, (A, b, c + dc), f"c_{j} (non-basic) up by its reduced cost + 0.1 %"),
        "row": (ROW, row, (np.vstack([A, row[:n]]), np.append(b, row[n + 1]), c), f"x_{bj} <= 0.99 x*_{bj}"),
        "col": (COL, col, (np.hstack([A, col[:m, None]]), b, np.append(c, col[m])),
                "new column: 1 in the three rows of largest shadow price, c_new = 1.01 x their sum"),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory for r06_session_reopt.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--m", type=int, default=4096)
    ap.add_argument("--n", type=int, default=8192)
    args = ap.parse_args()
    F.check(F.lib().lpx_init(0))
    F.lib().lpx_session_profile.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    A, b, c = workloads.large_c3(args.m, args.n)
    t0 = time.perf_counter()
    s = api.Session(A, b, c)
    st, base_piv = to_end(s)
    base_ms = (time.perf_counter() - t0) * 1e3
    assert st == F.OPTIMAL, st
    basis, x, z = s.solution()
    rep = s.sensitivity()
    res = dict(card=card(), shape=[args.m, args.n], base=dict(pivots=base_piv, ms_open_to_optimal=round(base_ms, 2)),
               rounds=args.rounds, queries={})
    qs = queries(A, b, c, x, basis, rep)
    for name, (kind, pay, (A2, b2, c2), what) in qs.items():
        warm_ms, cold_ms = [], []
        for _ in range(args.rounds):
            t0 = time.perf_counter()
            q = s.reoptimize(kind, pay)
            wst, wpiv = to_end(q)
            warm_ms.append((time.perf_counter() - t0) * 1e3)
            wz = q.solution()[2]
            q.close()
            t0 = time.perf_counter()
            cs = api.Session(A2, b2, c2)
            cst, cpiv = to_end(cs)
            cold_ms.append((time.perf_counter() - t0) * 1e3)
            cz = cs.solution()[2]
            cs.close()
        res["queries"][name] = dict(
            kind=kind, what=what, warm_status=wst, warm_pivots=wpiv, warm_ms_median=round(float(np.median(warm_ms)), 2),
            warm_ms=[round(v, 2) for v in warm_ms], cold_status=cst, cold_pivots=cpiv,
            cold_ms_median=round(float(np.median(cold_ms)), 2), cold_ms=[round(v, 2) for v in cold_ms], z_warm=wz,
            z_cold=cz, warm_faster=bool(np.median(warm_ms) < np.median(cold_ms)))
        print(name, json.dumps(res["queries"][name]), flush=True)
    # the Dual Simplex pair, timed pivot by pivot on a fresh query session (events around each kernel)
    kind, pay = qs["rhs_well_past"][:2]
    npiv = min(res["queries"]["rhs_well_past"]["warm_pivots"], 64)
    if npiv > 0:
        q = s.reoptimize(kind, pay)
        us = (C.c_double * 3)()
        F.check(F.lib().lpx_session_profile(q._h, npiv, us))
        q.close()
        res["dual_per_pivot_us"] = dict(pivots=npiv, select=round(us[0], 2), passes=round(us[1], 2),
                                        per_pivot=round(us[2], 2))
    s.close()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r06_session_reopt.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

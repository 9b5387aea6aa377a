"""Dual Simplex on a large LP in HBM -> <out>/r07_dual_session.json (default out: profiles/).

1. large_dual (2048 '=' rows x 8192, 4097 x 12289 tableau: C3's shape), per protocol: the per-pivot Dual Simplex pair
   (stream_protocol 1) and the blocked dual look-ahead with K = 8 and 16 (stream_protocol 4, the same kernels as 0):
   lpx_session_profile (CUDA events around each kernel, run back to back) gives the look-ahead / select time, the pass
   time and the time per block; per pivot = per block / K.
2. The cold Dual Simplex solve of the same model, open to terminal status (host clock, ends in a synchronise), per
   protocol, in alternated rounds; medians with the pivot counts.
3. The RHS query of r06 1 251 dual pivots from its C3 base (b_i to its range hi + 0.5 b_i), per-pivot against blocked,
   against the cold re-solve of the modified model by a fresh Primal Simplex session, in alternated rounds.
4. The per-CTA Dual Simplex (lpx_dual_solve, LPX_KERNEL_CTA_GLOBAL: one SM) against the stream (LPX_KERNEL_STREAM) on
   large_dual(1024, 4096), a shape both accept.
The card name, power limit and max SM clock are read in the same call.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402
from session_reopt_probe import card, queries, to_end  # noqa: E402

PROTOCOLS = {"per_pivot": dict(single_cta_select=1), "blocked_k8": dict(single_cta_select=4, kblock=8),
             "blocked_k16": dict(single_cta_select=4, kblock=16)}


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def med(v):
    return round(float(np.median(v)), 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory for r07_dual_session.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--skip-cta", action="store_true", help="skip the one-SM per-CTA comparison")
    args = ap.parse_args()
    F.check(F.lib().lpx_init(0))
    F.lib().lpx_session_profile.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    res = dict(card=card(), rounds=args.rounds)

    # 1. kernel times at C3's shape
    A, b, c, rel, sense = workloads.large_dual()
    prof = {}
    for name, opts in PROTOCOLS.items():
        s = api.Session(A, b, c, rel=rel, sense=sense, dual=True, **opts)
        k = opts.get("kblock", 1)
        nb = 64 if k == 1 else 128 // k
        s.step(16)  # past the first pivots, warmed up
        us = (C.c_double * 3)()
        F.check(F.lib().lpx_session_profile(s._h, nb, us))
        prof[name] = dict(units=nb, pivots_per_unit=k, lookahead_or_select_us=round(us[0], 2),
                          pass_us=round(us[1], 2), per_unit_us=round(us[2], 2), per_pivot_us=round(us[2] / k, 2))
        s.close()
        print(name, json.dumps(prof[name]), flush=True)
    res["large_dual_kernels"] = dict(shape=[2048, 8192], tableau=[4097, 12289], **prof)

    # 2. cold Dual Simplex solves, open to terminal status
    cold = {name: [] for name in PROTOCOLS}
    outcome = {}
    for _ in range(args.rounds):
        for name, opts in PROTOCOLS.items():
            def solve():
                s = api.Session(A, b, c, rel=rel, sense=sense, dual=True, **opts)
                st, tot = to_end(s)
                z = s.solution()[2]
                s.close()
                return st, tot, z
            ms, (st, tot, z) = timed(solve)
            cold[name].append(ms)
            outcome[name] = dict(status=st, pivots=tot, z=z)
    res["large_dual_cold_solve"] = {name: dict(ms_median=med(cold[name]), ms=[round(v, 2) for v in cold[name]],
                                               **outcome[name]) for name in PROTOCOLS}
    print(json.dumps(res["large_dual_cold_solve"]), flush=True)
    del A, b, c

    # 3. the RHS query 1 251 dual pivots from its C3 base, against its cold re-solve
    A, b, c = workloads.large_c3()
    s = api.Session(A, b, c)
    assert to_end(s)[0] == F.OPTIMAL
    basis, x, _ = s.solution()
    kind, pay, (A2, b2, c2), what = queries(A, b, c, x, basis, s.sensitivity())["rhs_well_past"]
    warm = {"per_pivot": [], "blocked_k8": [], "blocked_k16": []}
    cold_ms = []
    warm_out = {}
    for _ in range(args.rounds):
        for name in warm:
            def query():
                q = s.reoptimize(kind, pay, **PROTOCOLS[name])
                st, tot = to_end(q)
                z = q.solution()[2]
                q.close()
                return st, tot, z
            ms, (st, tot, z) = timed(query)
            warm[name].append(ms)
            warm_out[name] = dict(status=st, pivots=tot, z=z)
        def resolve():
            cs = api.Session(A2, b2, c2)
            st, tot = to_end(cs)
            z = cs.solution()[2]
            cs.close()
            return st, tot, z
        ms, (cst, cpiv, cz) = timed(resolve)
        cold_ms.append(ms)
    s.close()
    res["rhs_query"] = dict(what=what, cold_resolve=dict(status=cst, pivots=cpiv, z=cz, ms_median=med(cold_ms),
                                                          ms=[round(v, 2) for v in cold_ms]),
                            **{name: dict(ms_median=med(v), ms=[round(t, 2) for t in v], **warm_out[name])
                               for name, v in warm.items()})
    print(json.dumps(res["rhs_query"]), flush=True)
    del A, b, c, A2, b2, c2

    # 4. one SM (per-CTA global-memory kernel) against the whole GPU
    if not args.skip_cta:
        A, b, c, rel, sense = workloads.large_dual(1024, 4096)
        cta = {}
        for name, kernel in (("per_cta_global", F.KERNEL_CTA_GLOBAL), ("stream", F.KERNEL_STREAM)):
            ms, r = timed(lambda: api.dual_solve(A, b, c, rel, sense, kernel=kernel))
            cta[name] = dict(ms=round(ms, 2), status=r["status"], pivots=r["n_pivots"], z=r["z"])
        cta["same_bits"] = bool(np.array_equal(np.asarray(cta["per_cta_global"]["z"]).view(np.uint64),
                                               np.asarray(cta["stream"]["z"]).view(np.uint64)))
        res["per_cta_vs_stream"] = dict(shape=[1024, 4096], tableau=list(api.tableau_dims(1024, 4096, rel)), **cta)
        print(json.dumps(res["per_cta_vs_stream"]), flush=True)

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r07_dual_session.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

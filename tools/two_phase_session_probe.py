"""Two-phase session timings on one GPU -> <out>/r13_two_phase_session.json (default out: profiles/).

1. workloads.large_mixed(4096, 8192), Min ('<=' / '>=' / '=' rows, some b < 0; the batched call refuses it):
   open time (host clock around the synchronous open); Phase I, drive-out and Phase II pivots (a session stepped in
   blocks of 64 pivots, then one pivot at a time, until the phase turns 2 gives the Phase I pivots before the
   drive-out); the solve after open to the terminal status at K = 8 and 16 (default pass, host clock ending in a
   synchronise), bits checked equal across K; the first 4096 pivots at K = 1, 8 and 16 (host clock), since the whole
   solve at K = 1 takes minutes; look-ahead and pass microseconds per block from lpx_session_profile (CUDA events, 20
   blocks run back to back after the first 16 pivots).
2. One SM against the whole GPU: the same LP through lpx_two_phase_solve_batched (one CTA, global-memory tableau;
   host buffers, wall clock) and through the session (open + solve, wall clock), on large_mixed family members the
   batched call accepts; every output checked bit-equal.
3. large_c3: the two-phase session against the primal session (its default protocol, pipelined), open + solve,
   alternated rounds, medians and the ratio; outputs checked bit-equal.
The card name, power limit and max SM clock are read in the same call.
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
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402

RUNNING = F.RUNNING


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unavailable"


def solve(s):
    st = RUNNING
    while st == RUNNING:
        st, tot = s.step(512)
    return st, tot


def outputs(s, st, tot, cap):
    basis, x, z = s.solution()
    return dict(status=st, n_pivots=tot, phase1=s.two_phase_info()[1], pivots=s.pivots(cap), basis=basis, x=x,
                z=np.float64(z), tableau=s.tableau())


def same(a, b):
    for k in a:
        if k in b and np.asarray(a[k]).tobytes() != np.asarray(b[k]).tobytes():
            return False
    return True


def timed_session(A, b, c, rel, sense, cap, two_phase=True, **kw):
    t0 = time.perf_counter()
    s = api.Session(A, b, c, rel, sense, two_phase=two_phase, **kw)
    t1 = time.perf_counter()
    st, tot = solve(s)
    t2 = time.perf_counter()
    out = outputs(s, st, tot, cap) if two_phase else None
    if not two_phase:
        basis, x, z = s.solution()
        out = dict(status=st, n_pivots=tot, pivots=s.pivots(cap), basis=basis, x=x, z=np.float64(z),
                   tableau=s.tableau())
    s.close()
    return (t1 - t0) * 1e3, (t2 - t1) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    F.check(F.lib().lpx_init(0))
    F.lib().lpx_session_profile.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    res = dict(gpu=gpu_info(), rounds=args.rounds)
    cap, it = 2000000, 2000000

    # 1. the C3-sized mixed model
    A, b, c, rel, sense = workloads.large_mixed(4096, 8192)
    try:
        api.two_phase_solve_batched(A[None], b[None], c[None], rel, sense, pivots_cap=1, want_tableau=False)
        batched = "accepted"
    except F.LpxError as e:
        batched = f"refused, code {e.code}"
    r1 = dict(shape=[4096, 8192], sense="Min", batched_call=batched, rows_le_ge_eq=[int((rel == k).sum()) for k in range(3)],
              negative_b=int((b < 0).sum()), runs={})
    ref = None
    for K in (16, 8):
        to, ts, out = timed_session(A, b, c, rel, sense, cap, kblock=K, max_iterations=it)
        ref = ref or out
        assert same(out, ref), f"K={K}: outputs differ from K=16"
        r1["runs"][f"K={K}"] = dict(open_ms=round(to, 1), solve_ms=round(ts, 1))
        print("mixed", K, r1["runs"][f"K={K}"], flush=True)
    window = {}
    for K in (1, 8, 16):
        s = api.Session(A, b, c, rel, sense, kblock=K, max_iterations=it, two_phase=True)
        s.step(64)
        t0 = time.perf_counter()
        st, tot = s.step(4096)
        window[f"K={K}"] = dict(pivots=tot - 64, ms=round((time.perf_counter() - t0) * 1e3, 1),
                                us_per_pivot=round((time.perf_counter() - t0) * 1e6 / max(1, tot - 64), 1))
        s.close()
    r1["window_4096_pivots"] = window
    print("window", window, flush=True)
    # Phase I before the drive-out: the sync after each step turns the phase to 2 as soon as Phase I has ended, so
    # the pivot count at the first step that shows phase 2, stepping one pivot at a time, is Phase I's
    s = api.Session(A, b, c, rel, sense, kblock=16, max_iterations=it, two_phase=True)
    last = 0
    while s.two_phase_info()[0] == 1 and s.sync()[0] == RUNNING:
        last = s.sync()[1]
        s.step(64)
    s.close()
    s = api.Session(A, b, c, rel, sense, kblock=16, max_iterations=it, two_phase=True)
    st, tot = s.step(last)
    while s.two_phase_info()[0] == 1 and st == RUNNING:
        st, tot = s.step(1)
    ps = tot if s.two_phase_info()[0] == 2 else None
    s.close()
    r1.update(status=int(ref["status"]), n_pivots=int(ref["n_pivots"]), phase1_pivots=int(ref["phase1"]),
              phase1_simplex_pivots=ps, drive_out_pivots=None if ps is None else int(ref["phase1"]) - ps,
              phase2_pivots=int(ref["n_pivots"]) - int(ref["phase1"]), z=float(ref["z"]))
    prof = {}
    for K in (8, 16):
        s = api.Session(A, b, c, rel, sense, kblock=K, max_iterations=100000, two_phase=True)
        s.step(16)
        us = (C.c_double * 3)()
        F.check(F.lib().lpx_session_profile(s._h, 20, us))
        prof[f"K={K}"] = dict(lookahead_us=round(us[0], 1), pass_us=round(us[1], 1), per_block_us=round(us[2], 1),
                              per_pivot_us=round(us[2] / K, 1))
        s.close()
    r1["profile_phase1"] = prof
    print("mixed", json.dumps({k: v for k, v in r1.items() if k != "runs"}), flush=True)
    res["large_mixed"] = r1
    del A

    # 2. one SM against the whole GPU
    r2 = {}
    for m, n in ((512, 1024), (1024, 2048)):
        A, b, c, rel, sense = workloads.large_mixed(m, n)
        pc = 4 * (m + n)
        t0 = time.perf_counter()
        bat = api.two_phase_solve_batched(A[None], b[None], c[None], rel, sense, pivots_cap=pc, max_iterations=it)
        tb = (time.perf_counter() - t0) * 1e3
        to, ts, out = timed_session(A, b, c, rel, sense, pc, max_iterations=it)
        ok = (out["status"] == bat["status"][0] and out["n_pivots"] == bat["n_pivots"][0] and
              out["phase1"] == bat["phase1_pivots"][0] and
              all(np.asarray(out[k]).tobytes() == np.asarray(bat[k][0]).tobytes()
                  for k in ("pivots", "basis", "x", "z", "tableau")))
        r2[f"{m}x{n}"] = dict(batched_ms=round(tb, 1), session_open_ms=round(to, 1), session_solve_ms=round(ts, 1),
                              speedup=round(tb / (to + ts), 1), n_pivots=int(out["n_pivots"]),
                              phase1_pivots=int(out["phase1"]), status=int(out["status"]), bits_equal=bool(ok))
        print("one SM vs GPU", m, n, r2[f"{m}x{n}"], flush=True)
        assert ok
    res["one_sm_vs_gpu"] = r2

    # 3. C3: two-phase session against the primal session
    A, b, c = workloads.large_c3()
    tt, tp_ = [], []
    for _ in range(args.rounds):
        o1, s1, p = timed_session(A, b, c, None, 0, 10000, two_phase=False)
        o2, s2, q = timed_session(A, b, c, None, 0, 10000)
        tp_.append(o1 + s1)
        tt.append(o2 + s2)
        assert same({k: q[k] for k in p}, p), "C3: two-phase session differs from the primal session"
    res["c3"] = dict(primal_session_ms=round(float(np.median(tp_)), 1), two_phase_session_ms=round(float(np.median(tt)), 1),
                     ratio=round(float(np.median(tt)) / float(np.median(tp_)), 2), n_pivots=int(p["n_pivots"]),
                     all_primal_ms=[round(v, 1) for v in tp_], all_two_phase_ms=[round(v, 1) for v in tt],
                     bits_equal=True)
    print("c3", res["c3"], flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r13_two_phase_session.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

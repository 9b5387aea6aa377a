"""Parametric-analysis timings on one GPU -> <out>/r10_parametric.json (default out: profiles/).

Workloads (C2-shaped bases, workloads.batch_c2 64 x 128, dense integer directions in -5..5, theta_max = +inf,
seg_cap 64):
  rhs_one_base    one base x 4096 RHS directions          cost_one_base   the same for COST
  rhs_c2          4096 bases x 1 RHS direction each       cost_c2         the same for COST
Per workload:
  new       lpx_parametric_batched_dev (CUDA events around the launch, warmed up, median of the timed repeats) and
            lpx_parametric (host buffers, wall clock around the call, which solves the base and ends in a stream
            synchronise; one-base workloads only); checked bit-equal to the oracle
  today     what a user does without it: lpx_reoptimize_batched_dev RHS / COST what-if queries at as many theta points
            as the analysis returned segments (each segment's midpoint, or theta_lo + 1 for an infinite one) —
            values only, no breakpoints; timed with CUDA events, alternated with the new call, medians
  oracle    oracle/orc_param.cpp on one host thread and on all of them (ctypes releases the GIL)
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

CAP = 64


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--reps", type=int, default=15)
    args = ap.parse_args()
    import torch
    import orc_param_ffi as pm
    from test_gpu_reopt import device_bases

    F.check(F.lib().lpx_init(0))
    dev = torch.device("cuda:0")
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=11)
    bases = device_bases(A, b, c)
    hb = {k: bases[k].cpu().numpy() for k in ("status", "basis", "tableau")}
    rng = np.random.default_rng(2026)
    res = dict(gpu=gpu_info(), reps=args.reps, seg_cap=CAP, workloads={})
    stream = torch.cuda.current_stream()

    def events(fn):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e)

    for name, kind, one_base in (("rhs_one_base", 1, True), ("cost_one_base", 2, True), ("rhs_c2", 1, False),
                                 ("cost_c2", 2, False)):
        k = 64 if kind == 1 else 128
        D = rng.integers(-5, 6, size=(4096, k)).astype(float)
        pay = np.hstack([D, np.full((4096, 1), np.inf)])
        src = np.full(4096, 17, np.int32) if one_base else None
        rows, cols = api.parametric_dims(kind, 64, 128)
        t_pay = torch.from_numpy(pay).to(dev)
        t_src = None if src is None else torch.from_numpy(src).to(dev)
        o = dict(end=torch.zeros(4096, dtype=torch.int32, device=dev),
                 n_segments=torch.zeros(4096, dtype=torch.int32, device=dev),
                 n_pivots=torch.zeros(4096, dtype=torch.int32, device=dev),
                 segments=torch.zeros((4096, CAP, 260), dtype=torch.float64, device=dev),
                 seg_pivots=torch.zeros((4096, CAP, 2), dtype=torch.int32, device=dev),
                 basis=torch.zeros((4096, 64), dtype=torch.int32, device=dev),
                 tableau=torch.zeros((4096, rows, cols), dtype=torch.float64, device=dev))
        total = torch.zeros(1, dtype=torch.int64, device=dev)

        def new():
            api.parametric_batched_dev(kind, 4096, 64, 128, 0, None, bases["status"].data_ptr(),
                                       bases["basis"].data_ptr(), bases["tableau"].data_ptr(),
                                       None if t_src is None else t_src.data_ptr(), t_pay.data_ptr(), CAP,
                                       *[o[f].data_ptr() for f in ("end", "n_segments", "n_pivots", "segments",
                                                                    "seg_pivots", "basis")], None, total.data_ptr(),
                                       stream.cuda_stream)

        new()
        torch.cuda.synchronize()
        got = {f: v.cpu().numpy() for f, v in o.items() if f != "tableau"}
        t0 = time.perf_counter()
        want = pm.parametric(kind, 64, 128, hb["status"], hb["basis"], hb["tableau"], pay, None, 0, src, CAP)
        oracle_1 = time.perf_counter() - t0
        for f in ("end", "n_segments", "n_pivots", "seg_pivots", "basis"):
            assert np.array_equal(got[f], want[f]), (name, f)
        assert got["segments"].tobytes() == want["segments"].tobytes(), name
        nthreads = os.cpu_count() or 1
        chunks = np.array_split(np.arange(4096), nthreads)
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(nthreads) as ex:
            list(ex.map(lambda ix: pm.parametric(kind, 64, 128, hb["status"], hb["basis"], hb["tableau"], pay[ix],
                                                 None, 0, (src[ix] if src is not None else ix.astype(np.int32)),
                                                 CAP), chunks))
        oracle_all = time.perf_counter() - t0

        # today's route: what-if queries at one theta point per segment
        nseg = got["n_segments"]
        qsrc, qpay = [], []
        for q in range(4096):
            for s in range(nseg[q]):
                lo, hi = got["segments"][q, s, :2]
                t = (lo + hi) / 2 if np.isfinite(hi) else lo + 1.0
                qsrc.append(src[q] if src is not None else q)
                qpay.append(t * D[q])
        nq = len(qpay)
        r_pay = torch.from_numpy(np.ascontiguousarray(qpay)).to(dev)
        r_src = torch.from_numpy(np.asarray(qsrc, np.int32)).to(dev)
        r_out = dict(status=torch.zeros(nq, dtype=torch.int32, device=dev),
                     z=torch.zeros(nq, dtype=torch.float64, device=dev),
                     x=torch.zeros((nq, 128), dtype=torch.float64, device=dev))

        def today():
            api.reoptimize_batched_dev(kind, nq, 64, 128, 0, None, bases["status"].data_ptr(), bases["basis"].data_ptr(),
                                       bases["tableau"].data_ptr(), r_src.data_ptr(), r_pay.data_ptr(),
                                       r_out["status"].data_ptr(), None, None, 0, None, r_out["x"].data_ptr(),
                                       r_out["z"].data_ptr(), None, None, stream.cuda_stream)

        today()
        events(new)
        events(today)
        t_new, t_today = [], []
        for _ in range(args.reps):
            t_new.append(events(new))
            t_today.append(events(today))
        host = None
        if one_base:
            api.parametric(kind, A[17], b[17], c[17], D[:8], seg_cap=CAP, want_tableau=False)
            th = []
            for _ in range(5):
                t0 = time.perf_counter()
                hr = api.parametric(kind, A[17], b[17], c[17], D, seg_cap=CAP, want_tableau=False)
                th.append((time.perf_counter() - t0) * 1e3)
            assert hr["segments"].tobytes() == want["segments"].tobytes(), name
            host = float(np.median(th))
        kt = float(np.median(t_new))
        segs, pivs = int(nseg.sum()), int(got["n_pivots"].sum())
        ends = {str(e): int((got["end"] == e).sum()) for e in np.unique(got["end"])}
        res["workloads"][name] = dict(
            queries=4096, bases=1 if one_base else 4096, ends=ends, segments=segs, pivots=pivs,
            segments_per_query_mean=segs / 4096, segments_per_query_max=int(nseg.max()),
            kernel_ms_median=kt, kernel_ms_all=t_new, host_call_ms_median=host,
            queries_per_s=4096 / (kt * 1e-3), segments_per_s=segs / (kt * 1e-3), pivots_per_s=pivs / (kt * 1e-3),
            today_whatif_queries=nq, today_whatif_ms_median=float(np.median(t_today)), today_whatif_ms_all=t_today,
            oracle_one_thread_ms=oracle_1 * 1e3, oracle_all_threads_ms=oracle_all * 1e3, oracle_threads=nthreads,
            bits_equal_oracle=True)
        print(name, json.dumps({k: v for k, v in res["workloads"][name].items() if not k.endswith("_all")}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r10_parametric.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(res["gpu"])


if __name__ == "__main__":
    main()

"""Sensitivity report timings on the GPU (CUDA events, warm-ups); writes one JSON file.

  (a) the batched kernel over the 4096 C2 tableaux already on the device (lpx_sensitivity_batched_dev),
      against the HBM read bound of the 411 MB of tableaux;
  (b) end to end through host buffers, alternated: lpx_primal_solve_batched with tableaux,
      lpx_primal_solve_sensitivity_batched, and lpx_primal_solve_batched without tableaux (the floor);
  (c) a session stepped to OPTIMAL: lpx_session_sensitivity against lpx_session_read_tableau.

usage: python tools/sens_probe.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from linear_programming_solver_lpr381_b200 import _ffi as F  # noqa: E402
from linear_programming_solver_lpr381_b200 import api, workloads  # noqa: E402

HBM_TBS = 6.56  # the project's measured B200 HBM bandwidth (SURVEY 8d)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def kernel_over_c2():
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=1)
    count, m, n = A.shape
    dev = torch.device("cuda:0")
    tA, tb, tc = (torch.from_numpy(v).to(dev) for v in (A, b, c))
    st = torch.zeros(count, dtype=torch.int32, device=dev)
    npv = torch.zeros(count, dtype=torch.int32, device=dev)
    bas = torch.zeros((count, m), dtype=torch.int32, device=dev)
    x = torch.zeros((count, n), dtype=torch.float64, device=dev)
    z = torch.zeros(count, dtype=torch.float64, device=dev)
    T = torch.zeros((count, m + 1, n + m + 1), dtype=torch.float64, device=dev)
    rep = torch.zeros((count, api.sensitivity_stride(m, n)), dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # 256 MB, twice L2
    s = torch.cuda.current_stream()
    api.primal_solve_batched_dev(count, m, n, 0, tA.data_ptr(), None, tb.data_ptr(), tc.data_ptr(), st.data_ptr(),
                                 npv.data_ptr(), bas.data_ptr(), x.data_ptr(), z.data_ptr(), T.data_ptr(), None,
                                 s.cuda_stream)
    torch.cuda.synchronize()
    assert (st == 0).all()

    def launch():
        api.sensitivity_batched_dev(count, m, n, 0, None, tb.data_ptr(), tc.data_ptr(), st.data_ptr(), bas.data_ptr(),
                                    T.data_ptr(), rep.data_ptr(), s.cuda_stream)

    for _ in range(5):
        launch()
    times = []
    for _ in range(30):
        flush.zero_()  # overwrite L2 between timed passes: the tableaux come from HBM
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3)
    us = float(np.median(times))
    tbytes = count * (m + 1) * (n + m + 1) * 8
    bound_us = tbytes / (HBM_TBS * 1e12) * 1e6
    Tn = T.cpu().numpy()
    basis = bas.cpu().numpy()
    divs = 0
    for k in range(count):  # divisions actually performed: |g| > EPS entries of the slack block, |alpha| > EPS
        Tk = Tn[k]
        basic = np.zeros(n + m, dtype=bool)
        basic[basis[k]] = True
        divs += int((np.abs(Tk[:m, n:n + m]) > 1e-9).sum())
        rows = [r for r in range(m) if basis[k][r] < n]
        divs += int((np.abs(Tk[rows][:, :n + m][:, ~basic]) > 1e-9).sum())
    return dict(us_median=us, us_min=float(np.min(times)), tableau_bytes=tbytes, hbm_bound_us=bound_us,
                share_of_hbm_bound=bound_us / us, divisions=divs, divisions_bound=count * (m * m + m * n),
                l2="overwritten (256 MB) before every timed launch")


def end_to_end(runs=5):
    A, b, c = workloads.batch_c2(count=4096, m=64, n=128, seed=1)
    count, m, n = A.shape
    held = []  # the PinnedArray objects own the page-locked memory behind the numpy views

    def pinned(shape, dtype=np.float64, fill=None):
        p = F.PinnedArray(shape, dtype)
        held.append(p)
        if fill is not None:
            p.array[:] = fill
        return p.array

    Ap, bp, cp = pinned(A.shape, fill=A), pinned(b.shape, fill=b), pinned(c.shape, fill=c)
    out = dict(status=pinned((count,), np.int32), n_pivots=pinned((count,), np.int32),
               basis=pinned((count, m), np.int32), x=pinned((count, n)), z=pinned((count,)),
               tableau=pinned((count, m + 1, n + m + 1)))
    report = pinned((count, api.sensitivity_stride(m, n)))
    import ctypes as C
    opt = F.make_options()
    L = F.lib()
    total = C.c_longlong()

    def with_tableau():
        F.check(L.lpx_primal_solve_batched(count, m, n, 0, F.ptr(Ap), None, F.ptr(bp), F.ptr(cp), C.byref(opt),
                                           F.ptr(out["status"]), F.ptr(out["n_pivots"]), F.ptr(out["basis"]),
                                           F.ptr(out["x"]), F.ptr(out["z"]), F.ptr(out["tableau"]), C.byref(total)))

    def with_report():
        F.check(L.lpx_primal_solve_sensitivity_batched(count, m, n, 0, F.ptr(Ap), None, F.ptr(bp), F.ptr(cp),
                                                       C.byref(opt), F.ptr(out["status"]), F.ptr(out["n_pivots"]),
                                                       F.ptr(out["basis"]), F.ptr(out["x"]), F.ptr(out["z"]),
                                                       F.ptr(report), C.byref(total)))

    def floor():
        F.check(L.lpx_primal_solve_batched(count, m, n, 0, F.ptr(Ap), None, F.ptr(bp), F.ptr(cp), C.byref(opt),
                                           F.ptr(out["status"]), F.ptr(out["n_pivots"]), F.ptr(out["basis"]),
                                           F.ptr(out["x"]), F.ptr(out["z"]), None, C.byref(total)))

    legs = dict(solve_with_tableau=with_tableau, solve_with_report=with_report, solve_without_tableau=floor)
    for f in legs.values():
        f()
        f()
    ms = {k: [] for k in legs}
    for _ in range(runs):
        for k, f in legs.items():
            t0 = time.perf_counter()
            f()  # returns after the stream synchronise
            ms[k].append((time.perf_counter() - t0) * 1e3)
    res = {k: dict(ms_median=float(np.median(v)), ms_all=v) for k, v in ms.items()}
    res["input_bytes"] = int(A.nbytes + b.nbytes + c.nbytes)
    res["tableau_bytes"] = int(out["tableau"].nbytes)
    res["report_bytes"] = int(report.nbytes)
    res["runs_each"] = runs
    return res


def session(shapes=((1024, 2048), (2048, 4096), (4096, 8192))):
    best = None
    for m, n in shapes:
        A, b, c = workloads.large_c3(m, n) if (m, n) == (4096, 8192) else workloads.lp_integer(m, n, 31)
        s = api.Session(A, b, c)
        st, tot = F.RUNNING, 0
        while st == F.RUNNING and tot < 10000:
            st, tot = s.step(min(512, 10000 - tot))
        rec = dict(shape=[m, n], status=st, pivots=tot)
        if st == F.OPTIMAL:
            s.sensitivity()
            s.tableau()
            t_s, t_t = [], []
            for _ in range(5):
                t0 = time.perf_counter()
                s.sensitivity()
                t_s.append((time.perf_counter() - t0) * 1e3)
                t0 = time.perf_counter()
                s.tableau()
                t_t.append((time.perf_counter() - t0) * 1e3)
            rec.update(sensitivity_ms=float(np.median(t_s)), read_tableau_ms=float(np.median(t_t)),
                       tableau_bytes=s.rows * s.cols * 8, report_bytes=api.sensitivity_stride(m, n) * 8)
            best = rec
        s.close()
        print(json.dumps(rec), flush=True)
    return best


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_sensitivity.json")
    F.check(F.lib().lpx_init(0))
    res = dict(card=card())
    res["a_kernel_c2"] = kernel_over_c2()
    print(json.dumps(res["a_kernel_c2"]), flush=True)
    res["b_end_to_end_c2"] = end_to_end()
    print(json.dumps(res["b_end_to_end_c2"]), flush=True)
    res["c_session"] = session()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    json.dump(res, open(out, "w"), indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

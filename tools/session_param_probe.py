"""Parametric analysis of one large optimal session -> <out>/r11_session_parametric.json (default out: profiles/).

One C3 base (4096 x 8192, workloads.large_c3) solved to OPTIMAL in a streaming session.  Two directions: RHS d = -b
(b + theta d walks towards b = 0) and a dense COST direction with integers in -5..5, each analysed up to `seg_cap`
segments.  Per kind, in `rounds` alternating rounds (host clock around calls that end in a device synchronise):
  - lpx_session_parametric at K = 1, 8, 16 breakpoints per HBM pass, and at theta_max = 0 (one segment, no pivot: the
    fixed cost of a call, mostly the working session's allocation and build); per breakpoint = the median over rounds
    of (call - the same round's fixed call) / pivots;
  - today's alternatives: lpx_parametric_batched_dev on the downloaded tableau (one CTA, global-memory build) over
    `batched_segs` segments only, and lpx_session_reoptimize at one theta per segment (the midpoint of each of the
    first `reopt_segs` segments), stepped to its terminal status.
Every GPU result of the analysis is compared bit for bit across K.  The card name, power limit and max SM clock are
read in the same call.
"""
import argparse
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

RHS, COST = 1, 2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def to_end(s):
    st, tot = F.RUNNING, 0
    while st == F.RUNNING:
        st, tot = s.step(512)
    return st, tot


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t0) * 1e3, r


def batched_route(kind, T, basis, d, seg_cap):
    """lpx_parametric_batched_dev on the session's tableau uploaded as a base: ms including the upload."""
    import torch
    dev = torch.device("cuda:0")
    m, n = T.shape[0] - 1, T.shape[1] - T.shape[0]
    rows, cols = api.parametric_dims(kind, m, n)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bT = torch.from_numpy(T[None]).to(dev)
    bb = torch.from_numpy(np.ascontiguousarray(basis[None], np.int32)).to(dev)
    st = torch.zeros(1, dtype=torch.int32, device=dev)
    pay = torch.from_numpy(np.append(d, np.inf)[None]).to(dev)
    i32 = lambda k: torch.zeros(k, dtype=torch.int32, device=dev)  # noqa: E731
    end, ns, npv, spv, ob = i32(1), i32(1), i32(1), i32(2 * seg_cap), i32(m)
    seg = torch.zeros(seg_cap * (4 + 2 * n), dtype=torch.float64, device=dev)
    tab = torch.zeros(rows * cols, dtype=torch.float64, device=dev)
    api.parametric_batched_dev(kind, 1, m, n, 0, None, st.data_ptr(), bb.data_ptr(), bT.data_ptr(), None,
                               pay.data_ptr(), seg_cap, end.data_ptr(), ns.data_ptr(), npv.data_ptr(), seg.data_ptr(),
                               spv.data_ptr(), ob.data_ptr(), tab.data_ptr(), None, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    out = dict(end=int(end.item()), n_segments=int(ns.item()), segments=seg.cpu().numpy().reshape(seg_cap, -1))
    del bT, seg, tab
    torch.cuda.empty_cache()
    return ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory for r11_session_parametric.json")
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--seg-cap", type=int, default=32)
    ap.add_argument("--batched-segs", type=int, default=2)
    ap.add_argument("--reopt-segs", type=int, default=8)
    ap.add_argument("--m", type=int, default=4096)
    ap.add_argument("--n", type=int, default=8192)
    args = ap.parse_args()
    F.check(F.lib().lpx_init(0))
    A, b, c = workloads.large_c3(args.m, args.n)
    m, n = A.shape
    s = api.Session(A, b, c)
    st, base_piv = to_end(s)
    assert st == F.OPTIMAL, st
    basis = s.solution()[0]
    T = s.tableau()
    rng = np.random.default_rng(3)
    dirs = {RHS: ("rhs: d = -b", -b), COST: ("cost: dense integers in -5..5", rng.integers(-5, 6, size=n).astype(float))}
    res = dict(card=card(), shape=[m, n], tableau=[m + 1, n + m + 1], base_pivots=base_piv, rounds=args.rounds,
               seg_cap=args.seg_cap, kinds={})
    for kind, (what, d) in dirs.items():
        S = args.seg_cap
        ref = s.parametric(kind, d, seg_cap=S, want_tableau=False)  # warm-up, and the reference bits
        s.parametric(kind, d, 0.0, seg_cap=S, want_tableau=False)
        times = {k: [] for k in ("fixed", "K1", "K8", "K16")}
        for _ in range(args.rounds):
            ms, _ = timed(lambda: s.parametric(kind, d, 0.0, seg_cap=S, want_tableau=False))
            times["fixed"].append(ms)
            for K in (1, 8, 16):
                ms, got = timed(lambda: s.parametric(kind, d, seg_cap=S, want_tableau=False, kblock=K))
                times[f"K{K}"].append(ms)
                assert got["segments"].tobytes() == ref["segments"].tobytes(), (kind, K)
                assert got["end"] == ref["end"] and np.array_equal(got["seg_pivots"], ref["seg_pivots"])
        med = {k: float(np.median(v)) for k, v in times.items()}
        piv = max(ref["n_pivots"], 1)
        r = dict(direction=what, end=ref["end"], n_segments=ref["n_segments"], n_pivots=ref["n_pivots"],
                 ms_median={k: round(v, 2) for k, v in med.items()},
                 ms={k: [round(x, 2) for x in v] for k, v in times.items()},
                 ms_min={k: round(float(np.min(v)), 2) for k, v in times.items()},
                 # per round: (call - the same round's fixed call) / pivots; the median over rounds
                 us_per_breakpoint={f"K{K}": round(float(np.median(np.subtract(times[f"K{K}"], times["fixed"]))) * 1e3
                                                   / piv, 1) for K in (1, 8, 16)},
                 theta=[float(x) for x in ref["theta_hi"][:ref["n_segments"]]])
        # today's alternatives
        bs = args.batched_segs
        try:
            bms, bout = batched_route(kind, T, basis, d, bs)
            assert bout["segments"].tobytes() == ref["segments"][:bs].tobytes() or ref["n_segments"] < bs, kind
            r["batched_route"] = dict(seg_cap=bs, pivots=bout["n_segments"] - 1, ms_including_upload=round(bms, 1),
                                      ms_per_breakpoint=round(bms / max(bout["n_segments"] - 1, 1), 1))
        except F.LpxError as e:
            r["batched_route"] = dict(seg_cap=bs, refused=str(e))
        k_re = min(args.reopt_segs, ref["n_segments"])
        mids = [0.5 * (ref["theta_lo"][q] + (ref["theta_hi"][q] if np.isfinite(ref["theta_hi"][q])
                                             else ref["theta_lo"][q] + 1.0)) for q in range(k_re)]
        rms, agree = [], 0
        for q, th in enumerate(mids):
            def query():
                qs = s.reoptimize(kind, th * d)
                st_q, piv_q = to_end(qs)
                z = qs.solution()[2]
                qs.close()
                return st_q, piv_q, z
            ms, (st_q, piv_q, z) = timed(query)
            rms.append(ms)
            zp = ref["z0"][q] + th * ref["dz"][q]
            agree += int(st_q == F.OPTIMAL and abs(z - zp) <= 1e-6 * max(1.0, abs(zp)))
        r["reopt_route"] = dict(queries=k_re, ms_per_query_median=round(float(np.median(rms)), 1),
                                ms=[round(x, 1) for x in rms], z_matches_segment=agree)
        res["kinds"][kind] = r
        print(kind, json.dumps(r), flush=True)
    s.close()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r11_session_parametric.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py — simplex pivots/sec and B&B nodes/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload batched|large]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A step is one pass of the hot path over one batch of synthetic input:
  batched (default, BASELINE config 2): 4096 dense LPs of 64 x 128 per GPU, one launch of the
      per-tableau kernel; `value` = pivots/sec with inputs resident in HBM, `e2e` = the same through
      lpx_primal_solve_batched with pinned HOST buffers (H2D + D2H inside the timed call).
  large (BASELINE config 3): a window of pivots of one 4096 x 8192 LP, HBM-streamed.
The line also carries `large_tableau`, `bnb_simplex` and `bnb_knapsack` sections (configs 3-5).
Multi-GPU: independent problems per rank (weak scaling, no data-path collective); torch.distributed
only provides the barrier and the max-over-ranks of the timings.

--impl reference: the reference's own CPU implementation of the path.  The C# binary cannot run
here (no .NET); the timed code is the C++ restatement in oracle/ on all host threads.

--dump-outputs DIR: after the timed steps, rank 0 writes what the timed path returned in its last step
as DIR/<name>.npy (float64; int32 results are exact in it).  Inputs are seeded, so two builds run with
the same arguments can be compared array for array.  batched: status, n_pivots, basis, x, z of every
LP and the final tableaux of a fixed sample of DUMP_LPS LPs (`tableau`, their indices in
`tableau_index`).  large: basis, x, z and the objective row plus a fixed sample of DUMP_ROWS rows of
the tableau (`tableau`, `tableau_index`).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2 = dict(count=4096, m=64, n=128)
C3 = dict(m=4096, n=8192)
BNB_INSTANCES = 512             # C4 instances per GPU in the bnb_simplex section (SURVEY 8d: "e.g. 512")
KNAP_INSTANCES = 2368           # C5 instances per GPU in the bnb_knapsack section (16 per SM: one warp each)
KNAP_INSTANCES_FRACTIONAL = 148
POOLED = dict(seed=12, batch=4096)  # Mode B: one hard 60 x 120 instance (2.2e5 nodes), rounds of 4096 open nodes
DUMP_LPS = 256                  # --dump-outputs: batched tableaux kept (26 MB of the 411 MB)
DUMP_ROWS = 256                 # --dump-outputs: large-tableau constraint rows kept (25 MB of the 403 MB)
DUMP_LIMIT = 64 << 20           # --dump-outputs: bytes written at most
DUMP_SEED = 20261020            # the sample is the same in every run, so dumps compare element for element


def sample_index(count, k):
    """A fixed, seeded, sorted choice of k of range(count) (all of it when count <= k)."""
    if count <= k:
        return np.arange(count)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(count, k, replace=False))


def dump_outputs(dirname, arrays):
    """Each array as <dirname>/<name>.npy in float64."""
    out = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_LIMIT}")
    os.makedirs(dirname, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(dirname, k + ".npy"), v)


def dump_batched(dirname, res, tableaux):
    """`res`: status, n_pivots, basis, x, z of every LP; `tableaux(idx)` returns the final tableaux of LPs idx."""
    idx = sample_index(len(res["status"]), DUMP_LPS)
    dump_outputs(dirname, dict(res, tableau=tableaux(idx), tableau_index=idx))


def dump_large(dirname, T, basis, x, z):
    """The large LP's state: basis, x, z, and the objective row plus DUMP_ROWS sampled constraint rows of T."""
    m = T.shape[0] - 1
    idx = np.append(sample_index(m, DUMP_ROWS), m)
    dump_outputs(dirname, dict(basis=basis, x=x, z=[z], tableau=T[idx], tableau_index=idx))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            return json.load(f)[kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons while the timed region runs: NVML polled every 2 ms from a
    thread (the timed region of the default workload is ~10-50 ms, too short for `nvidia-smi -lms`),
    nvidia-smi only if NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None
        self.nv = None
        self.handle = None
        self.sm, self.bits, self.smax = [], 0, None
        self.run = False
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while self.run:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.sm, self.bits, self.run = [], 0, True
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nv:
            self.run = False
            self.th.join()
            nv = self.nv
            names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                     ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                     ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smax,
                    "reasons": sorted(nm for nm, bit in names if self.bits & bit), "samples": len(self.sm),
                    "source": "nvml, 2 ms polling inside the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------
# reference arm: the oracle (C++ restatement of the C# loops) on all host threads
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return None
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import orc_ffi
    from linear_programming_solver_lpr381_b200 import workloads
    cores = os.cpu_count() or 1
    if args.workload == "large":
        A, b, c = workloads.large_c3(**C3)
        m, n = A.shape
        T = np.zeros((m + 1, n + m + 1))
        T[:m, :n] = A
        T[:m, n:n + m] = np.eye(m)
        T[:m, -1] = b
        T[m, :n] = -c
        basis = np.arange(n, n + m, dtype=np.int32)
        per_step = 4
        times = []
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            orc_ffi.primal_core(T, basis, per_step)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
        total = per_step * len(times)
        value = total / sum(times)
        used, sample = 1, f"{per_step} pivots per step of the 4096x8192 tableau (single tableau: one thread, as upstream)"
        cfg = {"workload": "C3 single large dense LP 4096x8192, window of pivots", **C3}
        if args.dump_outputs:
            x = np.zeros(n)
            in_x = basis < n
            x[basis[in_x]] = T[:m, -1][in_x]
            dump_large(args.dump_outputs, T, basis, x, T[m, -1])
    else:
        A, b, c = workloads.batch_c2(**C2, seed=1)
        times, piv = [], 0
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = orc_ffi.primal_batch(A, b, c, threads=cores, with_format=False, want_tableau=True)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
                piv += int(r["total_pivots"])
        value = piv / sum(times)
        used, sample = cores, "full 4096-LP batch per step, arithmetic loop only (no per-iteration text formatting)"
        cfg = {"workload": "C2 batched dense LPs: 4096 x (64 constraints x 128 vars)", **C2}
        if args.dump_outputs:
            dump_batched(args.dump_outputs, {k: r[k] for k in ("status", "n_pivots", "basis", "x", "z")},
                         lambda idx: r["tableau"][idx])
    line = {
        "impl": "reference", "metric": "simplex pivots/sec", "value": value, "unit": "pivots/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "pivots/s", "cores": used, "kind": "port", "sample": sample,
                         "note": "C++ restatement of the reference's C# loops (oracle/); the C# binary cannot be "
                                 "built here (no .NET toolchain)"},
        "e2e": {"value": value, "unit": "pivots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    return line


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from linear_programming_solver_lpr381_b200 import _ffi as F
    from linear_programming_solver_lpr381_b200 import api, workloads

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    F.check(F.lib().lpx_init(local_rank))
    if world > 1:
        # the engine's own communicator (one tree over all ranks in the bnb_simplex_pooled section): rank 0
        # creates the id, torch.distributed ships the 128 bytes
        import ctypes as C
        uid = (C.c_byte * 128)()
        if rank == 0:
            F.check(F.lib().lpx_comm_unique_id(uid))
        obj = [bytes(uid)]
        dist.broadcast_object_list(obj, src=0)
        uid = (C.c_byte * 128).from_buffer_copy(obj[0])
        F.check(F.lib().lpx_comm_init(world, rank, uid))
    hbm_peak, peak_kind = load_peaks()
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    extras = {}
    sampler = ClockSampler(local_rank)

    # ---------------- config 3: large tableau (value when --workload large, else a section) ------
    def bench_large(steps, warmup, per_step, dump=None):
        import ctypes as C
        A, b, c = workloads.large_c3(**C3, seed=7 + rank)
        dA, db, dc = (torch.from_numpy(v).to(dev) for v in (A, b, c))
        torch.cuda.synchronize()
        kblock = 8  # the engine's default: 8 pivots per HBM pass, look-ahead pipelined with the pass
        s = api.Session(dA.data_ptr(), db.data_ptr(), dc.data_ptr(), device_ptrs=True, m=C3["m"], n=C3["n"],
                        max_iterations=1 << 30)
        del dA
        rows, cols = s.rows, s.cols
        sstream = torch.cuda.ExternalStream(s.stream)
        for _ in range(warmup):
            s.step_async(per_step)
        s.sync()
        barrier()
        l0 = F.lib().lpx_kernel_launches()
        # ONE event pair around the K steps: a timing event between steps makes the look-ahead of the
        # next block lose its head start on the pass (measured 31.6 vs 24.8 us per pivot)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        csamp = ClockSampler(local_rank)
        csamp.start()
        barrier()
        e0.record(sstream)
        for k in range(steps):
            s.step_async(per_step)
        e1.record(sstream)
        st, tot = s.sync()
        barrier()
        clocks = csamp.stop()
        launches = F.lib().lpx_kernel_launches() - l0 - 1
        ms = [e0.elapsed_time(e1)]
        total_ms = max_over_ranks(sum(ms))
        done = per_step * steps
        if st != F.RUNNING:
            raise SystemExit(f"large LP finished early (status {st}) inside the timed window")
        if dump:  # before lpx_session_profile, which pivots the session further
            dump_large(dump, s.tableau(), *s.solution())
        # the two kernels of a block, timed separately with CUDA events on the session stream
        us = (C.c_double * 3)()
        F.lib().lpx_session_profile.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        F.check(F.lib().lpx_session_profile(s._h, 8, us))
        lookahead_us, pass_us = us[0], us[1]
        bytes_per_pass = 2 * 8 * rows * cols
        pivots_s = world * done / (total_ms * 1e-3)
        ach = bytes_per_pass / (pass_us * 1e-6) / 1e9
        per_pivot_equiv = bytes_per_pass * done / (sum(ms) * 1e-3) / 1e9
        s.close()
        return dict(value=pivots_s, ms_per_step=total_ms / steps, launches=launches, rows=rows, cols=cols,
                    pivots_per_step=per_step, clocks=clocks,
                    roofline={"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                              "frac": ach / hbm_peak, "traffic": measured_traffic("stream_update_pipe_tma_kernel"),
                              "peak_source": peak_kind,
                              "kernel": "stream_update_pipe_tma_kernel (one TMA-staged HBM pass applying a block of pivots; "
                                        "timed alone, the look-ahead of the next block normally runs beside it)",
                              "algorithmic_bytes_per_launch": bytes_per_pass, "launch_us": pass_us,
                              "pivots_per_launch": kblock, "lookahead_us_per_block": lookahead_us,
                              "block_us_overlapped": 1e3 * sum(ms) / (done / kblock),
                              "per_pivot_roofline": {
                                  "note": "SURVEY 8d counts one read + one write of the tableau PER PIVOT "
                                          "(805.6 MB, 8137 pivots/s at the measured HBM peak).  The blocked "
                                          "look-ahead applies several pivots per pass with bit-identical "
                                          "arithmetic, so pivots/s exceeds that per-pivot bound; the kernel's own "
                                          "roofline (bytes it really streams per launch) is `achieved` above.",
                                  "equivalent_GBs": per_pivot_equiv, "x_of_per_pivot_bound": per_pivot_equiv / hbm_peak}})

    # ---------------- config 2: batched --------------------------------------------------------
    def bench_batched(steps, warmup, dump=None):
        A, b, c = workloads.batch_c2(**C2, seed=1 + rank)
        count, m, n = A.shape
        rows, cols = m + 1, n + m + 1
        dA, db, dc = (torch.from_numpy(v).to(dev) for v in (A, b, c))
        st = torch.zeros(count, dtype=torch.int32, device=dev)
        npv = torch.zeros(count, dtype=torch.int32, device=dev)
        basis = torch.zeros((count, m), dtype=torch.int32, device=dev)
        x = torch.zeros((count, n), dtype=torch.float64, device=dev)
        z = torch.zeros(count, dtype=torch.float64, device=dev)
        T = torch.zeros((count, rows, cols), dtype=torch.float64, device=dev)
        tot = torch.zeros(1, dtype=torch.int64, device=dev)

        def launch():
            api.primal_solve_batched_dev(count, m, n, 0, dA.data_ptr(), None, db.data_ptr(), dc.data_ptr(),
                                         st.data_ptr(), npv.data_ptr(), basis.data_ptr(), x.data_ptr(), z.data_ptr(),
                                         T.data_ptr(), tot.data_ptr(), stream.cuda_stream)

        for _ in range(warmup):
            launch()
        barrier()
        tot.zero_()
        l0 = F.lib().lpx_kernel_launches()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        sampler.start()
        barrier()
        for k in range(steps):
            ev[k][0].record(stream)
            launch()
            ev[k][1].record(stream)
        barrier()
        launches = F.lib().lpx_kernel_launches() - l0
        ms = [a.elapsed_time(bb) for a, bb in ev]
        total_ms = max_over_ranks(sum(ms))
        pivots = int(tot.item())
        all_pivots = sum_over_ranks(pivots)
        value = all_pivots / (total_ms * 1e-3)
        assert int((st != 0).sum().item()) == 0, "a batched LP did not reach OPTIMAL"

        # e2e: the reference-facing call, pinned host buffers in and out
        hA, hb, hc = F.PinnedArray(A.shape), F.PinnedArray(b.shape), F.PinnedArray(c.shape)
        hA.array[...] = A
        hb.array[...] = b
        hc.array[...] = c
        keep = dict(status=F.PinnedArray((count,), np.int32), n_pivots=F.PinnedArray((count,), np.int32),
                    basis=F.PinnedArray((count, m), np.int32), x=F.PinnedArray((count, n)),
                    z=F.PinnedArray((count,)), tableau=F.PinnedArray((count, rows, cols)))
        out = {k: v.array for k, v in keep.items()}  # `keep` owns the page-locked memory
        h2d = A.nbytes + b.nbytes + c.nbytes
        d2h = sum(v.nbytes for v in out.values())
        for _ in range(max(1, warmup)):
            api.primal_solve_batched(hA.array, hb.array, hc.array, out=out)
        barrier()
        t0 = time.perf_counter()
        e2e_piv = 0
        for _ in range(steps):
            r = api.primal_solve_batched(hA.array, hb.array, hc.array, out=out)
            e2e_piv += r["total_pivots"]
        torch.cuda.synchronize()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        clocks = sampler.stop()  # sampled across both timed regions (device-resident steps, then e2e steps)
        e2e_value = sum_over_ranks(e2e_piv) / e2e_s

        # roofline of the per-tableau kernel: on-chip, bounded by the unfused FP64 rate
        rate = F.C.c_double()
        F.check(F.lib().lpx_measure_fp64_rate(F.C.byref(rate)))
        flops_per_pivot = 2 * m * cols + cols
        ach_tf = flops_per_pivot * pivots / (sum(ms) * 1e-3) / 1e12
        hbm_bytes = (A.nbytes + b.nbytes + c.nbytes) + T.numel() * 8 + x.numel() * 8 + basis.numel() * 4
        roof = {"bound": "fp64", "achieved": ach_tf, "peak": rate.value, "unit": "TFLOP/s",
                "frac": ach_tf / rate.value if rate.value else None,
                "traffic": measured_traffic("reg_simplex_kernel"),
                "peak_source": "measured in this run: unfused DMUL+DADD issue rate (lpx_measure_fp64_rate); FMA is "
                               "excluded by the bit-exactness contract",
                "flops_per_pivot": flops_per_pivot,
                "kernel": "reg_simplex_kernel<8,8,2,2,3,cond>: one CTA per LP, three per SM, the CONDENSED tableau (n non-basic "
                          "columns + RHS) in registers / shared memory; the full tableau is put back together on the way out",
                "note": "flops_per_pivot is SURVEY 8d's count for the reference's FULL (m+1) x (n+m+1) tableau; the condensed "
                        "kernel executes (n+1)/(n+m+1) of them — the m basic columns are unit vectors nobody has to update",
                "hbm": {"bound": "hbm", "achieved": hbm_bytes * steps / (sum(ms) * 1e-3) / 1e9, "peak": hbm_peak,
                        "unit": "GB/s", "algorithmic_bytes_per_launch": hbm_bytes, "peak_source": peak_kind,
                        "note": "inputs read once + final tableaux/x/basis written once; the tableau lives on-chip "
                                "across all pivots, so this kernel is not HBM-bound"}}
        if dump:  # the device buffers still hold the last timed step: the e2e calls have their own
            res = dict(status=st, n_pivots=npv, basis=basis, x=x, z=z)
            dump_batched(dump, {k: v.cpu().numpy() for k, v in res.items()},
                         lambda idx: T[torch.from_numpy(idx).to(dev)].cpu().numpy())
        return dict(value=value, ms_per_step=total_ms / steps, launches=launches, clocks=clocks, pivots_per_step=pivots,
                    e2e={"value": e2e_value, "unit": "pivots/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                         "ms_per_step": 1e3 * e2e_s / steps}, roofline=roof, host=(A, b, c))

    # ---------------- configs 4 and 5 (sections) ------------------------------------------------
    def oracle():
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import orc_ffi
        orc_ffi.lib()
        return orc_ffi

    def timed_pool(fn, items, threads):
        """fn over items on `threads` host threads (the oracle's ctypes calls release the GIL)."""
        from concurrent.futures import ThreadPoolExecutor
        t0 = time.perf_counter()
        if threads <= 1:
            out = [fn(it) for it in items]
        else:
            with ThreadPoolExecutor(threads) as ex:
                out = list(ex.map(fn, items))
        return out, time.perf_counter() - t0

    port_note = "C++ restatement (oracle/) of the C# loops, not the C# binary (no .NET toolchain here)"
    with_cpu = rank == 0 and world == 1
    host_cores = os.cpu_count() or 1

    def fp64_rate():
        rate = F.C.c_double()
        F.check(F.lib().lpx_measure_fp64_rate(F.C.byref(rate)))
        return rate.value

    def bench_bnb(count):
        import ctypes as C
        As, bs, cs = zip(*[workloads.ip_c4(seed=1000 * rank + 11 + k) for k in range(count)])
        A, b, c = np.stack(As), np.stack(bs), np.stack(cs)
        api.bnb_simplex_batched(A, b, c)  # warm-up at full size: the node pool and pinned staging grow once
        barrier()
        l0 = F.lib().lpx_kernel_launches()
        t0 = time.perf_counter()
        r = api.bnb_simplex_batched(A, b, c)
        dt = max_over_ranks(time.perf_counter() - t0)
        st4 = (C.c_double * 4)()
        F.check(F.lib().lpx_bnb_last_stats(st4))
        flops, gpu_s, rounds = st4[0], st4[1], int(st4[3])
        nodes = sum_over_ranks(int(r["n_nodes"].sum()))
        rate = fp64_rate()
        ach = flops / gpu_s / 1e12 if gpu_s > 0 else 0.0
        out = {"metric": "B&B simplex nodes/sec (LP relaxations solved per second)", "value": nodes / dt,
               "unit": "nodes/s", "instances_per_gpu": count, "nodes": nodes, "lp_pivots": sum_over_ranks(int(r["lp_pivots"].sum())),
               "seconds": dt, "gpu_launches": F.lib().lpx_kernel_launches() - l0,
               "mode": "reference-exact tree (SURVEY F5), independent instances per GPU, host commit in DFS order",
               "timing": "end to end through lpx_bnb_simplex_batched (host buffers)",
               "roofline": {"bound": "fp64", "achieved": ach, "peak": rate, "unit": "TFLOP/s",
                            "frac": ach / rate if rate else None, "traffic": None,
                            "peak_source": "measured in this run: unfused DMUL+DADD issue rate",
                            "kernel": "cta_condensed_kernel (condensed tableau: non-basic columns + RHS; the open nodes of "
                                      "a quarter of the instances per round, one launch per occupancy class, four "
                                      "rounds in flight on four streams)",
                            "algorithmic_flops": flops, "gpu_seconds": gpu_s, "evaluation_rounds": rounds,
                            "note": "flops = sum over node LPs of pivots x (2 m_d (n+m_d+1) + (n+m_d+1)) at each node's "
                                    "own FULL-tableau shape, SURVEY 8d's count (rank 0's instances) — the condensed kernel "
                                    "does n+1 of those n+m+1 columns; gpu_seconds = the whole call: the GPU is busy "
                                    "throughout, the host commits one set's round while the others run"}}
        if with_cpu:
            orc = oracle()
            k1 = min(4, count)
            r1, t1 = timed_pool(lambda k: orc.bnb_simplex(As[k], bs[k], cs[k]), range(k1), 1)
            kn = min(count, 2 * host_cores)
            rn, tn = timed_pool(lambda k: orc.bnb_simplex(As[k], bs[k], cs[k]), range(kn), host_cores)
            out["cpu_baseline"] = {"value": sum(x["n_nodes"] for x in r1) / t1, "unit": "nodes/s", "cores": 1, "kind": "port",
                                   "sample": f"the first {k1} instances of the batch, one thread",
                                   "all_threads": {"value": sum(x["n_nodes"] for x in rn) / tn, "unit": "nodes/s",
                                                   "cores": host_cores, "sample": f"the first {kn} instances, one instance per thread"},
                                   "note": port_note}
        return out

    def bench_knap(count, kind="uncorrelated", label=None):
        ps, ws, caps = zip(*[workloads.knapsack_c5(seed=1000 * rank + 13 + k, kind=kind) for k in range(count)])
        p, w, cap = np.stack(ps), np.stack(ws), np.array(caps)
        api.bnb_knapsack_batched(p, w, cap)  # warm-up at full size
        barrier()
        l0 = F.lib().lpx_kernel_launches()
        t0 = time.perf_counter()
        r = api.bnb_knapsack_batched(p, w, cap)
        dt = max_over_ranks(time.perf_counter() - t0)
        nodes = sum_over_ranks(int(r["n_evals"].sum()))
        n_items = p.shape[1]
        bytes_per_node = 16 * n_items  # SURVEY 8d: 4n assigned read + 4n child assigned write + 8n relaxed write
        ach = nodes / world * bytes_per_node / dt / 1e9
        out = {"metric": "B&B knapsack nodes/sec (ComputeRelaxation evaluations committed per second)",
               "value": nodes / dt, "unit": "nodes/s", "instances_per_gpu": count, "items": n_items, "data": kind,
               "nodes": nodes, "seconds": dt, "gpu_launches": F.lib().lpx_kernel_launches() - l0,
               "timing": "end to end through lpx_bnb_knapsack_batched (host buffers)",
               "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                            "traffic": None, "peak_source": peak_kind, "algorithmic_bytes_per_node": bytes_per_node,
                            "note": "SURVEY 8d's per-node figure (the reference's int[n] assignment read and written, "
                                    "double[n] relaxed written) x committed evaluations / wall time of the call; the "
                                    "search is bound by the dependent pop -> evaluate -> push chain, not by HBM"}}
        if label:
            out["label"] = label
        if with_cpu:
            orc = oracle()
            k1 = min(4 if kind != "fractional" else 1, count)
            r1, t1 = timed_pool(lambda k: orc.knapsack(ps[k], ws[k], caps[k]), range(k1), 1)
            kn = min(count, 2 * host_cores)
            rn, tn = timed_pool(lambda k: orc.knapsack(ps[k], ws[k], caps[k]), range(kn), host_cores)
            out["cpu_baseline"] = {"value": sum(x["n_evals"] for x in r1) / t1, "unit": "nodes/s", "cores": 1, "kind": "port",
                                   "sample": f"the first {k1} instance(s) of the batch, one thread",
                                   "all_threads": {"value": sum(x["n_evals"] for x in rn) / tn, "unit": "nodes/s",
                                                   "cores": host_cores, "sample": f"the first {kn} instances, one instance per thread"},
                                   "note": port_note}
        return out

    def bench_pooled():
        """Mode B (NOT the reference's tree): ONE 60 x 120 IP, both children honoured, warm starts, the nodes of
        every round dealt over all ranks (strong scaling: the tree is the same for any N)."""
        A, b, c = workloads.ip_c4(seed=POOLED["seed"])
        api.bnb_pooled(A, b, c, batch=POOLED["batch"])  # warm-up: node pools allocated and mapped into the peers
        barrier()
        l0 = F.lib().lpx_kernel_launches()
        t0 = time.perf_counter()
        r = api.bnb_pooled(A, b, c, batch=POOLED["batch"])
        dt = max_over_ranks(time.perf_counter() - t0)
        out = {"metric": "B&B simplex nodes/sec, pooled tree (Mode B: both children, warm-started, one tree over all GPUs)",
               "value": r["n_nodes"] / dt, "unit": "nodes/s", "scaling": "strong", "nodes": int(r["n_nodes"]),
               "rounds": int(r["rounds"]), "dual_pivots": int(r["total_pivots"]), "best_z": r["best_z"], "seconds": dt,
               "gpu_launches": F.lib().lpx_kernel_launches() - l0, "n_gpus": world,
               "config": {"workload": "C4 one general IP 60 x 120 (seed %d), rounds of %d open nodes" %
                                      (POOLED["seed"], POOLED["batch"]), **POOLED},
               "note": "NOT the reference's tree (its '>=' children are never explored, SURVEY F5); checked node for "
                       "node against oracle/orc_pooled.cpp and against an independent MILP solver (tests/test_gpu_pooled.py); "
                       "every rank returns the same tree for any number of GPUs (tests/pooled_shard_check.py)"}
        if with_cpu:
            orc = oracle()
            t1 = time.perf_counter()
            ro = orc.bnb_pooled(A, b, c, batch=POOLED["batch"], max_nodes=40000, node_cap=1)
            d1 = time.perf_counter() - t1
            out["cpu_baseline"] = {"value": ro["n_nodes"] / d1, "unit": "nodes/s", "cores": 1, "kind": "port",
                                   "sample": f"the first {ro['n_nodes']} nodes of the same tree, one thread",
                                   "note": "oracle/orc_pooled.cpp: the same search on the CPU (there is no upstream code for this tree)"}
        return out

    def cpu_baseline_large():
        """The oracle's arithmetic loop on the same 4096 x 8192 tableau, one thread (a single tableau is one
        thread upstream)."""
        orc = oracle()
        A, b, c = workloads.large_c3(**C3, seed=7)
        m, n = A.shape
        T = np.zeros((m + 1, n + m + 1))
        T[:m, :n] = A
        T[:m, n:n + m] = np.eye(m)
        T[:m, -1] = b
        T[m, :n] = -c
        basis = np.arange(n, n + m, dtype=np.int32)
        orc.primal_core(T, basis, 4)
        t0 = time.perf_counter()
        done = 0
        while time.perf_counter() - t0 < 6.0:
            done += orc.primal_core(T, basis, 16)[1]
        dt = time.perf_counter() - t0
        return {"value": done / dt, "unit": "pivots/s", "cores": 1, "kind": "port",
                "sample": f"{done} pivots of the same 4097x12289 tableau after 4 warm-up pivots, one thread, arithmetic "
                          "loop only", "note": port_note}

    # ---------------- CPU baseline on rank 0, N = 1 ---------------------------------------------
    def cpu_baseline(host):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import orc_ffi
        A, b, c = host
        t0 = time.perf_counter()
        piv = 0
        reps = 0
        while time.perf_counter() - t0 < 8.0:
            piv += int(orc_ffi.primal_batch(A, b, c, threads=1)["total_pivots"])
            reps += 1
        dt = time.perf_counter() - t0
        sub = slice(0, 64)
        t1 = time.perf_counter()
        pf = int(orc_ffi.primal_batch(A[sub], b[sub], c[sub], threads=1, with_format=True)["total_pivots"])
        dtf = time.perf_counter() - t1
        return {"value": piv / dt, "unit": "pivots/s", "cores": 1, "kind": "port",
                "sample": f"the full 4096-LP C2 batch x {reps} passes, single thread, arithmetic loop only",
                "with_reference_text_formatting": {"value": pf / dtf, "unit": "pivots/s",
                                                   "sample": "first 64 LPs of the batch, one thread, including the "
                                                             "reference's unconditional per-iteration AppendTableau"},
                "host_cores_available": os.cpu_count(),
                "note": "C++ restatement (oracle/) of the C# loops, not the C# binary (no .NET toolchain here)"}

    dump = args.dump_outputs if rank == 0 else None
    if args.workload == "large":
        per_step = int(os.environ.get("LPX_BENCH_PERSTEP", "128"))
        L = bench_large(args.steps, args.warmup, per_step, dump)
        line = {"metric": "simplex pivots/sec", "value": L["value"], "unit": "pivots/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": L["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C3 single large dense LP 4096x8192 (tableau 4097x12289), window of "
                                       f"{per_step} pivots per step", **C3, "inputs_larger_than_L2": True},
                "roofline": L["roofline"], "gpu_launches": L["launches"], "clocks": L["clocks"],
                "cpu_baseline": cpu_baseline_large() if with_cpu else None,
                "e2e": {"value": L["value"], "unit": "pivots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                        "note": "the tableau is resident in HBM for the whole session; only 16 bytes of status "
                                "cross PCIe per step"}}
    else:
        Bm = bench_batched(args.steps, args.warmup, dump)
        host = Bm.pop("host")
        if not args.no_extras:
            try:
                Lg = bench_large(3, 3, 128)
                extras["large_tableau"] = {"metric": "simplex pivots/sec, one 4096x8192 LP (tableau 4097x12289)",
                                           "value": Lg["value"], "unit": "pivots/s", "ms_per_pivot":
                                           Lg["ms_per_step"] / Lg["pivots_per_step"], "roofline": Lg["roofline"],
                                           "gpu_launches": Lg["launches"],
                                           "cpu_baseline": cpu_baseline_large() if with_cpu else None}
            except Exception as e:  # a section must not take the headline down
                extras["large_tableau"] = {"error": str(e)}
            try:
                extras["bnb_simplex"] = bench_bnb(BNB_INSTANCES)
            except Exception as e:
                extras["bnb_simplex"] = {"error": str(e)}
            try:
                extras["bnb_knapsack"] = bench_knap(KNAP_INSTANCES)
            except Exception as e:
                extras["bnb_knapsack"] = {"error": str(e)}
            try:
                extras["bnb_simplex_pooled"] = bench_pooled()
            except Exception as e:
                extras["bnb_simplex_pooled"] = {"error": str(e)}
            try:  # non-integer data: every sum in the reference's order (the ordered-summation path)
                extras["bnb_knapsack_fractional"] = bench_knap(KNAP_INSTANCES_FRACTIONAL, kind="fractional",
                                                               label="ordered-summation path (non-integer data)")
            except Exception as e:
                extras["bnb_knapsack_fractional"] = {"error": str(e)}
        line = {"metric": "simplex pivots/sec", "value": Bm["value"], "unit": "pivots/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": Bm["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C2 batched dense LPs: 4096 x (64 constraints x 128 vars) per GPU, one CTA "
                                       "per tableau", **C2, "pivots_per_step_per_gpu": Bm["pivots_per_step"] // args.steps,
                           "inputs_larger_than_L2": True, "l2_note": "275 MB of inputs and 411 MB of result "
                           "tableaux per step exceed the 126 MB L2; no flush needed"},
                "roofline": Bm["roofline"], "e2e": Bm["e2e"], "gpu_launches": Bm["launches"], "clocks": Bm["clocks"],
                "cpu_baseline": cpu_baseline(host) if (rank == 0 and world == 1) else None}
        line.update(extras)
    if world > 1:
        F.lib().lpx_comm_destroy()
        dist.destroy_process_group()
    return line if rank == 0 else None


class OneJsonLine:
    """The driver parses stdout as ONE JSON line.  Libraries below us write there too (NCCL prints its version
    line to stdout when a communicator is created under NCCL_DEBUG=VERSION/WARN), so file descriptor 1 points at
    stderr while the benchmark runs and is restored only for the final print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="batched", choices=["batched", "large"])
    ap.add_argument("--no-extras", action="store_true", help="skip the configs 3-5 sections")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    with OneJsonLine() as guard:
        line = run_reference(args) if args.impl == "reference" else run_ours(args)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()

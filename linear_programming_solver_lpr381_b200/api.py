"""Thin numpy-level wrappers over the C ABI (one C call each).  Argument names and result fields
follow the reference's SimplexResult (R/Models/PrimalSimplex.cs:38-49): status, z (OptimalValue),
x (Solution), tableau, basis, plus the pivot list the parity tests compare.
"""
import ctypes as C

import numpy as np

from . import _ffi as F


def _prep(A, b, c, rel):
    A = np.ascontiguousarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    return A, b, c, rel


def tableau_dims(m, n, rel=None):
    rows, cols = C.c_int(), C.c_int()
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    F.check(F.lib().lpx_tableau_dims(m, n, F.ptr(rel), C.byref(rows), C.byref(cols)))
    return rows.value, cols.value


def primal_solve(A, b, c, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0, history=0,
                 pivots_cap=None, want_tableau=True):
    A, b, c, rel = _prep(A, b, c, rel)
    m, n = A.shape
    rows, cols = tableau_dims(m, n, rel)
    cap = max_iterations if pivots_cap is None else pivots_cap
    cap = min(cap, 1 << 20)
    opt = F.make_options(max_iterations, kernel, threads)
    status, npiv = C.c_int(), C.c_int()
    pivots = np.full((max(cap, 1), 2), -1, dtype=np.int32)
    basis = np.zeros(rows - 1, dtype=np.int32)
    x = np.zeros(n)
    z = C.c_double()
    T = np.zeros((rows, cols)) if want_tableau else None
    hist = np.zeros((history, rows, cols)) if history else None
    rc = F.lib().lpx_primal_solve(m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt),
                                  C.byref(status), C.byref(npiv), F.ptr(pivots), cap, F.ptr(basis), F.ptr(x),
                                  C.byref(z), F.ptr(T), F.ptr(hist), history)
    F.check(rc)
    out = dict(status=status.value, n_pivots=npiv.value, pivots=pivots[: min(npiv.value, cap)], basis=basis, x=x,
               z=z.value, tableau=T, rows=rows, cols=cols)
    if history:
        out["history"] = hist[: min(npiv.value + 1, history)]
    return out


def dual_solve(A, b, c, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0, history=0,
               pivots_cap=10200):
    A, b, c, rel = _prep(A, b, c, rel)
    m, n = A.shape
    rows, cols = tableau_dims(m, n, rel)
    opt = F.make_options(max_iterations, kernel, threads)
    status, npiv, silent = C.c_int(), C.c_int(), C.c_int()
    pivots = np.full((pivots_cap, 2), -1, dtype=np.int32)
    basis = np.zeros(rows - 1, dtype=np.int32)
    x = np.zeros(n)
    z = C.c_double()
    T = np.zeros((rows, cols))
    hist = np.zeros((history, rows, cols)) if history else None
    rc = F.lib().lpx_dual_solve(m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt), C.byref(status),
                                C.byref(npiv), C.byref(silent), F.ptr(pivots), pivots_cap, F.ptr(basis), F.ptr(x),
                                C.byref(z), F.ptr(T), F.ptr(hist), history)
    F.check(rc)
    out = dict(status=status.value, n_pivots=npiv.value, silent=silent.value,
               pivots=pivots[: min(npiv.value, pivots_cap)], basis=basis, x=x, z=z.value, tableau=T, rows=rows,
               cols=cols)
    if history:
        out["history"] = hist[: min(npiv.value - silent.value + 1, history)]
    return out


def revised_solve(A, b, c, rel=None, sense=0, max_iterations=10000, cap=16384, history=0, kernel=F.KERNEL_AUTO,
                  kblock=0, pass_variant=0):
    """lpx_revised_solve: RevisedPrimalSimplex numerics (pivots, theta, final basis state).  kernel: AUTO, STREAM
    (the whole GPU) or CTA_GLOBAL (one CTA); kblock / pass_variant: Gauss-Jordan steps per pass and the pass kernel
    of the whole-GPU inversion."""
    A, b, c, rel = _prep(A, b, c, rel)
    m, n = A.shape
    opt = F.make_options(max_iterations, kernel, kblock=kblock, pass_variant=pass_variant)
    status, n_iters = C.c_int(), C.c_int()
    pivots = np.full((cap, 2), -1, dtype=np.int32)
    theta = np.zeros(cap)
    basis, nonbasic = np.zeros(m, dtype=np.int32), np.zeros(n, dtype=np.int32)
    xB, Binv, x = np.zeros(m), np.zeros((m, m)), np.zeros(n)
    L = F.lib()
    L.lpx_revised_history_stride.restype = C.c_size_t
    hs = L.lpx_revised_history_stride(m, n)
    hist = np.zeros((history, hs)) if history else None
    rc = L.lpx_revised_solve(m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt), C.byref(status),
                             C.byref(n_iters), F.ptr(pivots), F.ptr(theta), cap, F.ptr(basis), F.ptr(nonbasic), F.ptr(xB),
                             F.ptr(Binv), F.ptr(x), F.ptr(hist), history)
    F.check(rc)
    k = min(n_iters.value, cap)
    out = dict(status=status.value, n_iters=n_iters.value, enter=pivots[:k, 0], leave=pivots[:k, 1], theta=theta[:k],
               basis=basis, nonbasic=nonbasic, xB=xB, Binv=Binv, x=x)
    if history:
        out["history"] = hist[: min(n_iters.value + 1, history)]
    return out


def primal_solve_batched(A, b, c, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0,
                         want_tableau=True, out=None, reg_variant=0):
    """Host buffers in, host buffers out (the reference-facing call).  `out` may carry
    preallocated (pinned) result arrays to reuse between calls."""
    A, b, c, rel = _prep(A, b, c, rel)
    count, m, n = A.shape
    rows, cols = tableau_dims(m, n, rel)
    opt = F.make_options(max_iterations, kernel, threads, reg_variant=reg_variant)
    o = out or {}
    status = o.get("status", None)
    if status is None:
        status = np.zeros(count, dtype=np.int32)
    npiv = o.get("n_pivots") if o.get("n_pivots") is not None else np.zeros(count, dtype=np.int32)
    basis = o.get("basis") if o.get("basis") is not None else np.zeros((count, rows - 1), dtype=np.int32)
    x = o.get("x") if o.get("x") is not None else np.zeros((count, n))
    z = o.get("z") if o.get("z") is not None else np.zeros(count)
    T = None
    if want_tableau:
        T = o.get("tableau") if o.get("tableau") is not None else np.zeros((count, rows, cols))
    total = C.c_longlong()
    rc = F.lib().lpx_primal_solve_batched(count, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c),
                                          C.byref(opt), F.ptr(status), F.ptr(npiv), F.ptr(basis), F.ptr(x), F.ptr(z),
                                          F.ptr(T), C.byref(total))
    F.check(rc)
    return dict(status=status, n_pivots=npiv, basis=basis, x=x, z=z, tableau=T, total_pivots=total.value)


def primal_solve_batched_dev(count, m, n, sense, dA, drel, db, dc, dstatus, dnpiv, dbasis, dx, dz, dtableau, dtotal,
                             stream, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0, reg_variant=0):
    """All arguments are raw device pointers (ints); asynchronous on `stream` (a cudaStream_t)."""
    opt = F.make_options(max_iterations, kernel, threads, reg_variant=reg_variant)
    rc = F.lib().lpx_primal_solve_batched_dev(count, m, n, sense, F.ptr(dA), F.ptr(drel), F.ptr(db), F.ptr(dc),
                                              C.byref(opt), F.ptr(dstatus), F.ptr(dnpiv), F.ptr(dbasis), F.ptr(dx),
                                              F.ptr(dz), F.ptr(dtableau), F.ptr(dtotal), F.ptr(stream or 0))
    F.check(rc)


SENSITIVITY_FIELDS = ("shadow", "slack", "rhs_lo", "rhs_hi", "reduced", "cost_lo", "cost_hi")


def sensitivity_stride(m, n):
    return int(F.lib().lpx_sensitivity_stride(m, n))


def split_sensitivity(report, m, n):
    """Named views of sensitivity records (include/lpx.h): shadow, slack, rhs_lo, rhs_hi (m each), reduced,
    cost_lo, cost_hi (n each); `report` is one record or (count, stride)."""
    out, o = {}, 0
    for name, k in zip(SENSITIVITY_FIELDS, (m, m, m, m, n, n, n)):
        out[name] = report[..., o:o + k]
        o += k
    return out


def primal_solve_sensitivity_batched(A, b, c, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO,
                                     threads=0, reg_variant=0):
    """primal_solve_batched without the tableaux, plus the sensitivity report of every OPTIMAL instance
    (NaN records for the others), computed on the GPU next to the tableaux: `report` (count, 4m + 3n) and its
    named (count, .) views."""
    A, b, c, rel = _prep(A, b, c, rel)
    count, m, n = A.shape
    rows, _ = tableau_dims(m, n, rel)
    opt = F.make_options(max_iterations, kernel, threads, reg_variant=reg_variant)
    status = np.zeros(count, dtype=np.int32)
    npiv = np.zeros(count, dtype=np.int32)
    basis = np.zeros((count, rows - 1), dtype=np.int32)
    x = np.zeros((count, n))
    z = np.zeros(count)
    report = np.zeros((count, sensitivity_stride(m, n)))
    total = C.c_longlong()
    rc = F.lib().lpx_primal_solve_sensitivity_batched(count, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c),
                                                      C.byref(opt), F.ptr(status), F.ptr(npiv), F.ptr(basis),
                                                      F.ptr(x), F.ptr(z), F.ptr(report), C.byref(total))
    F.check(rc)
    return dict(status=status, n_pivots=npiv, basis=basis, x=x, z=z, total_pivots=total.value, report=report,
                **split_sensitivity(report, m, n))


def sensitivity_batched_dev(count, m, n, sense, drel, db, dc, dstatus, dbasis, dtableau, dreport, stream):
    """lpx_sensitivity_batched_dev on the outputs of primal_solve_batched_dev: raw device pointers (ints),
    asynchronous on `stream`; dreport receives count x sensitivity_stride(m, n) doubles."""
    rc = F.lib().lpx_sensitivity_batched_dev(count, m, n, sense, F.ptr(drel), F.ptr(db), F.ptr(dc), F.ptr(dstatus),
                                             F.ptr(dbasis), F.ptr(dtableau), F.ptr(dreport), F.ptr(stream or 0))
    F.check(rc)


REOPT_KINDS = {"rhs": F.REOPT_RHS, "cost": F.REOPT_COST, "row": F.REOPT_ROW, "col": F.REOPT_COL}


def reopt_payload_stride(kind, m, n):
    return int(F.lib().lpx_reopt_payload_stride(REOPT_KINDS.get(kind, kind), m, n))


def reopt_dims(kind, m, n, rel=None):
    rows, cols = C.c_int(), C.c_int()
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    F.check(F.lib().lpx_reopt_dims(REOPT_KINDS.get(kind, kind), m, n, F.ptr(rel), C.byref(rows), C.byref(cols)))
    return rows.value, cols.value


def reoptimize(kind, A, b, c, payload, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0,
               pivots_cap=64, want_tableau=True):
    """lpx_reoptimize: one GPU Primal Simplex solve of the base, then len(payload) what-if queries of one kind
    ("rhs", "cost", "row", "col" or LPX_REOPT_*) re-solved warm from its final tableau (include/lpx.h).  payload:
    (count, reopt_payload_stride) doubles.  Returns base_status and per query status, n_pivots, pivots (count, cap, 2;
    -1 past the query's pivots), basis, x, z, tableau."""
    kind = REOPT_KINDS.get(kind, kind)
    A, b, c, rel = _prep(A, b, c, rel)
    m, n = A.shape
    stride = reopt_payload_stride(kind, m, n)
    pay = np.ascontiguousarray(payload, dtype=np.float64).reshape(-1, stride)
    count = pay.shape[0]
    rows, cols = reopt_dims(kind, m, n, rel)
    nx = n + 1 if kind == F.REOPT_COL else n
    opt = F.make_options(max_iterations, kernel, threads)
    base_status = C.c_int()
    status = np.zeros(count, np.int32)
    npiv = np.zeros(count, np.int32)
    pivots = np.full((count, max(pivots_cap, 1), 2), -1, np.int32)
    basis = np.zeros((count, rows - 1), np.int32)
    x = np.zeros((count, nx))
    z = np.zeros(count)
    T = np.zeros((count, rows, cols)) if want_tableau else None
    F.check(F.lib().lpx_reoptimize(kind, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt), count,
                                   F.ptr(pay), C.byref(base_status), F.ptr(status), F.ptr(npiv), F.ptr(pivots),
                                   pivots_cap, F.ptr(basis), F.ptr(x), F.ptr(z), F.ptr(T)))
    return dict(base_status=base_status.value, status=status, n_pivots=npiv, pivots=pivots, basis=basis, x=x, z=z,
                tableau=T)


def reoptimize_batched_dev(kind, count, m, n, sense, drel, dbase_status, dbase_basis, dbase_tableau, dsrc, dpayload,
                           dstatus, dnpiv, dpivots, pivots_cap, dbasis, dx, dz, dtableau, dtotal, stream,
                           max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0):
    """lpx_reoptimize_batched_dev: raw device pointers (ints, 0 / None for the nullable ones), asynchronous on
    `stream`; the bases are outputs of primal_solve_batched_dev."""
    opt = F.make_options(max_iterations, kernel, threads)
    F.check(F.lib().lpx_reoptimize_batched_dev(
        REOPT_KINDS.get(kind, kind), count, m, n, sense, F.ptr(drel), F.ptr(dbase_status), F.ptr(dbase_basis),
        F.ptr(dbase_tableau), F.ptr(dsrc), F.ptr(dpayload), C.byref(opt), F.ptr(dstatus), F.ptr(dnpiv),
        F.ptr(dpivots), pivots_cap, F.ptr(dbasis), F.ptr(dx), F.ptr(dz), F.ptr(dtableau), F.ptr(dtotal),
        F.ptr(stream or 0)))


def cutting_plane_dims(m, n, rel=None):
    """(max_rows, max_cols) = (m' + 50, n + m' + 50): the per-IP stride of the cutting-plane tableau output."""
    rows, cols = C.c_int(), C.c_int()
    rel = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
    F.check(F.lib().lpx_cutting_plane_dims(m, n, F.ptr(rel), C.byref(rows), C.byref(cols)))
    return rows.value, cols.value


def cutting_plane_batched(A, b, c, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0,
                          want_tableau=True):
    """lpx_cutting_plane_batched: CuttingPlane.Solve for `count` IPs of one shape (A (count, m, n), b (count, m),
    c (count, n)), every round on the GPU.  Returns end, n_rounds, n_cuts (count), lp_status / lp_pivots (count, 50),
    frac_var / cut_row (count, 50), cut_a (count, 50, n), cut_b (count, 50), and the final LP of the integral ends:
    basis (count, m' + 49), x, z and tableau (count, m' + 50, n + m' + 50; the final tableau compact at the start of
    each slot: tableau_of() reshapes it), plus total_pivots."""
    A, b, c, rel = _prep(A, b, c, rel)
    count, m, n = A.shape
    R = F.CUT_MAX_ROUNDS
    max_rows, max_cols = cutting_plane_dims(m, n, rel)
    opt = F.make_options(max_iterations, kernel, threads)
    out = dict(end=np.zeros(count, np.int32), n_rounds=np.zeros(count, np.int32), n_cuts=np.zeros(count, np.int32),
               lp_status=np.zeros((count, R), np.int32), lp_pivots=np.zeros((count, R), np.int32),
               frac_var=np.zeros((count, R), np.int32), cut_row=np.zeros((count, R), np.int32),
               cut_a=np.zeros((count, R, n)), cut_b=np.zeros((count, R)),
               basis=np.zeros((count, max_rows - 1), np.int32), x=np.zeros((count, n)), z=np.zeros(count),
               tableau=np.zeros((count, max_rows, max_cols)) if want_tableau else None)
    total = C.c_longlong()
    F.check(F.lib().lpx_cutting_plane_batched(
        count, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt),
        *[F.ptr(out[k]) for k in ("end", "n_rounds", "n_cuts", "lp_status", "lp_pivots", "frac_var", "cut_row",
                                  "cut_a", "cut_b", "basis", "x", "z", "tableau")], C.byref(total)))
    out["total_pivots"] = total.value
    return out


def cutting_plane(A, b, c, rel=None, sense=0, **kw):
    """One IP through cutting_plane_batched: the same fields without the leading count axis; `tableau` is the final
    LP's tableau (m' + n_cuts + 1, n + m' + n_cuts + 1) for an integral end, else None."""
    A = np.asarray(A, dtype=np.float64)
    r = cutting_plane_batched(A[None], np.asarray(b, np.float64)[None], np.asarray(c, np.float64)[None], rel, sense,
                              **kw)
    out = {k: (v[0] if isinstance(v, np.ndarray) else v) for k, v in r.items()}
    out["tableau"] = tableau_of(out, A.shape[1]) if out["end"] == F.CUT_INTEGER and r["tableau"] is not None else None
    return out


def tableau_of(one, n):
    """The compact final tableau at the start of one IP's tableau slot (an integral end only)."""
    slot = np.asarray(one["tableau"]).reshape(-1)
    mm = one["basis"].shape[-1] - 49
    rows, cols = mm + one["n_cuts"] + 1, n + mm + one["n_cuts"] + 1
    return slot[: rows * cols].reshape(rows, cols)


def cutting_plane_batched_dev(count, m, n, sense, dA, drel, db, dc, dend, dn_rounds, dn_cuts, dlp_status, dlp_pivots,
                              dfrac_var, dcut_row, dcut_a, dcut_b, dbasis, dx, dz, dtableau, dtotal, stream,
                              max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0):
    """lpx_cutting_plane_batched_dev: raw device pointers (ints, 0 / None for the nullable ones), asynchronous on
    `stream` (a cudaStream_t)."""
    opt = F.make_options(max_iterations, kernel, threads)
    F.check(F.lib().lpx_cutting_plane_batched_dev(
        count, m, n, sense, F.ptr(dA), F.ptr(drel), F.ptr(db), F.ptr(dc), C.byref(opt), F.ptr(dend),
        F.ptr(dn_rounds), F.ptr(dn_cuts), F.ptr(dlp_status), F.ptr(dlp_pivots), F.ptr(dfrac_var), F.ptr(dcut_row),
        F.ptr(dcut_a), F.ptr(dcut_b), F.ptr(dbasis), F.ptr(dx), F.ptr(dz), F.ptr(dtableau), F.ptr(dtotal),
        F.ptr(stream or 0)))


class Session:
    """Large single LP whose tableau lives in HBM (lpx_session_*).  dual=True: DualSimplex.Solve on the model
    (lpx_dual_session_open); the silent ForceDualFeasibility pivots run inside the constructor and `.silent` counts
    them.  A Dual Simplex session has no sensitivity report and cannot be a re-optimization base."""

    def __init__(self, A, b, c, rel=None, sense=0, max_iterations=10000, device_ptrs=False, m=None, n=None,
                 single_cta_select=0, kblock=0, pass_variant=0, dual=False):
        opt = F.make_options(max_iterations, single_cta_select=single_cta_select, kblock=kblock,
                             pass_variant=pass_variant)
        L = F.lib()
        if device_ptrs:
            self.m, self.n = m, n
            relp = None if rel is None else np.ascontiguousarray(rel, dtype=np.int32)
            open_dev = L.lpx_dual_session_open_dev if dual else L.lpx_session_open_dev
            self._h = open_dev(m, n, sense, F.ptr(A), F.ptr(relp), F.ptr(b), F.ptr(c), C.cast(C.byref(opt), C.c_void_p))
        else:
            A, b, c, rel = _prep(A, b, c, rel)
            self.m, self.n = A.shape
            open_host = L.lpx_dual_session_open if dual else L.lpx_session_open
            self._h = open_host(self.m, self.n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c),
                                C.cast(C.byref(opt), C.c_void_p))
        if not self._h:
            raise F.LpxError(F.E_CUDA, F.last_error())
        r, cc = C.c_int(), C.c_int()
        F.check(L.lpx_session_dims(self._h, C.byref(r), C.byref(cc)))
        self.rows, self.cols = r.value, cc.value
        silent = C.c_int()
        F.check(L.lpx_session_silent_pivots(self._h, C.byref(silent)))
        self.dual, self.silent = dual, silent.value

    def step(self, max_pivots):
        st, tot = C.c_int(), C.c_int()
        F.check(F.lib().lpx_session_step(self._h, max_pivots, C.byref(st), C.byref(tot)))
        return st.value, tot.value

    def step_async(self, max_pivots):
        F.check(F.lib().lpx_session_step_async(self._h, max_pivots))

    def sync(self):
        st, tot = C.c_int(), C.c_int()
        F.check(F.lib().lpx_session_sync(self._h, C.byref(st), C.byref(tot)))
        return st.value, tot.value

    @property
    def stream(self):
        return F.lib().lpx_session_stream(self._h)

    def tableau(self):
        T = np.zeros((self.rows, self.cols))
        F.check(F.lib().lpx_session_read_tableau(self._h, F.ptr(T)))
        return T

    def solution(self):
        basis = np.zeros(self.rows - 1, dtype=np.int32)
        x = np.zeros(self.n)
        z = C.c_double()
        F.check(F.lib().lpx_session_read_solution(self._h, F.ptr(basis), F.ptr(x), C.cast(C.byref(z), C.c_void_p)))
        return basis, x, z.value

    def reoptimize(self, kind, payload, **opts):
        """lpx_session_reoptimize: a new Session holding one what-if query ("rhs", "cost", "row", "col" or
        LPX_REOPT_*) against this session, which must be OPTIMAL and is left unchanged.  payload:
        reopt_payload_stride(kind, m, n) doubles.  opts (max_iterations, single_cta_select, kblock, pass_variant)
        select the Primal Simplex protocol of COST / COL queries; none given: this session's options."""
        kind = REOPT_KINDS.get(kind, kind)
        pay = np.ascontiguousarray(payload, dtype=np.float64).ravel()
        if kind in REOPT_KINDS.values() and pay.size != reopt_payload_stride(kind, self.m, self.n):
            raise F.LpxError(F.E_BAD_ARGS, "payload has %d doubles, kind %d needs %d" % (
                pay.size, kind, reopt_payload_stride(kind, self.m, self.n)))
        opt = F.make_options(**opts) if opts else None
        h = F.lib().lpx_session_reoptimize(self._h, kind, F.ptr(pay),
                                           None if opt is None else C.cast(C.byref(opt), C.c_void_p))
        if not h:
            raise F.LpxError(F.E_BAD_ARGS, F.last_error())
        q = Session.__new__(Session)
        q._h = h
        q.dual, q.silent = False, 0
        q.m = self.m + (kind == F.REOPT_ROW)
        q.n = self.n + (kind == F.REOPT_COL)
        r, cc = C.c_int(), C.c_int()
        F.check(F.lib().lpx_session_dims(h, C.byref(r), C.byref(cc)))
        q.rows, q.cols = r.value, cc.value
        return q

    def sensitivity(self):
        """Sensitivity report of the session's tableau (NaNs unless its status is OPTIMAL): `report` and its
        named views."""
        rep = np.zeros(sensitivity_stride(self.m, self.n))
        F.check(F.lib().lpx_session_sensitivity(self._h, F.ptr(rep)))
        return dict(report=rep, **split_sensitivity(rep, self.m, self.n))

    def pivots(self, cap):
        p = np.full((max(cap, 1), 2), -1, dtype=np.int32)
        F.check(F.lib().lpx_session_read_pivots(self._h, F.ptr(p), cap))
        return p

    def close(self):
        if self._h:
            F.lib().lpx_session_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bnb_simplex_batched(A, b, c, rel=None, sense=0, max_iterations=10000, kernel=F.KERNEL_AUTO, threads=0,
                        on_node=None, want_history=False):
    A, b, c, rel = _prep(A, b, c, rel)
    count, m, n = A.shape
    opt = F.make_options(max_iterations, kernel, threads)
    found = np.zeros(count, dtype=np.int32)
    best_z = np.zeros(count)
    best_x = np.zeros((count, n))
    n_nodes = np.zeros(count, dtype=np.int32)
    lp_piv = np.zeros(count, dtype=np.int64)
    root_status = np.zeros(count, dtype=np.int32)
    cb = F.BNB_NODE_FN(on_node) if on_node else None
    rc = F.lib().lpx_bnb_simplex_batched(count, m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.byref(opt),
                                         F.BNB_WANT_HISTORY if want_history else 0, F.ptr(found), F.ptr(best_z),
                                         F.ptr(best_x), F.ptr(n_nodes), F.ptr(lp_piv), F.ptr(root_status),
                                         C.cast(cb, C.c_void_p) if cb else None, None)
    F.check(rc)
    return dict(found=found.astype(bool), best_z=best_z, best_x=best_x, n_nodes=n_nodes, lp_pivots=lp_piv,
                root_status=root_status)


def bnb_simplex(A, b, c, rel=None, sense=0, trace=False, want_history=False, **kw):
    """Single IP.  With trace=True also returns the node records in the reference's order."""
    A = np.asarray(A, dtype=np.float64)
    nodes = []

    def on_node(p, _user):
        nd = p.contents
        n = A.shape[1]
        rec = dict(index=nd.index, depth=nd.depth, parent=nd.parent, is_ceil_child=nd.is_ceil_child,
                   id_path=[nd.id_path[i] for i in range(nd.id_path_len)], bound_var=nd.bound_var,
                   bound_val=nd.bound_val, algo=nd.algo, lp_status=nd.lp_status, outcome=nd.outcome,
                   n_pivots=nd.n_pivots, silent=nd.silent_pivots, rows=nd.rows, cols=nd.cols, z=nd.z,
                   x=np.array([nd.x[i] for i in range(n)]) if nd.x else None, branch_var=nd.branch_var,
                   floor_val=nd.floor_val, ceil_val=nd.ceil_val,
                   pivots=np.ctypeslib.as_array(nd.pivots, shape=(2 * nd.n_pivots,)).copy().reshape(-1, 2)
                   if nd.pivots and nd.n_pivots else None)
        if nd.n_history:
            cnt = nd.n_history * nd.rows * nd.cols
            rec["history"] = np.ctypeslib.as_array(nd.history, shape=(cnt,)).copy().reshape(nd.n_history, nd.rows,
                                                                                              nd.cols)
        nodes.append(rec)

    r = bnb_simplex_batched(A[None], np.asarray(b)[None], np.asarray(c)[None], rel, sense,
                            on_node=on_node if (trace or want_history) else None, want_history=want_history, **kw)
    out = dict(found=bool(r["found"][0]), best_z=float(r["best_z"][0]), best_x=r["best_x"][0],
               n_nodes=int(r["n_nodes"][0]), lp_pivots=int(r["lp_pivots"][0]), root_status=int(r["root_status"][0]))
    if trace or want_history:
        out["nodes"] = nodes
    return out


def bnb_pooled(A, b, c, rel=None, sense=0, batch=64, node_cap=1 << 20, threads=0):
    """Mode B, the pooled tree (lpx_bnb_pooled) — NOT the reference's tree.  After lpx_comm_init every rank must
    make the same call; every rank returns the same result."""
    A, b, c, rel = _prep(A, b, c, rel)
    m, n = A.shape
    opt = F.make_options(threads=threads)
    found = C.c_int()
    best_z = C.c_double()
    best_x = np.zeros(n)
    nn, npiv, nr = C.c_longlong(), C.c_longlong(), C.c_longlong()
    nid = np.zeros(node_cap, dtype=np.int32)
    oc = np.zeros(node_cap, dtype=np.int32)
    pv = np.zeros(node_cap, dtype=np.int32)
    nz = np.zeros(node_cap)
    L = F.lib()
    L.lpx_bnb_pooled.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    rc = L.lpx_bnb_pooled(m, n, sense, F.ptr(A), F.ptr(rel), F.ptr(b), F.ptr(c), C.cast(C.byref(opt), C.c_void_p), batch,
                          C.cast(C.byref(found), C.c_void_p), C.cast(C.byref(best_z), C.c_void_p), F.ptr(best_x),
                          C.cast(C.byref(nn), C.c_void_p), C.cast(C.byref(npiv), C.c_void_p),
                          C.cast(C.byref(nr), C.c_void_p), node_cap, F.ptr(nid), F.ptr(oc), F.ptr(pv), F.ptr(nz))
    F.check(rc)
    k = min(nn.value, node_cap)
    return dict(found=bool(found.value), best_z=best_z.value, best_x=best_x, n_nodes=nn.value, total_pivots=npiv.value,
                rounds=nr.value, node_id=nid[:k], outcome=oc[:k], pivots=pv[:k], z=nz[:k])


def bnb_knapsack(profit, weight, capacity, trace=False, spec_nodes=0, spec_depth=0, sequential=False,
                 shard_tree=False, warps=0):
    p = np.ascontiguousarray(profit, dtype=np.float64)
    w = np.ascontiguousarray(weight, dtype=np.float64)
    n = p.shape[0]
    # sequential=True forces the ordered-summation kernel path even for exactly summable integer data
    # shard_tree=True: all ranks of lpx_comm_init work on this ONE tree (see lpx_options.knap_shard_tree)
    # warps: 0 auto, 1 one warp per instance, 2 a main + helper pair (lpx_options.knap_warps)
    opt = F.make_options(spec_nodes=spec_nodes, spec_depth=spec_depth, ordered_sums=1 if sequential else 0,
                         shard_tree=1 if shard_tree else 0, knap_warps=warps)
    found = C.c_int()
    best = C.c_double()
    bx = np.zeros(n, dtype=np.int32)
    ne, npops = C.c_longlong(), C.c_longlong()
    rank = np.zeros(n, dtype=np.int32)
    pops = []

    def ev_dict(e):
        return dict(pop_index=e.pop_index, child=e.child, var=e.var, bound=e.bound, weight=e.weight,
                    frac_rank=e.frac_rank, frac=e.frac, break_rank=e.break_rank, decision=e.decision,
                    assigned=np.array([e.assigned[i] for i in range(n)], dtype=np.int8) if e.assigned else None)

    def on_pop(pp, l, r, _user):
        q = pp.contents
        pops.append(dict(pop_index=q.pop_index, label=[q.label[i] for i in range(q.label_len)],
                         relax=ev_dict(q.relax), closed=q.closed, left=ev_dict(l.contents) if l else None,
                         right=ev_dict(r.contents) if r else None))

    cb = F.KNAP_POP_FN(on_pop) if trace else None
    rc = F.lib().lpx_bnb_knapsack(n, F.ptr(p), F.ptr(w), float(capacity), C.cast(C.byref(opt), C.c_void_p),
                                  C.byref(found), C.byref(best), F.ptr(bx), C.byref(ne), C.byref(npops),
                                  F.ptr(rank), C.cast(cb, C.c_void_p) if cb else None, None)
    F.check(rc)
    out = dict(found=bool(found.value), best=best.value, best_x=bx, n_evals=ne.value, n_pops=npops.value,
               rank_order=rank)
    if trace:
        out["pops"] = pops
    return out


def bnb_knapsack_batched(profit, weight, capacity, spec_nodes=0, spec_depth=0, warps=0):
    p = np.ascontiguousarray(profit, dtype=np.float64)
    w = np.ascontiguousarray(weight, dtype=np.float64)
    cap = np.ascontiguousarray(capacity, dtype=np.float64)
    count, n = p.shape
    opt = F.make_options(spec_nodes=spec_nodes, spec_depth=spec_depth, knap_warps=warps)
    found = np.zeros(count, dtype=np.int32)
    best = np.zeros(count)
    bx = np.zeros((count, n), dtype=np.int32)
    ne = np.zeros(count, dtype=np.int64)
    npops = np.zeros(count, dtype=np.int64)
    rc = F.lib().lpx_bnb_knapsack_batched(count, n, F.ptr(p), F.ptr(w), F.ptr(cap), C.cast(C.byref(opt), C.c_void_p),
                                          F.ptr(found), F.ptr(best), F.ptr(bx), F.ptr(ne), F.ptr(npops))
    F.check(rc)
    return dict(found=found.astype(bool), best=best, best_x=bx, n_evals=ne, n_pops=npops)

"""ctypes view of liblpx.so (include/lpx.h) — the same C ABI the C# shim P/Invokes.

This module is the Python stand-in for the reference-side binding (see INTEGRATION.md); it adds
nothing to the data path: every call below is one C-ABI call on plain numpy buffers or raw
device pointers.  There is no CPU fallback: if liblpx.so is missing the import fails loudly, and
without a usable B200 every solve call raises LpxError.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblpx.so")

OPTIMAL, UNBOUNDED, INFEASIBLE, RUNNING = 0, 1, 2, 3
S_GE_ROW, S_NEG_RHS, S_ITER_LIMIT = -1, -2, -3
E_BAD_ARGS, E_CUDA, E_CAPACITY, E_NCCL = -4, -5, -8, -9
KERNEL_AUTO, KERNEL_CTA_SMEM, KERNEL_CTA_GLOBAL, KERNEL_STREAM, KERNEL_CTA_REG, KERNEL_CTA_CLUSTER = 0, 1, 2, 3, 4, 5
BNB_WANT_HISTORY = 1
REOPT_RHS, REOPT_COST, REOPT_ROW, REOPT_COL = 1, 2, 3, 4
CUT_INTEGER, CUT_INCOMPLETE, CUT_LP_ERROR, CUT_NONBASIC, CUT_MAX_ROUNDS = 0, 1, 2, 3, 50

# every symbol include/lpx.h declares; tests check that the library exports all of them
EXPORTS = [
    "lpx_default_options", "lpx_version", "lpx_last_error", "lpx_status_message", "lpx_device_count", "lpx_init",
    "lpx_shutdown", "lpx_host_alloc", "lpx_host_free", "lpx_tableau_dims", "lpx_primal_solve",
    "lpx_primal_solve_batched", "lpx_primal_solve_batched_dev", "lpx_dual_solve", "lpx_session_open",
    "lpx_session_open_dev", "lpx_session_step", "lpx_session_step_async", "lpx_session_sync", "lpx_session_stream",
    "lpx_session_dims", "lpx_session_read_tableau", "lpx_session_read_solution", "lpx_session_read_pivots",
    "lpx_session_close", "lpx_bnb_simplex_batched", "lpx_bnb_simplex", "lpx_bnb_instance", "lpx_bnb_knapsack",
    "lpx_bnb_knapsack_batched", "lpx_comm_unique_id", "lpx_comm_init", "lpx_comm_allreduce_max",
    "lpx_comm_allgather", "lpx_comm_destroy", "lpx_comm_world", "lpx_comm_rank", "lpx_kernel_launches",
    "lpx_reset_counters", "lpx_revised_solve", "lpx_revised_history_stride", "lpx_measure_fp64_rate", "lpx_measure_latencies", "lpx_session_profile", "lpx_session_debug_stamps",
    "lpx_bnb_last_stats", "lpx_bnb_pooled", "lpx_sensitivity_stride", "lpx_sensitivity_batched_dev",
    "lpx_primal_solve_sensitivity_batched", "lpx_session_sensitivity", "lpx_reopt_payload_stride", "lpx_reopt_dims",
    "lpx_reoptimize_batched_dev", "lpx_reoptimize", "lpx_session_reoptimize", "lpx_dual_session_open",
    "lpx_dual_session_open_dev", "lpx_session_silent_pivots", "lpx_cutting_plane_dims", "lpx_cutting_plane_batched",
    "lpx_cutting_plane_batched_dev",
]


class LpxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"lpx error {code}: {msg}")
        self.code = code


class Options(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("kernel", C.c_int), ("threads", C.c_int), ("knap_spec_nodes", C.c_int),
                ("knap_spec_depth", C.c_int), ("stream_protocol", C.c_int), ("reg_variant", C.c_int),
                ("stream_block", C.c_int), ("stream_pass_variant", C.c_int), ("knap_ordered_sums", C.c_int),
                ("knap_shard_tree", C.c_int), ("knap_warps", C.c_int), ("reserved", C.c_int * 4)]


class BnbNode(C.Structure):
    _fields_ = [
        ("index", C.c_int), ("depth", C.c_int), ("parent", C.c_int), ("is_ceil_child", C.c_int),
        ("id_path_len", C.c_int), ("id_path", C.POINTER(C.c_int)), ("bound_var", C.c_int), ("bound_val", C.c_int),
        ("algo", C.c_int), ("lp_status", C.c_int), ("outcome", C.c_int), ("n_pivots", C.c_int),
        ("silent_pivots", C.c_int), ("pivots", C.POINTER(C.c_int)), ("rows", C.c_int), ("cols", C.c_int),
        ("z", C.c_double), ("x", C.POINTER(C.c_double)), ("branch_var", C.c_int), ("floor_val", C.c_int),
        ("ceil_val", C.c_int), ("n_history", C.c_int), ("history", C.POINTER(C.c_double)),
    ]


class KnapEval(C.Structure):
    _fields_ = [
        ("pop_index", C.c_int), ("child", C.c_int), ("var", C.c_int), ("bound", C.c_double), ("weight", C.c_double),
        ("frac_rank", C.c_int), ("frac", C.c_double), ("break_rank", C.c_int), ("decision", C.c_int),
        ("assigned", C.POINTER(C.c_byte)),
    ]


class KnapPop(C.Structure):
    _fields_ = [("pop_index", C.c_int), ("label_len", C.c_int), ("label", C.POINTER(C.c_int)), ("relax", KnapEval),
                ("closed", C.c_int)]


BNB_NODE_FN = C.CFUNCTYPE(None, C.POINTER(BnbNode), C.c_void_p)
KNAP_POP_FN = C.CFUNCTYPE(None, C.POINTER(KnapPop), C.POINTER(KnapEval), C.POINTER(KnapEval), C.c_void_p)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_llp = C.POINTER(C.c_longlong)

_lib = None


def lib():
    """Load liblpx.so (built in-tree by __graft_entry__.build / csrc/Makefile).  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
            "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    L.lpx_version.restype = C.c_char_p
    L.lpx_last_error.restype = C.c_char_p
    L.lpx_status_message.restype = C.c_char_p
    L.lpx_status_message.argtypes = [C.c_int]
    L.lpx_host_alloc.restype = C.c_void_p
    L.lpx_host_alloc.argtypes = [C.c_size_t]
    L.lpx_host_free.argtypes = [C.c_void_p]
    L.lpx_kernel_launches.restype = C.c_longlong
    L.lpx_session_open.restype = C.c_void_p
    L.lpx_session_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p]
    L.lpx_session_open_dev.restype = C.c_void_p
    L.lpx_session_open_dev.argtypes = L.lpx_session_open.argtypes
    for f in ("lpx_dual_session_open", "lpx_dual_session_open_dev"):
        getattr(L, f).restype = C.c_void_p
        getattr(L, f).argtypes = L.lpx_session_open.argtypes
    L.lpx_session_silent_pivots.argtypes = [C.c_void_p, _ip]
    L.lpx_session_stream.restype = C.c_void_p
    L.lpx_session_stream.argtypes = [C.c_void_p]
    for f in ("lpx_session_step",):
        getattr(L, f).argtypes = [C.c_void_p, C.c_int, _ip, _ip]
    L.lpx_session_step_async.argtypes = [C.c_void_p, C.c_int]
    L.lpx_session_sync.argtypes = [C.c_void_p, _ip, _ip]
    L.lpx_session_dims.argtypes = [C.c_void_p, _ip, _ip]
    L.lpx_session_read_tableau.argtypes = [C.c_void_p, C.c_void_p]
    L.lpx_session_read_solution.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lpx_session_read_pivots.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.lpx_session_close.argtypes = [C.c_void_p]
    L.lpx_primal_solve.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, _ip, _ip, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int]
    L.lpx_dual_solve.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, _ip, _ip, _ip, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_int]
    L.lpx_primal_solve_batched.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, _llp]
    L.lpx_primal_solve_batched_dev.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p]
    L.lpx_sensitivity_stride.restype = C.c_size_t
    L.lpx_sensitivity_stride.argtypes = [C.c_int, C.c_int]
    L.lpx_sensitivity_batched_dev.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 8
    L.lpx_primal_solve_sensitivity_batched.argtypes = L.lpx_primal_solve_batched.argtypes
    L.lpx_session_sensitivity.argtypes = [C.c_void_p, C.c_void_p]
    L.lpx_reopt_payload_stride.restype = C.c_size_t
    L.lpx_reopt_payload_stride.argtypes = [C.c_int, C.c_int, C.c_int]
    L.lpx_reopt_dims.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, _ip, _ip]
    L.lpx_reoptimize_batched_dev.argtypes = ([C.c_int] * 5 + [C.c_void_p] * 9 + [C.c_void_p, C.c_int]
                                             + [C.c_void_p] * 6)
    L.lpx_reoptimize.argtypes = ([C.c_int] * 4 + [C.c_void_p] * 5 + [C.c_int] + [C.c_void_p] * 5 + [C.c_int]
                                 + [C.c_void_p] * 4)
    L.lpx_session_reoptimize.restype = C.c_void_p
    L.lpx_session_reoptimize.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.lpx_cutting_plane_dims.argtypes = [C.c_int, C.c_int, C.c_void_p, _ip, _ip]
    L.lpx_cutting_plane_batched.argtypes = [C.c_int] * 4 + [C.c_void_p] * 18 + [_llp]
    L.lpx_cutting_plane_batched_dev.argtypes = [C.c_int] * 4 + [C.c_void_p] * 20
    L.lpx_bnb_simplex_batched.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lpx_bnb_knapsack.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, _ip, _dp, C.c_void_p,
                                   _llp, _llp, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lpx_bnb_knapsack_batched.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lpx_comm_unique_id.argtypes = [C.c_void_p]
    L.lpx_comm_init.argtypes = [C.c_int, C.c_int, C.c_void_p]
    L.lpx_comm_allreduce_max.argtypes = [C.c_void_p, C.c_int]
    L.lpx_comm_allgather.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    _lib = L
    return L


def last_error():
    return lib().lpx_last_error().decode("utf-8", "replace")


def check(rc):
    if rc != 0:
        raise LpxError(rc, last_error())


def make_options(max_iterations=10000, kernel=KERNEL_AUTO, threads=0, spec_nodes=0, spec_depth=0, single_cta_select=0, reg_variant=0, kblock=0, pass_variant=0, ordered_sums=0, shard_tree=0, knap_warps=0):
    o = Options()
    lib().lpx_default_options(C.byref(o))
    o.max_iterations = max_iterations
    o.kernel = kernel
    o.threads = threads
    o.knap_spec_nodes = spec_nodes
    o.knap_spec_depth = spec_depth
    o.stream_protocol = single_cta_select  # 0 blocked look-ahead (cluster), 3 blocked (one CTA), 1 / 2 per pivot
    # (Dual Simplex sessions: 0 / 3 / 4 the blocked dual look-ahead, 1 / 2 per pivot)
    o.reg_variant = reg_variant
    o.stream_block = kblock
    o.stream_pass_variant = pass_variant
    o.knap_ordered_sums = ordered_sums
    o.knap_shard_tree = shard_tree
    o.knap_warps = knap_warps
    return o


def ptr(a):
    """numpy array -> void*; None -> NULL; int -> raw (device) pointer."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return C.c_void_p(a.ctypes.data)


def status_message(status):
    return lib().lpx_status_message(status).decode("utf-8")


class PinnedArray:
    """numpy view over lpx_host_alloc (page-locked) memory."""

    def __init__(self, shape, dtype=np.float64):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._p = lib().lpx_host_alloc(max(n, 16))
        if not self._p:
            raise LpxError(E_CUDA, last_error())
        buf = (C.c_byte * max(n, 16)).from_address(self._p)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p:
            self.array = None
            lib().lpx_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

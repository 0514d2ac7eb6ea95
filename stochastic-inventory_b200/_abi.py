"""ctypes binding of include/sdpb200.h (libsdpb200.so).

This is the same binding a Java maintainer would write with Panama FFM (INTEGRATION.md shows that
one); Python is used here because the build image has no JDK.  There is no fallback: if the
shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsdpb200.so")

# --- enums (include/sdpb200.h) -------------------------------------------------------------
SDPB_OK = 0
SDPB_ERR_ARG, SDPB_ERR_OFFGRID, SDPB_ERR_NO_DEVICE, SDPB_ERR_CUDA = -1, -2, -3, -4
SDPB_ERR_STATE, SDPB_ERR_NOMEM, SDPB_ERR_UNSOLVED, SDPB_ERR_PEER = -5, -6, -7, -8
STATUS_NAMES = {0: "SDPB_OK", -1: "SDPB_ERR_ARG", -2: "SDPB_ERR_OFFGRID", -3: "SDPB_ERR_NO_DEVICE",
                -4: "SDPB_ERR_CUDA", -5: "SDPB_ERR_STATE", -6: "SDPB_ERR_NOMEM", -7: "SDPB_ERR_UNSOLVED",
                -8: "SDPB_ERR_PEER"}
ABI_VERSION = 4
ALLOW_CLIPPED_SUCCESSORS, ALLOW_CAPPED_ACTIONS = 1, 2
PEER_BLOB_BYTES = 256

COST_BACKORDER, COST_CASH_DEPOSIT, COST_CASH_OVERDRAFT, COST_CASH_XR = 0, 1, 2, 3
COST_CASH_OD_LIMIT, COST_CASH_OD_TESTING, COST_CASH_LOAN, COST_CASH_TWO_PRODUCT, COST_STAFF = 4, 5, 6, 7, 8
REC_EXPECT, REC_SURVIVAL = 0, 1
MIN, MAX = 0, 1
Q_DIV, Q_LONGDIV, Q_TRUNC = 0, 1, 2
F_CLAMP_INV, F_LOST_SALES, F_GY_MODE, F_NO_ORDER_LAST, F_CASH_LIMITED_ACTIONS = 1, 2, 4, 8, 16
KERNEL_AUTO, KERNEL_GENERIC, KERNEL_TILED, KERNEL_STAGED, KERNEL_CASH_INT, KERNEL_TILED2, KERNEL_LEAD_SLAB = 0, 1, 2, 3, 4, 5, 6
KERNEL_LEAD_COL, KERNEL_CASH_DIAG, KERNEL_LEAD_Q2, KERNEL_TWO_PRODUCT_ROW, KERNEL_FUSED, KERNEL_CASH_ROW = 7, 8, 9, 10, 11, 12
KERNEL_CASH_TAIL = 13
KERNEL_LEAD_Q2M = 14  # reported only
KERNEL_COLLAPSED = 15  # request only: opt-in, ~1e-13 relative, not bit-identical

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class SdpbModel(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("cost_kind", C.c_int32), ("recursion", C.c_int32),
        ("direction", C.c_int32), ("T", C.c_int32), ("lead_time", C.c_int32), ("flags", C.c_uint32),
        ("max_order_idx", C.c_int32), ("gamma", C.c_double),
        ("pmf_len", _ip), ("pmf_d", _dp), ("pmf_p", _dp),
        ("inv_min", C.c_double), ("inv_max", C.c_double), ("step", C.c_double),
        ("cash_min", C.c_double), ("cash_max", C.c_double),
        ("quantiser", C.c_int32), ("q_from_period", C.c_int32),
        ("q_mul", C.c_double), ("q_div", C.c_double),
        ("fixed_cost", C.c_double), ("vari_cost", C.c_double), ("hold_cost", C.c_double),
        ("penalty_cost", C.c_double), ("price", C.c_double), ("salvage", C.c_double),
        ("deposit_rate", C.c_double), ("overhead_rate", C.c_double), ("overhead", C.c_double),
        ("r0", C.c_double), ("r2", C.c_double), ("r3", C.c_double), ("od_limit", C.c_double),
        ("interest_free", C.c_double),
        ("price_t", _dp), ("vari_cost_t", _dp), ("overhead_t", _dp), ("reserve_t", _dp),
        ("reserve2", C.c_double),
        ("price2", C.c_double), ("vari_cost2", C.c_double), ("salvage2", C.c_double), ("pmf_d2", _dp),
        ("tie_tolerance", C.c_double),
        ("apmf_len", _ip), ("apmf_p", _dp), ("min_level_t", _dp),
        ("terminal_value", _dp),
    ]


class SdpbOptions(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("shard_rank", C.c_int32),
        ("shard_count", C.c_int32), ("kernel", C.c_int32), ("dedup", C.c_int32), ("stream", C.c_void_p),
        ("allow", C.c_uint32), ("strict_cash_bounds", C.c_int32), ("profile", C.c_int32), ("reserved", C.c_int32),
    ]


class SdpbGrid(C.Structure):
    _fields_ = [
        ("ndim", C.c_int32), ("n_inv", C.c_int32), ("n_cash", C.c_int32), ("n_q", C.c_int32),
        ("n_states", C.c_int64), ("shard_lo", C.c_int64), ("shard_hi", C.c_int64),
        ("n_actions", C.c_int32), ("T", C.c_int32), ("cash_k_min", C.c_int64),
        ("window_lo", C.c_int64), ("window_hi", C.c_int64), ("device_bytes", C.c_int64),
    ]


class SdpbStats(C.Structure):
    _fields_ = [
        ("evals", C.c_double), ("solve_ms", C.c_double), ("kernel_ms", C.c_double),
        ("launches", C.c_int32), ("kernel_used", C.c_int32), ("fp64_ops", C.c_double),
        ("evals_executed", C.c_double),
        ("clipped_successors", C.c_double), ("capped_action_sets", C.c_double), ("cash_bound_hits", C.c_double),
        ("exchange_ms", C.c_double),
    ]


class SdpbReachedModel(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("kind", C.c_int32), ("T", C.c_int32), ("q_bound", C.c_int32),
        ("n_demands", C.c_int32), ("reserved", C.c_int32),
        ("d1", _dp), ("d2", _dp), ("p", _dp), ("overhead_t", _dp),
        ("price", C.c_double * 2), ("vari_cost", C.c_double * 2), ("salvage", C.c_double * 2),
        ("r0", C.c_double), ("r1", C.c_double), ("r2", C.c_double), ("limit", C.c_double), ("interest_free", C.c_double),
        ("deposit_rate", C.c_double),
        ("min_inv", C.c_double), ("max_inv", C.c_double), ("min_cash", C.c_double), ("max_cash", C.c_double),
        ("gamma", C.c_double), ("tie_tolerance", C.c_double),
        ("fixed_cost", C.c_double), ("hold_cost", C.c_double), ("min_cash_required", C.c_double), ("state_q", C.c_double),
        ("n_demands_t", _ip),
    ]


class SdpbTopdownOptions(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("allow", C.c_uint32), ("reserved", C.c_int32),
        ("scratch_bytes", C.c_int64),
    ]


REACHED_MULTILEAD, REACHED_MULTI_XR, REACHED_MULTI_YR, REACHED_CASH_ROUNDED = 0, 1, 2, 3

# every symbol include/sdpb200.h declares
EXPORTS = [
    "sdpb_abi_version", "sdpb_sizeof_model", "sdpb_sizeof_options", "sdpb_create", "sdpb_destroy",
    "sdpb_last_error", "sdpb_grid_info", "sdpb_solve", "sdpb_solve_async", "sdpb_solve_period_async", "sdpb_sync",
    "sdpb_value", "sdpb_period_tables", "sdpb_device_tables", "sdpb_state_of_index", "sdpb_reach",
    "sdpb_opt_table", "sdpb_stats_get", "sdpb_eval_triples", "sdpb_microbench", "sdpb_simulate", "sdpb_shard_reads",
    "sdpb_sizeof_grid", "sdpb_sizeof_stats", "sdpb_reachable_hull", "sdpb_peer_export", "sdpb_peer_attach",
    "sdpb_peer_traffic", "sdpb_period_profile", "sdpb_shard_tables", "sdpb_group_create", "sdpb_group_destroy",
    "sdpb_group_last_error", "sdpb_group_solve", "sdpb_group_shard", "sdpb_group_value", "sdpb_group_period_tables",
    "sdpb_group_stats", "sdpb_solve_batch", "sdpb_trim_pool", "sdpb_reached_solve", "sdpb_reached_last_error",
    "sdpb_topdown_solve", "sdpb_topdown_destroy", "sdpb_topdown_last_error", "sdpb_topdown_value",
    "sdpb_topdown_opt_table", "sdpb_topdown_states", "sdpb_topdown_stats", "sdpb_topdown_extend",
    "sdpb_topdown_simulate", "sdpb_reached_open", "sdpb_reached_destroy", "sdpb_reached_value", "sdpb_reached_extend",
    "sdpb_reached_opt_table", "sdpb_reached_states", "sdpb_reached_stats", "sdpb_reached_simulate",
]

_lib = None


class SdpbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{STATUS_NAMES.get(code, code)}: {msg}")
        self.code = code


def microbench(device=-1):
    """-> dict(nofma_tops, fma_tflops, lds_gbs): the fp64 / shared-memory roofline denominators."""
    lib = load()
    a, b, c = C.c_double(), C.c_double(), C.c_double()
    rc = lib.sdpb_microbench(device, C.byref(a), C.byref(b), C.byref(c))
    if rc != SDPB_OK:
        raise SdpbError(rc, "sdpb_microbench failed")
    return {"nofma_tops": a.value, "fma_tflops": b.value, "lds_gbs": c.value}


def load():
    """Load libsdpb200.so (built in-tree by `make -C stochastic-inventory_b200/csrc`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.sdpb_abi_version.restype = C.c_int
    lib.sdpb_sizeof_model.restype = C.c_size_t
    lib.sdpb_sizeof_options.restype = C.c_size_t
    lib.sdpb_create.argtypes = [C.POINTER(SdpbModel), C.POINTER(SdpbOptions), C.POINTER(vp)]
    lib.sdpb_destroy.argtypes = [vp]
    lib.sdpb_destroy.restype = None
    lib.sdpb_last_error.argtypes = [vp]
    lib.sdpb_last_error.restype = C.c_char_p
    lib.sdpb_grid_info.argtypes = [vp, C.POINTER(SdpbGrid)]
    lib.sdpb_shard_reads.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.sdpb_solve.argtypes = [vp]
    lib.sdpb_solve_async.argtypes = [vp]
    lib.sdpb_solve_period_async.argtypes = [vp, C.c_int]
    lib.sdpb_sync.argtypes = [vp]
    lib.sdpb_value.argtypes = [vp, C.c_int, _dp, C.c_int, _dp, _dp]
    lib.sdpb_period_tables.argtypes = [vp, C.c_int, _dp, _dp]
    lib.sdpb_device_tables.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp)]
    lib.sdpb_state_of_index.argtypes = [vp, C.c_int64, _dp]
    lib.sdpb_reach.argtypes = [vp, _dp, C.c_int]
    lib.sdpb_opt_table.argtypes = [vp, _dp, C.POINTER(C.c_size_t)]
    lib.sdpb_stats_get.argtypes = [vp, C.POINTER(SdpbStats)]
    lib.sdpb_eval_triples.argtypes = [vp, C.c_int, _dp, _ip, _dp, C.c_int, _dp, _dp, _ip]
    lib.sdpb_microbench.argtypes = [C.c_int, _dp, _dp, _dp]
    lib.sdpb_simulate.argtypes = [vp, _dp, _dp, C.c_int, C.c_double, _dp]
    lib.sdpb_sizeof_grid.restype = C.c_size_t
    lib.sdpb_sizeof_stats.restype = C.c_size_t
    lib.sdpb_reachable_hull.argtypes = [C.POINTER(SdpbModel), _dp, C.c_int, _dp, _dp]
    lib.sdpb_peer_export.argtypes = [vp, vp]
    lib.sdpb_peer_attach.argtypes = [vp, vp, C.c_int]
    lib.sdpb_peer_traffic.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.sdpb_period_profile.argtypes = [vp, _dp]
    lib.sdpb_shard_tables.argtypes = [vp, C.c_int, _dp, _dp]
    lib.sdpb_group_create.argtypes = [C.POINTER(SdpbModel), C.POINTER(SdpbOptions), _ip, C.c_int, C.POINTER(vp)]
    lib.sdpb_group_destroy.argtypes = [vp]
    lib.sdpb_group_destroy.restype = None
    lib.sdpb_group_last_error.argtypes = [vp]
    lib.sdpb_group_last_error.restype = C.c_char_p
    lib.sdpb_group_solve.argtypes = [vp]
    lib.sdpb_group_shard.argtypes = [vp, C.c_int]
    lib.sdpb_group_shard.restype = vp
    lib.sdpb_group_value.argtypes = [vp, C.c_int, _dp, C.c_int, _dp, _dp]
    lib.sdpb_group_period_tables.argtypes = [vp, C.c_int, _dp, _dp]
    lib.sdpb_group_stats.argtypes = [vp, C.POINTER(SdpbStats)]
    lib.sdpb_solve_batch.argtypes = [C.POINTER(vp), C.c_int]
    lib.sdpb_trim_pool.argtypes = [C.c_int]
    lib.sdpb_reached_solve.argtypes = [C.POINTER(SdpbReachedModel), C.c_int, _dp, _dp, _dp, _dp,
                                       C.POINTER(C.c_int64), _dp]
    lib.sdpb_reached_last_error.restype = C.c_char_p
    lib.sdpb_reached_open.argtypes = [C.POINTER(SdpbReachedModel), C.c_int, C.c_int64, _dp, C.c_int, C.POINTER(vp)]
    lib.sdpb_reached_destroy.argtypes = [vp]
    lib.sdpb_reached_destroy.restype = None
    lib.sdpb_reached_value.argtypes = [vp, C.c_int, _dp, C.c_int, _dp, _dp, _dp]
    lib.sdpb_reached_extend.argtypes = [vp, C.c_int, _dp, C.c_int]
    lib.sdpb_reached_opt_table.argtypes = [vp, _dp, C.POINTER(C.c_size_t)]
    lib.sdpb_reached_states.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.sdpb_reached_stats.argtypes = [vp, C.POINTER(SdpbStats)]
    lib.sdpb_reached_simulate.argtypes = [vp, _dp, _dp, C.c_int, C.c_double, _dp]
    lib.sdpb_topdown_solve.argtypes = [C.POINTER(SdpbModel), C.POINTER(SdpbTopdownOptions), _dp, C.c_int, C.POINTER(vp)]
    lib.sdpb_topdown_destroy.argtypes = [vp]
    lib.sdpb_topdown_destroy.restype = None
    lib.sdpb_topdown_last_error.argtypes = [vp]
    lib.sdpb_topdown_last_error.restype = C.c_char_p
    lib.sdpb_topdown_value.argtypes = [vp, C.c_int, _dp, C.c_int, _dp, _dp]
    lib.sdpb_topdown_opt_table.argtypes = [vp, _dp, C.POINTER(C.c_size_t)]
    lib.sdpb_topdown_states.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.sdpb_topdown_stats.argtypes = [vp, C.POINTER(SdpbStats)]
    lib.sdpb_topdown_extend.argtypes = [vp, C.c_int, _dp, C.c_int]
    lib.sdpb_topdown_simulate.argtypes = [vp, _dp, _dp, C.c_int, C.c_double, _dp]
    if (lib.sdpb_sizeof_model() != C.sizeof(SdpbModel) or lib.sdpb_sizeof_options() != C.sizeof(SdpbOptions)
            or lib.sdpb_sizeof_grid() != C.sizeof(SdpbGrid) or lib.sdpb_sizeof_stats() != C.sizeof(SdpbStats)
            or lib.sdpb_abi_version() != ABI_VERSION):
        raise ImportError("libsdpb200.so struct layout / ABI version differs from the ctypes binding")
    _lib = lib
    return lib

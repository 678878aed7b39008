"""ctypes binding of ``libctb.so`` (declared in ``include/ctb.h``).

The library is built in-tree by ``__graft_entry__.build()``.  There is no CPU
fallback: if the shared object is missing this module raises at first use.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CTB_LIBRARY: path of a development build of the library (bench_micro/ experiments)
LIB_PATH = os.environ.get("CTB_LIBRARY") or os.path.join(_HERE, "libctb.so")

OK, ERR_LABEL_NOT_FOUND, ERR_CUDA, ERR_INVALID, ERR_UNSUPPORTED = range(5)
F32, F64 = 0, 1
LAYOUT_TIME_MAJOR, LAYOUT_CELL_MAJOR = 0, 1
TR_IDENTITY, TR_POLY, TR_EDD, TR_GDD, TR_BINS, TR_RCSPLINE = range(6)
MAX_OUT = 4
VARIANT_AUTO, VARIANT_STAGED, VARIANT_DIRECT = 0, 1, 2
VARIANT_MAPPED_HOST = 0x100   # or-ed into a variant: x0 / x1 are mapped pinned host memory, read in place
DAILY_MEAN, DAILY_MIN, DAILY_MAX = 1, 2, 4
STEP_EDD, STEP_GDD, STEP_BINS = 1, 2, 3

# every symbol include/ctb.h declares (tests check the .so exports each one)
SYMBOLS = (
    "ctb_version", "ctb_last_error", "ctb_launch_count", "ctb_plan_build", "ctb_plan_free",
    "ctb_plan_get_info", "ctb_plan_row_cells", "ctb_plan_den", "ctb_plan_row_weights", "ctb_plan_region_order",
    "ctb_aggregate_workspace_bytes", "ctb_aggregate", "ctb_transform", "ctb_gather_rows",
    "ctb_host_pack", "ctb_pull_pack", "ctb_pull_pack_daily", "ctb_pull_pack_daily_steps",
    "ctb_pull_pack_decode", "ctb_pull_pack_daily_decode", "ctb_pull_pack_daily_steps_decode",
    "ctb_copy_rows_to_host", "ctb_time_groups_create", "ctb_time_groups_free", "ctb_time_groups_count",
    "ctb_aggregate_grouped_workspace_bytes", "ctb_aggregate_grouped", "ctb_aggregate_ex",
    "ctb_ipc_alloc", "ctb_ipc_open", "ctb_ipc_close", "ctb_ipc_free", "ctb_push_rows", "ctb_fingerprint",
)


class PlanOpts(C.Structure):
    _fields_ = [("stage_bytes_per_cell_day", C.c_int32), ("smem_budget_bytes", C.c_int32),
                ("compact", C.c_int32), ("elem_bytes", C.c_int32), ("reserved", C.c_int32 * 4),
                ("cell_gate", C.c_void_p)]


class AggOpts(C.Structure):
    _fields_ = [("groups", C.c_void_p), ("t_begin", C.c_int64), ("flush", C.c_int32), ("n_peer_out", C.c_int32),
                ("day_of_year", C.c_void_p), ("peer_out", C.POINTER(C.c_void_p)), ("peer_row", C.c_void_p)]


class Decode(C.Structure):
    """``ctb_decode``: CF packing of an int16 source (scale, offset, decoded dtype, fill values)."""
    _fields_ = [("scale", C.c_double), ("offset", C.c_double), ("dtype", C.c_int32), ("n_fill", C.c_int32),
                ("fill", C.c_int16 * 4)]


PUSH_SM, PUSH_COPY_ENGINE = 0, 1
MAX_PEERS = 8
IPC_HANDLE_BYTES = 64


GATE_ALWAYS = 511 << 9
GATE_NEVER = 511          # empty interval, no wrap


def gate_word(first, last, wrap):
    """first_day | last_day << 9 | wrap << 18 (include/ctb.h, ctb_plan_opts.cell_gate)."""
    return int(first) | (int(last) << 9) | (int(bool(wrap)) << 18)


class PlanInfo(C.Structure):
    _fields_ = [
        ("n_rows", C.c_int64), ("nnz", C.c_int64), ("n_cells_distinct", C.c_int64),
        ("n_cells_grid", C.c_int64), ("n_regions", C.c_int32), ("n_bundles", C.c_int32),
        ("n_pieces", C.c_int64), ("n_pieces_distinct", C.c_int64),
        ("n_split_regions", C.c_int32), ("n_scratch_slots", C.c_int32),
        ("cap_cells", C.c_int32), ("max_bundle_cells", C.c_int32), ("time_block", C.c_int32),
        ("max_region_rows", C.c_int32), ("max_meta_bytes", C.c_int32), ("n_packed_cells", C.c_int32),
        ("n_quads", C.c_int64), ("n_quads_conflict", C.c_int64),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


_lib = None


def lib():
    """Load (once) and return the shared library; fail loudly if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "climate_toolbox_b200: native library {} is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` from the repo root. "
            "There is no CPU fallback for the aggregation path.".format(LIB_PATH))
    L = C.CDLL(LIB_PATH)
    p, i32, i64, dp, ip, vp = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_double), \
        C.POINTER(C.c_int32), C.c_void_p
    L.ctb_version.restype = C.c_int
    L.ctb_last_error.restype = C.c_char_p
    L.ctb_launch_count.restype = i64
    L.ctb_plan_build.restype = C.c_int
    L.ctb_plan_build.argtypes = [dp, i32, ip, i32, dp, i32, ip, i32, dp, dp, ip, dp, dp, i64, i32,
                                 C.POINTER(PlanOpts), C.c_int, C.POINTER(p), C.POINTER(i64),
                                 C.POINTER(i32)]
    L.ctb_plan_free.restype = None
    L.ctb_plan_free.argtypes = [p]
    L.ctb_plan_get_info.restype = C.c_int
    L.ctb_plan_get_info.argtypes = [p, C.POINTER(PlanInfo)]
    for name, ptr in (("ctb_plan_row_cells", ip), ("ctb_plan_den", dp), ("ctb_plan_row_weights", dp),
                      ("ctb_plan_region_order", ip)):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [p, ptr]
    L.ctb_aggregate_workspace_bytes.restype = C.c_size_t
    L.ctb_aggregate_workspace_bytes.argtypes = [p, i64, C.c_int]
    L.ctb_aggregate.restype = C.c_int
    L.ctb_aggregate.argtypes = [p, vp, vp, C.c_int, C.c_int, i64, vp, i64, C.c_int, dp, C.c_int,
                                C.c_int, vp, i64, vp, C.c_size_t, C.c_int, vp]
    L.ctb_aggregate_ex.restype = C.c_int
    L.ctb_aggregate_ex.argtypes = [p, vp, vp, C.c_int, C.c_int, i64, vp, i64, C.c_int, dp, C.c_int,
                                   C.c_int, C.POINTER(AggOpts), vp, i64, vp, C.c_size_t, C.c_int, vp]
    L.ctb_ipc_alloc.restype = C.c_int
    L.ctb_ipc_alloc.argtypes = [C.c_size_t, C.c_int, C.POINTER(vp), vp]
    L.ctb_ipc_open.restype = C.c_int
    L.ctb_ipc_open.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.ctb_ipc_close.restype = C.c_int
    L.ctb_ipc_close.argtypes = [vp, C.c_int]
    L.ctb_ipc_free.restype = C.c_int
    L.ctb_ipc_free.argtypes = [vp, C.c_int]
    L.ctb_fingerprint.restype = C.c_uint64
    L.ctb_fingerprint.argtypes = [vp, C.c_size_t]
    L.ctb_push_rows.restype = C.c_int
    L.ctb_push_rows.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.POINTER(vp), C.c_int, vp]
    L.ctb_transform.restype = C.c_int
    L.ctb_transform.argtypes = [vp, vp, C.c_int, i64, C.c_int, dp, C.c_int, C.c_int, vp, vp]
    L.ctb_gather_rows.restype = C.c_int
    L.ctb_gather_rows.argtypes = [p, vp, C.c_int, C.c_int, i64, vp, i64, vp, vp]
    L.ctb_pull_pack.restype = C.c_int
    L.ctb_pull_pack.argtypes = [p, vp, C.c_int, i64, vp, i64, i64, vp, vp]
    L.ctb_pull_pack_daily.restype = C.c_int
    L.ctb_pull_pack_daily.argtypes = [p, vp, C.c_int, i64, C.c_int, vp, i64, i64, C.c_int, vp, vp, vp, vp]
    L.ctb_pull_pack_daily_steps.restype = C.c_int
    L.ctb_pull_pack_daily_steps.argtypes = [p, vp, C.c_int, i64, C.c_int, vp, i64, i64, C.c_int, vp, C.c_int, C.c_int,
                                            vp, vp]
    dec = C.POINTER(Decode)
    L.ctb_pull_pack_decode.restype = C.c_int
    L.ctb_pull_pack_decode.argtypes = [p, vp, i64, dec, vp, i64, i64, vp, vp]
    L.ctb_pull_pack_daily_decode.restype = C.c_int
    L.ctb_pull_pack_daily_decode.argtypes = [p, vp, i64, dec, C.c_int, vp, i64, i64, C.c_int, vp, vp, vp, vp]
    L.ctb_pull_pack_daily_steps_decode.restype = C.c_int
    L.ctb_pull_pack_daily_steps_decode.argtypes = [p, vp, i64, dec, C.c_int, vp, i64, i64, C.c_int, vp, C.c_int,
                                                   C.c_int, vp, vp]
    L.ctb_copy_rows_to_host.restype = C.c_int
    L.ctb_copy_rows_to_host.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_size_t, C.c_size_t, vp]
    L.ctb_time_groups_create.restype = C.c_int
    L.ctb_time_groups_create.argtypes = [ip, i64, C.c_int, C.POINTER(p)]
    L.ctb_time_groups_free.restype = None
    L.ctb_time_groups_free.argtypes = [p]
    L.ctb_time_groups_count.restype = i32
    L.ctb_time_groups_count.argtypes = [p]
    L.ctb_aggregate_grouped_workspace_bytes.restype = C.c_size_t
    L.ctb_aggregate_grouped_workspace_bytes.argtypes = [p, p, C.c_int]
    L.ctb_aggregate_grouped.restype = C.c_int
    L.ctb_aggregate_grouped.argtypes = [p, vp, vp, C.c_int, C.c_int, i64, vp, i64, C.c_int, dp, C.c_int,
                                        C.c_int, p, i64, C.c_int, vp, i64, vp, C.c_size_t, C.c_int, vp]
    L.ctb_host_pack.restype = C.c_int
    L.ctb_host_pack.argtypes = [p, vp, C.c_int, i64, C.POINTER(C.c_int64), i64, i64, vp, C.c_int]
    _lib = L
    return L


def last_error():
    return (lib().ctb_last_error() or b"").decode("utf-8", "replace")


class CtbError(RuntimeError):
    pass


def check(rc):
    """Map a status code to the exception the reference raises at that point."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_LABEL_NOT_FOUND:
        raise KeyError(msg)           # xarray .sel miss, aggregations.py:27
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise CtbError(msg)

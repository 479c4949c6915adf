"""ctypes binding of libevgsched.so (include/evg_sched.h).

The library is the product; this module only loads it and mirrors its structs.
There is no fallback: if the shared object is missing, or no sm_100 device is
usable, every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libevgsched.so")

EVG_TIME_ZERO = -(2 ** 63)

EVG_OK = 0
EVG_ERR_INVALID, EVG_ERR_CUDA, EVG_ERR_NOMEM, EVG_ERR_STATE = -1, -2, -3, -4
EVG_ALLOC_OK, EVG_ALLOC_ERR_FUTURE_FRACTION, EVG_ALLOC_ERR_POOL_SIZE, EVG_ALLOC_ERR_PARENT_MISSING = 0, 1, 2, 3

EVG_TF_REQ_OTHER, EVG_TF_REQ_PATCH, EVG_TF_REQ_MERGE_QUEUE = 0, 1, 2
EVG_TF_GENERATE, EVG_TF_STEPBACK, EVG_TF_DEPS_MET, EVG_TF_OTHER_DISTRO = 0x4, 0x8, 0x10, 0x20
EVG_HF_RUNNING, EVG_HF_TEARDOWN, EVG_HF_RT_FOUND = 0x1, 0x2, 0x4
EVG_HG_NONE, EVG_HG_UNQUEUED = -1, -2
EVG_PROVIDER_STATIC, EVG_PROVIDER_EPHEMERAL, EVG_PROVIDER_DOCKER = 0, 1, 2
EVG_OPT_BREAKDOWN = 0x1
EVG_BD_N = 13
(EVG_BD_TASK_GROUP_LENGTH, EVG_BD_TOTAL_VALUE, EVG_BD_P_INITIAL, EVG_BD_P_TASK_GROUP, EVG_BD_P_GENERATOR,
 EVG_BD_P_COMMIT_QUEUE, EVG_BD_R_COMMIT_QUEUE, EVG_BD_R_NUM_DEPENDENTS, EVG_BD_R_ESTIMATED_RUNTIME,
 EVG_BD_R_MAINLINE_WAIT, EVG_BD_R_STEPBACK, EVG_BD_R_PATCH, EVG_BD_R_PATCH_WAIT) = range(13)
MAX_TASKS_PER_DISTRO = (1 << 21) - 1

# numpy mirrors of the POD structs (all naturally aligned, no padding)
DISTRO_CFG_DTYPE = np.dtype([
    ("patch_factor", "<i8"), ("patch_time_in_queue_factor", "<i8"), ("commit_queue_factor", "<i8"),
    ("mainline_time_in_queue_factor", "<i8"), ("expected_runtime_factor", "<i8"),
    ("generate_task_factor", "<i8"), ("stepback_task_factor", "<i8"), ("num_dependents_factor", "<f8"),
    ("target_time_ns", "<i8"), ("group_versions", "<i4"), ("includes_dependencies", "<i4"),
    ("n_versions", "<i4"), ("_reserved", "<i4")])
GROUP_INFO_FIELDS = ("count", "count_free", "count_required", "max_hosts", "expected_duration",
                     "count_duration_over_threshold", "count_wait_over_threshold",
                     "count_dep_filled_merge_queue_tasks", "duration_over_threshold")
GROUP_INFO_DTYPE = np.dtype([(f, "<i8") for f in GROUP_INFO_FIELDS])
QUEUE_INFO_DTYPE = np.dtype([
    ("length", "<i8"), ("length_with_dependencies_met", "<i8"), ("count_dep_filled_merge_queue_tasks", "<i8"),
    ("expected_duration", "<i8"), ("max_duration_threshold", "<i8"), ("count_duration_over_threshold", "<i8"),
    ("duration_over_threshold", "<i8"), ("count_wait_over_threshold", "<i8"), ("secondary_queue", "<i8"),
    ("has_ungrouped", "<i8"), ("ungrouped", GROUP_INFO_DTYPE)])
ALLOC_CFG_DTYPE = np.dtype([
    ("future_host_fraction", "<f8"), ("provider", "<i4"), ("disabled", "<i4"), ("minimum_hosts", "<i4"),
    ("maximum_hosts", "<i4"), ("round_up", "<i4"), ("waits_over_thresh_feedback", "<i4"), ("has_pool", "<i4"),
    ("pool_max_containers", "<i4"), ("parent_found", "<i4"), ("parent_maximum_hosts", "<i4")])
ALLOC_RESULT_DTYPE = np.dtype([("new_hosts", "<i4"), ("free_hosts", "<i4"), ("deficit_ns", "<i8")])
QUEUE_ITEM_DTYPE = np.dtype([("task", "<i4"), ("group_index", "<i4"), ("group_max_hosts", "<i4"), ("flags", "<u4"),
                             ("priority", "<i8"), ("expected_ns", "<i8"), ("total_value", "<i8")])
EVG_QI_DEPS_MET = 0x1
EVG_PERSISTED_QUEUE_CAP = 10000
assert QUEUE_ITEM_DTYPE.itemsize == 40
assert DISTRO_CFG_DTYPE.itemsize == 88 and GROUP_INFO_DTYPE.itemsize == 72
assert QUEUE_INFO_DTYPE.itemsize == 152 and ALLOC_CFG_DTYPE.itemsize == 48 and ALLOC_RESULT_DTYPE.itemsize == 16


class StrColStruct(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("off", C.c_void_p)]


class StringColsStruct(C.Structure):
    _fields_ = [("n_tasks", C.c_int64), ("n_distros", C.c_int32), ("task_off", C.c_void_p), ("id", StrColStruct),
                ("version", StrColStruct), ("group_key", StrColStruct), ("group_max_hosts", C.c_void_p),
                ("dep_off", C.c_void_p), ("dep_id", StrColStruct)]


class InternOutStruct(C.Structure):
    _fields_ = [("group_id", C.c_void_p), ("version_id", C.c_void_p), ("group_off", C.c_void_p), ("n_versions", C.c_void_p),
                ("group_max_hosts", C.c_void_p), ("group_first", C.c_void_p), ("dep_off", C.c_void_p), ("dep_idx", C.c_void_p)]


class TaskSoAStruct(C.Structure):
    _fields_ = [("n_tasks", C.c_int64), ("n_edges", C.c_int64),
                ("priority", C.c_void_p), ("expected_ns", C.c_void_p), ("queue_basis_ns", C.c_void_p),
                ("wait_basis_ns", C.c_void_p), ("num_dependents", C.c_void_p), ("task_group_order", C.c_void_p),
                ("group_id", C.c_void_p), ("version_id", C.c_void_p), ("flags", C.c_void_p),
                ("dep_off", C.c_void_p), ("dep_idx", C.c_void_p)]


class DistroTableStruct(C.Structure):
    _fields_ = [("n_distros", C.c_int32), ("_reserved", C.c_int32), ("task_off", C.c_void_p),
                ("group_off", C.c_void_p), ("cfg", C.c_void_p), ("group_max_hosts", C.c_void_p)]


class PlanOutStruct(C.Structure):
    _fields_ = [("order", C.c_void_p), ("total_value", C.c_void_p), ("breakdown", C.c_void_p),
                ("info", C.c_void_p), ("group_info", C.c_void_p)]


class HostSoAStruct(C.Structure):
    _fields_ = [("n_hosts", C.c_int64), ("flags", C.c_void_p), ("group_id", C.c_void_p),
                ("expected_ns", C.c_void_p), ("std_ns", C.c_void_p), ("start_ns", C.c_void_p)]


class DepsInStruct(C.Structure):
    _fields_ = [("n_tasks", C.c_int64), ("n_deps", C.c_int64), ("dep_off", C.c_void_p), ("dep_kind", C.c_void_p),
                ("dep_ref", C.c_void_p), ("dep_want", C.c_void_p), ("task_state", C.c_void_p), ("task_pre", C.c_void_p),
                ("ext_state", C.c_void_p), ("n_ext", C.c_int64)]


EVG_DEP_IN_QUEUE, EVG_DEP_EXTERNAL, EVG_DEP_MISSING = 0, 1, 2
EVG_WANT_SUCCESS, EVG_WANT_FAILED, EVG_WANT_ANY, EVG_WANT_OTHER = 0, 1, 2, 3
EVG_TS_BLOCKED = 0x4
EVG_TP_OVERRIDE, EVG_TP_MET_TIME = 0x1, 0x2


class RunnableInStruct(C.Structure):
    _fields_ = [("n_tasks", C.c_int64), ("n_distros", C.c_int32), ("n_projects", C.c_int32), ("task_off", C.c_void_p),
                ("sched", C.c_void_p), ("project", C.c_void_p), ("project_flags", C.c_void_p), ("valid_off", C.c_void_p),
                ("valid_idx", C.c_void_p), ("finder", C.c_void_p), ("deps", C.POINTER(DepsInStruct))]


EVG_SQ_ACTIVATED, EVG_SQ_UNDISPATCHED, EVG_SQ_PRIORITY_OK, EVG_SQ_HOST_PLATFORM = 0x01, 0x02, 0x04, 0x08
EVG_SQ_UNATTAINABLE, EVG_SQ_OVERRIDE_DEPS, EVG_SQ_GITHUB_PR, EVG_SQ_PATCH_REQUEST = 0x10, 0x20, 0x40, 0x80
EVG_PF_ENABLED, EVG_PF_HIDDEN, EVG_PF_DISPATCHING_DISABLED, EVG_PF_PATCHING_DISABLED = 0x1, 0x2, 0x4, 0x8
EVG_FINDER_NO_DEPS, EVG_FINDER_LEGACY, EVG_FINDER_ALTERNATE = 0, 1, 2


class DurationRowsStruct(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_keys", C.c_int32), ("_reserved", C.c_int32), ("key", C.c_void_p),
                ("time_taken_ns", C.c_void_p), ("start_ns", C.c_void_p), ("finish_ns", C.c_void_p), ("flags", C.c_void_p),
                ("window_start_ns", C.c_int64), ("window_end_ns", C.c_int64)]


EVG_DR_COMPLETED, EVG_DR_TIMED_OUT = 0x1, 0x2
DURATION_STAT_DTYPE = np.dtype([("count", np.int64), ("mean_ns", np.float64), ("stddev_ns", np.float64)])


class LegacySoAStruct(C.Structure):
    _fields_ = [("n_tasks", C.c_int64), ("priority", C.c_void_p), ("ingest_ns", C.c_void_p), ("expected_ns", C.c_void_p),
                ("num_dependents", C.c_void_p), ("revision_order", C.c_void_p), ("project_id", C.c_void_p),
                ("tg_rank", C.c_void_p), ("tg_pair_id", C.c_void_p), ("task_group_order", C.c_void_p),
                ("presort_rank", C.c_void_p), ("flags", C.c_void_p)]


EVG_LF_REQ_SYSTEM, EVG_LF_REQ_PATCH, EVG_LF_REQ_OTHER, EVG_LF_GENERATE, EVG_LF_MERGE_QUEUE_VERSION = 0, 1, 2, 0x4, 0x8
EVG_LEGACY_MODE_INGEST, EVG_LEGACY_MODE_REVISION, EVG_LEGACY_MODE_LITERAL = 0, 1, 2
EVG_LEGACY_OK, EVG_LEGACY_NOT_DECOMPOSABLE = 0, 1


class DagInStruct(C.Structure):
    _fields_ = [("n_items", C.c_int64), ("n_deps", C.c_int64), ("dep_off", C.c_void_p), ("dep_item", C.c_void_p),
                ("group_id", C.c_void_p), ("group_index", C.c_void_p)]


class AllocOutStruct(C.Structure):
    _fields_ = [("result", C.c_void_p), ("status", C.c_void_p)]


class EvgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libevgsched error {code}: {msg}")
        self.code = code


# every symbol include/evg_sched.h declares: (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "evg_init": (C.c_int, [C.c_int, _P, C.POINTER(_P)]),
    "evg_shutdown": (None, [_P]),
    "evg_last_error": (C.c_char_p, []),
    "evg_abi_version": (C.c_int, []),
    "evg_host_alloc": (_P, [C.c_uint64]),
    "evg_host_free": (None, [_P]),
    "evg_plan_batch": (C.c_int, [_P, _P, _P, C.c_int64, C.c_uint32, _P]),
    "evg_alloc_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int64, _P]),
    "evg_plan_and_alloc_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_uint32, _P, _P]),
    "evg_upload": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "evg_upload_device": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "evg_update_tasks": (C.c_int, [_P, C.c_int64, _P, _P]),
    "evg_plan_from_finder": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, _P, _P]),
    "evg_intern_columns": (C.c_int, [_P, _P, C.c_int32]),
    "evg_run_resident": (C.c_int, [_P, C.c_int64, C.c_uint32]),
    "evg_download": (C.c_int, [_P, _P, _P]),
    "evg_download_queue": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int64]),
    "evg_run_resident_head": (C.c_int, [_P, C.c_int64, C.c_uint32, C.c_int32]),
    "evg_download_queue_bd": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int64]),
    "evg_device_result_ptr": (_P, [_P]),
    "evg_bind_result_buffer": (C.c_int, [_P, _P, C.c_int64]),
    "evg_last_launch_count": (C.c_int64, [_P]),
    "evg_last_timing_ms": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "evg_kernel_timing_ms": (C.c_int, [_P, C.POINTER(C.c_float), C.c_int32]),
    "evg_general_timing_ms": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "evg_deps_met_batch": (C.c_int, [_P, _P, _P]),
    "evg_upload_with_deps": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int64]),
    "evg_download_deps": (C.c_int, [_P, _P, _P]),
    "evg_find_runnable_batch": (C.c_int, [_P, _P, _P, _P]),
    "evg_expected_durations_batch": (C.c_int, [_P, _P, _P]),
    "evg_prioritize_legacy_batch": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P, _P]),
    "evg_dag_rebuild_batch": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P]),
    "evg_plan_distro": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int64, C.c_uint32, _P]),
    "evg_alloc_distro": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int64, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load libevgsched.so (built in-tree by __graft_entry__.build()). Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). evergreen_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if lib.evg_abi_version() != 1:
        raise ImportError("libevgsched.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    return (load().evg_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc != EVG_OK:
        raise EvgError(rc, last_error())


def ptr(a) -> int:
    """Address of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"], "columns must be C-contiguous"
    return a.ctypes.data

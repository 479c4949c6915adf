"""Host-side mirror of the reference `scheduler` package's plug points, backed by
libevgsched.so (CUDA, sm_100a).  Same names, argument meaning and error
behaviour as the Go interfaces this path sits behind:

* ``PrioritizeTasks`` / ``TaskPlanner``      scheduler/scheduler.go:25-51
* ``GetDistroQueueInfo``                      scheduler/scheduler.go:56-159
* ``HostAllocator`` / ``GetHostAllocator``    scheduler/host_allocator.go:15-32
* ``UtilizationBasedHostAllocator``           scheduler/utilization_based_host_allocator.go:26-130
* ``PlanDistro`` (planner half, DB-free)      scheduler/wrapper.go:30-130

plus the batched entry the GPU wants (one call per 15 s tick instead of one
amboy job per distro, units/crons.go:303-332).  Nothing here computes scores,
orders or host counts on the CPU; the host code only marshals and un-marshals.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from . import model as M
from . import soa as S

RUNNER_NAME = "scheduler"  # scheduler/scheduler.go:53
# new plug names a maintainer registers next to the existing ones
# (globals.go:1080-1100: ValidTaskPlannerVersions / ValidHostAllocators)
PLANNER_VERSION_GPU_TUNABLE = "gpu-tunable"
HOST_ALLOCATOR_GPU_UTILIZATION = "gpu-utilization"


class AllocatorError(Exception):
    """The `error` UtilizationBasedHostAllocator returns for data problems."""
    MESSAGES = {
        L.EVG_ALLOC_ERR_FUTURE_FRACTION: "future host factor cannot be greater than 1",   # allocator.go:302-304
        L.EVG_ALLOC_ERR_POOL_SIZE: "unable to plan hosts for distro due to pool size",     # allocator.go:200-202
        L.EVG_ALLOC_ERR_PARENT_MISSING: "error finding parent distros",                    # allocator.go:151-158
    }

    def __init__(self, status: int, distro_id: str = ""):
        super().__init__(f"error calculating hosts for distro {distro_id}: {self.MESSAGES.get(status, status)}")
        self.status = status


class Engine:
    """One evg_ctx: device buffers + stream.  Thread-compatible (one tick at a time).

    Result arrays live in pinned host buffers owned by the engine and are REUSED by the next
    call: copy what must outlive the next tick."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self.lib = L.load()
        h = C.c_void_p()
        L.check(self.lib.evg_init(int(device), C.c_void_p(stream) if stream else None, C.byref(h)))
        self.ctx = h
        self._n_tasks = self._n_distros = self._n_groups = 0
        self._has_hosts = False
        self._pinned = {}  # name -> (address, capacity in bytes): result buffers reused across ticks

    def close(self) -> None:
        if getattr(self, "ctx", None):
            for addr, _ in self._pinned.values():
                self.lib.evg_host_free(C.c_void_p(addr))
            self._pinned = {}
            self.lib.evg_shutdown(self.ctx)
            self.ctx = None

    def _out(self, name: str, shape, dtype) -> np.ndarray:
        """A result array in pinned host memory (evg_host_alloc), cached by name and grown on demand.
        The returned view is only valid until the next call that produces the same result."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
        nbytes = max(n * dtype.itemsize, 1)
        addr, cap = self._pinned.get(name, (0, 0))
        if cap < nbytes:
            if addr:
                self.lib.evg_host_free(C.c_void_p(addr))
            cap = nbytes + nbytes // 8
            addr = self.lib.evg_host_alloc(cap)
            if not addr:
                raise L.EvgError(L.EVG_ERR_NOMEM, L.last_error())
            self._pinned[name] = (addr, cap)
        buf = (C.c_uint8 * nbytes).from_address(addr)
        return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)

    def _plan_output(self, T: int, D: int, G: int, breakdown: bool) -> S.PlanOutput:
        info = self._out("info", D, L.QUEUE_INFO_DTYPE)
        ginfo = self._out("group_info", G, L.GROUP_INFO_DTYPE)
        return S.PlanOutput(self._out("order", T, np.int32), self._out("total_value", T, np.int64), info, ginfo,
                            self._out("breakdown", (T, L.EVG_BD_N), np.int64) if breakdown else None)

    def _alloc_output(self, D: int) -> S.AllocOutput:
        return S.AllocOutput(self._out("result", D, L.ALLOC_RESULT_DTYPE), self._out("status", D, np.int32))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- resident API ------------------------------------------------------
    def upload(self, tasks: S.TaskSoA, distros: S.DistroTable, hosts: Optional[S.HostSoA] = None) -> None:
        ts, ds = tasks.struct(), distros.struct()
        if hosts is not None:
            hs = hosts.struct()
            L.check(self.lib.evg_upload(self.ctx, C.byref(ts), C.byref(ds), C.byref(hs), L.ptr(hosts.host_off),
                                        L.ptr(hosts.cfg) if hosts.cfg.shape[0] else None))
        else:
            L.check(self.lib.evg_upload(self.ctx, C.byref(ts), C.byref(ds), None, None, None))
        self._n_tasks, self._n_distros, self._n_groups = tasks.n_tasks, distros.n_distros, distros.n_groups
        self._has_hosts = hosts is not None

    def upload_with_deps(self, tasks: S.TaskSoA, distros: S.DistroTable, hosts: Optional[S.HostSoA], deps: "S.DepsTable",
                         dep_finished: Optional[np.ndarray], now: int) -> None:
        """evg_upload_with_deps: the device evaluates Task.DependenciesMet and writes the deps-met bit and the stamped
        wait basis of the resident columns itself."""
        ts, ds, dp = tasks.struct(), distros.struct(), deps.struct()
        fin = None
        if dep_finished is not None and dep_finished.shape[0]:
            fin = np.ascontiguousarray(dep_finished, dtype=np.int64)
        if hosts is not None:
            hs = hosts.struct()
            L.check(self.lib.evg_upload_with_deps(self.ctx, C.byref(ts), C.byref(ds), C.byref(hs), L.ptr(hosts.host_off),
                                                  L.ptr(hosts.cfg) if hosts.cfg.shape[0] else None, C.byref(dp), L.ptr(fin), int(now)))
        else:
            L.check(self.lib.evg_upload_with_deps(self.ctx, C.byref(ts), C.byref(ds), None, None, None, C.byref(dp), L.ptr(fin), int(now)))
        self._n_tasks, self._n_distros, self._n_groups = tasks.n_tasks, distros.n_distros, distros.n_groups
        self._has_hosts = hosts is not None

    def download_deps(self):
        """(met, met_time): the device's Task.DependenciesMet verdicts and DependenciesMetTime stamps of the resident tick."""
        met = self._out("deps_met", self._n_tasks, np.uint8)
        stamp = self._out("deps_stamp", self._n_tasks, np.int64)
        L.check(self.lib.evg_download_deps(self.ctx, L.ptr(met) if self._n_tasks else None, L.ptr(stamp) if self._n_tasks else None))
        return met, stamp

    def upload_device(self, cols: dict, n_tasks: int, distros: S.DistroTable, hosts: Optional[S.HostSoA] = None,
                      n_edges: int = 0) -> None:
        """evg_upload_device: the task columns already live in device memory.  `cols` maps the evg_task_soa column
        names to device addresses (16-byte aligned, readable 8 rows past the end); nothing is copied, the caller
        keeps the memory alive until the next upload."""
        ts = L.TaskSoAStruct(int(n_tasks), int(n_edges), *[cols.get(name) for name, _ in S.TaskSoA.COLUMNS],
                             cols.get("dep_off"), cols.get("dep_idx"))
        ds = distros.struct()
        if hosts is not None:
            hs = hosts.struct()
            L.check(self.lib.evg_upload_device(self.ctx, C.byref(ts), C.byref(ds), C.byref(hs), L.ptr(hosts.host_off),
                                               L.ptr(hosts.cfg) if hosts.cfg.shape[0] else None))
        else:
            L.check(self.lib.evg_upload_device(self.ctx, C.byref(ts), C.byref(ds), None, None, None))
        self._n_tasks, self._n_distros, self._n_groups = int(n_tasks), distros.n_distros, distros.n_groups
        self._has_hosts = hosts is not None

    def update_tasks(self, rows: np.ndarray, values: S.TaskSoA) -> None:
        """evg_update_tasks: the per-task scalars of `rows` (task slots of the resident table) take the values of
        `values`' rows; group / version / dependency structure stays.  48 B per changed row cross PCIe."""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        values = values.normalize()
        if values.n_tasks != rows.shape[0]:
            raise ValueError("one value row per updated task slot")
        vs = values.struct()
        L.check(self.lib.evg_update_tasks(self.ctx, int(rows.shape[0]), L.ptr(rows), C.byref(vs)))

    def run(self, now: int, opts: int = 0) -> None:
        L.check(self.lib.evg_run_resident(self.ctx, int(now), int(opts)))

    def download(self, want_breakdown: bool = False, want_alloc: Optional[bool] = None):
        T, D, G = self._n_tasks, self._n_distros, self._n_groups
        po = self._plan_output(T, D, G, want_breakdown)
        ps = L.PlanOutStruct(L.ptr(po.order), L.ptr(po.total_value),
                             L.ptr(po.breakdown) if want_breakdown else None, L.ptr(po.info), L.ptr(po.group_info))
        ao = None
        if want_alloc is None:
            want_alloc = self._has_hosts
        if want_alloc:
            ao = self._alloc_output(D)
            as_ = L.AllocOutStruct(L.ptr(ao.result), L.ptr(ao.status))
            L.check(self.lib.evg_download(self.ctx, C.byref(ps), C.byref(as_)))
        else:
            L.check(self.lib.evg_download(self.ctx, C.byref(ps), None))
        return po, ao

    def download_queue(self, cap: int = 0, task_off=None):
        """evg_download_queue: (item_off, items) -- the TaskQueueItem rows of the first min(length, cap) ranks of every
        distro (cap 0 = the reference's 10 000), projected on the device; only those rows cross PCIe."""
        D = self._n_distros
        item_off = self._out("queue_item_off", D + 1, np.int64)
        cap_eff = cap or L.EVG_PERSISTED_QUEUE_CAP
        n = self._n_tasks if task_off is None else int(np.minimum(np.diff(task_off), cap_eff).sum())
        items = self._out("queue_items", max(n, 1), L.QUEUE_ITEM_DTYPE)
        L.check(self.lib.evg_download_queue(self.ctx, int(cap), L.ptr(item_off), L.ptr(items), int(max(n, 1))))
        return item_off, items[: int(item_off[D])]

    def bind_result_buffer(self, device_ptr: int, capacity_rows: int) -> None:
        """The allocator kernel writes evg_alloc_result rows straight into this device buffer
        (the all-gather send buffer, evergreen_b200.dist)."""
        L.check(self.lib.evg_bind_result_buffer(self.ctx, C.c_void_p(device_ptr) if device_ptr else None, int(capacity_rows)))

    def device_result_ptr(self) -> int:
        return int(self.lib.evg_device_result_ptr(self.ctx) or 0)

    def last_launch_count(self) -> int:
        return int(self.lib.evg_last_launch_count(self.ctx))

    def last_timing_ms(self) -> Tuple[float, float]:
        a, b = C.c_float(), C.c_float()
        L.check(self.lib.evg_last_timing_ms(self.ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def general_timing_ms(self) -> Tuple[float, float]:
        """(k_gtask ms, segmented sort ms) of the last resident run; raises when it had no general-path distro."""
        a, b = C.c_float(), C.c_float()
        L.check(self.lib.evg_general_timing_ms(self.ctx, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def kernel_timing_ms(self, n: int):
        """Per-run device time of the dominant kernel (k_plan_smem<1024,12>) for the last n resident runs."""
        buf = (C.c_float * max(n, 1))()
        L.check(self.lib.evg_kernel_timing_ms(self.ctx, buf, int(n)))
        return [buf[k] for k in range(n)]

    # -- one-shot batch API (host buffers in, host buffers out) ---------------
    def plan_batch(self, tasks: S.TaskSoA, distros: S.DistroTable, now: int, breakdown: bool = False) -> S.PlanOutput:
        T, D, G = tasks.n_tasks, distros.n_distros, distros.n_groups
        po = self._plan_output(T, D, G, breakdown)
        ps = L.PlanOutStruct(L.ptr(po.order), L.ptr(po.total_value), L.ptr(po.breakdown) if breakdown else None,
                             L.ptr(po.info), L.ptr(po.group_info))
        ts, ds = tasks.struct(), distros.struct()
        L.check(self.lib.evg_plan_batch(self.ctx, C.byref(ts), C.byref(ds), int(now),
                                        L.EVG_OPT_BREAKDOWN if breakdown else 0, C.byref(ps)))
        self._n_tasks, self._n_distros, self._n_groups, self._has_hosts = T, D, G, False
        return po

    def plan_and_alloc_batch(self, tasks: S.TaskSoA, distros: S.DistroTable, hosts: S.HostSoA, now: int,
                             breakdown: bool = False):
        T, D, G = tasks.n_tasks, distros.n_distros, distros.n_groups
        po = self._plan_output(T, D, G, breakdown)
        ao = self._alloc_output(D)
        ps = L.PlanOutStruct(L.ptr(po.order), L.ptr(po.total_value), L.ptr(po.breakdown) if breakdown else None,
                             L.ptr(po.info), L.ptr(po.group_info))
        as_ = L.AllocOutStruct(L.ptr(ao.result), L.ptr(ao.status))
        ts, ds, hs = tasks.struct(), distros.struct(), hosts.struct()
        L.check(self.lib.evg_plan_and_alloc_batch(self.ctx, C.byref(ts), C.byref(ds), C.byref(hs), L.ptr(hosts.host_off),
                                                  L.ptr(hosts.cfg) if hosts.cfg.shape[0] else None, int(now),
                                                  L.EVG_OPT_BREAKDOWN if breakdown else 0, C.byref(ps), C.byref(as_)))
        self._n_tasks, self._n_distros, self._n_groups, self._has_hosts = T, D, G, True
        return po, ao

    def deps_met_batch(self, deps: "S.DepsTable") -> np.ndarray:
        """Task.DependenciesMet for every task of the tick on the device (evg_deps_met_batch)."""
        met = self._out("deps_met", deps.n_tasks, np.uint8)
        st = deps.struct()
        L.check(self.lib.evg_deps_met_batch(self.ctx, C.byref(st), L.ptr(met) if deps.n_tasks else None))
        return met

    def find_runnable_batch(self, table: "S.RunnableTable"):
        """The task finders' filter for every distro at once (evg_find_runnable_batch):
        -> (runnable [n_tasks] distro-local indices compacted per distro, -1 padded; count [n_distros])."""
        runnable = self._out("runnable", table.n_tasks, np.int32)
        count = self._out("runnable_count", table.n_distros, np.int64)
        st, keep = table.struct()
        L.check(self.lib.evg_find_runnable_batch(self.ctx, C.byref(st), L.ptr(runnable) if table.n_tasks else None,
                                                 L.ptr(count) if table.n_distros else None))
        del keep
        return runnable, count

    def plan_from_finder(self, table: "S.RunnableTable", candidates: S.TaskSoA, distros: S.DistroTable,
                         hosts: Optional[S.HostSoA], dep_finished: Optional[np.ndarray], now: int):
        """evg_plan_from_finder: finder -> dependency predicate -> compaction -> resident planner inputs on the device.
        -> (runnable, count) as find_runnable_batch; the context then holds the tick of the KEPT tasks (run / download).
        Its group slots are the candidate groups that kept a task: `self.group_slots` lists them as rows of the
        candidate distro table, `self.group_slot_off` cuts that list per distro (see kept_group_slots)."""
        if table.deps is None:
            raise ValueError("plan_from_finder needs the candidates' dependency table")
        runnable = self._out("runnable", table.n_tasks, np.int32)
        count = self._out("runnable_count", table.n_distros, np.int64)
        st, keep = table.struct()
        ts, ds = candidates.normalize().struct(), distros.struct()
        fin = None if dep_finished is None else np.ascontiguousarray(dep_finished, dtype=np.int64)
        hargs = (None, None, None)
        if hosts is not None:
            hs = hosts.struct()
            hargs = (C.byref(hs), L.ptr(hosts.host_off), L.ptr(hosts.cfg) if hosts.cfg.shape[0] else None)
        L.check(self.lib.evg_plan_from_finder(self.ctx, C.byref(st), C.byref(ts), C.byref(ds), *hargs,
                                              L.ptr(fin) if fin is not None and fin.shape[0] else None, int(now),
                                              L.ptr(runnable) if table.n_tasks else None, L.ptr(count) if table.n_distros else None))
        del keep
        self.group_slots, self.group_slot_off = kept_group_slots(table.task_off, runnable, count, candidates.group_id,
                                                                 distros.group_off)
        self._n_tasks, self._n_distros, self._n_groups = int(count.sum()), distros.n_distros, int(self.group_slot_off[-1])
        self._has_hosts = hosts is not None
        return runnable, count

    def expected_durations_batch(self, rows: "S.DurationRows") -> np.ndarray:
        """{$avg, $stdDevPop} of TimeTaken per key (evg_expected_durations_batch) -> DURATION_STAT_DTYPE[n_keys]."""
        out = self._out("duration_stats", rows.n_keys, L.DURATION_STAT_DTYPE)
        st = rows.struct()
        L.check(self.lib.evg_expected_durations_batch(self.ctx, C.byref(st), L.ptr(out) if rows.n_keys else None))
        return out

    def prioritize_legacy_batch(self, table: "S.LegacyTable"):
        """evg_prioritize_legacy_batch: (order, count, status) of CmpBasedTaskPrioritizer over every distro of the table."""
        T, D = table.n_tasks, table.n_distros
        order = self._out("legacy_order", T, np.int32)
        count = self._out("legacy_count", D, np.int64)
        status = self._out("legacy_status", D, np.int32)
        ts = table.struct()
        L.check(self.lib.evg_prioritize_legacy_batch(self.ctx, C.byref(ts), L.ptr(table.task_off), L.ptr(table.list_mode), D,
                                                     L.ptr(order) if T else None, L.ptr(count), L.ptr(status)))
        return order, count, status

    def dag_rebuild_batch(self, item_off, group_off, dep_off, dep_item, group_id, group_index):
        """evg_dag_rebuild_batch -> (sorted, n_sorted, n_cycles, unit_items, unit_off)."""
        D = int(item_off.shape[0]) - 1
        N, E, G = int(item_off[-1]), int(dep_off[-1]) if dep_off.shape[0] else 0, int(group_off[-1])
        st = L.DagInStruct(N, E, L.ptr(dep_off), L.ptr(dep_item) if E else None, L.ptr(group_id) if N else None,
                           L.ptr(group_index) if N else None)
        sorted_ = self._out("dag_sorted", max(N, 1), np.int32)
        n_sorted, n_cycles = self._out("dag_nsorted", D, np.int32), self._out("dag_ncycles", D, np.int32)
        unit_items, unit_off = self._out("dag_unit_items", max(N, 1), np.int32), self._out("dag_unit_off", G + D, np.int32)
        L.check(self.lib.evg_dag_rebuild_batch(self.ctx, C.byref(st), L.ptr(item_off), L.ptr(group_off), D, L.ptr(sorted_) if N else None,
                                               L.ptr(n_sorted), L.ptr(n_cycles), L.ptr(unit_items) if N else None, L.ptr(unit_off)))
        return sorted_[:N], n_sorted, n_cycles, unit_items[:N], unit_off

    def alloc_batch(self, hosts: S.HostSoA, qinfo: np.ndarray, ginfo: np.ndarray, group_off: np.ndarray, now: int):
        D = int(qinfo.shape[0])
        ao = self._alloc_output(D)
        as_ = L.AllocOutStruct(L.ptr(ao.result), L.ptr(ao.status))
        hs = hosts.struct()
        qinfo = np.ascontiguousarray(qinfo, dtype=L.QUEUE_INFO_DTYPE)
        ginfo = np.ascontiguousarray(ginfo, dtype=L.GROUP_INFO_DTYPE)
        group_off = np.ascontiguousarray(group_off, dtype=np.int64)
        L.check(self.lib.evg_alloc_batch(self.ctx, C.byref(hs), L.ptr(hosts.host_off),
                                         L.ptr(hosts.cfg) if D else None, L.ptr(qinfo) if D else None,
                                         L.ptr(ginfo) if ginfo.shape[0] else None, L.ptr(group_off), D, int(now),
                                         C.byref(as_)))
        return ao, ginfo


def kept_group_slots(task_off, runnable, count, group_id, group_off):
    """The group slots evg_plan_from_finder leaves resident (include/evg_sched.h): per distro, the candidate groups
    that kept at least one task, in id order.  -> (their rows in the candidate distro table, offsets per distro)."""
    task_off, group_off = np.asarray(task_off, np.int64), np.asarray(group_off, np.int64)
    D, T = int(task_off.shape[0]) - 1, int(task_off[-1])
    used = np.zeros(int(group_off[-1]), dtype=bool)
    if T > 0 and used.shape[0] > 0:
        dist = np.repeat(np.arange(D), np.diff(task_off))
        kept = (np.arange(T) - task_off[dist]) < np.asarray(count, np.int64)[dist]
        g = np.asarray(group_id)[task_off[dist[kept]] + np.asarray(runnable)[kept]]
        live = g >= 0
        used[group_off[dist[kept][live]] + g[live]] = True
    slots = np.nonzero(used)[0]
    return slots, np.searchsorted(slots, group_off).astype(np.int64)


_default_engine: Optional[Engine] = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(0)
    return _default_engine


# ---------------------------------------------------------------------------
# reference-shaped API
# ---------------------------------------------------------------------------

@dataclass
class TaskPlannerOptions:  # scheduler/scheduler.go:18-23
    id: str = ""
    is_secondary_queue: bool = False
    includes_dependencies: bool = False
    started_at: int = M.ZERO_TIME


def _queue_info_from_rows(q, groups, names: Sequence[str]) -> M.DistroQueueInfo:
    infos: List[M.TaskGroupInfo] = []
    if int(q["has_ungrouped"]):
        u = q["ungrouped"]
        infos.append(M.TaskGroupInfo("", *[int(u[f]) for f in L.GROUP_INFO_FIELDS]))
    for name, g in zip(names, groups):
        infos.append(M.TaskGroupInfo(name, *[int(g[f]) for f in L.GROUP_INFO_FIELDS]))
    return M.DistroQueueInfo(
        length=int(q["length"]), length_with_dependencies_met=int(q["length_with_dependencies_met"]),
        count_dep_filled_merge_queue_tasks=int(q["count_dep_filled_merge_queue_tasks"]),
        expected_duration=int(q["expected_duration"]), max_duration_threshold=int(q["max_duration_threshold"]),
        count_duration_over_threshold=int(q["count_duration_over_threshold"]),
        duration_over_threshold=int(q["duration_over_threshold"]),
        count_wait_over_threshold=int(q["count_wait_over_threshold"]), task_group_infos=infos,
        secondary_queue=bool(q["secondary_queue"]))


def _upload_with_device_deps(eng: Engine, batch, soa, table, hosts, now: int, dependency_db) -> None:
    """Upload a marshalled tick and let the device evaluate Task.DependenciesMet (scheduler.go:161-168) for it; the
    DependenciesMetTime stamps it made are written back on the Task objects, like tasks[i] = task (scheduler.go:137)."""
    pairs = [(d, t) for d, t in ((b[0], b[1]) for b in batch)]
    eng.upload_with_deps(soa, table, hosts, S.marshal_deps(pairs, dependency_db), S.marshal_dep_finished(pairs), now)
    _, stamp = eng.download_deps()
    k = 0
    for _, tasks in pairs:
        for t in tasks:
            if int(stamp[k]) != M.ZERO_TIME:
                t.dependencies_met_time = int(stamp[k])
            k += 1


def plan_distros(batch: Sequence[Tuple[M.Distro, List[M.Task]]], now: int, *, engine: Optional[Engine] = None,
                 dependency_db: Optional[Dict[str, M.Task]] = None, breakdown: bool = True,
                 secondary: bool = False):
    """Batched runTunablePlanner minus persistence (scheduler/scheduler.go:34-51):
    returns, per distro, (ranked [Task] with SortingValueBreakdown stamped,
    DistroQueueInfo)."""
    eng = engine or default_engine()
    soa, table, keys = S.marshal_tasks(batch, now, dependency_db)
    _upload_with_device_deps(eng, batch, soa, table, None, now, dependency_db)
    eng.run(now, L.EVG_OPT_BREAKDOWN if breakdown else 0)
    po, _ = eng.download(want_breakdown=breakdown, want_alloc=False)
    out = []
    for d, (distro, tasks) in enumerate(batch):
        a, b = int(table.task_off[d]), int(table.task_off[d + 1])
        ga, gb = int(table.group_off[d]), int(table.group_off[d + 1])
        ranked = []
        for r in range(a, b):
            t = tasks[int(po.order[r])]
            if breakdown:
                t.sorting_value_breakdown = M.SortingValueBreakdown.from_row(po.breakdown[r])  # planner.go:475
            else:
                t.sorting_value_breakdown = M.SortingValueBreakdown(total_value=int(po.total_value[r]))
            ranked.append(t)
        info = _queue_info_from_rows(po.info[d], po.group_info[ga:gb], keys[d].group_names)
        info.secondary_queue = secondary  # scheduler.go:44
        out.append((ranked, info))
    return out


def persist_task_queues(batch: Sequence[Tuple[M.Distro, List[M.Task]]], now: int, *, engine: Optional[Engine] = None,
                        dependency_db: Optional[Dict[str, M.Task]] = None, cap: int = 0) -> List[M.TaskQueue]:
    """Batched PersistTaskQueue minus the upsert (scheduler/task_queue_persister.go:14-42, TaskQueue.Save
    model/task_queue.go:216-219): plan every distro, then build each distro's TaskQueue document from the
    TaskQueueItem rows the device projected for the first min(length, 10 000) ranks -- only those rows are copied
    back -- plus the strings of the shim's own Task objects.  Tasks are stamped like the reference leaves them
    (ExpectedDuration scheduler.go:98, DependenciesMetTime task.go:653, ScheduledTime / DependenciesMetTime
    task.go:1164-1195 at `now`)."""
    eng = engine or default_engine()
    soa, table, keys = S.marshal_tasks(batch, now, dependency_db)
    _upload_with_device_deps(eng, batch, soa, table, None, now, dependency_db)
    eng.run(now)
    po, _ = eng.download(want_alloc=False)
    item_off, items = eng.download_queue(cap, table.task_off)
    out = []
    for d, (distro, tasks) in enumerate(batch):
        ga, gb = int(table.group_off[d]), int(table.group_off[d + 1])
        info = _queue_info_from_rows(po.info[d], po.group_info[ga:gb], keys[d].group_names)
        incl = distro.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
        queue = []
        for row in items[int(item_off[d]):int(item_off[d + 1])]:
            t = tasks[int(row["task"])]
            met = bool(int(row["flags"]) & L.EVG_QI_DEPS_MET)
            if met or not incl:  # GetDistroQueueInfo stamps ExpectedDuration only on the tasks it counts (scheduler.go:98)
                t.expected_duration = int(row["expected_ns"])
            t.sorting_value_breakdown = M.SortingValueBreakdown(total_value=int(row["total_value"]))
            queue.append(M.TaskQueueItem(
                id=t.id, display_name=t.display_name, build_variant=t.build_variant,
                revision_order_number=t.revision_order_number, requester=t.requester, revision=t.revision, project=t.project,
                expected_duration=t.expected_duration, priority=int(row["priority"]),
                sorting_value_breakdown=t.sorting_value_breakdown, group=t.task_group,
                group_max_hosts=t.task_group_max_hosts, group_index=int(row["group_index"]), version=t.version,
                activated_by=t.activated_by, dependencies=[dep.task_id for dep in t.depends_on],
                dependencies_met=met))
        for t in tasks:  # SetTasksScheduledAndDepsMetTime (model/task/task.go:1164-1195), every prioritised task
            if M.is_zero_time(t.scheduled_time):
                t.scheduled_time = now
            if t.has_dependencies_met() and M.is_zero_time(t.dependencies_met_time):
                t.dependencies_met_time = now
        out.append(M.TaskQueue(distro=distro.id, generated_at=now, queue=queue, distro_queue_info=info))
    return out


def PersistTaskQueue(distro: M.Distro, tasks: List[M.Task], *, now: int, engine: Optional[Engine] = None,
                     dependency_db: Optional[Dict[str, M.Task]] = None) -> M.TaskQueue:
    """scheduler.PersistTaskQueue for one distro; the caller upserts the returned document."""
    return persist_task_queues([(distro, tasks)], now, engine=engine, dependency_db=dependency_db)[0]


def PlanDistro(distro: M.Distro, find_tasks, *, now: int, engine: Optional[Engine] = None,
               dependency_db: Optional[Dict[str, M.Task]] = None, existing_queue_length: int = 0):
    """scheduler.PlanDistro (scheduler/wrapper.go:30-130) without its Mongo calls: a disabled distro is not planned
    -- its persisted queue is cleared when it has one (wrapper.go:45-78; returns (None, True iff cleared)) --
    otherwise the task finder runs and the queue is planned and projected (returns (TaskQueue, False)).
    Unscheduling of stale tasks (underwaterUnschedule, wrapper.go:41) is a database update and stays with the caller."""
    if distro.disabled:
        return None, existing_queue_length > 0
    tasks = list(find_tasks(distro))
    return PersistTaskQueue(distro, tasks, now=now, engine=engine, dependency_db=dependency_db), False


def hosts_to_request(distro: M.Distro, info: M.DistroQueueInfo, n_provisioning_hosts: int, allocate) -> Tuple[int, int]:
    """The allocator call of hostAllocatorJob.Run (units/host_allocator.go:180-196): a single-task distro spawns one
    host per queued task whose dependencies are met, minus the hosts already provisioning (:182-184); every other distro
    asks the HostAllocator (`allocate()` -> (new_hosts, free_hosts))."""
    if distro.single_task_distro:
        return info.length_with_dependencies_met - n_provisioning_hosts, 0
    return allocate()


def PrioritizeTasks(d: M.Distro, tasks: List[M.Task], opts: Optional[TaskPlannerOptions] = None, *, now: int,
                    engine: Optional[Engine] = None, dependency_db: Optional[Dict[str, M.Task]] = None):
    """scheduler.PrioritizeTasks (scheduler/scheduler.go:27-32) for one distro.
    Returns (plan, DistroQueueInfo); the reference persists the info instead
    of returning it (scheduler.go:43-48)."""
    opts = opts or TaskPlannerOptions()
    (plan, info), = plan_distros([(d, tasks)], now, engine=engine, dependency_db=dependency_db,
                                 secondary=opts.is_secondary_queue)
    info.plan_created_at = opts.started_at
    return plan, info


def GetDistroQueueInfo(distro: M.Distro, tasks: List[M.Task], max_duration_threshold: int,
                       opts: Optional[TaskPlannerOptions] = None, *, now: int, engine: Optional[Engine] = None,
                       dependency_db: Optional[Dict[str, M.Task]] = None) -> M.DistroQueueInfo:
    """scheduler.GetDistroQueueInfo (scheduler/scheduler.go:56-159).  Every
    quantity is a commutative sum, so the plan order does not matter."""
    opts = opts or TaskPlannerOptions()
    import copy
    d = copy.deepcopy(distro)
    d.planner_settings.target_time = max_duration_threshold
    d.dispatcher_settings.version = (M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
                                     if opts.includes_dependencies else "")
    eng = engine or default_engine()
    soa, table, keys = S.marshal_tasks([(d, tasks)], now, dependency_db)
    _upload_with_device_deps(eng, [(d, tasks)], soa, table, None, now, dependency_db)
    eng.run(now)
    po, _ = eng.download(want_alloc=False)
    info = _queue_info_from_rows(po.info[0], po.group_info, keys[0].group_names)
    return info


def dependencies_met(batch: Sequence[Tuple[M.Distro, List[M.Task]]], *, engine: Optional[Engine] = None,
                     dependency_db: Optional[Dict[str, M.Task]] = None) -> List[List[bool]]:
    """Task.DependenciesMet (model/task/task.go:632-671) for every queued task, per distro: the predicate the
    task finders filter on and the bit the planner takes as EVG_TF_DEPS_MET."""
    eng = engine or default_engine()
    met = eng.deps_met_batch(S.marshal_deps(batch, dependency_db))
    out, a = [], 0
    for _, tasks in batch:
        out.append([bool(x) for x in met[a:a + len(tasks)]])
        a += len(tasks)
    return out


def find_runnable_tasks(batch: Sequence[Tuple[M.Distro, List[M.Task]]], project_refs: Sequence[M.ProjectRef], *,
                        finder: str = "legacy", dependency_db: Optional[Dict[str, M.Task]] = None,
                        engine: Optional[Engine] = None) -> List[List[M.Task]]:
    """LegacyFindRunnableTasks / AlternateTaskFinder / ParallelTaskFinder (scheduler/task_finder.go:40-317) for every
    distro of the tick: `batch` holds each distro's candidates (the rows the tasks collection has for it), the result
    the tasks each finder returns, in candidate order."""
    eng = engine or default_engine()
    table = S.marshal_runnable(batch, project_refs, finder, dependency_db)
    runnable, count = eng.find_runnable_batch(table)
    out = []
    for i, (_, tasks) in enumerate(batch):
        a = int(table.task_off[i])
        out.append([tasks[int(j)] for j in runnable[a:a + int(count[i])]])
    return out


def plan_candidates(batch: Sequence[Tuple[M.Distro, List[M.Task]]], project_refs: Sequence[M.ProjectRef], now: int, *,
                    finder: str = "legacy", dependency_db: Optional[Dict[str, M.Task]] = None,
                    engine: Optional[Engine] = None):
    """The finder -> checkDependenciesMet -> PrioritizeTasks hand-over of scheduler.PlanDistro (wrapper.go:60-118,
    scheduler.go:56-168) without the host in the middle: `batch` holds every distro's CANDIDATES; the device filters them,
    evaluates their dependencies, compacts the planner's columns and plans (evg_plan_from_finder).  Returns, per distro,
    (ranked kept tasks with TotalValue stamped, DistroQueueInfo); the TaskGroupInfos are those of the groups that kept a
    task, group slot k naming the k-th such candidate group."""
    eng = engine or default_engine()
    table = S.marshal_runnable(batch, project_refs, finder, dependency_db)
    if table.deps is None:
        table.deps = S.marshal_deps(batch, dependency_db)
    soa, dtable, keys = S.marshal_tasks(batch, now, dependency_db)
    runnable, count = eng.plan_from_finder(table, soa, dtable, None, S.marshal_dep_finished(batch), now)
    eng.run(now)
    po, _ = eng.download(want_alloc=False)
    out, a_new = [], 0
    for d, (_, tasks) in enumerate(batch):
        a = int(table.task_off[d])
        kept = [tasks[int(j)] for j in runnable[a:a + int(count[d])]]
        ranked = []
        for r in range(a_new, a_new + len(kept)):
            t = kept[int(po.order[r])]
            t.sorting_value_breakdown = M.SortingValueBreakdown(total_value=int(po.total_value[r]))
            ranked.append(t)
        a_new += len(kept)
        ga, gb = int(eng.group_slot_off[d]), int(eng.group_slot_off[d + 1])
        names = [keys[d].group_names[int(g - dtable.group_off[d])] for g in eng.group_slots[ga:gb]]
        out.append((ranked, _queue_info_from_rows(po.info[d], po.group_info[ga:gb], names)))
    return out


def LegacyFindRunnableTasks(d: M.Distro, candidates: List[M.Task], project_refs: Sequence[M.ProjectRef], **kw) -> List[M.Task]:
    """scheduler/task_finder.go:40-106 for one distro."""
    return find_runnable_tasks([(d, candidates)], project_refs, finder="legacy", **kw)[0]


def AlternateTaskFinder(d: M.Distro, candidates: List[M.Task], project_refs: Sequence[M.ProjectRef], **kw) -> List[M.Task]:
    """scheduler/task_finder.go:108-197 for one distro."""
    return find_runnable_tasks([(d, candidates)], project_refs, finder="alternate", **kw)[0]


def get_expected_durations_for_window(tasks: Sequence[M.Task], window_start: int, window_end: int, *,
                                      engine: Optional[Engine] = None) -> Dict[tuple, Tuple[float, float]]:
    """getExpectedDurationsForWindow (model/task/expected_duration.go:36-96) for every (project, build variant) at
    once: {(project, build_variant, display_name): (exp_dur ns, std_dev ns)} over the finished tasks given; keys
    whose rows all fail the $match are absent, as they are from the aggregation's result."""
    eng = engine or default_engine()
    rows, keys = S.marshal_durations(tasks, window_start, window_end)
    stats = eng.expected_durations_batch(rows)
    return {k: (float(stats["mean_ns"][i]), float(stats["stddev_ns"][i])) for i, k in enumerate(keys) if stats["count"][i] > 0}


def allocate_distros(datas: Sequence[M.HostAllocatorData], now: int, *, engine: Optional[Engine] = None):
    """Batched UtilizationBasedHostAllocator: [(new_hosts, free_hosts, status)].
    Mutates each DistroQueueInfo.TaskGroupInfos[i].CountFree/CountRequired like
    the reference (utilization_based_host_allocator.go:107-110)."""
    eng = engine or default_engine()
    qrows, grows, goff, names = S.queue_info_rows([d.distro_queue_info for d in datas])
    hosts = S.marshal_hosts(datas, names)
    ao, ginfo = eng.alloc_batch(hosts, qrows, grows, goff, now)
    out = []
    for i, data in enumerate(datas):
        st = int(ao.status[i])
        if st == L.EVG_ALLOC_OK:
            lookup = {n: k for k, n in enumerate(names[i])}
            for g in data.distro_queue_info.task_group_infos:
                k = lookup.get(g.name)
                if k is not None:
                    row = ginfo[int(goff[i]) + k]
                    g.count_free, g.count_required = int(row["count_free"]), int(row["count_required"])
        out.append((int(ao.result[i]["new_hosts"]), int(ao.result[i]["free_hosts"]), st))
    return out


def UtilizationBasedHostAllocator(data: M.HostAllocatorData, *, now: int, engine: Optional[Engine] = None):
    """HostAllocator (scheduler/host_allocator.go:15): (newHostsNeeded, estimatedFreeHosts) or raises."""
    (n, f, st), = allocate_distros([data], now, engine=engine)
    if st != L.EVG_ALLOC_OK:
        raise AllocatorError(st, data.distro.id)
    return n, f


HostAllocator = Callable[..., Tuple[int, int]]


def GetHostAllocator(name: str) -> HostAllocator:
    """scheduler.GetHostAllocator (scheduler/host_allocator.go:25-32): every name resolves to the utilization allocator."""
    return UtilizationBasedHostAllocator


def plan_and_allocate(batch: Sequence[Tuple[M.Distro, List[M.Task], M.HostAllocatorData]], now: int, *,
                      engine: Optional[Engine] = None, dependency_db: Optional[Dict[str, M.Task]] = None):
    """The fused tick: distroSchedulerJob + hostAllocatorJob for every distro
    (units/scheduler.go:57-87, units/host_allocator.go:76-196) in one call; the
    queue info stays on the device between the two halves."""
    eng = engine or default_engine()
    soa, table, keys = S.marshal_tasks([(d, t) for d, t, _ in batch], now, dependency_db)
    hosts = S.marshal_hosts([h for _, _, h in batch], [k.group_names for k in keys])
    _upload_with_device_deps(eng, batch, soa, table, hosts, now, dependency_db)
    eng.run(now)
    po, ao = eng.download()
    out = []
    for i, (distro, tasks, _) in enumerate(batch):
        a, b = int(table.task_off[i]), int(table.task_off[i + 1])
        ga, gb = int(table.group_off[i]), int(table.group_off[i + 1])
        ranked = [tasks[int(po.order[r])] for r in range(a, b)]
        info = _queue_info_from_rows(po.info[i], po.group_info[ga:gb], keys[i].group_names)
        out.append((ranked, info, int(ao.result[i]["new_hosts"]), int(ao.result[i]["free_hosts"]), int(ao.status[i])))
    return out


# ---------------------------------------------------------------------------------------------------------------
class NotDecomposableError(Exception):
    """The legacy comparator chain is not a strict weak order on some list of the distro (commit builds of several
    projects in one list, zero and non-zero expected durations mixed): the reference's result then depends on the exact
    steps of Go's sort.Stable, which this library does not reproduce.  The order it did compute is attached."""

    def __init__(self, distro_id: str, tasks):
        super().__init__(f"distro {distro_id!r}: the comparator chain is not a strict weak order on this queue")
        self.tasks = tasks


class CmpBasedTaskPrioritizer:
    """scheduler.TaskPrioritizer (scheduler/task_prioritizer.go:20-25) implemented by the legacy comparator
    prioritiser on the GPU.  PrioritizeTasks returns (tasks in run order, orderingLogic, error) like the reference;
    orderingLogic -- the reference's map of per-comparison reason strings -- is always empty here."""

    def __init__(self, runtime_id: str = "", engine: Optional[Engine] = None, now: Optional[int] = None):
        self.runtime_id = runtime_id
        self.engine = engine
        self.now = now

    def prioritize_batch(self, batch):
        """(distro_id, tasks, versions) per distro -> list of (sorted tasks, status)."""
        eng = self.engine or default_engine()
        table = S.marshal_legacy(batch, self.now)
        order, count, status = eng.prioritize_legacy_batch(table)
        out = []
        for d, (_, tasks, _) in enumerate(batch):
            a = int(table.task_off[d])
            out.append(([tasks[int(i)] for i in order[a:a + int(count[d])]], int(status[d])))
        return out

    def PrioritizeTasks(self, distro_id: str, tasks, versions=None):
        (sorted_tasks, status), = self.prioritize_batch([(distro_id, list(tasks), versions)])
        if status != L.EVG_LEGACY_OK:
            return None, None, NotDecomposableError(distro_id, sorted_tasks)
        return sorted_tasks, {}, None


# ---------------------------------------------------------------------------------------------------------------
def rebuild_dag_dispatchers(queues: Sequence[M.TaskQueue], *, engine: Optional[Engine] = None):
    """basicCachedDAGDispatcherImpl.rebuild for a batch of persisted queues (model/task_queue_service_dependency.go:
    153-252).  Per queue: (sorted item ids with None for each dependency cycle's placeholder, number of cycles,
    {composite group id: [item ids by GroupIndex]})."""
    eng = engine or default_engine()
    item_off, group_off, dep_off, dep_item, group_id, group_index, names = [0], [0], [0], [], [], [], []
    for q in queues:
        pos = {it.id: k for k, it in enumerate(q.queue)}
        groups: Dict[str, int] = {}
        for it in q.queue:
            for dep in it.dependencies:
                dep_item.append(pos.get(dep, -1))
            dep_off.append(len(dep_item))
            if it.group:
                gid = f"{it.group}_{it.build_variant}_{it.project}_{it.version}"  # compositeGroupID
                group_id.append(groups.setdefault(gid, len(groups)))
            else:
                group_id.append(-1)
            group_index.append(it.group_index)
        names.append(list(groups))
        item_off.append(item_off[-1] + len(q.queue))
        group_off.append(group_off[-1] + len(groups))
    a = lambda x, t: np.ascontiguousarray(np.array(x, dtype=t))  # noqa: E731
    io, go = a(item_off, np.int64), a(group_off, np.int64)
    srt, n_sorted, n_cycles, unit_items, unit_off = eng.dag_rebuild_batch(io, go, a(dep_off, np.int64), a(dep_item, np.int32),
                                                                            a(group_id, np.int32), a(group_index, np.int32))
    out = []
    for d, q in enumerate(queues):
        b = int(io[d])
        order = [None if int(i) < 0 else q.queue[int(i)].id for i in srt[b:b + int(n_sorted[d])]]
        u = int(go[d]) + d
        units = {name: [q.queue[int(i)].id for i in unit_items[b + int(unit_off[u + g]):b + int(unit_off[u + g + 1])]]
                 for g, name in enumerate(names[d])}
        out.append((order, int(n_cycles[d]), units))
    return out

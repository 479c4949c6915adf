"""SoA tables (numpy) that cross the C-ABI, and the marshalling of
reference-shaped structs (evergreen_b200.model) into them.

This is what the Go shim does on the reference side of the boundary
(INTEGRATION.md): intern the string keys the planner hashes
(task-group string, version, task id -> dense distro-local ids), resolve the
per-task inputs the reference fetches lazily (expected duration, dependency
state) and lay everything out column-wise.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import ctypes as C

import numpy as np

from . import _lib as L
from . import model as M


@dataclass
class TaskSoA:
    """evg_task_soa (include/evg_sched.h). 48 B per task."""
    priority: np.ndarray
    expected_ns: np.ndarray
    queue_basis_ns: np.ndarray
    wait_basis_ns: np.ndarray
    num_dependents: np.ndarray
    task_group_order: np.ndarray
    group_id: np.ndarray
    version_id: np.ndarray
    flags: np.ndarray
    dep_off: Optional[np.ndarray] = None
    dep_idx: Optional[np.ndarray] = None

    COLUMNS = (("priority", np.int32), ("expected_ns", np.int64), ("queue_basis_ns", np.int64),
               ("wait_basis_ns", np.int64), ("num_dependents", np.int32), ("task_group_order", np.int32),
               ("group_id", np.int32), ("version_id", np.int32), ("flags", np.uint32))

    @property
    def n_tasks(self) -> int:
        return int(self.priority.shape[0])

    @property
    def n_edges(self) -> int:
        return 0 if self.dep_idx is None else int(self.dep_idx.shape[0])

    def normalize(self) -> "TaskSoA":
        for name, dt in self.COLUMNS:
            setattr(self, name, np.ascontiguousarray(getattr(self, name), dtype=dt))
        if self.dep_idx is not None and self.dep_idx.shape[0] > 0:
            self.dep_off = np.ascontiguousarray(self.dep_off, dtype=np.int64)
            self.dep_idx = np.ascontiguousarray(self.dep_idx, dtype=np.int32)
        else:
            self.dep_off, self.dep_idx = None, None
        return self

    def struct(self) -> L.TaskSoAStruct:
        s = L.TaskSoAStruct()
        s.n_tasks, s.n_edges = self.n_tasks, self.n_edges
        for name, _ in self.COLUMNS:
            setattr(s, name, L.ptr(getattr(self, name)))
        s.dep_off, s.dep_idx = L.ptr(self.dep_off), L.ptr(self.dep_idx)
        return s

    def nbytes(self) -> int:
        n = sum(getattr(self, name).nbytes for name, _ in self.COLUMNS)
        if self.dep_idx is not None:
            n += self.dep_off.nbytes + self.dep_idx.nbytes
        return n


@dataclass
class DistroTable:
    """evg_distro_table."""
    task_off: np.ndarray
    group_off: np.ndarray
    cfg: np.ndarray              # L.DISTRO_CFG_DTYPE
    group_max_hosts: np.ndarray

    @property
    def n_distros(self) -> int:
        return int(self.cfg.shape[0])

    @property
    def n_groups(self) -> int:
        return int(self.group_off[-1]) if self.group_off.shape[0] else 0

    def normalize(self) -> "DistroTable":
        self.task_off = np.ascontiguousarray(self.task_off, dtype=np.int64)
        self.group_off = np.ascontiguousarray(self.group_off, dtype=np.int64)
        self.cfg = np.ascontiguousarray(self.cfg, dtype=L.DISTRO_CFG_DTYPE)
        self.group_max_hosts = np.ascontiguousarray(self.group_max_hosts, dtype=np.int32)
        return self

    def struct(self) -> L.DistroTableStruct:
        s = L.DistroTableStruct()
        s.n_distros = self.n_distros
        s.task_off, s.group_off = L.ptr(self.task_off), L.ptr(self.group_off)
        s.cfg = L.ptr(self.cfg) if self.n_distros else None
        s.group_max_hosts = L.ptr(self.group_max_hosts) if self.group_max_hosts.shape[0] else None
        return s

    def nbytes(self) -> int:
        return self.task_off.nbytes + self.group_off.nbytes + self.cfg.nbytes + self.group_max_hosts.nbytes


@dataclass
class HostSoA:
    """evg_host_soa + host_off + evg_alloc_cfg[]. 32 B per host."""
    flags: np.ndarray
    group_id: np.ndarray
    expected_ns: np.ndarray
    std_ns: np.ndarray
    start_ns: np.ndarray
    host_off: np.ndarray
    cfg: np.ndarray              # L.ALLOC_CFG_DTYPE

    COLUMNS = (("flags", np.uint32), ("group_id", np.int32), ("expected_ns", np.int64), ("std_ns", np.int64),
               ("start_ns", np.int64))

    @property
    def n_hosts(self) -> int:
        return int(self.flags.shape[0])

    def normalize(self) -> "HostSoA":
        for name, dt in self.COLUMNS:
            setattr(self, name, np.ascontiguousarray(getattr(self, name), dtype=dt))
        self.host_off = np.ascontiguousarray(self.host_off, dtype=np.int64)
        self.cfg = np.ascontiguousarray(self.cfg, dtype=L.ALLOC_CFG_DTYPE)
        return self

    def struct(self) -> L.HostSoAStruct:
        s = L.HostSoAStruct()
        s.n_hosts = self.n_hosts
        for name, _ in self.COLUMNS:
            setattr(s, name, L.ptr(getattr(self, name)) if self.n_hosts else None)
        return s

    def nbytes(self) -> int:
        return sum(getattr(self, name).nbytes for name, _ in self.COLUMNS) + self.host_off.nbytes + self.cfg.nbytes


@dataclass
class PlanOutput:
    order: np.ndarray          # int32 [T]
    total_value: np.ndarray    # int64 [T]
    info: np.ndarray           # QUEUE_INFO_DTYPE [D]
    group_info: np.ndarray     # GROUP_INFO_DTYPE [G]
    breakdown: Optional[np.ndarray] = None  # int64 [T, 13]

    def nbytes(self) -> int:
        n = self.order.nbytes + self.total_value.nbytes + self.info.nbytes + self.group_info.nbytes
        return n + (self.breakdown.nbytes if self.breakdown is not None else 0)


@dataclass
class AllocOutput:
    result: np.ndarray         # ALLOC_RESULT_DTYPE [D]
    status: np.ndarray         # int32 [D]

    def nbytes(self) -> int:
        return self.result.nbytes + self.status.nbytes


# ---------------------------------------------------------------------------
# marshalling reference-shaped structs -> SoA
# ---------------------------------------------------------------------------

def planner_cfg_row(d: M.Distro, includes_dependencies: bool, n_versions: int) -> tuple:
    ps = d.planner_settings
    return (ps.patch_factor, ps.patch_time_in_queue_factor, ps.commit_queue_factor,
            ps.mainline_time_in_queue_factor, ps.expected_runtime_factor, ps.generate_task_factor,
            ps.stepback_task_factor, float(ps.num_dependents_factor), d.get_target_time(),
            int(ps.should_group_versions()), int(includes_dependencies), n_versions, 0)


def requester_class(r: str) -> int:
    if M.is_github_merge_queue_requester(r):
        return L.EVG_TF_REQ_MERGE_QUEUE
    if M.is_patch_requester(r):
        return L.EVG_TF_REQ_PATCH
    return L.EVG_TF_REQ_OTHER


def satisfies_dependency(dep: M.Dependency, dep_task: M.Task) -> bool:
    """Task.SatisfiesDependency (model/task/task.go:529-543)."""
    if dep.status in (M.TASK_SUCCEEDED, ""):
        return dep_task.status == M.TASK_SUCCEEDED
    if dep.status == M.TASK_FAILED:
        return dep_task.status == M.TASK_FAILED
    if dep.status == M.ALL_STATUSES:
        return dep_task.status in (M.TASK_FAILED, M.TASK_SUCCEEDED) or dep_task.blocked()
    return False


def dependencies_met(t: M.Task, in_queue: Dict[str, M.Task], db: Optional[Dict[str, M.Task]],
                     now: Optional[int] = None) -> bool:
    """Task.DependenciesMet (model/task/task.go:632-671) against the in-queue
    cache first, then `db` (the tasks collection lookup); a missing dependency
    is the lookup error checkDependenciesMet turns into false (scheduler.go:161-168).
    With `now`, a fresh evaluation that comes out met stamps DependenciesMetTime on the task like the reference
    does (setDependenciesMetTime, task.go:653,673-684): the latest non-zero FinishedAt of its dependencies, else now."""
    if t.has_dependencies_met():
        return True
    for dep in t.depends_on:
        dep_task = in_queue.get(dep.task_id)
        if dep_task is None and db is not None:
            dep_task = db.get(dep.task_id)
        if dep_task is None:
            return False
        if not satisfies_dependency(next(x for x in t.depends_on if x.task_id == dep.task_id), dep_task):  # the first one naming it
            return False
    if now is not None:
        best = M.ZERO_TIME
        for dep in t.depends_on:
            if not M.is_zero_time(dep.finished_at) and dep.finished_at > best:
                best = dep.finished_at
        t.dependencies_met_time = now if M.is_zero_time(best) else best
    return True


@dataclass
class MarshalledDistro:
    """Key tables the shim keeps to translate results back to strings."""
    group_names: List[str] = field(default_factory=list)
    versions: List[str] = field(default_factory=list)


def marshal_tasks(batch: Sequence[tuple], now: int, dependency_db: Optional[Dict[str, M.Task]] = None,
                  duration_history: Optional[dict] = None, resolve_deps: bool = False):
    """[(Distro, [Task])] -> (TaskSoA, DistroTable, [MarshalledDistro]).

    Per task this resolves FetchExpectedDuration (PopulateCaches, setup_funcs.go:20-67).  Task.DependenciesMet
    (scheduler.go:161-168) is the DEVICE's job: the product path pairs these columns with marshal_deps() and
    Engine.upload_with_deps(), which sets the EVG_TF_DEPS_MET bit and the stamped wait basis on the GPU.
    resolve_deps=True evaluates it here instead (host restatement, kept for tests and for callers of the plain
    one-shot entry points that want self-contained columns)."""
    cols = {name: [] for name, _ in TaskSoA.COLUMNS}
    dep_off, dep_idx = [0], []
    task_off, group_off, cfg_rows, gmax, keys = [0], [0], [], [], []
    for d, tasks in batch:
        if len(tasks) > L.MAX_TASKS_PER_DISTRO:
            raise ValueError(f"distro {d.id!r}: {len(tasks)} tasks exceed {L.MAX_TASKS_PER_DISTRO}")
        incl = d.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES  # scheduler.go:28
        index = {t.id: i for i, t in enumerate(tasks)}
        by_id = {t.id: t for t in tasks}
        groups: Dict[str, int] = {}
        versions: Dict[str, int] = {}
        md = MarshalledDistro()
        for t in tasks:
            hist = None if duration_history is None else duration_history.get((t.project, t.build_variant, t.display_name))
            avg, _ = M.fetch_expected_duration(t, now, hist)
            gid = -1
            if t.task_group != "":
                name = t.get_task_group_string()
                gid = groups.get(name)
                if gid is None:
                    gid = groups[name] = len(groups)
                    md.group_names.append(name)
                    gmax.append(t.task_group_max_hosts)
                elif gmax[group_off[-1] + gid] != t.task_group_max_hosts:
                    # TaskGroupInfo.MaxHosts is the value of the group's first task in PLAN order (scheduler.go:87-90);
                    # a per-group table can only carry one value, so members must agree (they do: it is a project setting)
                    raise ValueError(f"task group {name!r}: TaskGroupMaxHosts differs between members "
                                     f"({gmax[group_off[-1] + gid]} vs {t.task_group_max_hosts} on {t.id!r})")
            vid = versions.get(t.version)
            if vid is None:
                vid = versions[t.version] = len(versions)
                md.versions.append(t.version)
            qb = t.activated_time if t.activated_time != M.ZERO_TIME else t.ingest_time  # planner.go:318-322
            # checkDependenciesMet runs first (scheduler.go:82-98) and, on a fresh evaluation, stamps DependenciesMetTime
            # on the task (task.go:653); the wait is measured after that (scheduler.go:119-123)
            deps_met = dependencies_met(t, by_id, dependency_db, now) if resolve_deps else False
            wb = max(t.scheduled_time, t.dependencies_met_time)  # ZERO_TIME sorts first
            fl = requester_class(t.requester)
            if t.generate_task:
                fl |= L.EVG_TF_GENERATE
            if t.activated_by == M.STEPBACK_TASK_ACTIVATOR:
                fl |= L.EVG_TF_STEPBACK
            if deps_met:
                fl |= L.EVG_TF_DEPS_MET
            if t.distro_id != d.id:
                fl |= L.EVG_TF_OTHER_DISTRO
            if not -2 ** 31 <= t.priority < 2 ** 31 or not -2 ** 31 <= t.num_dependents < 2 ** 31:
                # evg_task_soa carries both as int32; Go's Task.Priority is an int64 whose valid range ends at
                # evergreen.MaxTaskPriority (100, globals.go:185), so a value out here is a corrupt document
                raise ValueError(f"task {t.id!r}: priority {t.priority} / num_dependents {t.num_dependents} outside int32")
            cols["priority"].append(t.priority)
            cols["expected_ns"].append(avg)
            cols["queue_basis_ns"].append(qb)
            cols["wait_basis_ns"].append(wb)
            cols["num_dependents"].append(t.num_dependents)
            cols["task_group_order"].append(t.task_group_order)
            cols["group_id"].append(gid)
            cols["version_id"].append(vid)
            cols["flags"].append(fl)
            for dep in t.depends_on:  # only dependencies that are in this queue join units (planner.go:453)
                j = index.get(dep.task_id)
                if j is not None:
                    dep_idx.append(j)
            dep_off.append(len(dep_idx))
        task_off.append(task_off[-1] + len(tasks))
        group_off.append(group_off[-1] + len(groups))
        cfg_rows.append(planner_cfg_row(d, incl, len(versions)))
        keys.append(md)
    soa = TaskSoA(**{name: np.array(cols[name], dtype=dt) for name, dt in TaskSoA.COLUMNS},
                  dep_off=np.array(dep_off, dtype=np.int64), dep_idx=np.array(dep_idx, dtype=np.int32)).normalize()
    table = DistroTable(np.array(task_off, dtype=np.int64), np.array(group_off, dtype=np.int64),
                        np.array(cfg_rows, dtype=L.DISTRO_CFG_DTYPE), np.array(gmax, dtype=np.int32)).normalize()
    return soa, table, keys


def pack_strings(strings: Sequence[str]):
    """[str] -> (uint8 bytes, int64 offsets[n+1]): an evg_str_col."""
    enc = [x.encode() for x in strings]
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    if enc:
        np.cumsum([len(b) for b in enc], out=off[1:])
    return np.frombuffer(b"".join(enc), dtype=np.uint8).copy() if enc else np.zeros(0, np.uint8), off


def intern_columns(batch: Sequence[tuple], threads: int = 0):
    """evg_intern_columns over a tick: the string work of marshal_tasks (task-group keys and versions to dense ids in
    first-appearance order, dependency ids to queue indices) in the library's C++ instead of Python dicts.
    -> dict(group_id, version_id, group_off, n_versions, group_max_hosts, group_first, dep_off, dep_idx)."""
    lib = L.load()
    tasks = [t for _, ts in batch for t in ts]
    T, D = len(tasks), len(batch)
    task_off = np.zeros(D + 1, dtype=np.int64)
    if D:
        np.cumsum([len(ts) for _, ts in batch], out=task_off[1:])
    idb, ido = pack_strings([t.id for t in tasks])
    vb, vo = pack_strings([t.version for t in tasks])
    gb, go = pack_strings([t.get_task_group_string() if t.task_group != "" else "" for t in tasks])
    gmax = np.array([t.task_group_max_hosts for t in tasks], dtype=np.int32)
    dep_off = np.zeros(T + 1, dtype=np.int64)
    if T:
        np.cumsum([len(t.depends_on) for t in tasks], out=dep_off[1:])
    db, do = pack_strings([dep.task_id for t in tasks for dep in t.depends_on])
    E = int(dep_off[-1])
    out = dict(group_id=np.empty(T, np.int32), version_id=np.empty(T, np.int32), group_off=np.zeros(D + 1, np.int64),
               n_versions=np.zeros(D, np.int32), group_max_hosts=np.empty(max(T, 1), np.int32), group_first=np.empty(max(T, 1), np.int64),
               dep_off=np.zeros(T + 1, np.int64), dep_idx=np.empty(max(E, 1), np.int32))
    col = lambda b, o: L.StrColStruct(L.ptr(b) if b.shape[0] else None, L.ptr(o))  # noqa: E731
    ins = L.StringColsStruct(T, D, L.ptr(task_off), col(idb, ido), col(vb, vo), col(gb, go), L.ptr(gmax) if T else None,
                             L.ptr(dep_off), col(db, do))
    outs = L.InternOutStruct(*[L.ptr(out[k]) for k in ("group_id", "version_id", "group_off", "n_versions", "group_max_hosts",
                                                       "group_first", "dep_off", "dep_idx")])
    import ctypes as C
    L.check(lib.evg_intern_columns(C.byref(ins), C.byref(outs), int(threads)))
    G, En = int(out["group_off"][D]), int(out["dep_off"][T])
    out["group_max_hosts"], out["group_first"], out["dep_idx"] = out["group_max_hosts"][:G], out["group_first"][:G], out["dep_idx"][:En]
    return out


def provider_class(provider: str) -> int:
    if provider == M.PROVIDER_DOCKER:
        return L.EVG_PROVIDER_DOCKER
    if provider in M.PROVIDER_SPAWNABLE:
        return L.EVG_PROVIDER_EPHEMERAL
    return L.EVG_PROVIDER_STATIC


def alloc_cfg_row(data: M.HostAllocatorData) -> tuple:
    d = data.distro
    hs = d.host_allocator_settings
    pool = data.container_pool
    return (float(hs.future_host_fraction), provider_class(d.provider), int(d.disabled), hs.minimum_hosts,
            hs.maximum_hosts, int(hs.rounding_rule == M.HOST_ALLOCATOR_ROUND_UP),
            int(hs.feedback_rule == M.HOST_ALLOCATOR_WAITS_OVER_THRESH_FEEDBACK),
            int(pool is not None), pool.max_containers if pool else 0,
            int(data.parent_distro_maximum_hosts is not None),
            data.parent_distro_maximum_hosts if data.parent_distro_maximum_hosts is not None else 0)


def marshal_hosts(datas: Sequence[M.HostAllocatorData], group_names: Sequence[Sequence[str]]) -> HostSoA:
    """[HostAllocatorData] -> HostSoA.  `group_names[d]` is the distro's group
    table (slot order of its TaskGroupInfos); hosts are bucketed like
    groupByTaskGroup (utilization_based_host_allocator.go:223-260)."""
    fl, gid, exp, std, start, off, rows = [], [], [], [], [], [0], []
    for data, names in zip(datas, group_names):
        lookup = {n: i for i, n in enumerate(names)}
        for h in data.existing_hosts:
            f = 0
            g = L.EVG_HG_NONE
            e = s = 0
            st = M.ZERO_TIME
            if h.running_task != "":
                f |= L.EVG_HF_RUNNING
                rt = data.running_tasks.get(h.running_task)
                if rt is not None and rt.found:
                    f |= L.EVG_HF_RT_FOUND
                    e, s, st = rt.expected, rt.std_dev, rt.start_time
                if h.running_task_group != "":
                    g = lookup.get(h.get_task_group_string(), L.EVG_HG_UNQUEUED)
            if h.task_group_teardown_start_time != M.ZERO_TIME:
                f |= L.EVG_HF_TEARDOWN
            fl.append(f); gid.append(g); exp.append(e); std.append(s); start.append(st)
        off.append(len(fl))
        rows.append(alloc_cfg_row(data))
    return HostSoA(np.array(fl, dtype=np.uint32), np.array(gid, dtype=np.int32), np.array(exp, dtype=np.int64),
                   np.array(std, dtype=np.int64), np.array(start, dtype=np.int64), np.array(off, dtype=np.int64),
                   np.array(rows, dtype=L.ALLOC_CFG_DTYPE)).normalize()


def queue_info_rows(infos: Sequence[M.DistroQueueInfo]):
    """[DistroQueueInfo] -> (QUEUE_INFO rows, GROUP_INFO rows, group_off, names per distro).
    Later duplicates of a name win, like the map built at allocator.go:243-246."""
    qrows = np.zeros(len(infos), dtype=L.QUEUE_INFO_DTYPE)
    grows, goff, names_all = [], [0], []
    for i, qi in enumerate(infos):
        q = qrows[i]
        q["length"] = qi.length
        q["length_with_dependencies_met"] = qi.length_with_dependencies_met
        q["count_dep_filled_merge_queue_tasks"] = qi.count_dep_filled_merge_queue_tasks
        q["expected_duration"] = qi.expected_duration
        q["max_duration_threshold"] = qi.max_duration_threshold
        q["count_duration_over_threshold"] = qi.count_duration_over_threshold
        q["duration_over_threshold"] = qi.duration_over_threshold
        q["count_wait_over_threshold"] = qi.count_wait_over_threshold
        q["secondary_queue"] = int(qi.secondary_queue)
        by_name = {}
        for g in qi.task_group_infos:
            by_name[g.name] = g
        names = []
        for name, g in by_name.items():
            row = tuple(getattr(g, f) for f in L.GROUP_INFO_FIELDS)
            if name == "":
                q["has_ungrouped"] = 1
                q["ungrouped"] = row
            else:
                names.append(name)
                grows.append(row)
        goff.append(len(grows))
        names_all.append(names)
    return qrows, np.array(grows, dtype=L.GROUP_INFO_DTYPE).reshape(-1), np.array(goff, dtype=np.int64), names_all


# ---------------------------------------------------------------------------
# dependency filter tables (evg_deps_in)
# ---------------------------------------------------------------------------

def _task_state(t: M.Task) -> int:
    st = 0 if t.status == M.TASK_SUCCEEDED else 1 if t.status == M.TASK_FAILED else 2
    return st | (L.EVG_TS_BLOCKED if t.blocked() else 0)


def _want(status: str) -> int:
    if status in (M.TASK_SUCCEEDED, ""):
        return L.EVG_WANT_SUCCESS
    if status == M.TASK_FAILED:
        return L.EVG_WANT_FAILED
    if status == M.ALL_STATUSES:
        return L.EVG_WANT_ANY
    return L.EVG_WANT_OTHER


@dataclass
class DepsTable:
    """evg_deps_in: every direct dependency of every task of the tick (all distros concatenated)."""
    dep_off: np.ndarray
    dep_kind: np.ndarray
    dep_ref: np.ndarray
    dep_want: np.ndarray
    task_state: np.ndarray
    task_pre: np.ndarray
    ext_state: np.ndarray

    @property
    def n_tasks(self) -> int:
        return int(self.task_state.shape[0])

    def struct(self) -> L.DepsInStruct:
        s = L.DepsInStruct()
        s.n_tasks, s.n_deps, s.n_ext = self.n_tasks, int(self.dep_ref.shape[0]), int(self.ext_state.shape[0])
        s.dep_off = L.ptr(self.dep_off)
        for f in ("dep_kind", "dep_ref", "dep_want"):
            setattr(s, f, L.ptr(getattr(self, f)) if s.n_deps else None)
        s.task_state, s.task_pre = L.ptr(self.task_state), L.ptr(self.task_pre)
        s.ext_state = L.ptr(self.ext_state) if s.n_ext else None
        return s


def marshal_dep_finished(batch: Sequence[tuple]) -> np.ndarray:
    """Dependency.FinishedAt of every dependency, in marshal_deps' order (what setDependenciesMetTime reads)."""
    return np.array([d.finished_at for _, tasks in batch for t in tasks for d in t.depends_on], dtype=np.int64)


def marshal_deps(batch: Sequence[tuple], dependency_db: Optional[Dict[str, M.Task]] = None) -> DepsTable:
    """[(Distro, [Task])] -> DepsTable.  A dependency resolves against the distro's own queue first (the
    depCache of scheduler.go:61-64), then against `dependency_db` (the tasks collection), else it is MISSING."""
    dep_off, kind, ref, want, tstate, pre, ext_state = [0], [], [], [], [], [], []
    ext_index: Dict[str, int] = {}
    db = dependency_db or {}
    base = 0
    for _, tasks in batch:
        index = {t.id: i for i, t in enumerate(tasks)}
        for t in tasks:
            tstate.append(_task_state(t))
            pre.append((L.EVG_TP_OVERRIDE if t.override_dependencies else 0) |
                       (0 if M.is_zero_time(t.dependencies_met_time) else L.EVG_TP_MET_TIME))
            first: Dict[str, str] = {}
            for d in t.depends_on:
                # SatisfiesDependency judges a dependency task by the FIRST Dependency naming it (task.go:529-543)
                want.append(_want(first.setdefault(d.task_id, d.status)))
                j = index.get(d.task_id)
                if j is not None:
                    kind.append(L.EVG_DEP_IN_QUEUE); ref.append(base + j)
                elif d.task_id in db:
                    k = ext_index.get(d.task_id)
                    if k is None:
                        k = ext_index[d.task_id] = len(ext_state)
                        ext_state.append(_task_state(db[d.task_id]))
                    kind.append(L.EVG_DEP_EXTERNAL); ref.append(k)
                else:
                    kind.append(L.EVG_DEP_MISSING); ref.append(0)
            dep_off.append(len(ref))
        base += len(tasks)
    return DepsTable(np.array(dep_off, np.int64), np.array(kind, np.uint8), np.array(ref, np.int32),
                     np.array(want, np.uint8), np.array(tstate, np.uint8), np.array(pre, np.uint8),
                     np.array(ext_state, np.uint8))


@dataclass
class RunnableTable:
    """evg_runnable_in: every candidate task of every distro, plus the project-ref cache and the per-distro rules."""
    task_off: np.ndarray
    sched: np.ndarray
    project: np.ndarray
    project_flags: np.ndarray
    valid_off: np.ndarray
    valid_idx: np.ndarray
    finder: np.ndarray
    deps: Optional[DepsTable]

    @property
    def n_tasks(self) -> int:
        return int(self.sched.shape[0])

    @property
    def n_distros(self) -> int:
        return int(self.finder.shape[0])

    def struct(self):
        """-> (RunnableInStruct, keepalive): the nested evg_deps_in must outlive the call."""
        s = L.RunnableInStruct()
        s.n_tasks, s.n_distros, s.n_projects = self.n_tasks, self.n_distros, int(self.project_flags.shape[0])
        s.task_off, s.valid_off, s.finder = L.ptr(self.task_off), L.ptr(self.valid_off), L.ptr(self.finder)
        s.sched = L.ptr(self.sched) if s.n_tasks else None
        s.project = L.ptr(self.project) if s.n_tasks else None
        s.project_flags = L.ptr(self.project_flags) if s.n_projects else None
        s.valid_idx = L.ptr(self.valid_idx) if self.valid_idx.shape[0] else None
        keep = None
        if self.deps is not None:
            keep = self.deps.struct()
            s.deps = C.pointer(keep)
        return s, keep


def sched_bits(t: M.Task) -> int:
    """The EVG_SQ_* byte of one task: the fields of schedulableHostTasksQuery (model/task/db.go:671-689) and the
    requester classes ProjectCanDispatchTask looks at."""
    b = 0
    if t.activated:
        b |= L.EVG_SQ_ACTIVATED
    if t.status == M.TASK_UNDISPATCHED:
        b |= L.EVG_SQ_UNDISPATCHED
    if t.priority > M.DISABLED_TASK_PRIORITY:
        b |= L.EVG_SQ_PRIORITY_OK
    if t.execution_platform in ("", "host"):
        b |= L.EVG_SQ_HOST_PLATFORM
    if t.unattainable_dependency:
        b |= L.EVG_SQ_UNATTAINABLE
    if t.override_dependencies:
        b |= L.EVG_SQ_OVERRIDE_DEPS
    if t.requester == M.GITHUB_PR_REQUESTER:
        b |= L.EVG_SQ_GITHUB_PR
    if M.is_patch_requester(t.requester):
        b |= L.EVG_SQ_PATCH_REQUEST
    return b


def project_bits(p: M.ProjectRef) -> int:
    return ((L.EVG_PF_ENABLED if p.enabled else 0) | (L.EVG_PF_HIDDEN if p.hidden else 0) |
            (L.EVG_PF_DISPATCHING_DISABLED if p.dispatching_disabled else 0) |
            (L.EVG_PF_PATCHING_DISABLED if p.patching_disabled else 0))


def marshal_runnable(batch: Sequence[tuple], project_refs: Sequence[M.ProjectRef], finder: str = "legacy",
                     dependency_db: Optional[Dict[str, M.Task]] = None) -> RunnableTable:
    """[(Distro, [candidate Task])] + the project-ref cache (getProjectRefCache, task_finder.go:46) -> RunnableTable.
    `finder`: "legacy" (LegacyFindRunnableTasks) or "alternate" (AlternateTaskFinder / ParallelTaskFinder)."""
    prow = {p.id: i for i, p in enumerate(project_refs)}
    flavour = {"legacy": L.EVG_FINDER_LEGACY, "alternate": L.EVG_FINDER_ALTERNATE, "parallel": L.EVG_FINDER_ALTERNATE}[finder]
    task_off, valid_off, valid_idx, fnd, sched, proj = [0], [0], [], [], [], []
    for d, tasks in batch:
        for t in tasks:
            sched.append(sched_bits(t))
            proj.append(prow.get(t.project, -1))
        task_off.append(len(sched))
        valid_idx.extend(prow.get(name, -1) for name in d.valid_projects)
        valid_off.append(len(valid_idx))
        fnd.append(L.EVG_FINDER_NO_DEPS
                   if d.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES else flavour)
    deps = marshal_deps(batch, dependency_db) if any(f != L.EVG_FINDER_NO_DEPS for f in fnd) else None
    return RunnableTable(np.array(task_off, np.int64), np.array(sched, np.uint8), np.array(proj, np.int32),
                         np.array([project_bits(p) for p in project_refs], np.uint8), np.array(valid_off, np.int64),
                         np.array(valid_idx, np.int32), np.array(fnd, np.uint8), deps)


@dataclass
class DurationRows:
    """evg_duration_rows: finished tasks, the interned group-by key of each, and the aggregation window."""
    key: np.ndarray
    time_taken_ns: np.ndarray
    start_ns: np.ndarray
    finish_ns: np.ndarray
    flags: np.ndarray
    n_keys: int
    window_start_ns: int
    window_end_ns: int

    @property
    def n_rows(self) -> int:
        return int(self.key.shape[0])

    def struct(self) -> L.DurationRowsStruct:
        s = L.DurationRowsStruct()
        s.n_rows, s.n_keys, s._reserved = self.n_rows, int(self.n_keys), 0
        for f in ("key", "time_taken_ns", "start_ns", "finish_ns", "flags"):
            setattr(s, f, L.ptr(getattr(self, f)) if s.n_rows else None)
        s.window_start_ns, s.window_end_ns = int(self.window_start_ns), int(self.window_end_ns)
        return s


def marshal_durations(tasks: Sequence[M.Task], window_start: int, window_end: int):
    """Finished tasks -> (DurationRows, keys): keys[i] = (project, build_variant, display_name) of key row i, in
    first-appearance order.  The $match of expected_duration.go:37-55 is evaluated on the device from the flags
    and the two timestamps; here a row only says what the task document says."""
    index: Dict[tuple, int] = {}
    key, taken, start, finish, flags = [], [], [], [], []
    for t in tasks:
        k = (t.project, t.build_variant, t.display_name)
        key.append(index.setdefault(k, len(index)))
        taken.append(t.time_taken); start.append(t.start_time); finish.append(t.finish_time)
        flags.append((L.EVG_DR_COMPLETED if t.status in M.TASK_COMPLETED_STATUSES else 0) |
                     (L.EVG_DR_TIMED_OUT if t.timed_out else 0))
    rows = DurationRows(np.array(key, np.int32), np.array(taken, np.int64), np.array(start, np.int64),
                        np.array(finish, np.int64), np.array(flags, np.uint8), len(index), window_start, window_end)
    return rows, list(index)


# ---------------------------------------------------------------------------------------------------------------
# legacy comparator prioritiser (scheduler/task_prioritizer.go, task_priority_cmp.go, setup_funcs.go:72-87)
@dataclass
class LegacyTable:
    """evg_legacy_soa + task_off + list_mode for a batch of distros."""
    priority: np.ndarray
    ingest_ns: np.ndarray
    expected_ns: np.ndarray
    num_dependents: np.ndarray
    revision_order: np.ndarray
    project_id: np.ndarray
    tg_rank: np.ndarray
    tg_pair_id: np.ndarray
    task_group_order: np.ndarray
    presort_rank: np.ndarray
    flags: np.ndarray
    task_off: np.ndarray
    list_mode: np.ndarray  # uint8 [3 * n_distros]: high priority, patch, repotracker

    COLUMNS = (("priority", np.int64), ("ingest_ns", np.int64), ("expected_ns", np.int64), ("num_dependents", np.int32),
               ("revision_order", np.int32), ("project_id", np.int32), ("tg_rank", np.int32), ("tg_pair_id", np.int32),
               ("task_group_order", np.int32), ("presort_rank", np.int32), ("flags", np.uint32))

    @property
    def n_tasks(self) -> int:
        return int(self.priority.shape[0])

    @property
    def n_distros(self) -> int:
        return int(self.task_off.shape[0]) - 1

    def struct(self) -> "L.LegacySoAStruct":
        s = L.LegacySoAStruct()
        s.n_tasks = self.n_tasks
        for name, _ in self.COLUMNS:
            setattr(s, name, L.ptr(getattr(self, name)))
        return s


def legacy_list_of(t: M.Task) -> int:
    """splitTasksByRequester (task_prioritizer.go:214-247): 0 high priority, 1 patch, 2 repotracker, 3 dropped."""
    if t.priority > M.MAX_TASK_PRIORITY:
        return 0
    if t.requester in M.SYSTEM_VERSION_REQUESTER_TYPES:
        return 2
    if M.is_patch_requester(t.requester):
        return 1
    return 3


def legacy_list_mode(tasks: Sequence[M.Task], expected: Sequence[int]) -> int:
    """Is the comparator chain a strict weak order on this list, and which byAge branch does it take
    (task_priority_cmp.go:73-95)?  Only tasks outside task groups reach byAge / byRuntime."""
    plain = [(t, e) for t, e in zip(tasks, expected) if t.task_group == ""]
    if any(e == 0 for _, e in plain) and any(e != 0 for _, e in plain):
        return L.EVG_LEGACY_MODE_LITERAL  # byRuntime ties a zero duration with everything (:109-111)
    commit = [t for t, _ in plain if t.requester in M.SYSTEM_VERSION_REQUESTER_TYPES]
    projects = [t.project for t in commit]
    if len(set(projects)) == len(projects):
        return L.EVG_LEGACY_MODE_INGEST      # no pair takes the revision-order branch
    if len(commit) == len(plain) and len(set(projects)) == 1:
        return L.EVG_LEGACY_MODE_REVISION    # every pair takes it
    return L.EVG_LEGACY_MODE_LITERAL


def marshal_legacy(batch: Sequence[tuple], now: Optional[int] = None) -> LegacyTable:
    """batch: (distro_id, tasks, versions) per distro; `versions` maps a version id to its Requester (what byCommitQueue
    reads of model.Version).  Resolves FetchExpectedDuration, interns the strings, decides each list's mode."""
    cols = {name: [] for name, _ in LegacyTable.COLUMNS}
    task_off, modes = [0], []
    for _, tasks, versions in batch:
        versions = versions or {}
        expected = [M.fetch_expected_duration(t, now)[0] if now is not None else t.expected_duration for t in tasks]
        fmt = [f"{t.build_id}-{t.task_group}" for t in tasks]
        grouped = sorted({f for f, t in zip(fmt, tasks) if t.task_group != ""})
        rank = {f: k for k, f in enumerate(grouped)}
        pairs: Dict[tuple, int] = {}
        by_fmt: Dict[str, set] = {}
        for f, t in zip(fmt, tasks):
            if t.task_group != "":
                pairs.setdefault((t.task_group, t.build_id), len(pairs))
                by_fmt.setdefault(f, set()).add((t.task_group, t.build_id))
        collision = any(len(v) > 1 for v in by_fmt.values())
        keys = sorted(range(len(tasks)), key=lambda k: f"{fmt[k]}-{tasks[k].id}", reverse=True)
        presort = [0] * len(tasks)
        for pos, k in enumerate(keys):
            presort[k] = pos
        projects: Dict[str, int] = {}
        lists = [legacy_list_of(t) for t in tasks]
        for k, t in enumerate(tasks):
            if not -(2 ** 63) <= t.priority < 2 ** 63:
                raise ValueError(f"task {t.id!r}: priority {t.priority} is outside int64")
            rq = (L.EVG_LF_REQ_SYSTEM if t.requester in M.SYSTEM_VERSION_REQUESTER_TYPES else
                  L.EVG_LF_REQ_PATCH if M.is_patch_requester(t.requester) else L.EVG_LF_REQ_OTHER)
            fl = rq | (L.EVG_LF_GENERATE if t.generate_task else 0)
            if versions.get(t.version, "") == M.GITHUB_MERGE_REQUESTER:
                fl |= L.EVG_LF_MERGE_QUEUE_VERSION
            cols["priority"].append(t.priority); cols["ingest_ns"].append(t.ingest_time); cols["expected_ns"].append(expected[k])
            cols["num_dependents"].append(t.num_dependents); cols["revision_order"].append(t.revision_order_number)
            cols["project_id"].append(projects.setdefault(t.project, len(projects)))
            cols["tg_rank"].append(rank[fmt[k]] if t.task_group != "" else -1)
            cols["tg_pair_id"].append(pairs[(t.task_group, t.build_id)] if t.task_group != "" else -1)
            cols["task_group_order"].append(t.task_group_order); cols["presort_rank"].append(presort[k]); cols["flags"].append(fl)
        for lst in (0, 1, 2):
            sel = [k for k in range(len(tasks)) if lists[k] == lst]
            m = legacy_list_mode([tasks[k] for k in sel], [expected[k] for k in sel])
            modes.append(L.EVG_LEGACY_MODE_LITERAL if collision else m)
        task_off.append(task_off[-1] + len(tasks))
    return LegacyTable(**{name: np.array(cols[name], dtype=dt) for name, dt in LegacyTable.COLUMNS},
                       task_off=np.array(task_off, dtype=np.int64), list_mode=np.array(modes, dtype=np.uint8))

"""What a caller receives after the host allocator, against the CPU oracle: the finder -> planner -> allocator hand-over
of evg_plan_from_finder, the persisted TaskQueueItem rows of evg_download_queue (against oracle/oracle_persist.py), and
evg_dag_rebuild_batch at the edges of its C-ABI (against oracle/oracle_dag.py)."""
import copy
import random
from collections import Counter

import numpy as np
import pytest

from evergreen_b200 import _lib as L
from evergreen_b200 import model as M
from evergreen_b200 import scheduler as S
from evergreen_b200 import soa, synth
from oracle import oracle as O
from oracle import oracle_dag as OD
from oracle import oracle_persist as OP
from test_gpu_parity import random_finder_batch
from test_host_logic import random_tasks

pytestmark = pytest.mark.gpu

NOW = synth.NOW_NS
QINFO_FIELDS = ("length", "length_with_dependencies_met", "count_dep_filled_merge_queue_tasks", "expected_duration",
                "max_duration_threshold", "count_duration_over_threshold", "duration_over_threshold",
                "count_wait_over_threshold")


def _group_rows(infos):
    """TaskGroupInfos as a multiset: the reference builds the list from a map (scheduler.go:139-142)."""
    return Counter(tuple([g.name] + [getattr(g, f) for f in L.GROUP_INFO_FIELDS]) for g in infos)


# ---------------------------------------------------------------- A. finder -> planner -> allocator
def _clean(prefix, n, rng, project="p1", group=None):
    """n tasks every finder keeps (activated, undispatched, a dispatchable project, no dependencies)."""
    out = []
    for i in range(n):
        t = M.Task(id=f"{prefix}{i}", project=project, version=f"v{i % 3}", build_variant="bv", activated=True,
                   status="undispatched", requester=rng.choice([M.PATCH_VERSION_REQUESTER, M.REPOTRACKER_VERSION_REQUESTER]),
                   priority=rng.randrange(4), num_dependents=rng.randrange(3), expected_duration=rng.randrange(1, 90) * M.MINUTE,
                   activated_time=NOW - rng.randrange(10 ** 13), scheduled_time=NOW - rng.randrange(10 ** 12))
        if group is not None and rng.random() < 0.3:
            t.task_group, t.task_group_order, t.task_group_max_hosts = f"{group}{i % 4}", i % 5, 1 + i % 4 % 3
            t.version = "v0"
        out.append(t)
    return out


def _hosts_for(d, tasks, rng, n):
    """Free hosts, hosts running ungrouped tasks, hosts running tasks of the distro's task groups (kept or dropped)."""
    groups = sorted({(t.task_group, t.build_variant, t.project, t.version) for t in tasks if t.task_group})
    hosts, running = [], {}
    for k in range(n):
        h = M.Host(id=f"{d.id}-h{k}")
        r = rng.random()
        if r < 0.6 or not tasks:
            if r < 0.3:
                h.running_task = f"{d.id}-run{k}"
                running[h.running_task] = M.RunningTaskStats(found=rng.random() < 0.9, expected=rng.randrange(1, 60) * M.MINUTE,
                                                             std_dev=rng.randrange(0, 5) * M.MINUTE, start_time=NOW - rng.randrange(40) * M.MINUTE)
        elif groups:
            g = groups[k % len(groups)]
            h.running_task = f"{d.id}-run{k}"
            h.running_task_group, h.running_task_build_variant, h.running_task_project, h.running_task_version = g
            running[h.running_task] = M.RunningTaskStats(found=True, expected=rng.randrange(1, 60) * M.MINUTE, std_dev=0,
                                                         start_time=NOW - rng.randrange(40) * M.MINUTE)
        hosts.append(h)
    d.provider = M.PROVIDER_EC2_FLEET
    d.host_allocator_settings = M.HostAllocatorSettings(maximum_hosts=200, future_host_fraction=0.5, minimum_hosts=rng.randrange(3))
    return M.HostAllocatorData(distro=d, existing_hosts=hosts, distro_queue_info=M.DistroQueueInfo(), running_tasks=running)


def _handover_batch(seed, includes_dependencies, group_versions):
    rng = random.Random(seed)
    batch, refs, db = random_finder_batch(rng, 5)
    # every route of the planner by kept count: warp (<= 32), the k_plan_cta classes (384 / 1280 / 5120 / 10240),
    # the general path (> 10240)
    for n in (32, 33, 384, 385, 1280, 1281, 5120, 5121, 10240):
        tasks = _clean(f"r{n}-", n, rng, group="rg")
        tasks += [M.Task(id=f"r{n}-off{k}", project="p1", activated=False) for k in range(7)]  # dropped: the compaction moves rows
        rng.shuffle(tasks)
        batch.append((M.Distro(id=f"route{n}"), tasks))
    big, db2 = random_tasks(rng, 16000)
    for k, t in enumerate(big):
        t.id = "big-" + t.id
        t.project = "p1"
        t.depends_on = [dep for dep in t.depends_on if k % 5 == 0]
        for dep in t.depends_on:
            if dep.task_id.startswith("t"):
                dep.task_id = "big-" + dep.task_id
    batch.append((M.Distro(id="big"), big)); db.update(db2)
    # task groups whose every member the finder drops, next to groups that keep some
    tg = _clean("grp-", 300, rng, group="tg")
    for t in tg:
        if t.task_group in ("tg0", "tg2"):
            t.activated = False
    batch.append((M.Distro(id="dropped-groups"), tg))
    # kept members that all wait on dependencies: under IncludesDependencies a legitimate Count 0 group
    wait = _clean("wait-", 60, rng)
    for k, t in enumerate(wait):
        t.task_group, t.task_group_order, t.task_group_max_hosts = ("wg", k, 2) if k % 2 else ("", 0, 0)
        t.version = "v0"
        if k % 2:
            t.depends_on = [M.Dependency(f"wait-{k - 1}")]  # an undispatched task of the queue: never met
    batch.append((M.Distro(id="waiting-group"), wait))
    # many candidate groups, few survivors: the phantom slots would route the distro past the 64-thread k_plan_cta
    many = _clean("many-", 900, rng)
    for k, t in enumerate(many):
        t.task_group, t.task_group_order, t.task_group_max_hosts, t.version = f"mg{k // 2}", k % 2, 1 + (k // 2) % 3, "v0"
        t.activated = k % 40 < 2
    batch.append((M.Distro(id="many-groups"), many))
    alldrop = _clean("none-", 30, rng, group="ng")
    for t in alldrop:
        t.activated = False
    batch.append((M.Distro(id="all-dropped"), alldrop))
    batch.append((M.Distro(id="empty"), []))
    for d, _ in batch:
        if includes_dependencies:
            d.dispatcher_settings.version = M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
        elif d.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES:
            d.dispatcher_settings.version = ""
        d.planner_settings.group_versions = group_versions
        d.planner_settings.target_time = rng.choice([0, 20 * M.MINUTE, 2 * M.HOUR])
    db.update({t.id: t for _, ts in batch for t in ts})  # a dropped candidate is still a task document
    datas = [_hosts_for(d, ts, rng, 40 if d.id == "dropped-groups" else rng.choice([0, 3, 40, 90])) for d, ts in batch]
    return batch, refs, db, datas


def oracle_handover(d, candidates, refs, db, finder, data):
    """The reference's path for one distro: finder -> PrepareTasksForPlanning -> GetDistroQueueInfo -> the allocator."""
    kept = O.find_runnable(d, candidates, refs, db, finder)
    order, bd, _ = O.plan(d, kept, NOW)
    incl = d.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
    info = O.queue_info(d.id, kept, d.get_target_time(), incl, NOW, db, order=order)
    data = copy.copy(data)
    data.distro_queue_info = info
    new, free, status = O.allocate(data, NOW)
    return kept, order, bd[:, L.EVG_BD_TOTAL_VALUE], info, (new, free, status)


def _kept_group_names(keys, soa_, task_off, runnable, count):
    """Group slot k of distro d = the k-th candidate group of d, in id order, that kept a task (include/evg_sched.h)."""
    out = []
    for d in range(len(keys)):
        a = int(task_off[d])
        gids = sorted({int(g) for g in soa_.group_id[a + runnable[a:a + int(count[d])]] if g >= 0})
        out.append([keys[d].group_names[g] for g in gids])
    return out


@pytest.mark.parametrize("group_versions", [False, True], ids=["units", "group_versions"])
@pytest.mark.parametrize("includes_dependencies", [False, True], ids=["finder_deps", "includes_deps"])
@pytest.mark.parametrize("finder", ["legacy", "alternate"])
def test_finder_handover_matches_the_oracle(engine, finder, includes_dependencies, group_versions):
    """evg_plan_from_finder with hosts, then evg_run_resident + evg_download: per distro the kept ids in rank order,
    TotalValue, every DistroQueueInfo scalar, the whole TaskGroupInfo list (no group the finder emptied, Count 0 groups
    of waiting members kept), the allocator's (new, free, status) and CountFree / CountRequired -- all equal to the
    oracle's finder -> planner -> GetDistroQueueInfo -> allocator."""
    seed = 900 + 4 * (finder == "alternate") + 2 * includes_dependencies + group_versions
    batch, refs, db, datas = _handover_batch(seed, includes_dependencies, group_versions)
    dev = copy.deepcopy(batch)
    table = soa.marshal_runnable(dev, refs, finder, db)
    if table.deps is None:
        table.deps = soa.marshal_deps(dev, db)
    soa_, dtable, keys = soa.marshal_tasks(dev, NOW, db)
    hosts = soa.marshal_hosts(datas, [k.group_names for k in keys])
    runnable, count = engine.plan_from_finder(table, soa_, dtable, hosts, soa.marshal_dep_finished(dev), NOW)
    runnable, count = runnable.copy(), count.copy()
    engine.run(NOW)
    po, ao = copy.deepcopy(engine.download())
    names = _kept_group_names(keys, soa_, table.task_off, runnable, count)
    infos = {}
    a_new = g_new = 0
    for d, ((dist, cands), data) in enumerate(zip(batch, datas)):
        kept, order, tv, info, alloc = oracle_handover(dist, copy.deepcopy(cands), refs, db, finder, data)
        a, n = int(table.task_off[d]), int(count[d])
        assert n == len(kept), dist.id
        dkept = [dev[d][1][int(j)] for j in runnable[a:a + n]]
        assert [dkept[int(i)].id for i in po.order[a_new:a_new + n]] == [kept[int(i)].id for i in order], dist.id
        assert po.total_value[a_new:a_new + n].tolist() == tv.tolist(), dist.id
        ng = len(names[d])
        got = S._queue_info_from_rows(po.info[d], po.group_info[g_new:g_new + ng], names[d])
        for f in QINFO_FIELDS:
            assert getattr(got, f) == getattr(info, f), (dist.id, f)
        assert _group_rows(got.task_group_infos) == _group_rows(info.task_group_infos), dist.id
        assert (int(ao.result[d]["new_hosts"]), int(ao.result[d]["free_hosts"]), int(ao.status[d])) == alloc, dist.id
        infos[dist.id] = got
        a_new += n
        g_new += ng
    assert {32, 33, 384, 385, 1280, 1281, 5120, 5121, 10240} <= set(count.tolist()) and int(count.max()) > 10240
    by = {dist.id: d for d, (dist, _) in enumerate(batch)}
    dropped = {t.get_task_group_string() for t in batch[by["dropped-groups"]][1] if t.task_group in ("tg0", "tg2")}
    assert dropped and not dropped & set(names[by["dropped-groups"]])
    assert any(h.running_task_group in ("tg0", "tg2") for h in datas[by["dropped-groups"]].existing_hosts)
    assert len(names[by["many-groups"]]) < 60 < len(keys[by["many-groups"]].group_names)
    assert int(count[by["all-dropped"]]) == 0 and names[by["all-dropped"]] == [] and int(count[by["empty"]]) == 0
    if includes_dependencies:  # the waiting members are kept, counted nowhere
        assert [g.count for g in infos["waiting-group"].task_group_infos if g.name.startswith("wg_")] == [0]
    # the persisted rows of the compacted tick: indices into the kept queue, GroupMaxHosts through the kept group slots
    item_off, items = engine.download_queue(0, np.cumsum([0] + count.tolist()))
    for d, (dist, cands) in enumerate(batch):
        a, n = int(table.task_off[d]), int(count[d])
        okept = O.find_runnable(dist, copy.deepcopy(cands), refs, db, finder)
        order, bd, _ = O.plan(dist, okept, NOW)
        planned = [okept[int(i)] for i in order]
        incl = dist.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
        want = OP.saved_queue(OP.task_queue_items(OP.stamp_planned_tasks(planned, incl, NOW, db)))
        rows = items[int(item_off[d]):int(item_off[d + 1])]
        dkept = [dev[d][1][int(j)] for j in runnable[a:a + n]]
        assert [dkept[int(r)].id for r in rows["task"]] == [w.id for w in want], dist.id
        assert rows["group_max_hosts"].tolist() == [w.group_max_hosts if w.group else 0 for w in want], dist.id
        assert ((rows["flags"] & L.EVG_QI_DEPS_MET) != 0).tolist() == [w.dependencies_met for w in want], dist.id


# ---------------------------------------------------------------- B. the persisted queue against the restatement
def _persist_tasks(rng, n, tag, distro_id):
    out = []
    for k in range(n):
        t = M.Task(id=f"{tag}{k}", display_name=f"dn{k % 17}", build_variant=f"bv{k % 2}", project="p", version=f"v{k % 3}",
                   requester=rng.choice([M.PATCH_VERSION_REQUESTER, M.REPOTRACKER_VERSION_REQUESTER, M.GITHUB_MERGE_REQUESTER]),
                   revision=f"r{k % 5}", revision_order_number=k % 11, priority=rng.randrange(5), num_dependents=rng.randrange(3),
                   activated_time=NOW - rng.randrange(10 ** 13), distro_id=distro_id, activated_by=rng.choice(["", "user", "stepback"]),
                   expected_duration=rng.choice([0, rng.randrange(1, 60) * M.MINUTE]),
                   scheduled_time=rng.choice([M.ZERO_TIME, NOW - rng.randrange(10 ** 12)]),
                   dependencies_met_time=rng.choice([M.ZERO_TIME, M.ZERO_TIME, NOW - rng.randrange(10 ** 12)]),
                   override_dependencies=rng.random() < 0.05)
        if rng.random() < 0.2:
            g = rng.randrange(3)
            t.task_group, t.task_group_order = f"tg{g}", rng.randrange(-2, 6)
            t.task_group_max_hosts = 1 + (g + k % 2 + k % 3) % 4  # uniform per (group, variant, version)
        elif rng.random() < 0.05:
            t.task_group_max_hosts = 7  # outside a task group: persisted literally, not through the group table
        for _ in range(rng.choice([0, 0, 0, 1, 2])):
            t.depends_on.append(M.Dependency(rng.choice([f"{tag}{rng.randrange(max(n, 1))}", "ext-ok", "ext-bad", "missing"]),
                                             finished_at=rng.choice([M.ZERO_TIME, NOW - rng.randrange(10 ** 12)])))
        out.append(t)
    return out


def _compare_rows(rows, tasks, want, fresh, incl):
    """evg_queue_item rows against the restatement's items (same ranks); `fresh` = FetchExpectedDuration per task id,
    which the row carries for every task (the persisted ExpectedDuration differs only where GetDistroQueueInfo did not
    count the task: no EVG_QI_DEPS_MET under IncludesDependencies)."""
    assert [tasks[int(r)].id for r in rows["task"]] == [w.id for w in want]
    assert rows["priority"].tolist() == [w.priority for w in want]
    assert rows["group_index"].tolist() == [w.group_index for w in want]
    assert rows["total_value"].tolist() == [w.sorting_value_breakdown.total_value for w in want]
    met = ((rows["flags"] & L.EVG_QI_DEPS_MET) != 0).tolist()
    assert met == [w.dependencies_met for w in want]
    assert rows["group_max_hosts"].tolist() == [w.group_max_hosts if w.group else 0 for w in want]
    assert rows["expected_ns"].tolist() == [fresh[w.id] for w in want]
    assert all(w.expected_duration == fresh[w.id] for w, m in zip(want, met) if m or not incl)


def _oracle_queue(dist, tasks, db):
    planned_src = copy.deepcopy(tasks)
    order, bd, _ = O.plan(dist, planned_src, NOW)
    planned = [planned_src[int(i)] for i in order]
    for t, row in zip(planned, bd):
        t.sorting_value_breakdown = M.SortingValueBreakdown.from_row(row)
    incl = dist.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
    return OP.task_queue_items(OP.stamp_planned_tasks(planned, incl, NOW, db))


def test_persisted_queue_matches_the_restatement(engine):
    """PersistTaskQueue / TaskQueue.Save through the device (evg_download_queue rows, persist_task_queues documents)
    against oracle/oracle_persist.py applied to the oracle's plan: queue lengths around the 10 000 cap, caps 0 / 1 /
    10 000 / 10 001, task groups with MaxHosts, OverrideDependencies, earlier DependenciesMetTime stamps,
    IncludesDependencies; then again after evg_update_tasks."""
    rng = random.Random(41)
    sizes = (0, 1, 9999, 10000, 10001, 12000, 100000)
    db = {"ext-ok": M.Task(id="ext-ok", status="success"), "ext-bad": M.Task(id="ext-bad", status="failed")}
    batch = [(M.Distro(id=f"q{n}"), _persist_tasks(rng, n, f"q{n}-", f"q{n}")) for n in sizes]
    batch[2][0].dispatcher_settings.version = ""  # one distro without IncludesDependencies
    fresh = {t.id: O.fetch_expected_duration(copy.deepcopy(t), NOW)[0] for _, ts in batch for t in ts}
    want = [_oracle_queue(d, ts, db) for d, ts in batch]
    dev = copy.deepcopy(batch)
    docs = S.persist_task_queues(dev, NOW, engine=engine, dependency_db=db)
    task_off = np.cumsum([0] + [len(ts) for _, ts in batch])
    for (dist, _), doc, w in zip(batch, docs, want):
        saved = OP.saved_queue(w)
        assert len(doc.queue) == len(saved) == min(len(w), 10000)
        for got, exp in zip(doc.queue, saved):
            g, e = dict(vars(got)), dict(vars(exp))
            gv, ev = g.pop("sorting_value_breakdown"), e.pop("sorting_value_breakdown")
            assert g == e, (dist.id, got.id)
            assert gv.total_value == ev.total_value, (dist.id, got.id)
    for cap in (0, 1, 10000, 10001):
        item_off, items = engine.download_queue(cap, task_off)
        for d, (dist, _) in enumerate(batch):
            n = min(len(want[d]), cap or 10000)
            assert int(item_off[d + 1] - item_off[d]) == n
            incl = dist.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
            _compare_rows(items[int(item_off[d]):int(item_off[d + 1])], dev[d][1], want[d][:n], fresh, incl)
    # a tick whose priorities changed in place (evg_update_tasks): the rows follow the edited plan
    soa_, _, _ = soa.marshal_tasks(copy.deepcopy(batch), NOW, db)
    met, stamp = (x.copy() for x in engine.download_deps())
    rows = np.sort(np.random.default_rng(4).choice(int(task_off[-1]), size=int(task_off[-1]) // 10, replace=False)).astype(np.int64)
    vals = soa.TaskSoA(**{name: getattr(soa_, name)[rows].copy() for name, _ in soa_.COLUMNS})
    vals.priority = np.random.default_rng(5).integers(0, 101, rows.shape[0]).astype(np.int32)
    vals.flags = (vals.flags & ~np.uint32(L.EVG_TF_DEPS_MET)) | np.where(met[rows] != 0, L.EVG_TF_DEPS_MET, 0).astype(np.uint32)
    vals.wait_basis_ns = np.maximum(vals.wait_basis_ns, stamp[rows])
    engine.update_tasks(rows, vals)
    engine.run(NOW)
    edited = copy.deepcopy(batch)
    flat = [t for _, ts in edited for t in ts]
    for r, p in zip(rows.tolist(), vals.priority.tolist()):
        flat[r].priority = p
    item_off, items = engine.download_queue(0, task_off)
    for d, (dist, ts) in enumerate(edited):
        w = OP.saved_queue(_oracle_queue(dist, ts, db))
        incl = dist.dispatcher_settings.version == M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES
        _compare_rows(items[int(item_off[d]):int(item_off[d + 1])], ts, w, fresh, incl)


# ---------------------------------------------------------------- C. the DAG rebuild at its ABI edges
def _dag_batch(queues):
    """[(items, [group names])] -> evg_dag_in columns; a queue may declare groups no item is in."""
    item_off, group_off, dep_off, dep_item, group_id, group_index = [0], [0], [0], [], [], []
    for items, names in queues:
        pos = {it["id"]: k for k, it in enumerate(items)}
        gid = {g: k for k, g in enumerate(names)}
        for it in items:
            dep_item += [pos.get(x, -1) for x in it.get("dependencies", [])]
            dep_off.append(len(dep_item))
            key = f'{it.get("group", "")}_{it.get("build_variant", "")}_{it.get("project", "")}_{it.get("version", "")}'  # compositeGroupID
            group_id.append(gid[key] if it.get("group") else -1)
            group_index.append(it.get("group_index", 0))
        item_off.append(item_off[-1] + len(items))
        group_off.append(group_off[-1] + len(names))
    a = lambda x, t: np.ascontiguousarray(np.array(x, dtype=t))  # noqa: E731
    return (a(item_off, np.int64), a(group_off, np.int64), a(dep_off, np.int64), a(dep_item, np.int32), a(group_id, np.int32),
            a(group_index, np.int32))


def _check_dag(engine, queues):
    cols = _dag_batch(queues)
    srt, n_sorted, n_cycles, unit_items, unit_off = [np.array(x, copy=True) for x in engine.dag_rebuild_batch(*cols)]
    io, go = cols[0], cols[1]
    for d, (items, names) in enumerate(queues):
        want_order, want_cycles, want_units = OD.rebuild(items)
        b = int(io[d])
        assert [None if int(i) < 0 else items[int(i)]["id"] for i in srt[b:b + int(n_sorted[d])]] == want_order
        assert int(n_cycles[d]) == len(want_cycles)
        u = int(go[d]) + d
        got = {name: [items[int(i)]["id"] for i in unit_items[b + int(unit_off[u + g]):b + int(unit_off[u + g + 1])]]
               for g, name in enumerate(names)}
        assert got == {name: want_units.get(name, []) for name in names}
        assert all(int(unit_off[u + g]) <= int(unit_off[u + g + 1]) for g in range(len(names)))
    return n_cycles


def _item(k, group="", gi=0, deps=()):
    return {"id": str(k), "group": group, "build_variant": "", "project": "", "version": "", "group_index": gi,
            "dependencies": [str(x) for x in deps]}


def test_dag_rebuild_empty_groups(engine):
    """Declared groups no item is in -- at the start, the middle and the end of a distro, in a distro without items, and
    in a batch without any item (N == 0, G > 0): each is the empty range where the next group starts."""
    key = lambda g: f"{g}___"  # noqa: E731  compositeGroupID of (group, "", "", "")
    rnd = random.Random(3)
    items = [_item(k, rnd.choice(["b", "d", ""]), rnd.randrange(-3, 4), [rnd.randrange(k)] if k and rnd.random() < 0.4 else [])
             for k in range(40)]
    names = [key(g) for g in "abcde"]
    queues = [(items, names), ([], [key("x"), key("y")]), ([_item(0, "only")], [key("only"), key("z")]),
              ([_item(k) for k in range(5)], [key("q")])]
    _check_dag(engine, queues)
    _check_dag(engine, [([], [key("x")]), ([], [key("y"), key("z")]), ([], [])])


def test_dag_rebuild_group_index_extremes(engine):
    """GroupIndex at the int32 extremes inside one group (the key flips the sign bit): INT32_MIN, -1, 0, INT32_MAX in
    a shuffled, repeated mix, ties kept in queue order."""
    rnd = random.Random(8)
    vals = [-2 ** 31, -1, 0, 2 ** 31 - 1] * 6
    rnd.shuffle(vals)
    items = [_item(k, "g", v) for k, v in enumerate(vals)] + [_item(100 + k, "h", v) for k, v in enumerate(vals[::-1])]
    _check_dag(engine, [(items, ["g___", "h___"])])


def test_dag_rebuild_long_chains(engine):
    """A single 200 000-item dependency chain in both directions, and the same chain closed into one cycle."""
    n = 200_000
    fwd = [_item(k, deps=[k - 1] if k else []) for k in range(n)]
    bwd = [_item(k, deps=[k + 1] if k + 1 < n else []) for k in range(n)]
    cyc = [_item(k, deps=[(k - 1) % n]) for k in range(n)]
    assert _check_dag(engine, [(fwd, []), (bwd, []), (cyc, [])]).tolist() == [0, 0, 1]


def test_dag_rebuild_rejects_group_ids_outside_the_distro(engine):
    """A group_id below -1 or at / past its distro's group count is an error, found before anything runs."""
    for bad in (2, -2):
        cols = list(_dag_batch([([_item(0, "a"), _item(1, "b")], ["a___", "b___"]), ([_item(0, "c")], ["c___"])]))
        cols[4][1] = bad
        with pytest.raises(L.EvgError):
            engine.dag_rebuild_batch(*cols)
    cols = list(_dag_batch([([_item(0, "a")], ["a___"]), ([_item(0)], [])]))
    cols[4][1] = 0  # distro 1 declares no group
    with pytest.raises(L.EvgError):
        engine.dag_rebuild_batch(*cols)
    _check_dag(engine, [([_item(0, "a"), _item(1, "b")], ["a___", "b___"])])  # the context is still usable

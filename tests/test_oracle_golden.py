"""The oracle (oracle/evg_oracle.cpp) against every known answer the
reference's own tests hold for this path (SURVEY.md §8c).  CPU only."""
import copy
import itertools

import pytest

import golden_loader as G
from evergreen_b200 import model as M
from oracle import oracle as O

KATS = G.load("planner_kats.json")
ALLOC = G.load("allocator_scenarios.json")
NOW, EL = KATS["now"], KATS["elapsed_ns"]


def verify_rank_breakdown(b: M.SortingValueBreakdown):
    """verifyRankBreakdown (scheduler/planner_test.go:563-576)."""
    rank = (b.stepback_impact + b.patch_impact + b.patch_wait_time_impact + b.mainline_wait_time_impact +
            b.estimated_runtime_impact + b.num_dependents_impact + b.rank_commit_queue_impact)
    prio = (b.initial_priority_impact + b.priority_commit_queue_impact + b.generator_task_impact + b.task_group_impact)
    assert prio + b.task_group_length + rank * prio == b.total_value


@pytest.mark.parametrize("case", KATS["unit_values"], ids=lambda c: c["name"])
def test_unit_value_kats(case):
    tasks = [G.make_task(t, NOW, EL) for t in case["tasks"]]
    b = O.unit_value(G.make_distro(case), tasks, NOW)
    if "total" in case:
        assert b.total_value == case["total"], case["ref"]
    for f, v in case.get("fields", {}).items():
        assert getattr(b, f) == v, (case["ref"], f)
    verify_rank_breakdown(b)


def test_mainline_kat_needs_elapsed_time():
    """planner_test.go:247-252 expects 178; with zero elapsed test time the formula gives 179."""
    t = M.Task(id="foo", requester=M.REPOTRACKER_VERSION_REQUESTER, activated_time=NOW - M.HOUR)
    assert O.unit_value(M.Distro(), [t], NOW).total_value == 179
    t.activated_time -= 1
    assert O.unit_value(M.Distro(), [t], NOW).total_value == 178


def _run_plan(case):
    tasks = [G.make_task(t, NOW, EL) for t in case["tasks"]]
    order, bd, n_units = O.plan(G.make_distro(case), tasks, NOW)
    return tasks, [tasks[i] for i in order], bd, n_units


@pytest.mark.parametrize("case", KATS["plans"], ids=lambda c: c["name"])
def test_plan_kats(case):
    tasks, out, bd, n_units = _run_plan(case)
    ids = [t.id for t in out]
    assert len(set(ids)) == len(ids)
    if "order" in case:
        assert ids == case["order"], case["ref"]
    if "n_units" in case:
        assert n_units == case["n_units"], case["ref"]
    if "n_out" in case:
        assert len(ids) == case["n_out"]
    if "head_task_groups" in case:
        assert [t.task_group for t in out[:len(case["head_task_groups"])]] == case["head_task_groups"]
    if "last" in case:
        assert ids[-1] == case["last"]
    if "head_set" in case:
        assert set(ids[:len(case["head_set"])]) == set(case["head_set"])
    for a, b in case.get("before", []):
        assert ids.index(a) < ids.index(b), case["ref"]
    for row in bd:
        verify_rank_breakdown(M.SortingValueBreakdown.from_row(row))


def test_plan_deduplicates():
    """TaskPlan/Deduplicates (planner_test.go:430-433): the same task in two units is emitted once.
    Restated through dependencies: 'b' sits in its own unit and in a's."""
    tasks = [M.Task(id="a"), M.Task(id="b", depends_on=[M.Dependency("a")])]
    order, _, n_units = O.plan(M.Distro(), tasks, NOW)
    assert n_units == 2 and sorted(order.tolist()) == [0, 1]


@pytest.mark.parametrize("case", KATS["task_lists"], ids=lambda c: c["name"])
def test_task_list_kats(case):
    """TaskList.Less: tasks of one unit (a shared version under GroupVersions) come out in comparator order."""
    case = dict(case, group_versions=True)
    for t in case["tasks"]:
        t["version"] = "v"
    _, out, _, n_units = _run_plan(case)
    assert n_units == 1
    assert [t.id for t in out] == case["order"], case["ref"]


@pytest.mark.parametrize("case", KATS["queue_infos"], ids=lambda c: c["name"])
def test_queue_info_kats(case):
    tasks = [G.make_task(t, NOW, EL) for t in case["tasks"]]
    info = O.queue_info(case["distro_id"], tasks, case["threshold"], False, NOW)
    assert info.length == case["length"]
    assert info.length_with_dependencies_met == case["length_with_dependencies_met"], case["ref"]
    assert [O.fetch_expected_duration(t, NOW)[0] for t in tasks] == case["expected_durations"]
    assert info.expected_duration == sum(case["expected_durations"])
    assert info.max_duration_threshold == case["threshold"]


@pytest.mark.parametrize("case", KATS["group_by"], ids=lambda c: c["name"])
def test_group_by_task_group(case):
    hosts = [M.Host(**h) for h in case["hosts"]]
    infos = [M.TaskGroupInfo(**g) for g in case["infos"]]
    buckets = O.group_by_task_group(hosts, infos)
    assert set(buckets) == set(case["buckets"]), case["ref"]
    for name, want in case["buckets"].items():
        idx, info = buckets[name]
        assert [hosts[i].id for i in idx] == want["hosts"]
        assert (info.count if info else 0) == want["count"]


@pytest.mark.parametrize("v", [v for v in ALLOC["vectors"] if v["fn"] == "calcNewHostsNeeded"],
                         ids=lambda v: "-".join(str(a) for a in v["args"]))
def test_calc_new_hosts_needed(v):
    assert O.calc_new_hosts_needed(*v["args"]) == v["expect"], v["ref"]


def test_calc_existing_free_hosts():
    (v,) = [v for v in ALLOC["vectors"] if v["fn"] == "calcExistingFreeHosts"]
    hosts = [G.go_host(h) for h in v["hosts"]]
    running = {t["Id"]: G.go_running_task(t, ALLOC["now"], O.fetch_expected_duration) for t in v["tasks"]}
    free, st = O.calc_existing_free_hosts(hosts, running, v["fraction"], v["threshold"], ALLOC["now"])
    assert st == 0 and free == v["expect"] == 3, v["ref"]


@pytest.mark.parametrize("s", ALLOC["scenarios"], ids=lambda s: s["test"])
def test_allocator_scenarios(s):
    data = G.go_allocator_data(s, O.fetch_expected_duration)
    n, f, st = O.allocate(data, s["now"])
    assert st == 0
    assert (n, f) == (s["expect_new_hosts"], s["expect_free_hosts"]), s["ref"]


def test_allocator_scenarios_cover_the_reference_suite():
    names = {s["test"] for s in ALLOC["scenarios"]}
    assert len(names) == 23
    for must in ("TestNoExistingHosts", "TestRoundingUp", "TestRealisticScenarioWithContainers2",
                 "TestRealisticScenarioWithTaskGroups", "TestHostsWithLongTasks"):
        assert must in names


def test_allocator_data_errors():
    """The two data errors (utilization_based_host_allocator.go:200-202,302-304) and the missing parent (:151-158)."""
    s = next(x for x in ALLOC["scenarios"] if x["test"] == "TestNoExistingHosts")
    d = G.go_allocator_data(s, O.fetch_expected_duration)
    d.distro.host_allocator_settings.future_host_fraction = 1.5
    assert O.allocate(d, s["now"])[2] == 1
    d = G.go_allocator_data(s, O.fetch_expected_duration)
    d.distro.provider = M.PROVIDER_DOCKER
    d.distro.host_allocator_settings.maximum_hosts = 0
    assert O.allocate(d, s["now"])[2] == 2
    d = G.go_allocator_data(s, O.fetch_expected_duration)
    d.container_pool = M.ContainerPool("p", "nowhere", 10)
    assert O.allocate(d, s["now"])[2] == 3


def test_host_allocator_property_bounds():
    """host_allocator_fuzzer_test.go:154-172: 0 <= new <= queue length on random cases (seeded here)."""
    import random
    rng = random.Random(7)
    for _ in range(100):
        n_tasks = rng.randint(0, 200)
        durs = [rng.randint(1, 7200) * M.SECOND for _ in range(n_tasks)]
        thr = 30 * M.MINUTE
        over = [d for d in durs if d > thr]
        g = M.TaskGroupInfo("", count=n_tasks, expected_duration=sum(durs), count_duration_over_threshold=len(over),
                            duration_over_threshold=sum(over))
        qi = M.DistroQueueInfo(length=n_tasks, length_with_dependencies_met=n_tasks, expected_duration=sum(durs),
                               max_duration_threshold=thr, count_duration_over_threshold=len(over),
                               duration_over_threshold=sum(over), task_group_infos=[g] if n_tasks else [])
        hosts, running = [], {}
        for h in range(rng.randint(0, 50)):
            if rng.random() < 0.7:
                hosts.append(M.Host(id=f"h{h}", running_task=f"t{h}"))
                running[f"t{h}"] = M.RunningTaskStats(True, rng.randint(60, 7200) * M.SECOND, 0,
                                                      NOW - rng.randint(0, 7200) * M.SECOND)
            else:
                hosts.append(M.Host(id=f"h{h}"))
        d = M.Distro(id="d", provider=M.PROVIDER_EC2_FLEET,
                     host_allocator_settings=M.HostAllocatorSettings(maximum_hosts=1000, future_host_fraction=0.5))
        n, f, st = O.allocate(M.HostAllocatorData(d, hosts, qi, running_tasks=running), NOW)
        assert st == 0 and 0 <= n <= n_tasks and f >= 0


# ---------------------------------------------------------------- task finders (SURVEY.md §8f.1)
FINDER = G.load("task_finder.json")


@pytest.mark.parametrize("finder", ["legacy", "alternate"])
@pytest.mark.parametrize("case", FINDER["cases"], ids=lambda c: c["name"])
def test_task_finder_cases(case, finder):
    """What scheduler/task_finder_test.go asserts (every finder of the suite must satisfy it)."""
    d, tasks, refs = G.finder_case(case)
    got = [t.id for t in O.find_runnable(d, tasks, refs, finder=finder)]
    if "expect_len" in case:
        assert len(got) == case["expect_len"]
    if "expect_ids" in case:
        assert sorted(got) == sorted(case["expect_ids"])


@pytest.mark.parametrize("seed", range(20))
def test_task_finders_agree_on_fuzzy_tasks(seed):
    """TaskFinderComparisonSuite.TestFindRunnableHostsIsIdentical (task_finder_test.go:309-334) on the fuzzy
    generator: legacy and alternate finders return the same ids."""
    import random
    tasks = G.random_finder_tasks(random.Random(seed))
    refs = [M.ProjectRef(**r) for r in FINDER["cases"][-1]["project_refs"]]
    a = sorted(t.id for t in O.find_runnable(M.Distro(), tasks, refs, finder="legacy"))
    b = sorted(t.id for t in O.find_runnable(M.Distro(), tasks, refs, finder="alternate"))
    assert a == b
    assert all(t.startswith("task") for t in a)


def test_task_finders_differ_only_by_the_short_circuit():
    """DependenciesMet trusts DependenciesMetTime / OverrideDependencies (task.go:3393-3395); AllDependenciesSatisfied
    walks anyway (task.go:795-821)."""
    dep = M.Task(id="dep", status="failed", activated=True, project="exists")
    t = M.Task(id="t", activated=True, project="exists", dependencies_met_time=5,
               depends_on=[M.Dependency(task_id="dep", status="success")])
    refs = [M.ProjectRef(id="exists", enabled=True)]
    assert [x.id for x in O.find_runnable(M.Distro(), [t, dep], refs, finder="legacy")] == ["t"]
    assert [x.id for x in O.find_runnable(M.Distro(), [t, dep], refs, finder="alternate")] == []
    d = M.Distro(dispatcher_settings=M.DispatcherSettings(version="revised-with-dependencies"))
    assert [x.id for x in O.find_runnable(d, [t, dep], refs, finder="alternate")] == ["t"]


# ---------------------------------------------------------------- expected-duration statistics (SURVEY.md §8f.2)
DURATION = G.load("expected_duration.json")


def duration_case(case):
    return [G.make_task(t, 0, 0) for t in case["tasks"]], case["window_start"], case["window_end"]


@pytest.mark.parametrize("case", DURATION["cases"], ids=lambda c: c["name"])
def test_expected_duration_kat(case):
    tasks, w0, w1 = duration_case(case)
    got = O.expected_durations_for_window(tasks, w0, w1)
    e = case["expect"]
    n, mean, std, _ = got[tuple(e["key"])]
    assert len(got) == 1 and n == len(tasks)
    assert mean == e["mean_ns"]                                   # EqualValues: exact
    assert abs(std - e["stddev_ns"]) <= e["stddev_delta_ns"]      # InDelta(…, 0.01 minute)


def test_expected_duration_match_stage():
    """The $match of expected_duration.go:37-55: completed, not timed out, StartTime > start (strict), FinishTime <= end."""
    MIN, now = 60 * 10 ** 9, 10 ** 18
    base = dict(build_variant="bv", project="p", display_name="n", status="success", finish_time=now, start_time=now - MIN, time_taken=MIN)
    rows = [M.Task(**base), M.Task(**dict(base, status="undispatched")), M.Task(**dict(base, timed_out=True)),
            M.Task(**dict(base, start_time=now - 60 * MIN)), M.Task(**dict(base, finish_time=now + 1)),
            M.Task(**dict(base, status="failed", time_taken=3 * MIN))]
    got = O.expected_durations_for_window(rows, now - 60 * MIN, now)
    assert got[("p", "bv", "n")][:3] == (2, 2.0 * MIN, 1.0 * MIN)


# ---------------------------------------------------------------- Task.DependenciesMet (model/task/task_test.go)
DEPS = G.load("dependencies_met.json")


@pytest.mark.parametrize("case", DEPS["cases"], ids=lambda c: c["name"])
def test_dependencies_met_cases(case):
    """TestDependenciesMet: the C++ oracle (evo_deps_met), the finder restatement's walk and the host mirror."""
    from evergreen_b200 import soa
    t, db = G.deps_case(case)
    if "met" in case:
        assert bool(O.deps_met([t], 0, db)[0]) == case["met"]
        assert O._deps_walk(t, dict(db), shortcut=True) == case["met"]
        assert soa.dependencies_met(t, {t.id: t}, db) == case["met"]
    if "all_satisfied" in case:
        assert O._deps_walk(t, dict(db), shortcut=False) == case["all_satisfied"]


@pytest.mark.parametrize("case", DEPS["blocked"], ids=lambda c: c["name"])
def test_blocked_cases(case):
    t = M.Task(id="t1", depends_on=[M.Dependency(task_id="", unattainable=u) for u in case["unattainable"]])
    assert t.blocked() == case["expect"]


# ---------------------------------------------------------------- PersistTaskQueue (scheduler/task_queue_persister_test.go)
def test_task_queue_persister_golden():
    """TestDBTaskQueuePersister: the persisted items of the two queues, their fields copied from the tasks, t5's
    ExpectedDuration the ten-minute default, and the two queue infos the test checks first."""
    from oracle import oracle_persist as OP
    g = G.load("task_queue_persister.json")
    now = 10 ** 18
    for q in g["queues"]:
        src = {t["id"]: t for t in g["tasks"]}
        tasks = [G.make_task(src[i], now, 0) for i in q["tasks"]]
        info = O.queue_info(q["distro"], [G.make_task(src[i], now, 0) for i in q["tasks"]], g["max_duration_threshold_ns"], False, now)
        assert (info.length, info.length_with_dependencies_met) == (q["length"], q["length_with_dependencies_met"]), q["ref"]
        items = OP.saved_queue(OP.task_queue_items(OP.stamp_planned_tasks(tasks, False, now)))
        assert [it.id for it in items] == q["tasks"], q["ref"]
        assert [it.expected_duration for it in items] == q["expected_durations"], q["ref"]
        for it in items:
            s = src[it.id]
            assert (it.display_name, it.build_variant, it.revision_order_number, it.requester, it.revision, it.project,
                    it.activated_by) == (s["display_name"], s["build_variant"], s["revision_order_number"], s["requester"],
                                         s["revision"], s["project"], s["activated_by"])
            assert it.dependencies == [d["task_id"] for d in s.get("depends_on", [])]
            assert it.dependencies_met == (not s.get("depends_on"))  # "someTask" does not exist: never met
    # Save keeps 10 000 items; the projection itself keeps every task
    many = [M.Task(id=f"t{k}") for k in range(10001)]
    assert len(OP.task_queue_items(many)) == 10001 and [it.id for it in OP.saved_queue(OP.task_queue_items(many))] == [t.id for t in many[:10000]]


def test_persister_restatement_stamps_like_get_distro_queue_info():
    """GetDistroQueueInfo's writes the persisted items read: a fresh met verdict stamps DependenciesMetTime (latest
    FinishedAt, else now), an earlier stamp is kept, and under IncludesDependencies a task whose dependencies are not
    met keeps its own ExpectedDuration."""
    from oracle import oracle_persist as OP
    now, MIN = 10 ** 18, 60 * 10 ** 9
    db = {"ok": M.Task(id="ok", status="success"), "bad": M.Task(id="bad", status="failed")}
    mk = lambda i, **kw: M.Task(id=i, expected_duration=0, **kw)  # noqa: E731
    tasks = [mk("a", depends_on=[M.Dependency("ok", finished_at=now - 5 * MIN), M.Dependency("ok", finished_at=now - 9 * MIN)]),
             mk("b", depends_on=[M.Dependency("ok")]),
             mk("c", depends_on=[M.Dependency("bad")]),
             mk("d", depends_on=[M.Dependency("bad")], dependencies_met_time=now - MIN),
             mk("e", depends_on=[M.Dependency("bad")], override_dependencies=True)]
    for incl in (False, True):
        ts = OP.stamp_planned_tasks(copy.deepcopy(tasks), incl, now, db)
        assert [t.dependencies_met_time for t in ts] == [now - 5 * MIN, now, M.ZERO_TIME, now - MIN, M.ZERO_TIME]
        assert [it.dependencies_met for it in OP.task_queue_items(ts)] == [True, True, False, True, True]
        assert [t.expected_duration for t in ts] == [10 * MIN, 10 * MIN, 0 if incl else 10 * MIN, 10 * MIN, 10 * MIN]

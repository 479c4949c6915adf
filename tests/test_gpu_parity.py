"""Parity of the CUDA path (through the C-ABI) with the oracle: the committed
golden vectors, seeded synthetic ticks in every BASELINE shape, edge cases, and
size-independent properties at full size.  Integer / index work: bit-exact."""
import copy

import numpy as np
import pytest

import golden_loader as G
import parity
from evergreen_b200 import _lib as L
from evergreen_b200 import model as M
from evergreen_b200 import scheduler as S
from evergreen_b200 import soa, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

KATS = G.load("planner_kats.json")
ALLOC = G.load("allocator_scenarios.json")
NOW, EL = KATS["now"], KATS["elapsed_ns"]


def run(engine, w, breakdown=False):
    if w.hosts is not None:
        return engine.plan_and_alloc_batch(w.tasks, w.distros, w.hosts, w.now, breakdown=breakdown)
    return engine.plan_batch(w.tasks, w.distros, w.now, breakdown=breakdown), None


# ---------------------------------------------------------------- golden vectors
@pytest.mark.parametrize("case", KATS["unit_values"], ids=lambda c: c["name"])
def test_unit_value_kats(engine, case):
    """planner_test.go:199-406 through the product: the tasks of each unit are
    queued so that they form exactly that unit (one version under GroupVersions,
    or their task group), and the stamped breakdown is compared."""
    case = dict(case)
    tasks = [G.make_task(t, NOW, EL) for t in case["tasks"]]
    if len(tasks) > 1 and not tasks[0].task_group:
        case["group_versions"] = True
        for t in tasks:
            t.version = "v"
    d = G.make_distro(case)
    plan, _ = S.PrioritizeTasks(d, tasks, now=NOW, engine=engine)
    b = plan[0].sorting_value_breakdown
    want = O.unit_value(d, tasks, NOW)
    assert b.row() == want.row()
    if "total" in case:
        assert b.total_value == case["total"], case["ref"]
    for f, v in case.get("fields", {}).items():
        assert getattr(b, f) == v


@pytest.mark.parametrize("case", KATS["plans"] + [dict(c, group_versions=True, _one_version=True) for c in KATS["task_lists"]],
                         ids=lambda c: c["name"])
def test_plan_kats(engine, case):
    tasks = [G.make_task(t, NOW, EL) for t in case["tasks"]]
    if case.get("_one_version"):
        for t in tasks:
            t.version = "v"
    d = G.make_distro(case)
    opts = S.TaskPlannerOptions(is_secondary_queue=bool(case.get("secondary_queue")))
    plan, info = S.PrioritizeTasks(d, tasks, opts, now=NOW, engine=engine)
    ids = [t.id for t in plan]
    order, bd, _ = O.plan(d, tasks, NOW)
    assert ids == [tasks[i].id for i in order]
    assert [t.sorting_value_breakdown.row() for t in plan] == bd.tolist()
    if "order" in case:
        assert ids == case["order"], case["ref"]
    if "n_out" in case:
        assert len(ids) == case["n_out"]
    if "last" in case:
        assert ids[-1] == case["last"]
    if "head_set" in case:
        assert set(ids[:len(case["head_set"])]) == set(case["head_set"])
    if "head_task_groups" in case:
        assert [t.task_group for t in plan[:2]] == case["head_task_groups"]
    for a, b in case.get("before", []):
        assert ids.index(a) < ids.index(b)
    assert info.secondary_queue == bool(case.get("secondary_queue"))


@pytest.mark.parametrize("case", KATS["queue_infos"], ids=lambda c: c["name"])
def test_queue_info_kats(engine, case):
    tasks = [G.make_task(t, NOW, EL) for t in case["tasks"]]
    info = S.GetDistroQueueInfo(M.Distro(id=case["distro_id"]), tasks, case["threshold"], now=NOW, engine=engine)
    assert (info.length, info.length_with_dependencies_met) == (case["length"], case["length_with_dependencies_met"])
    assert info.expected_duration == sum(case["expected_durations"])
    want = O.queue_info(case["distro_id"], [G.make_task(t, NOW, EL) for t in case["tasks"]], case["threshold"], False, NOW)
    key = lambda g: g.name
    assert sorted(info.task_group_infos, key=key) == sorted(want.task_group_infos, key=key)


@pytest.mark.parametrize("s", ALLOC["scenarios"], ids=lambda s: s["test"])
def test_allocator_scenarios(engine, s):
    data = G.go_allocator_data(s, M.fetch_expected_duration)
    odata = G.go_allocator_data(s, O.fetch_expected_duration)
    n, f = S.UtilizationBasedHostAllocator(data, now=s["now"], engine=engine)
    assert (n, f) == (s["expect_new_hosts"], s["expect_free_hosts"]), s["ref"]
    O.allocate(odata, s["now"])
    assert data.distro_queue_info.task_group_infos == odata.distro_queue_info.task_group_infos


@pytest.mark.parametrize("v", [v for v in ALLOC["vectors"] if v["fn"] == "calcNewHostsNeeded"],
                         ids=lambda v: "-".join(str(a) for a in v["args"]))
def test_calc_new_hosts_needed(engine, v):
    """utilization_based_host_allocator_test.go:160-170 reached through the allocator:
    one "" bucket whose numbers are exactly the vector's arguments."""
    short, thr, exp_free, n_long, overdue, mq, round_down = v["args"]
    g = M.TaskGroupInfo("", count=10 ** 6, expected_duration=short, count_duration_over_threshold=n_long,
                        count_wait_over_threshold=overdue, count_dep_filled_merge_queue_tasks=mq)
    qi = M.DistroQueueInfo(length=10 ** 6, length_with_dependencies_met=10 ** 6, expected_duration=short,
                           max_duration_threshold=thr, task_group_infos=[g])
    d = M.Distro(id="d", provider=M.PROVIDER_EC2_FLEET, host_allocator_settings=M.HostAllocatorSettings(
        maximum_hosts=10 ** 6, future_host_fraction=0.5,
        rounding_rule=M.HOST_ALLOCATOR_ROUND_DOWN if round_down else M.HOST_ALLOCATOR_ROUND_UP,
        feedback_rule=M.HOST_ALLOCATOR_WAITS_OVER_THRESH_FEEDBACK))
    hosts = [M.Host(id=f"h{i}") for i in range(exp_free)]
    n, f = S.UtilizationBasedHostAllocator(M.HostAllocatorData(d, hosts, qi), now=NOW, engine=engine)
    assert (n, f) == (v["expect"], exp_free), v["ref"]


def test_allocator_data_errors(engine):
    s = next(x for x in ALLOC["scenarios"] if x["test"] == "TestNoExistingHosts")
    for mutate, code in ((lambda d: setattr(d.distro.host_allocator_settings, "future_host_fraction", 1.5), 1),
                         (lambda d: (setattr(d.distro, "provider", M.PROVIDER_DOCKER),
                                     setattr(d.distro.host_allocator_settings, "maximum_hosts", 0)), 2),
                         (lambda d: setattr(d, "container_pool", M.ContainerPool("p", "nowhere", 10)), 3)):
        d = G.go_allocator_data(s, M.fetch_expected_duration)
        mutate(d)
        with pytest.raises(S.AllocatorError) as e:
            S.UtilizationBasedHostAllocator(d, now=s["now"], engine=engine)
        assert e.value.status == code
        assert O.allocate(copy.deepcopy(d), s["now"])[2] == code


# ---------------------------------------------------------------- synthetic ticks vs oracle
@pytest.mark.parametrize("k,scale", [(1, 1), (2, 0.004), (3, 0.05), (4, 0.03), (5, 0.02)])
def test_config_parity(engine, k, scale):
    w = synth.config(k, scale)
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)
    parity.check_properties(w, po, ao)


@pytest.mark.parametrize("seed", range(4))
def test_mixed_parity(engine, seed):
    """Everything at once: task groups, GroupVersions on half the distros, met and unmet
    in-queue dependencies, custom factors, ragged sizes incl. empty and single-task distros."""
    rng = synth.Rng(1000 + seed)
    sizes = np.concatenate([[0, 1, 2, 0, 3], rng.integers(40, 1, 400), [2049, 4097, 0]])
    w = synth.make(sizes, 7000 + seed, zipf_priority=True, unmet_dep_frac=0.06, met_dep_frac=0.04, tg_frac=0.2,
                   group_versions_frac=0.5, custom_factor_frac=0.5, includes_dependencies=bool(seed & 1),
                   n_hosts=300, providers=(0.6, 0.2, 0.2))
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)
    parity.check_properties(w, po, ao)


def test_breakdown_parity(engine):
    w = synth.make(np.array([300, 7, 1, 900]), 99, zipf_priority=True, unmet_dep_frac=0.05, met_dep_frac=0.05,
                   tg_frac=0.3, group_versions_frac=0.5, custom_factor_frac=1.0)
    po, _ = run(engine, w, breakdown=True)
    assert np.array_equal(po.breakdown[:, L.EVG_BD_TOTAL_VALUE], po.total_value)
    b = po.breakdown
    prio = b[:, 2] + b[:, 3] + b[:, 4] + b[:, 5]
    rank = b[:, 6:].sum(axis=1)
    # verifyRankBreakdown (planner_test.go:563-576).  The reference's bookkeeping drops the unit length for
    # units that are all-task-group AND contain a generator (planner.go:285-293, SURVEY.md App. A.2): skip those.
    ok = ~((b[:, L.EVG_BD_P_TASK_GROUP] != 0) & (b[:, L.EVG_BD_P_GENERATOR] != 0))
    assert ok.sum() > 1000
    assert np.array_equal((prio + b[:, 0] + rank * prio)[ok], b[:, 1][ok])
    ref = parity.check_against_oracle(w, po, None)
    assert np.array_equal(po.breakdown, ref["breakdown"])


def test_task_group_order_fallbacks(engine):
    """The list-free task-group path needs unique TaskGroupOrder < 64 inside each group; distros that break
    that (duplicates, large or zero orders) must fall back to the unit lists and still match the oracle."""
    w = synth.make(np.array([900, 3000, 9000, 9000, 500]), 55, tg_frac=0.2, zipf_priority=True, n_hosts=40)
    toff = w.distros.task_off
    t = w.tasks
    t.task_group_order[toff[0]:toff[1]] = 0                       # all equal (the reference's TaskGroup KAT shape)
    sel = np.arange(toff[1], toff[2])[::5]
    t.task_group_order[sel] = 70                                  # beyond the presence mask
    t.task_group_order[toff[2]:toff[3]] = np.minimum(t.task_group_order[toff[2]:toff[3]], 2)  # duplicates
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)


def test_route_boundaries(engine):
    """Distro sizes on both sides of every on-chip capacity class (1024 / 4096 / 12288 tasks) in one tick,
    so the three k_plan_smem variants and the general path all run in the same call."""
    sizes = np.array([1023, 1024, 1025, 4095, 4096, 4097, 12287, 12288, 12289, 1, 0, 33])
    w = synth.make(sizes, 21, zipf_priority=True, tg_frac=0.15, unmet_dep_frac=0.03, met_dep_frac=0.02,
                   custom_factor_frac=0.5, includes_dependencies=True, n_hosts=120, providers=(0.7, 0.2, 0.1))
    po, ao = run(engine, w, breakdown=True)
    ref = parity.check_against_oracle(w, po, ao)
    assert np.array_equal(po.breakdown, ref["breakdown"])
    parity.check_properties(w, po, ao)


def test_wide_value_range(engine):
    """TotalValue ranges beyond 32 bits (factors of 100 and priorities up to 100) take the two-word key path."""
    w = synth.make(np.array([9000, 700, 12000]), 31, zipf_priority=True, custom_factor_frac=1.0, tg_frac=0.1)
    for f in ("patch_time_in_queue_factor", "generate_task_factor", "expected_runtime_factor"):
        w.distros.cfg[f] = 100
    w.tasks.priority[::7] = 1000
    po, _ = run(engine, w)
    assert int(po.total_value.max() - po.total_value.min()) > 2 ** 33
    parity.check_against_oracle(w, po, None)


def test_large_distros_multi_tile(engine):
    """Distros far larger than one sort tile, with heavy TotalValue ties."""
    w = synth.make(np.array([70_000, 5, 33_000]), 5, tg_frac=0.1, unmet_dep_frac=0.02, includes_dependencies=True,
                   n_hosts=50)
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)


def test_group_versions_big_units(engine):
    """GroupVersions with ~50-task version units and task groups nested in them."""
    w = synth.make(np.full(6, 1500), 11, tg_frac=0.15, group_versions_frac=1.0, met_dep_frac=0.03, unmet_dep_frac=0.03)
    po, _ = run(engine, w)
    parity.check_against_oracle(w, po, None)


def test_dependency_fan(engine):
    """One task everyone depends on (fan-in) and one task depending on everyone (fan-out)."""
    n = 400
    w = synth.make(np.array([n]), 3, tg_frac=0.0)
    t = w.tasks
    dep_off = np.zeros(n + 1, dtype=np.int64)
    idx = []
    for i in range(n):
        if i == 7:
            idx += [j for j in range(n) if j != 7]      # fan-out: task 7 depends on all
        elif i % 3 == 0:
            idx += [5]                                   # fan-in: a third of the tasks depend on 5
        dep_off[i + 1] = len(idx)
    t.dep_off, t.dep_idx = dep_off, np.array(idx, dtype=np.int32)
    t.flags = t.flags | np.uint32(L.EVG_TF_DEPS_MET)
    t.normalize()
    po, _ = run(engine, w)
    parity.check_against_oracle(w, po, None)


def test_edge_inputs(engine):
    # no distros at all
    w = synth.make(np.zeros(0, dtype=np.int64), 1)
    po, _ = run(engine, w)
    assert po.order.shape == (0,) and po.info.shape == (0,)
    # only empty distros
    w = synth.make(np.zeros(3, dtype=np.int64), 1, n_hosts=0)
    po, _ = run(engine, w)
    assert np.all(po.info["length"] == 0) and np.all(po.info["has_ungrouped"] == 0)
    # all keys equal: order must be the input order
    w = synth.make(np.array([3000]), 2, tg_frac=0.0)
    for col in ("expected_ns", "queue_basis_ns", "wait_basis_ns"):
        getattr(w.tasks, col)[:] = getattr(w.tasks, col)[0]
    w.tasks.num_dependents[:] = 0
    w.tasks.flags[:] = L.EVG_TF_DEPS_MET
    po, _ = run(engine, w)
    assert np.array_equal(po.order, np.arange(3000))
    # negative priority (disabled tasks are -1): MaxPriority floors at 0 (planner.go:325-327)
    w = synth.make(np.array([50]), 4)
    w.tasks.priority[:] = -1
    po, _ = run(engine, w)
    parity.check_against_oracle(w, po, None)
    # Go-zero and Unix-epoch times
    w = synth.make(np.array([64]), 6)
    w.tasks.queue_basis_ns[::2] = M.ZERO_TIME
    w.tasks.queue_basis_ns[1::4] = 0
    w.tasks.wait_basis_ns[::3] = M.ZERO_TIME
    po, _ = run(engine, w)
    parity.check_against_oracle(w, po, None)


@pytest.mark.parametrize("now", [5, -(10 ** 18), 2 ** 62])
def test_odd_clocks(engine, now):
    """Clocks outside the usual range (before the threshold, negative, far future) take the literal
    saturating time.Since path instead of the cutoff comparison."""
    w = synth.make(np.array([700, 2000, 5000]), 17, tg_frac=0.1, unmet_dep_frac=0.03, includes_dependencies=True, n_hosts=30)
    w.now = now
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)


@pytest.mark.parametrize("seed", range(3))
def test_tiny_distros_warp_path(engine, seed):
    """Distros of 0..32 tasks are planned one warp each (k_plan_warp): task groups, GroupVersions, met and
    unmet in-queue dependencies, custom factors, all mixed; plus the breakdown, which reroutes them on-chip."""
    rng = synth.Rng(300 + seed)
    sizes = rng.integers(3000, 0, 32)
    w = synth.make(sizes, 9000 + seed, zipf_priority=True, unmet_dep_frac=0.08, met_dep_frac=0.05, tg_frac=0.3,
                   group_versions_frac=0.4, custom_factor_frac=0.5, includes_dependencies=bool(seed & 1),
                   n_hosts=2000, providers=(0.6, 0.2, 0.2))
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)
    parity.check_properties(w, po, ao)
    order, tv = po.order.copy(), po.total_value.copy()
    po2, _ = run(engine, w, breakdown=True)
    assert np.array_equal(order, po2.order) and np.array_equal(tv, po2.total_value)
    ref = parity.check_against_oracle(w, po2, None)
    assert np.array_equal(po2.breakdown, ref["breakdown"])


def test_out_of_range_ids_are_rejected(engine):
    """Distro-local ids index device tables: the library range-checks them once per upload (k_validate)."""
    for mutate in (lambda w: w.tasks.group_id.__setitem__(5, 10 ** 6),
                   lambda w: w.tasks.version_id.__setitem__(7, 10 ** 6),
                   lambda w: w.tasks.group_id.__setitem__(3, -5),
                   lambda w: w.tasks.dep_idx.__setitem__(0, 10 ** 6)):
        w = synth.make(np.array([200, 50, 3000]), 8, tg_frac=0.2, unmet_dep_frac=0.1, includes_dependencies=True)
        mutate(w)
        with pytest.raises(L.EvgError) as e:
            engine.plan_batch(w.tasks, w.distros, w.now)
        assert e.value.code == L.EVG_ERR_INVALID
    w = synth.make(np.array([200, 50, 3000]), 8, tg_frac=0.2)
    po, _ = run(engine, w)  # the context recovers
    parity.check_against_oracle(w, po, None)


@pytest.mark.parametrize("seed", range(3))
def test_dependency_filter_parity(engine, seed):
    """evg_deps_met_batch (SURVEY.md §8f.1) against the oracle's Task.DependenciesMet restatement and the host mirror."""
    import random
    from test_host_logic import random_tasks
    rng = random.Random(40 + seed)
    batch, db_all = [], {}
    for d in range(6):
        tasks, db = random_tasks(rng, rng.choice([0, 1, 7, 150, 900]))
        for t in tasks:
            t.id = f"d{d}-{t.id}"
            for dep in t.depends_on:
                if dep.task_id.startswith("t"):
                    dep.task_id = f"d{d}-{dep.task_id}"
        batch.append((M.Distro(id=f"d{d}"), tasks))
        db_all.update(db)
    got = S.dependencies_met(batch, engine=engine, dependency_db=db_all)
    for (dist, tasks), g in zip(batch, got):
        by_id = {t.id: t for t in tasks}
        assert g == [soa.dependencies_met(t, by_id, db_all) for t in tasks]
        assert g == O.deps_met(tasks, NOW, db_all).tolist()


@pytest.mark.parametrize("case", G.load("dependencies_met.json")["cases"], ids=lambda c: c["name"])
def test_dependencies_met_cases(engine, case):
    """TestDependenciesMet (model/task/task_test.go:249-434) through evg_deps_met_batch, and its
    AllDependenciesSatisfied assertions through the alternate finder of evg_find_runnable_batch."""
    t, db = G.deps_case(case)
    if "met" in case:
        assert S.dependencies_met([(M.Distro(id="d"), [t])], engine=engine, dependency_db=db) == [[case["met"]]]
    if "all_satisfied" in case:
        t.project = "p"
        got = S.AlternateTaskFinder(M.Distro(id="d"), [t], [M.ProjectRef(id="p", enabled=True)], dependency_db=db, engine=engine)
        assert [x.id for x in got] == (["t1"] if case["all_satisfied"] else [])


def test_dependency_filter_at_scale(engine):
    """1e6 tasks with ~1.5e6 dependencies: device result vs a numpy restatement of the same table."""
    rng = np.random.default_rng(5)
    T = 1_000_000
    n_dep = rng.integers(0, 4, T)
    off = np.zeros(T + 1, np.int64); np.cumsum(n_dep, out=off[1:])
    E = int(off[-1])
    deps = soa.DepsTable(off, rng.integers(0, 3, E).astype(np.uint8), rng.integers(0, 5000, E).astype(np.int32),
                         rng.integers(0, 4, E).astype(np.uint8), rng.integers(0, 8, T).astype(np.uint8) & 7,
                         (rng.random(T) < 0.1).astype(np.uint8) | ((rng.random(T) < 0.1).astype(np.uint8) << 1),
                         rng.integers(0, 8, 5000).astype(np.uint8))
    deps.task_state &= 0x7
    deps.task_state[(deps.task_state & 3) == 3] -= 1
    deps.ext_state[(deps.ext_state & 3) == 3] -= 1
    got = engine.deps_met_batch(deps).copy()
    st = np.where(deps.dep_kind == 0, deps.task_state[deps.dep_ref], deps.ext_state[deps.dep_ref])
    status, blocked = st & 3, (st & 4) != 0
    sat = np.where(deps.dep_want == 0, status == 0, np.where(deps.dep_want == 1, status == 1,
                   np.where(deps.dep_want == 2, (status < 2) | blocked, False)))
    sat &= deps.dep_kind != 2
    unsat = np.add.reduceat(np.concatenate([(~sat).astype(np.int64), [0]]), np.minimum(off[:-1], E))[:T] * (n_dep > 0)
    want = (n_dep == 0) | (deps.task_pre != 0) | (unsat == 0)
    assert np.array_equal(got.astype(bool), want)


# ---------------------------------------------------------------- task finders (SURVEY.md §8f.1)
FINDER = G.load("task_finder.json")


def random_finder_batch(rng, n_distros):
    """Candidates with every field the finders read randomised, plus project refs of every flag combination."""
    from test_host_logic import random_tasks
    refs = [M.ProjectRef(id=f"p{k}", enabled=bool(k & 1), hidden=bool(k & 2) or None, dispatching_disabled=bool(k & 4) or None,
                         patching_disabled=bool(k & 8) or None) for k in range(16)]
    batch, db_all = [], {}
    for d in range(n_distros):
        tasks, db = random_tasks(rng, rng.choice([0, 1, 40, 300, 700]))
        for t in tasks:
            t.id = f"d{d}-{t.id}"
            for dep in t.depends_on:
                if dep.task_id.startswith("t"):
                    dep.task_id = f"d{d}-{dep.task_id}"
            t.project = rng.choice([f"p{rng.randrange(16)}", f"p{rng.randrange(16)}", "p1", "p1", "nowhere"])
            t.activated = rng.random() < 0.9
            t.status = rng.choice(["undispatched"] * 8 + ["started", "success"])
            t.execution_platform = rng.choice(["", "", "host", "container"])
            t.unattainable_dependency = rng.random() < 0.1
        dist = M.Distro(id=f"d{d}", valid_projects=rng.choice([[], [], ["p1"], ["p1", "p3", "ghost"], ["ghost"]]),
                        dispatcher_settings=M.DispatcherSettings(version=rng.choice(["", "revised", "revised-with-dependencies"])))
        batch.append((dist, tasks))
        db_all.update(db)
    return batch, refs, db_all


@pytest.mark.parametrize("finder", ["legacy", "alternate"])
@pytest.mark.parametrize("case", FINDER["cases"], ids=lambda c: c["name"])
def test_task_finder_cases(engine, case, finder):
    """What scheduler/task_finder_test.go asserts, through evg_find_runnable_batch."""
    d, tasks, refs = G.finder_case(case)
    got = [t.id for t in S.find_runnable_tasks([(d, tasks)], refs, finder=finder, engine=engine)[0]]
    if "expect_len" in case:
        assert len(got) == case["expect_len"]
    if "expect_ids" in case:
        assert sorted(got) == sorted(case["expect_ids"])
    assert got == [t.id for t in O.find_runnable(d, tasks, refs, finder=finder)]  # same tasks, same order


@pytest.mark.parametrize("seed", range(6))
def test_task_finders_agree_on_fuzzy_tasks(engine, seed):
    """TaskFinderComparisonSuite (task_finder_test.go:309-334) on its fuzzy generator: every finder returns the same ids."""
    import random
    tasks = G.random_finder_tasks(random.Random(seed))
    refs = [M.ProjectRef(**r) for r in FINDER["cases"][-1]["project_refs"]]
    a = [t.id for t in S.LegacyFindRunnableTasks(M.Distro(), tasks, refs, engine=engine)]
    b = [t.id for t in S.AlternateTaskFinder(M.Distro(), tasks, refs, engine=engine)]
    assert a == b == [t.id for t in O.find_runnable(M.Distro(), tasks, refs)]


@pytest.mark.parametrize("finder", ["legacy", "alternate"])
@pytest.mark.parametrize("seed", range(3))
def test_task_finder_parity(engine, seed, finder):
    import random
    batch, refs, db = random_finder_batch(random.Random(70 + seed), 9)
    got = S.find_runnable_tasks(batch, refs, finder=finder, dependency_db=db, engine=engine)
    for (d, tasks), g in zip(batch, got):
        assert [t.id for t in g] == [t.id for t in O.find_runnable(d, tasks, refs, db, finder)]


def test_task_finder_at_scale(engine):
    """2e6 candidates over 3000 distros: device result vs a numpy restatement of the same table (stable compaction)."""
    rng = np.random.default_rng(9)
    D, P = 3000, 64
    sizes = rng.integers(0, 1400, D)
    sizes[7] = 40_000
    off = np.zeros(D + 1, np.int64); np.cumsum(sizes, out=off[1:])
    T = int(off[-1])
    sched = (rng.integers(0, 256, T) | 0x0F * (rng.random(T) < 0.85)).astype(np.uint8)
    project = rng.integers(-1, P, T).astype(np.int32)
    pflags = rng.integers(0, 16, P).astype(np.uint8) | np.uint8(1) * (rng.random(P) < 0.7).astype(np.uint8)
    nvalid = np.where(rng.random(D) < 0.3, rng.integers(1, 6, D), 0)
    voff = np.zeros(D + 1, np.int64); np.cumsum(nvalid, out=voff[1:])
    vidx = rng.integers(-1, P, int(voff[-1])).astype(np.int32)
    finder = rng.integers(0, 3, D).astype(np.uint8)
    n_dep = rng.integers(0, 3, T)
    doff = np.zeros(T + 1, np.int64); np.cumsum(n_dep, out=doff[1:])
    E = int(doff[-1])
    deps = soa.DepsTable(doff, rng.integers(0, 3, E).astype(np.uint8), rng.integers(0, 4000, E).astype(np.int32),
                         rng.integers(0, 4, E).astype(np.uint8), rng.integers(0, 3, T).astype(np.uint8) | (4 * (rng.random(T) < 0.2)).astype(np.uint8),
                         (rng.random(T) < 0.1).astype(np.uint8) | ((rng.random(T) < 0.1).astype(np.uint8) << 1),
                         rng.integers(0, 3, 4000).astype(np.uint8))
    table = soa.RunnableTable(off, sched, project, pflags, voff, vidx, finder, deps)
    runnable, count = engine.find_runnable_batch(table)
    runnable, count = runnable.copy(), count.copy()
    # numpy restatement
    st = np.where(deps.dep_kind == 0, deps.task_state[deps.dep_ref], deps.ext_state[deps.dep_ref])
    status, blocked = st & 3, (st & 4) != 0
    sat = np.where(deps.dep_want == 0, status == 0, np.where(deps.dep_want == 1, status == 1,
                   np.where(deps.dep_want == 2, (status < 2) | blocked, False)))
    sat &= deps.dep_kind != 2
    unsat = np.add.reduceat(np.concatenate([(~sat).astype(np.int64), [0]]), np.minimum(doff[:-1], E))[:T] * (n_dep > 0)
    walk_ok = unsat == 0
    met_legacy = walk_ok | (deps.task_pre != 0)
    dist_of = np.repeat(np.arange(D), sizes)
    q = ((sched & 1) != 0) & ((sched & 2) != 0) & ((sched & 4) != 0) & ((sched & 8) != 0) & (((sched & 16) == 0) | ((sched & 32) != 0))
    pf = pflags[np.maximum(project, 0)]
    can = (((pf & 1) != 0) | (((sched & 64) != 0) & ((pf & 2) != 0))) & ((pf & 4) == 0) & ~(((sched & 128) != 0) & ((pf & 8) != 0))
    keep = q & (project >= 0) & can
    has_valid = nvalid[dist_of] > 0
    in_valid = np.zeros(T, bool)
    for d in np.nonzero(nvalid)[0]:
        a, b = off[d], off[d + 1]
        in_valid[a:b] = np.isin(project[a:b], vidx[voff[d]:voff[d + 1]])
    keep &= ~has_valid | in_valid
    f = finder[dist_of]
    keep &= (f == 0) | ((f == 1) & met_legacy) | ((f == 2) & walk_ok)
    assert np.array_equal(count, np.add.reduceat(np.concatenate([keep.astype(np.int64), [0]]), np.minimum(off[:-1], T))[:D] * (sizes > 0))
    local = np.arange(T) - off[dist_of]
    want = np.full(T, -1, np.int32)
    pos = np.cumsum(keep) - keep  # exclusive, global
    base_pos = pos[np.minimum(off[:-1], T - 1)]
    dst = off[dist_of] + pos - base_pos[dist_of]
    want[dst[keep]] = local[keep]
    assert np.array_equal(runnable, want)
    assert engine.last_launch_count() == 2  # k_deps_met + k_runnable


# ---------------------------------------------------------------- expected-duration statistics (SURVEY.md §8f.2)
def test_expected_duration_kat(engine):
    """model/task/expected_duration_test.go:14-69 through evg_expected_durations_batch."""
    for case in G.load("expected_duration.json")["cases"]:
        tasks = [G.make_task(t, 0, 0) for t in case["tasks"]]
        got = S.get_expected_durations_for_window(tasks, case["window_start"], case["window_end"], engine=engine)
        e = case["expect"]
        mean, std = got[tuple(e["key"])]
        assert len(got) == 1 and mean == e["mean_ns"] and abs(std - e["stddev_ns"]) <= e["stddev_delta_ns"]


@pytest.mark.parametrize("seed", range(3))
def test_expected_duration_parity(engine, seed):
    """Random finished-task history: bit-equal to the oracle's canonical roundings, and within 1e-12 (relative) of the
    exactly rounded population standard deviation."""
    import random
    rng = random.Random(90 + seed)
    now = 1_800_000_000 * 10 ** 9
    tasks = []
    for i in range(4000):
        taken = rng.choice([rng.randrange(10 ** 9, 4 * 3600 * 10 ** 9), rng.randrange(1, 10 ** 6), 7 * 10 ** 9])
        tasks.append(M.Task(id=f"t{i}", project=f"p{rng.randrange(3)}", build_variant=f"bv{rng.randrange(4)}",
                            display_name=f"n{rng.randrange(25)}", status=rng.choice(["success", "failed", "failed", "undispatched", "started"]),
                            timed_out=rng.random() < 0.05, time_taken=taken,
                            start_time=now - rng.randrange(0, 9 * 24 * 3600 * 10 ** 9), finish_time=now - rng.randrange(-10 ** 9, 10 ** 12)))
    w0, w1 = now - 7 * 24 * 3600 * 10 ** 9, now
    got = S.get_expected_durations_for_window(tasks, w0, w1, engine=engine)
    want = O.expected_durations_for_window(tasks, w0, w1)
    assert set(got) == set(want)
    for k, (n, mean, std, exact) in want.items():
        assert got[k] == (mean, std), k
        assert abs(std - exact) <= 1e-12 * max(exact, 1.0) + 1e-3


def test_expected_duration_at_scale(engine):
    """8e6 rows over 200k keys against numpy (float64 two-pass): means equal, standard deviations within 1e-9 relative."""
    rng = np.random.default_rng(3)
    R, K = 8_000_000, 200_000
    key = rng.integers(0, K, R).astype(np.int32)
    taken = rng.integers(10 ** 9, 3 * 3600 * 10 ** 9, R)
    flags = (rng.random(R) < 0.9).astype(np.uint8) | ((rng.random(R) < 0.05).astype(np.uint8) << 1)
    now = 10 ** 18
    start = now - rng.integers(0, 8 * 24 * 3600 * 10 ** 9, R)
    finish = start + taken
    rows = soa.DurationRows(key, taken, start, finish, flags, K, now - 7 * 24 * 3600 * 10 ** 9, now)
    st = engine.expected_durations_batch(rows).copy()
    ok = ((flags & 1) != 0) & ((flags & 2) == 0) & (start > rows.window_start_ns) & (finish <= rows.window_end_ns)
    cnt = np.bincount(key[ok], minlength=K)
    ssum = np.bincount(key[ok], weights=taken[ok].astype(np.float64), minlength=K)
    assert np.array_equal(st["count"], cnt)
    have = cnt > 0
    mean = ssum[have] / cnt[have]
    assert np.allclose(st["mean_ns"][have], mean, rtol=1e-12, atol=0)
    dev = taken[ok].astype(np.float64) - (ssum / np.maximum(cnt, 1))[key[ok]]
    var = np.bincount(key[ok], weights=dev * dev, minlength=K)[have] / cnt[have]
    assert np.allclose(st["stddev_ns"][have], np.sqrt(var), rtol=1e-9, atol=1e-3)
    assert not st["mean_ns"][~have].any() and not st["stddev_ns"][~have].any()
    assert engine.last_launch_count() == 3


def test_bad_arguments_are_errors(engine):
    w = synth.make(np.array([10]), 1)
    bad = copy.deepcopy(w)
    bad.distros.task_off[-1] = 11
    with pytest.raises(L.EvgError) as e:
        engine.plan_batch(bad.tasks, bad.distros, w.now)
    assert e.value.code == L.EVG_ERR_INVALID
    big = soa.DistroTable(np.array([0, L.MAX_TASKS_PER_DISTRO + 1]), np.array([0, 0]),
                          np.zeros(1, L.DISTRO_CFG_DTYPE), np.zeros(0, np.int32)).normalize()
    t = w.tasks
    with pytest.raises(L.EvgError):
        engine.plan_batch(t, big, w.now)


def test_resident_rerun_is_idempotent(engine):
    w = synth.config(3, 0.02)
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now)
    a_po, a_ao = copy.deepcopy(engine.download())  # result buffers are reused by the next call
    engine.run(w.now)
    engine.run(w.now)
    b_po, b_ao = engine.download()
    assert np.array_equal(a_po.order, b_po.order) and np.array_equal(a_po.info, b_po.info)
    assert np.array_equal(a_ao.result, b_ao.result)
    assert engine.last_launch_count() > 0


def test_all_routes_in_one_tick(engine):
    """One tick holding every planner route at once -- warp, the three on-chip classes at their boundaries, the
    general path -- with task groups, GroupVersions, dependencies and hosts: each distro against the oracle."""
    sizes = np.array([3, 31, 32, 33, 0, 900, 1024, 1025, 4000, 4096, 4097, 12288, 12289, 20000, 1, 7])
    w = synth.make(sizes, 91, tg_frac=0.12, unmet_dep_frac=0.03, met_dep_frac=0.02, group_versions_frac=0.25,
                   custom_factor_frac=0.4, zipf_priority=True, includes_dependencies=True, n_hosts=400,
                   providers=(0.6, 0.2, 0.2))
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao)
    po, _ = run(engine, w, breakdown=True)
    parity.check_against_oracle(w, po, None)


def test_resident_reruns_follow_the_clock(engine):
    """Upload once, run at three different clocks (evg_run_resident): every run equals the oracle at that clock."""
    w = synth.make(np.array([5000, 40, 13000, 700]), 92, tg_frac=0.1, met_dep_frac=0.02, n_hosts=60)
    engine.upload(w.tasks, w.distros, w.hosts)
    for now in (w.now, w.now + 3 * 3600 * 10 ** 9, w.now + 9 * 24 * 3600 * 10 ** 9):
        engine.run(now)
        po, ao = engine.download()
        w2 = copy.copy(w)
        w2.now = now
        parity.check_against_oracle(w2, po, ao)


def test_bound_result_buffer_receives_the_rows(engine):
    """evg_bind_result_buffer: the allocator writes its rows into a caller-owned device buffer (the all-gather
    send buffer) -- same bytes as the context-owned one."""
    import torch
    w = synth.config(3, 0.01)
    po, ao = run(engine, w)
    want = ao.result.copy()
    D = w.distros.n_distros
    buf = torch.zeros((D + 5) * 16, dtype=torch.uint8, device="cuda:0")
    try:
        engine.bind_result_buffer(buf.data_ptr(), D + 5)
        po2, ao2 = run(engine, w)
        got = np.frombuffer(buf.cpu().numpy().tobytes(), dtype=L.ALLOC_RESULT_DTYPE)
        assert np.array_equal(got[:D], want) and not got[D:].view(np.uint8).any()
        assert np.array_equal(ao2.result, want)  # the host copy comes from the bound buffer too
        with pytest.raises(L.EvgError):
            engine.bind_result_buffer(buf.data_ptr(), D - 1)
            run(engine, w)
    finally:
        engine.bind_result_buffer(0, 0)
    po3, ao3 = run(engine, w)
    assert np.array_equal(ao3.result, want)


def test_alloc_only_call_matches_the_fused_tick(engine):
    """evg_alloc_batch on the queue infos a planner call returned (the reference's two-job topology) gives the same
    decisions as the fused tick, including a distro with thousands of task groups (block-per-distro allocator)."""
    w = synth.make(np.array([60000, 300, 5, 9000]), 93, tg_frac=0.15, n_hosts=500, providers=(0.7, 0.2, 0.1))
    po, ao = run(engine, w)
    want, want_status = ao.result.copy(), ao.status.copy()
    qinfo, ginfo = po.info.copy(), po.group_info.copy()
    ginfo["count_free"] = 0
    ginfo["count_required"] = 0
    assert int(np.diff(w.distros.group_off).max()) > 1024
    ao2, g2 = engine.alloc_batch(w.hosts, qinfo, ginfo, w.distros.group_off, w.now)
    assert np.array_equal(ao2.result, want) and np.array_equal(ao2.status, want_status)
    assert np.array_equal(g2["count_required"], po.group_info["count_required"])
    assert np.array_equal(g2["count_free"], po.group_info["count_free"])


def test_pipelined_one_shot_equals_resident(engine):
    """Ticks of >= 2^21 tasks take the chunked H2D / kernels / D2H pipeline inside evg_plan_and_alloc_batch;
    its results must equal the upload -> run -> download path bit for bit."""
    rng = synth.Rng(77)
    sizes = rng.integers(330, 2000, 12000)
    w = synth.make(sizes, 78, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.02, met_dep_frac=0.01,
                   custom_factor_frac=0.3, includes_dependencies=True, n_hosts=3000, providers=(0.7, 0.2, 0.1))
    assert w.n_tasks >= 2 ** 21
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now)
    a_po, a_ao = copy.deepcopy(engine.download())
    b_po, b_ao = engine.plan_and_alloc_batch(w.tasks, w.distros, w.hosts, w.now)
    for f in ("order", "total_value", "info", "group_info"):
        assert np.array_equal(getattr(a_po, f), getattr(b_po, f)), f
    assert np.array_equal(a_ao.result, b_ao.result) and np.array_equal(a_ao.status, b_ao.status)
    parity.check_against_oracle(w, b_po, b_ao, distros=[0, 1, 2, 150, 329])


# ---------------------------------------------------------------- full-size configs
@pytest.mark.parametrize("k", [3, 4, 5])
def test_configs_full_distro_counts(engine, k):
    """BASELINE configs[2..4] at their full DISTRO counts (10k / 10k / 100k distros; the "N tasks" of configs[2]
    and [3] read as the tick total, see SURVEY.md §8d), every distro compared bit-exactly with the oracle."""
    w = synth.config(k, 1.0)
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao, threads=32)


def test_config3_per_distro_reading_scaled(engine):
    """configs[2] read per distro (100k tasks in ONE distro queue): 24 such distros take the general
    (global-memory) path; oracle on all of them."""
    w = synth.config(3, 0.0024, each=True)
    assert w.distros.n_distros == 24 and w.n_tasks == 2_400_000
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao, threads=32)


# ---------------------------------------------------------------- full-size properties
def test_c2_full_size_properties(engine):
    """BASELINE configs[1] at full size: 1000 distros x 10k tasks (1e7 tasks).  The oracle checks a
    sample of distros bit-exactly; the rest is covered by the size-independent invariants."""
    w = synth.config(2, 1.0)
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao, distros=[0, 1, 499, 998, 999])


def test_c2_full_size_every_distro_every_tick(engine):
    """The same tick, ALL 1000 distros bit-exact against the oracle, eight resident ticks in a row.  A staging race in
    k_plan_cta (a shared-memory slot refilled by TMA before a lagging warp's loads had read it) corrupted one warp's
    tasks in roughly one CTA out of ten thousand: invisible to a handful of sampled distros or to a single tick."""
    w = synth.config(2, 1.0)
    job = O.SoAJob(w.tasks, w.distros, w.hosts, None)
    ref = job.run(w.now, 32)
    engine.upload(w.tasks, w.distros, w.hosts)
    for tick in range(8):
        engine.run(w.now)
        po, ao = engine.download()
        k = parity.first_diff(po.order, ref["order"])
        assert k < 0, f"tick {tick}: order differs at table row {k} (distro {int(np.searchsorted(w.distros.task_off, k, side='right')) - 1})"
        assert parity.first_diff(po.total_value, ref["total_value"]) < 0, f"tick {tick}: TotalValue differs"
        assert np.array_equal(ao.result["new_hosts"], ref["new_hosts"]) and np.array_equal(ao.result["free_hosts"], ref["free_hosts"])


# ---------------------------------------------------------------- round 2: second-generation planners
def test_cta_class_boundaries(engine):
    """Sizes on both sides of every k_plan_cta class (384 / 1280 / 5120 / 10240 tasks) and of the k_plan_smem class above
    it, with task groups only (the shape k_plan_cta plans) -- and the same sizes with in-queue dependencies, which
    must be routed to k_plan_smem / the general path instead."""
    sizes = np.array([33, 1279, 1280, 1281, 5119, 5120, 5121, 10239, 10240, 10241, 12288, 12289, 64, 0, 1, 383, 384, 385, 129])
    w = synth.make(sizes, 201, zipf_priority=True, tg_frac=0.15, custom_factor_frac=0.4, n_hosts=150, providers=(0.7, 0.2, 0.1))
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao)
    w = synth.make(sizes, 202, zipf_priority=True, tg_frac=0.15, met_dep_frac=0.02, unmet_dep_frac=0.02,
                   includes_dependencies=True, n_hosts=150)
    po, ao = run(engine, w)
    parity.check_against_oracle(w, po, ao)


def test_sparse_classes_on_their_own_kernels(engine, monkeypatch):
    """A k_plan_smem class of 1025+ task distros that cannot fill the GPU is planned by the general path
    (EVG_SPARSE_CLASS, default 64).  With the rule switched off every class runs on its own kernel: both
    routings must give the oracle's answer on the same ticks."""
    sizes = np.array([33, 1023, 1025, 4095, 4096, 4097, 10241, 12288, 12289, 700, 2500, 9000])
    for seed, kw in ((211, dict(met_dep_frac=0.03, unmet_dep_frac=0.02, includes_dependencies=True)),
                     (212, dict(group_versions_frac=1.0)), (213, dict(met_dep_frac=0.02, group_versions_frac=0.5))):
        w = synth.make(sizes, seed, zipf_priority=True, tg_frac=0.15, n_hosts=80, **kw)
        for rule in ("0", "64"):
            monkeypatch.setenv("EVG_SPARSE_CLASS", rule)
            po, ao = run(engine, w)
            parity.check_against_oracle(w, po, ao)
            pb, _ = run(engine, w, breakdown=True)
            ref = parity.check_against_oracle(w, pb, None)
            assert np.array_equal(pb.breakdown, ref["breakdown"])  # the general path's breakdown reads the unit table
    monkeypatch.delenv("EVG_SPARSE_CLASS")


def test_cta_misaligned_distro_starts(engine):
    """TMA tiles start at multiples of four tasks; distros start anywhere.  Every start residue mod 4, first and
    last distro of the table, sizes around one and two tiles of each class."""
    sizes = np.array([1, 510, 513, 3, 127, 129, 2, 255, 257, 5, 1023, 1025, 6, 2049, 9999, 7, 10240])
    w = synth.make(sizes, 203, tg_frac=0.1, zipf_priority=True, n_hosts=60)
    assert len({int(x) % 4 for x in w.distros.task_off[:-1]}) == 4
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao)


def test_cta_hands_back_what_it_cannot_hold(engine):
    """Distros k_plan_cta starts and then hands back to k_plan_smem on the device: TotalValue beyond 32 bits,
    TaskGroupOrder >= 64 or repeated inside a group, more task-group tasks than its work list holds -- next to
    distros it keeps, in one tick."""
    sizes = np.array([9000, 3000, 9000, 700, 4000, 9000, 2000])
    w = synth.make(sizes, 204, tg_frac=0.12, zipf_priority=True, n_hosts=70)
    toff, t = w.distros.task_off, w.tasks
    w.distros.cfg["patch_time_in_queue_factor"][0] = 100      # distro 0: values beyond 2^32
    w.distros.cfg["generate_task_factor"][0] = 100
    w.distros.cfg["expected_runtime_factor"][0] = 100
    t.priority[toff[0]:toff[1]:5] = 30000
    t.flags[toff[0]:toff[1]:3] |= L.EVG_TF_GENERATE
    t.task_group_order[np.arange(toff[1], toff[2])[::4]] = 70  # distro 1: order beyond the presence mask
    t.task_group_order[toff[2]:toff[3]] = np.minimum(t.task_group_order[toff[2]:toff[3]], 2)  # distro 2: duplicates
    w2 = synth.make(np.array([4000]), 205, tg_frac=0.6, zipf_priority=True)  # distro 4's shape: 60 % task-group tasks
    po, ao = run(engine, w)
    assert int(po.total_value[toff[0]:toff[1]].max()) > 2 ** 32
    parity.check_against_oracle(w, po, ao)
    po2, _ = run(engine, w2)
    parity.check_against_oracle(w2, po2, None)


def test_cta_digit_widths(engine):
    """Value ranges from one value (no pass) through every pass count of the 10/9/8-bit digit classes."""
    for seed, prio_step, factor in ((206, 0, 0), (207, 1, 0), (208, 50, 20), (209, 1000, 100)):
        w = synth.make(np.array([10000, 5000, 1200, 300]), seed, tg_frac=0.05, custom_factor_frac=0.0)
        if prio_step == 0:  # every task identical: a single TotalValue, ties broken by input order only
            t = w.tasks
            t.priority[:] = 0; t.expected_ns[:] = 600 * 10 ** 9; t.queue_basis_ns[:] = w.now; t.num_dependents[:] = 0
            t.flags[:] = L.EVG_TF_DEPS_MET; t.group_id[:] = -1
            w.distros.group_off[:] = 0
            w.distros.group_max_hosts = w.distros.group_max_hosts[:0]
        else:
            w.tasks.priority[:] = (np.arange(w.n_tasks) % 7) * prio_step
            for f in ("patch_time_in_queue_factor", "mainline_time_in_queue_factor", "expected_runtime_factor"):
                w.distros.cfg[f] = factor
        po, _ = run(engine, w)
        parity.check_against_oracle(w, po, None)


def test_one_million_task_distro(engine):
    """A single queue of a million tasks (configs[3]'s per-distro reading) with task groups and in-queue
    dependencies, bit-exact against the oracle: ~490 general-path tiles, the 2^21-1 index space half used."""
    w = synth.make(np.array([1_000_000, 17]), 210, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.03, met_dep_frac=0.01,
                   includes_dependencies=True, n_hosts=300)
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao, threads=32)


def test_general_path_shapes(engine):
    """General-path distros of every kind in one tick: plain (identity pre-arrangement inside a tick that needs
    e[] elsewhere), task groups, GroupVersions, dependency edges, a value range beyond 32 bits (two key words),
    a single repeated value (no sort pass), start residues mod 4."""
    sizes = np.array([13001, 1, 20003, 2, 15000, 3, 14001, 30000])
    w = synth.make(sizes, 211, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.03, met_dep_frac=0.02,
                   group_versions_frac=0.0, includes_dependencies=True, n_hosts=100)
    toff, t = w.distros.task_off, w.tasks
    w.distros.cfg["group_versions"][2] = 1
    for f in ("patch_time_in_queue_factor", "generate_task_factor", "expected_runtime_factor"):
        w.distros.cfg[f][4] = 100
    t.priority[toff[4]:toff[5]:7] = 100000
    t.flags[toff[4]:toff[5]:3] |= L.EVG_TF_GENERATE
    po, ao = run(engine, w)
    assert int(po.total_value[toff[4]:toff[5]].max() - po.total_value[toff[4]:toff[5]].min()) > 2 ** 33
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao)
    # no multi-member unit anywhere: the scan-free placement
    w = synth.make(np.array([40000, 13000]), 212, tg_frac=0.0, zipf_priority=True)
    po, _ = run(engine, w)
    parity.check_against_oracle(w, po, None)
    t = w.tasks
    t.priority[:] = 0; t.expected_ns[:] = 600 * 10 ** 9; t.queue_basis_ns[:] = w.now; t.num_dependents[:] = 0
    t.flags[:] = L.EVG_TF_DEPS_MET
    po, _ = run(engine, w)
    assert np.array_equal(po.order[:40000], np.arange(40000))
    parity.check_against_oracle(w, po, None)


def test_config3_each_bigger_sample(engine):
    """configs[2] per-distro reading at 100 distros x 100k tasks (1e7 tasks through the general path): invariants on
    everything, the oracle on a sample."""
    w = synth.config(3, 0.01, each=True)
    assert w.n_tasks == 10_000_000
    po, ao = run(engine, w)
    parity.check_properties(w, po, ao)
    parity.check_against_oracle(w, po, ao, distros=[0, 1, 50, 99], threads=32)


def test_upload_device_equals_upload(engine):
    """evg_upload_device: task columns that already live in device memory are planned in place."""
    import torch
    w = synth.make(np.array([9000, 40, 15000, 3, 700, 2000]), 213, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.02,
                   met_dep_frac=0.02, includes_dependencies=True, n_hosts=80)
    po, ao = run(engine, w)
    want = copy.deepcopy((po, ao))
    keep, cols = [], {}
    names = [n for n, _ in w.tasks.COLUMNS] + ["dep_off", "dep_idx"]
    for name in names:
        a = getattr(w.tasks, name)
        pad = np.zeros(a.shape[0] + 8, dtype=a.dtype)
        pad[:a.shape[0]] = a
        v = pad.view(np.int32) if pad.dtype == np.uint32 else pad
        tdev = torch.from_numpy(v).to("cuda:0")
        keep.append(tdev)
        cols[name] = tdev.data_ptr()
    torch.cuda.synchronize()
    engine.upload_device(cols, w.n_tasks, w.distros, w.hosts, n_edges=w.tasks.n_edges)
    engine.run(w.now)
    po2, ao2 = engine.download()
    for f in ("order", "total_value", "info", "group_info"):
        assert np.array_equal(getattr(want[0], f), getattr(po2, f)), f
    assert np.array_equal(want[1].result, ao2.result)
    engine.upload(w.tasks, w.distros, w.hosts)  # the context owns its columns again
    engine.run(w.now)
    po3, _ = engine.download()
    assert np.array_equal(want[0].order, po3.order)
    del keep


@pytest.mark.parametrize("finder", ["legacy", "alternate"])
def test_planner_consumes_the_finders_device_output(engine, finder):
    """evg_plan_from_finder: candidates in, ranked queues out, with the finder's verdict, the dependency predicate and the
    compaction of the planner's columns all on the device -- equal to the route through the host (find_runnable_tasks ->
    the kept tasks marshalled again -> plan_distros) on ranked ids, TotalValue and every DistroQueueInfo field."""
    import random
    rng = random.Random(23)
    NOWT = synth.NOW_NS
    batch, refs, db = random_finder_batch(rng, 9)
    big, db2 = __import__("test_host_logic").random_tasks(rng, 15000)  # a general-path queue among the small ones
    for t in big:
        t.id = "big-" + t.id
        for dep in t.depends_on:
            if dep.task_id.startswith("t"):
                dep.task_id = "big-" + dep.task_id
        t.project = "p1"
    batch.append((M.Distro(id="big"), big)); db.update(db2)
    # a candidate the finder drops is still a task document: the host route finds it in the database (task.go:632-671 reads
    # missing dependencies from the collection), the device route sees it in the candidate table -- same status either way
    db.update({t.id: t for _, ts in batch for t in ts})
    host_side = copy.deepcopy(batch)
    kept = S.find_runnable_tasks(host_side, refs, finder=finder, dependency_db=db, engine=engine)
    want = S.plan_distros([(d, k) for (d, _), k in zip(host_side, kept)], NOWT, engine=engine, dependency_db=db, breakdown=False)
    got = S.plan_candidates(copy.deepcopy(batch), refs, NOWT, finder=finder, dependency_db=db, engine=engine)
    n_kept = 0
    for (wr, wi), (gr, gi) in zip(want, got):
        assert [t.id for t in gr] == [t.id for t in wr]
        assert [t.sorting_value_breakdown.total_value for t in gr] == [t.sorting_value_breakdown.total_value for t in wr]
        n_kept += len(wr)
        for f in ("length", "length_with_dependencies_met", "count_dep_filled_merge_queue_tasks", "expected_duration",
                  "max_duration_threshold", "count_duration_over_threshold", "duration_over_threshold", "count_wait_over_threshold"):
            assert getattr(gi, f) == getattr(wi, f), f
        every = lambda infos: sorted((g.name, g.count, g.max_hosts, g.expected_duration, g.count_duration_over_threshold,  # noqa: E731
                                      g.count_wait_over_threshold) for g in infos)
        assert every(gi.task_group_infos) == every(wi.task_group_infos)
    assert 2000 < n_kept < sum(len(t) for _, t in batch)


def test_plan_from_finder_edges_of_the_input(engine):
    """evg_plan_from_finder on empty and degenerate inputs: no candidates, distros whose candidates are all dropped,
    a single kept task, candidates without any in-queue edge."""
    NOWT = synth.NOW_NS
    refs = [M.ProjectRef(id="p", enabled=True)]
    def task(i, **kw):
        return M.Task(id=f"t{i}", project="p", version="v", build_variant="bv", distro_id="d", activated=True, status="undispatched",
                      requester=M.REPOTRACKER_VERSION_REQUESTER, priority=1 + i % 3, expected_duration=(1 + i % 7) * M.MINUTE,
                      activated_time=NOWT - (1 + i) * M.MINUTE, scheduled_time=NOWT - M.HOUR, **kw)
    # no candidates at all, one and three distros
    for batch in ([(M.Distro(id="d"), [])], [(M.Distro(id=f"d{k}"), []) for k in range(3)]):
        got = S.plan_candidates(batch, refs, NOWT, engine=engine)
        assert [(len(r), i.length) for r, i in got] == [(0, 0)] * len(batch)
    # everything dropped in one distro (inactive), one task kept in another, 40 kept without edges in a third
    batch = [(M.Distro(id="a"), [task(i, ) for i in range(30)]), (M.Distro(id="b"), [task(0)]), (M.Distro(id="c"), [task(i) for i in range(40)])]
    for t in batch[0][1]:
        t.activated = False
    want = S.plan_distros([(d, k) for (d, _), k in zip(batch, S.find_runnable_tasks(copy.deepcopy(batch), refs, engine=engine))],
                          NOWT, engine=engine, breakdown=False)
    got = S.plan_candidates(copy.deepcopy(batch), refs, NOWT, engine=engine)
    assert [len(r) for r, _ in got] == [0, 1, 40]
    for (wr, wi), (gr, gi) in zip(want, got):
        assert [t.id for t in gr] == [t.id for t in wr]
        assert (gi.length, gi.length_with_dependencies_met, gi.expected_duration) == (wi.length, wi.length_with_dependencies_met, wi.expected_duration)


def test_update_tasks_equals_a_fresh_upload(engine):
    """evg_update_tasks: after scattering changed rows into the resident table (every route: tiny, on-chip, general),
    the tick equals the tick of a fresh upload of the edited table and the oracle's; bad row indices are errors."""
    sizes = np.array([20, 700, 3000, 9000, 14000, 1, 40000])
    w = synth.make(sizes, 221, zipf_priority=True, tg_frac=0.12, met_dep_frac=0.02, unmet_dep_frac=0.03, includes_dependencies=True, n_hosts=50)
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now)
    rng = np.random.default_rng(5)
    t = w.tasks
    for round_ in range(3):
        rows = np.sort(rng.choice(t.n_tasks, size=t.n_tasks // 15, replace=False)).astype(np.int64)
        vals = soa.TaskSoA(**{name: getattr(t, name)[rows].copy() for name, _ in t.COLUMNS})
        vals.priority = rng.integers(0, 101, rows.shape[0]).astype(np.int32)
        vals.expected_ns = (vals.expected_ns + rng.integers(0, 10 ** 10, rows.shape[0])).astype(np.int64)
        vals.flags = (vals.flags | np.where(rng.uniform(size=rows.shape[0]) < 0.5, L.EVG_TF_DEPS_MET, 0)).astype(np.uint32)
        vals.wait_basis_ns = (vals.wait_basis_ns - rng.integers(0, 10 ** 12, rows.shape[0])).astype(np.int64)
        vals.num_dependents = rng.integers(0, 30, rows.shape[0]).astype(np.int32)
        for name in ("priority", "expected_ns", "flags", "wait_basis_ns", "num_dependents", "queue_basis_ns", "task_group_order"):
            getattr(t, name)[rows] = getattr(vals, name)
        engine.update_tasks(rows, vals)
        engine.run(w.now)
        po, ao = engine.download()
        parity.check_against_oracle(w, po, ao)  # w.tasks was edited in step: the oracle plans the same table
    with pytest.raises(L.EvgError):
        engine.update_tasks(np.array([t.n_tasks], dtype=np.int64), soa.TaskSoA(**{name: getattr(t, name)[:1].copy() for name, _ in t.COLUMNS}))


def test_two_contexts_two_threads(engine):
    """Entry points are called from arbitrary OS threads (cgo): two contexts planning different ticks at the same
    time, and two threads sharing ONE context (serialised by its lock), all bit-equal to the single-threaded run."""
    import threading
    from evergreen_b200 import scheduler
    ws = [synth.make(np.array([3000, 50, 14000, 900]), 220 + k, tg_frac=0.1, zipf_priority=True, met_dep_frac=0.02, n_hosts=50)
          for k in range(2)]
    want = []
    for w in ws:
        po, ao = engine.plan_and_alloc_batch(w.tasks, w.distros, w.hosts, w.now)
        want.append((po.order.copy(), ao.result.copy()))
    engines = [scheduler.Engine(0), scheduler.Engine(0)]
    errs = []

    def work(k, eng, reps):
        try:
            for _ in range(reps):
                po, ao = eng.plan_and_alloc_batch(ws[k].tasks, ws[k].distros, ws[k].hosts, ws[k].now)
                if not (np.array_equal(po.order, want[k][0]) and np.array_equal(ao.result, want[k][1])):
                    errs.append(f"context {k}: results differ")
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))
    th = [threading.Thread(target=work, args=(k, engines[k], 5)) for k in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    for e in engines:
        e.close()
    assert not errs, errs
    # one context, two threads: raw C-ABI calls interleave, the lock keeps each call whole
    lib = engine.lib
    rcs = []

    def resident(reps):
        for _ in range(reps):
            rcs.append(lib.evg_run_resident(engine.ctx, int(ws[0].now), 0))
    engine.upload(ws[0].tasks, ws[0].distros, ws[0].hosts)
    th = [threading.Thread(target=resident, args=(10,)) for _ in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert rcs == [0] * 20
    po, ao = engine.download()
    assert np.array_equal(po.order, want[0][0]) and np.array_equal(ao.result, want[0][1])


def test_persisted_queue_projection(engine):
    """evg_download_queue (SURVEY.md §8 f.4): TaskQueueItem rows of the first min(length, cap) ranks, projected on the
    device -- equal to gathering the same fields on the host from the full download; the default cap is the
    reference's 10 000 (TaskQueue.Save, model/task_queue.go:216-219)."""
    w = synth.make(np.array([700, 0, 30, 15000, 12000, 3]), 230, zipf_priority=True, tg_frac=0.15, unmet_dep_frac=0.1,
                   includes_dependencies=True, n_hosts=30)
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now)
    po, _ = copy.deepcopy(engine.download())
    toff, goff = w.distros.task_off, w.distros.group_off
    for cap in (0, 50, 1):
        item_off, items = engine.download_queue(cap, toff)
        eff = cap or 10000
        assert np.array_equal(np.diff(item_off), np.minimum(np.diff(toff), eff))
        for d in range(w.distros.n_distros):
            rows = items[int(item_off[d]):int(item_off[d + 1])]
            n = rows.shape[0]
            a = int(toff[d])
            idx = po.order[a:a + n].astype(np.int64)
            assert np.array_equal(rows["task"], po.order[a:a + n])
            assert np.array_equal(rows["total_value"], po.total_value[a:a + n])
            g = a + idx
            assert np.array_equal(rows["priority"], w.tasks.priority[g]) and np.array_equal(rows["expected_ns"], w.tasks.expected_ns[g])
            assert np.array_equal(rows["group_index"], w.tasks.task_group_order[g])
            assert np.array_equal((rows["flags"] & L.EVG_QI_DEPS_MET) != 0, (w.tasks.flags[g] & L.EVG_TF_DEPS_MET) != 0)
            gid = w.tasks.group_id[g]
            want_max = np.where(gid >= 0, w.distros.group_max_hosts[np.clip(int(goff[d]) + gid, 0, None)], 0)
            assert np.array_equal(rows["group_max_hosts"], want_max)
    with pytest.raises(L.EvgError):
        buf = np.zeros(3, dtype=L.QUEUE_ITEM_DTYPE)
        off = np.zeros(w.distros.n_distros + 1, dtype=np.int64)
        L.check(engine.lib.evg_download_queue(engine.ctx, 0, L.ptr(off), L.ptr(buf), 3))


def test_persist_task_queue_mirror(engine):
    """scheduler.PersistTaskQueue / PlanDistro mirrors: TaskQueue documents with the reference's item fields, a
    12 000-task queue truncated to 10 000, a disabled distro cleared instead of planned, the single-task-distro bypass."""
    rng = np.random.default_rng(3)
    def tasks(n, tag):
        return [M.Task(id=f"{tag}{k}", display_name=f"dn{k}", build_variant="bv", project="p", version=f"v{k % 7}",
                       requester=M.PATCH_VERSION_REQUESTER if k % 3 else M.REPOTRACKER_VERSION_REQUESTER, revision=f"r{k % 5}",
                       revision_order_number=k % 11, priority=int(rng.integers(0, 5)), num_dependents=int(rng.integers(0, 3)),
                       activated_time=synth.NOW_NS - int(rng.integers(0, 10 ** 13)), distro_id=tag, activated_by="user",
                       expected_duration=int(rng.integers(1, 60)) * M.MINUTE,
                       depends_on=[M.Dependency("nowhere")] if k % 50 == 7 else []) for k in range(n)]
    da, db = M.Distro(id="a"), M.Distro(id="b")
    ta, tb = tasks(12000, "a"), tasks(40, "b")
    tb_again, tb_third = copy.deepcopy(tb), copy.deepcopy(tb)
    qa, qb = S.persist_task_queues([(da, ta), (db, tb)], synth.NOW_NS, engine=engine)
    assert len(qa.queue) == 10000 and len(qb.queue) == 40 and qa.distro == "a"
    assert qa.distro_queue_info.length == 12000 and qb.distro_queue_info.length == 40
    plan, info = S.PrioritizeTasks(db, tb_again, now=synth.NOW_NS, engine=engine)
    assert [i.id for i in qb.queue] == [t.id for t in plan]
    by_id = {t.id: t for t in tb}
    for it, t in zip(qb.queue, plan):
        src = by_id[it.id]
        assert (it.display_name, it.build_variant, it.requester, it.revision, it.project, it.version, it.activated_by) == \
               (src.display_name, "bv", src.requester, src.revision, "p", src.version, "user")
        assert it.revision_order_number == src.revision_order_number and it.priority == src.priority
        assert it.expected_duration == src.expected_duration and it.dependencies == [d.task_id for d in src.depends_on]
        assert it.dependencies_met == (not src.depends_on)
        assert it.sorting_value_breakdown.total_value == t.sorting_value_breakdown.total_value
    assert all(t.scheduled_time == synth.NOW_NS for t in tb)  # SetTasksScheduledAndDepsMetTime
    assert all((t.dependencies_met_time == synth.NOW_NS) == (not t.depends_on) for t in tb)
    # PlanDistro: disabled distro
    q, cleared = S.PlanDistro(M.Distro(id="x", disabled=True), lambda d: 1 / 0, now=synth.NOW_NS, engine=engine, existing_queue_length=5)
    assert q is None and cleared
    q, cleared = S.PlanDistro(db, lambda d: tb_third, now=synth.NOW_NS, engine=engine)
    assert [i.id for i in q.queue] == [i.id for i in qb.queue] and not cleared
    # units/host_allocator.go:182-184
    assert S.hosts_to_request(M.Distro(id="s", single_task_distro=True), qb.distro_queue_info, 3, lambda: 1 / 0) == \
           (qb.distro_queue_info.length_with_dependencies_met - 3, 0)
    assert S.hosts_to_request(db, qb.distro_queue_info, 3, lambda: (7, 2)) == (7, 2)


def test_device_side_dependency_wiring(engine):
    """evg_upload_with_deps: the device evaluates Task.DependenciesMet and writes the EVG_TF_DEPS_MET bit and the
    stamped wait basis of the resident columns itself -- equal to the host restatement (marshal_tasks
    resolve_deps=True), on tasks, queue info and allocator decisions; the stamps come back for the write-back."""
    import random
    rng = random.Random(17)
    NOWT = synth.NOW_NS
    batch, db = [], {}
    for di in range(4):
        n = [60, 0, 400, 1500][di]
        tasks = []
        for i in range(n):
            t = M.Task(id=f"d{di}t{i}", version=f"v{i % 5}", project="p", build_variant="bv", distro_id=f"d{di}",
                       requester=rng.choice([M.PATCH_VERSION_REQUESTER, M.REPOTRACKER_VERSION_REQUESTER, M.GITHUB_MERGE_REQUESTER]),
                       priority=rng.randrange(3), num_dependents=rng.randrange(3), expected_duration=rng.randrange(1, 90) * M.MINUTE,
                       activated_time=NOWT - rng.randrange(10 ** 13), scheduled_time=rng.choice([M.ZERO_TIME, NOWT - rng.randrange(4 * M.HOUR)]),
                       dependencies_met_time=rng.choice([M.ZERO_TIME, M.ZERO_TIME, NOWT - rng.randrange(3 * M.HOUR)]),
                       override_dependencies=rng.random() < 0.05)
            for _ in range(rng.choice([0, 0, 0, 1, 2])):
                target = rng.choice([f"d{di}t{rng.randrange(n)}", f"ext{rng.randrange(8)}", "missing"])
                t.depends_on.append(M.Dependency(target, status=rng.choice(["", "success", "failed", "*"]),
                                                 finished_at=rng.choice([M.ZERO_TIME, 0, NOWT - rng.randrange(2 * M.HOUR)])))
            tasks.append(t)
        d = M.Distro(id=f"d{di}", dispatcher_settings=M.DispatcherSettings(M.DISPATCHER_VERSION_REVISED_WITH_DEPENDENCIES if di % 2 else ""))
        batch.append((d, tasks))
    for k in range(8):
        db[f"ext{k}"] = M.Task(id=f"ext{k}", status=rng.choice([M.TASK_SUCCEEDED, M.TASK_FAILED, "started"]))
    host_side = copy.deepcopy(batch)
    soa_h, table_h, _ = soa.marshal_tasks(host_side, NOWT, db, resolve_deps=True)
    po_h = copy.deepcopy(engine.plan_batch(soa_h, table_h, NOWT))
    soa_d, table_d, _ = soa.marshal_tasks(batch, NOWT, db)
    assert not (soa_d.flags & L.EVG_TF_DEPS_MET).any()
    engine.upload_with_deps(soa_d, table_d, None, soa.marshal_deps(batch, db), soa.marshal_dep_finished(batch), NOWT)
    engine.run(NOWT)
    po_d, _ = engine.download(want_alloc=False)
    for f in ("order", "total_value", "info", "group_info"):
        assert np.array_equal(getattr(po_h, f), getattr(po_d, f)), f
    met, stamp = engine.download_deps()
    want_met = [(f & L.EVG_TF_DEPS_MET) != 0 for f in soa_h.flags.tolist()]
    assert met.astype(bool).tolist() == want_met
    flat_h = [t for _, ts in host_side for t in ts]
    flat_d = [t for _, ts in batch for t in ts]
    n_stamped = 0
    for th, td, s in zip(flat_h, flat_d, stamp.tolist()):
        if th.dependencies_met_time != td.dependencies_met_time:  # the host restatement stamped the task: so did the device
            assert s == th.dependencies_met_time
            n_stamped += 1
        else:
            assert s == M.ZERO_TIME
    assert n_stamped > 20
    # the reference-shaped mirrors take the same route and write the stamps back
    plan, info = S.PrioritizeTasks(batch[2][0], batch[2][1], now=NOWT, engine=engine, dependency_db=db)
    assert [t.dependencies_met_time for t in batch[2][1]] == [t.dependencies_met_time for t in host_side[2][1]]
    assert info.length_with_dependencies_met == int(po_h.info[2]["length_with_dependencies_met"])


def test_pipelined_one_shot_with_general_path_distros(engine):
    """The chunked one-shot call also carries general-path distros (each chunk runs the general path on its own
    tiles): equal to upload -> run -> download, and to the oracle on a sample."""
    sizes = np.array([60000, 900, 130000, 20, 250000, 13000, 5000, 400000, 70000, 33, 300000, 90000, 512, 450000, 200000, 180000])
    w = synth.make(sizes, 240, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.03, met_dep_frac=0.01, includes_dependencies=True,
                   n_hosts=200, providers=(0.7, 0.2, 0.1))
    assert w.n_tasks >= 2 ** 21
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now)
    a_po, a_ao = copy.deepcopy(engine.download())
    b_po, b_ao = engine.plan_and_alloc_batch(w.tasks, w.distros, w.hosts, w.now)
    for f in ("order", "total_value", "info", "group_info"):
        assert np.array_equal(getattr(a_po, f), getattr(b_po, f)), f
    assert np.array_equal(a_ao.result, b_ao.result) and np.array_equal(a_ao.status, b_ao.status)
    parity.check_properties(w, b_po, b_ao)
    parity.check_against_oracle(w, b_po, b_ao, distros=[0, 1, 2, 3, 5, 8, 9], threads=16)

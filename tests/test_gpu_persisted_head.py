"""The persisted-head tick (evg_run_resident_head): only the first min(length, cap) ranks of every distro are ordered.
Its queue rows, breakdown rows, queue info, group info and allocator result must be the full tick's, and the oracle's."""
import copy

import numpy as np
import pytest

import parity
from evergreen_b200 import _lib as L
from evergreen_b200 import model as M
from evergreen_b200 import scheduler as S
from evergreen_b200 import soa, synth
from oracle import oracle_persist as OP
from test_gpu_handover_parity import NOW, _handover_batch, _oracle_queue, _persist_tasks

pytestmark = pytest.mark.gpu

CAPS = (1, 9999, 10000)


def _tick(engine, w, cap, head, opts=0):
    """One tick on the resident inputs; everything a caller can read after it, copied out of the reused buffers."""
    if head:
        engine.run_head(w.now, cap, opts)
    else:
        engine.run(w.now, opts)
    po, ao = engine.download(ranks=not head)
    bd = bool(opts & L.EVG_OPT_BREAKDOWN)
    q = engine.download_queue(cap, w.distros.task_off, breakdown=bd)
    return {"info": po.info.tobytes(), "ginfo": po.group_info.tobytes(),
            "alloc": None if ao is None else (ao.result.tobytes(), ao.status.tobytes()),
            "off": q[0].copy(), "items": q[1].copy(), "bd": q[2].copy() if bd else None}


def _same(a, b):
    assert np.array_equal(a["off"], b["off"])
    assert a["items"].tobytes() == b["items"].tobytes()
    assert a["info"] == b["info"] and a["ginfo"] == b["ginfo"] and a["alloc"] == b["alloc"]
    if a["bd"] is not None or b["bd"] is not None:
        assert np.array_equal(a["bd"], b["bd"])


def _against_ref(w, got, ref, cap):
    """The head rows against the oracle's first min(length, cap) ranks of every distro."""
    toff, rt = w.distros.task_off, ref["task_off"]
    for d in range(w.distros.n_distros):
        n = min(int(toff[d + 1] - toff[d]), cap or L.EVG_PERSISTED_QUEUE_CAP)
        rows = got["items"][int(got["off"][d]):int(got["off"][d + 1])]
        assert rows.shape[0] == n, d
        ra = int(rt[d])
        assert np.array_equal(rows["task"], ref["order"][ra:ra + n]), d
        assert np.array_equal(rows["total_value"], ref["total_value"][ra:ra + n]), d
        if got["bd"] is not None:
            assert np.array_equal(got["bd"][int(got["off"][d]):int(got["off"][d + 1])], ref["breakdown"][ra:ra + n]), d


def _check_head(engine, w, caps=CAPS, oracle=True):
    """Full tick (checked against the oracle), then for every cap a full and a head tick of the same inputs."""
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now)
    po, ao = copy.deepcopy(engine.download())
    ref = parity.check_against_oracle(w, po, ao) if oracle else None
    for cap in caps:
        full = _tick(engine, w, cap, head=False)
        head = _tick(engine, w, cap, head=True)
        _same(full, head)
        if ref is not None:
            _against_ref(w, head, ref, cap)
    return ref


def _flat(w, priority):
    """Every value of the tick decided by `priority` alone (everything else equal, no task groups or edges)."""
    t = w.tasks
    t.priority[:] = priority
    t.expected_ns[:] = 600 * 10 ** 9
    t.queue_basis_ns[:] = w.now
    t.num_dependents[:] = 0
    t.flags[:] = L.EVG_TF_DEPS_MET
    return w


# ---------------------------------------------------------------- 1. head ranks = full ranks = oracle
def test_mixed_tick_every_route(engine):
    """Warp, k_plan_cta, k_plan_smem and general-path distros in one tick with hosts, task groups and dependencies."""
    sizes = np.array([20, 300, 1200, 5000, 10000, 12288, 0, 12289, 30000, 700, 23000])
    w = synth.make(sizes, 301, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.03, met_dep_frac=0.02,
                   includes_dependencies=True, n_hosts=80)
    _check_head(engine, w)


def test_general_path_units_and_wide_keys(engine):
    """General-path distros with task groups, GroupVersions, in-queue dependency edges, and one whose value range needs
    a second key word."""
    sizes = np.array([13001, 20003, 15000, 14001, 30000])
    w = synth.make(sizes, 302, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.03, met_dep_frac=0.02,
                   includes_dependencies=True, n_hosts=60)
    toff, t = w.distros.task_off, w.tasks
    w.distros.cfg["group_versions"][1] = 1
    for f in ("patch_time_in_queue_factor", "generate_task_factor", "expected_runtime_factor"):
        w.distros.cfg[f][3] = 100
    t.priority[toff[3]:toff[4]:7] = 100000
    t.flags[toff[3]:toff[4]:3] |= L.EVG_TF_GENERATE
    ref = _check_head(engine, w)
    tv = ref["total_value"][int(ref["task_off"][3]):int(ref["task_off"][4])]
    assert int(tv.max() - tv.min()) > 2 ** 33


# ---------------------------------------------------------------- 2. ties at the cut
def test_one_repeated_value(engine):
    """20 000 tasks of one value: theta = 0 and every taken key comes from the tie run (buffer order)."""
    w = _flat(synth.make(np.array([20000, 13000]), 303, tg_frac=0.0), 0)
    _check_head(engine, w)
    engine.run_head(w.now)
    _, items = engine.download_queue(0, w.distros.task_off)
    assert np.array_equal(items["task"][:10000], np.arange(10000))


def test_ties_straddle_and_end_at_the_cut(engine):
    """Three values of ~10 000 tasks each (ties straddle ranks 1, 9 999 and 10 000), and a distro whose top value is
    held by exactly 10 000 tasks (the cut at cap 10 000 falls at the end of that tie run)."""
    rng = np.random.default_rng(7)
    w = synth.make(np.array([30000, 25000]), 304, tg_frac=0.0)
    pri = rng.integers(0, 3, w.n_tasks).astype(np.int32)
    top = rng.permutation(25000)[:10000]
    pri[30000:] = 0
    pri[30000 + top] = 5
    _flat(w, pri)
    _check_head(engine, w)


# ---------------------------------------------------------------- 3. sizes
def test_sizes_around_the_routes(engine):
    """12 288 tasks (on-chip) next to 12 289 (general), a 1M-task distro and empty distros in one tick."""
    sizes = np.array([0, 12288, 12289, 0, 1_000_000, 5, 0])
    w = synth.make(sizes, 305, zipf_priority=True, tg_frac=0.05, unmet_dep_frac=0.02, includes_dependencies=True, n_hosts=30)
    _check_head(engine, w)


@pytest.mark.parametrize("rule", ["0", "64"])
def test_sparse_class_distros_shorter_than_the_cap(engine, monkeypatch, rule):
    """2000- and 10 000-task distros with dependency edges and a few task groups: with EVG_SPARSE_CLASS on they take the
    general path although the head is the whole distro (next to a 25 000-task distro, so the tick selects), with it off
    they stay on-chip."""
    monkeypatch.setenv("EVG_SPARSE_CLASS", rule)
    w = synth.make(np.array([2000, 10000, 25000, 2000, 40]), 306, zipf_priority=True, tg_frac=0.02, met_dep_frac=0.03,
                   unmet_dep_frac=0.02, includes_dependencies=True, n_hosts=20)
    _check_head(engine, w)
    engine.run_head(w.now)
    engine.general_timing_ms()  # the 25 000-task distro


def test_short_general_distros_take_the_full_sort(engine):
    """No general-path distro longer than twice the cap: the head tick sorts them whole and its rows are still the
    full tick's, at every cap."""
    w = synth.make(np.array([12289, 15000, 20000, 700]), 310, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.02,
                   includes_dependencies=True, n_hosts=20)
    _check_head(engine, w, caps=(1, 7500, 9999, 10000))


# ---------------------------------------------------------------- 4. breakdown
def test_breakdown_rows(engine):
    """evg_download_queue_bd after a head run with EVG_OPT_BREAKDOWN = the full run's breakdown at the same ranks = the
    oracle's; on-chip and general-path distros, units of every kind."""
    sizes = np.array([33, 900, 5000, 12289, 26000, 0, 14000])
    w = synth.make(sizes, 307, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.03, met_dep_frac=0.02,
                   group_versions_frac=0.3, includes_dependencies=True, n_hosts=40)
    engine.upload(w.tasks, w.distros, w.hosts)
    engine.run(w.now, L.EVG_OPT_BREAKDOWN)
    po, ao = copy.deepcopy(engine.download(want_breakdown=True))
    ref = parity.check_against_oracle(w, po, ao)
    assert np.array_equal(po.breakdown, ref["breakdown"])
    for cap in CAPS:
        full = _tick(engine, w, cap, head=False, opts=L.EVG_OPT_BREAKDOWN)
        head = _tick(engine, w, cap, head=True, opts=L.EVG_OPT_BREAKDOWN)
        _same(full, head)
        _against_ref(w, head, ref, cap)


def test_persisted_heads_match_the_restatement(engine):
    """persist_task_queue_heads documents = oracle/oracle_persist.py's saved queue, field by field, the whole
    SortingValueBreakdown included; the tasks are stamped as persist_task_queues stamps them."""
    import random
    rng = random.Random(42)
    sizes = (0, 1, 9999, 10001, 13000, 30000)
    db = {"ext-ok": M.Task(id="ext-ok", status="success"), "ext-bad": M.Task(id="ext-bad", status="failed")}
    batch = [(M.Distro(id=f"h{n}"), _persist_tasks(rng, n, f"h{n}-", f"h{n}")) for n in sizes]
    batch[3][0].dispatcher_settings.version = ""  # one distro without IncludesDependencies
    want = [_oracle_queue(d, ts, db) for d, ts in batch]
    dev, dev_full = copy.deepcopy(batch), copy.deepcopy(batch)
    docs = S.persist_task_queue_heads(dev, NOW, engine=engine, dependency_db=db)
    full = S.persist_task_queues(dev_full, NOW, engine=engine, dependency_db=db)
    for (dist, _), doc, w, f in zip(batch, docs, want, full):
        saved = OP.saved_queue(w)
        assert len(doc.queue) == len(saved) == min(len(w), 10000)
        for got, exp in zip(doc.queue, saved):
            assert vars(got) == vars(exp), (dist.id, got.id)
        assert vars(doc.distro_queue_info) == vars(f.distro_queue_info), dist.id
    for (_, a), (_, b) in zip(dev, dev_full):  # ScheduledTime, DependenciesMetTime, ExpectedDuration stamps
        assert [(t.scheduled_time, t.dependencies_met_time, t.expected_duration) for t in a] == \
               [(t.scheduled_time, t.dependencies_met_time, t.expected_duration) for t in b]


# ---------------------------------------------------------------- 5. state
def test_head_run_state_contract(engine):
    w = synth.make(np.array([15000, 300, 0, 4000]), 308, zipf_priority=True, tg_frac=0.1, n_hosts=20)
    engine.upload(w.tasks, w.distros, w.hosts)
    first = _tick(engine, w, 0, head=False)
    engine.run(w.now)
    po1, _ = copy.deepcopy(engine.download())
    engine.run_head(w.now, 100)
    with pytest.raises(L.EvgError) as e:
        engine.download()
    assert e.value.code == L.EVG_ERR_STATE
    engine.download(ranks=False)  # queue info, group info, allocator result
    engine.download_queue(100, w.distros.task_off)
    for cap in (101, 0):
        with pytest.raises(L.EvgError) as e:
            engine.download_queue(cap, w.distros.task_off)
        assert e.value.code == L.EVG_ERR_STATE
    for cap in (-1, 10001):
        with pytest.raises(L.EvgError) as e:
            engine.run_head(w.now, cap)
        assert e.value.code == L.EVG_ERR_INVALID
    with pytest.raises(L.EvgError) as e:  # no EVG_OPT_BREAKDOWN in the last run
        engine.download_queue(100, w.distros.task_off, breakdown=True)
    assert e.value.code == L.EVG_ERR_STATE
    engine.run(w.now)
    with pytest.raises(L.EvgError) as e:
        engine.download_queue(0, w.distros.task_off, breakdown=True)
    assert e.value.code == L.EVG_ERR_STATE
    # full, head, full: the last full run is the first one
    last = _tick(engine, w, 0, head=False)
    _same(first, last)
    engine.run(w.now)
    po2, _ = engine.download()
    assert np.array_equal(po1.order, po2.order) and np.array_equal(po1.total_value, po2.total_value)


def test_head_ticks_follow_update_tasks(engine):
    """Head ticks before and after evg_update_tasks: each equals the full tick of the table as it stands, and the
    oracle on the edited inputs."""
    w = synth.make(np.array([14000, 3000, 25000]), 309, zipf_priority=True, tg_frac=0.1, unmet_dep_frac=0.02,
                   includes_dependencies=True, n_hosts=30)
    _check_head(engine, w, caps=(0,))
    rng = np.random.default_rng(3)
    rows = np.sort(rng.choice(w.n_tasks, size=w.n_tasks // 10, replace=False)).astype(np.int64)
    vals = soa.TaskSoA(**{name: getattr(w.tasks, name)[rows].copy() for name, _ in w.tasks.COLUMNS})
    vals.priority = rng.integers(0, 101, rows.shape[0]).astype(np.int32)
    vals.expected_ns = (vals.expected_ns + rng.integers(0, 10 ** 9, rows.shape[0])).astype(np.int64)
    engine.update_tasks(rows, vals)
    head = _tick(engine, w, 0, head=True)
    full = _tick(engine, w, 0, head=False)
    _same(full, head)
    w.tasks.priority[rows] = vals.priority
    w.tasks.expected_ns[rows] = vals.expected_ns
    engine.run(w.now)
    po, ao = engine.download()
    ref = parity.check_against_oracle(w, po, ao)
    _against_ref(w, head, ref, 10000)


def test_head_tick_after_plan_from_finder(engine):
    """evg_plan_from_finder leaves a resident tick of the kept tasks: a head run on it agrees with a full run."""
    batch, refs, db, datas = _handover_batch(905, True, False)
    batch = copy.deepcopy(batch)
    table = soa.marshal_runnable(batch, refs, "alternate", db)
    if table.deps is None:
        table.deps = soa.marshal_deps(batch, db)
    soa_, dtable, keys = soa.marshal_tasks(batch, NOW, db)
    hosts = soa.marshal_hosts(datas, [k.group_names for k in keys])
    _, count = engine.plan_from_finder(table, soa_, dtable, hosts, soa.marshal_dep_finished(batch), NOW)
    kept_off = np.cumsum([0] + count.tolist())
    assert int(count.max()) > 10240
    out = {}
    for head in (True, False):
        if head:
            engine.run_head(NOW, 0, L.EVG_OPT_BREAKDOWN)
        else:
            engine.run(NOW, L.EVG_OPT_BREAKDOWN)
        po, ao = engine.download(ranks=not head)
        off, items, bd = engine.download_queue(0, kept_off, breakdown=True)
        out[head] = (po.info.tobytes(), po.group_info.tobytes(), ao.result.tobytes(), ao.status.tobytes(), off.copy(),
                     items.tobytes(), bd.copy())
    for a, b in zip(out[True], out[False]):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b

"""CPU restatement of the persisted task queue -- test infrastructure only.

Only tests/ may import this module.

PersistTaskQueue (scheduler/task_queue_persister.go:14-42) turns the planned tasks into one TaskQueueItem each, every
field copied literally from the Task; TaskQueue.Save keeps the first 10 000 (model/task_queue.go:216-219).  The tasks it
reads are the plan's tasks as GetDistroQueueInfo left them (runTunablePlanner, scheduler/scheduler.go:34-51):
  * Task.DependenciesMet ran on every task, and a fresh evaluation that came out met stamped DependenciesMetTime
    (scheduler.go:82-98,161-168; model/task/task.go:632-684), so HasDependenciesMet (task.go:3393-3395) sees it;
  * ExpectedDuration = FetchExpectedDuration().Average, but only for the tasks GetDistroQueueInfo counts
    (scheduler.go:98): all of them, or under IncludesDependencies only those whose dependencies are met -- the others
    keep the ExpectedDuration their document had.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

from evergreen_b200 import model as M
from oracle import oracle as O

SAVED_QUEUE_CAP = 10000  # TaskQueue.Save (model/task_queue.go:216-219)


def _dependencies_met(t: M.Task, cache: Dict[str, M.Task], now: int) -> bool:
    """Task.DependenciesMet (task.go:632-671) with setDependenciesMetTime (:673-684) on a fresh met verdict."""
    if t.has_dependencies_met():
        return True
    if not O._deps_walk(t, cache, shortcut=False):
        return False
    finished = [d.finished_at for d in t.depends_on if not M.is_zero_time(d.finished_at)]
    t.dependencies_met_time = max(finished) if finished else now
    return True


def stamp_planned_tasks(tasks: Sequence[M.Task], includes_dependencies: bool, now: int,
                        dependency_db: Optional[Dict[str, M.Task]] = None) -> Sequence[M.Task]:
    """What GetDistroQueueInfo (scheduler.go:56-143) writes on the plan's tasks, in place.  Its depCache holds the plan's
    tasks; a dependency outside them is looked up in the tasks collection (`dependency_db`)."""
    cache = dict(dependency_db or {})
    cache.update({t.id: t for t in tasks})
    for t in tasks:
        met = _dependencies_met(t, cache, now)
        if not includes_dependencies or met:
            t.expected_duration = O.fetch_expected_duration(t, now)[0]
    return tasks


def task_queue_items(tasks: Sequence[M.Task]) -> List[M.TaskQueueItem]:
    """PersistTaskQueue's projection (task_queue_persister.go:18-40), before TaskQueue.Save truncates it."""
    return [M.TaskQueueItem(
        id=t.id, display_name=t.display_name, build_variant=t.build_variant, revision_order_number=t.revision_order_number,
        requester=t.requester, revision=t.revision, project=t.project, expected_duration=t.expected_duration,
        priority=t.priority, sorting_value_breakdown=t.sorting_value_breakdown, group=t.task_group,
        group_max_hosts=t.task_group_max_hosts, group_index=t.task_group_order, version=t.version,
        activated_by=t.activated_by, dependencies=[d.task_id for d in t.depends_on],
        dependencies_met=t.has_dependencies_met()) for t in tasks]


def saved_queue(items: Sequence[M.TaskQueueItem]) -> List[M.TaskQueueItem]:
    """TaskQueue.Save: the first 10 000 items."""
    return list(items[:SAVED_QUEUE_CAP])

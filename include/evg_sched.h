/*
 * evg_sched.h -- C-ABI of libevgsched.so: the B200 (sm_100a) implementation of
 * Evergreen's scheduler hot path (scheduler.PlanDistro: tunable planner +
 * DistroQueueInfo + utilization host allocator), batched over distros.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch/CUDA types.
 * A Go maintainer binds it with cgo from package `scheduler` (INTEGRATION.md
 * shows the stub); the Python mirror in evergreen_b200/ binds it with ctypes.
 * Every entry point cites the reference interface it replaces; paths are
 * relative to the evergreen-ci/evergreen checkout.
 *
 * Layout: all distros of one scheduler tick are concatenated.  Distro d owns
 * tasks  [task_off[d],  task_off[d+1]),  hosts [host_off[d], host_off[d+1]) and
 * task-group slots [group_off[d], group_off[d+1]).  Indices inside a distro
 * (dep_idx, group_id, version_id, order[]) are distro-local.
 *
 * Determinism: `now_ns` replaces every time.Now()/time.Since on the path
 * (planner.go:318-322, scheduler.go:123, utilization_based_host_allocator.go:360).
 * Ties the reference leaves to map order / unstable sort are broken by the
 * canonical policy of DESIGN.md §3 (units: TotalValue desc, then the unit's
 * anchor -- the smallest input index among the tasks whose own key the unit is
 * filed under -- asc; tasks in a unit: the TaskList.Less chain, then input
 * index asc).
 *
 * There is no CPU fallback: every compute entry point fails with
 * EVG_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef EVG_SCHED_H
#define EVG_SCHED_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVG_ABI_VERSION 1

/* Go's zero time.Time (year 1).  0 is the Unix epoch, which time.Time.IsZero
 * reports as NON-zero; other values are ns since the Unix epoch. */
#define EVG_TIME_ZERO INT64_MIN

/* library status codes (negative = failure; message via evg_last_error()) */
enum {
  EVG_OK = 0,
  EVG_ERR_INVALID = -1, /* bad argument / inconsistent offsets */
  EVG_ERR_CUDA = -2,    /* no usable sm_100 device, or a CUDA call failed */
  EVG_ERR_NOMEM = -3,   /* device or pinned allocation failed */
  EVG_ERR_STATE = -4    /* resident call without a prior evg_upload */
};

/* per-distro allocator status: the data errors UtilizationBasedHostAllocator
 * returns as `error` (utilization_based_host_allocator.go:151-160,200-202,302-304) */
enum {
  EVG_ALLOC_OK = 0,
  EVG_ALLOC_ERR_FUTURE_FRACTION = 1, /* "future host factor cannot be greater than 1" */
  EVG_ALLOC_ERR_POOL_SIZE = 2,       /* "unable to plan hosts ... due to pool size" (maxHosts < 1) */
  EVG_ALLOC_ERR_PARENT_MISSING = 3   /* container pool parent distro not found */
};

/* evg_task_soa.flags */
#define EVG_TF_REQ_MASK 0x3u       /* requester class */
#define EVG_TF_REQ_OTHER 0u        /*   anything else -> mainline branch (planner.go:234) */
#define EVG_TF_REQ_PATCH 1u        /*   IsPatchRequester && !merge queue (globals.go:1179) */
#define EVG_TF_REQ_MERGE_QUEUE 2u  /*   IsGithubMergeQueueRequester (globals.go:1195) */
#define EVG_TF_GENERATE 0x4u       /* Task.GenerateTask */
#define EVG_TF_STEPBACK 0x8u       /* Task.ActivatedBy == "stepback" (globals.go:219) */
#define EVG_TF_DEPS_MET 0x10u      /* Task.DependenciesMet(...) (model/task/task.go:632) */
#define EVG_TF_OTHER_DISTRO 0x20u  /* Task.DistroId != distro id (scheduler.go:75) */

/* Task records, SoA (replaces []task.Task, model/task/task.go:83-350; the
 * fields are those SURVEY.md §8a row A20 lists).  48 B per task. */
typedef struct {
  int64_t n_tasks;
  int64_t n_edges;
  const int32_t* priority;         /* Task.Priority (int64 in Go; the shim saturates to int32) */
  const int64_t* expected_ns;      /* Task.FetchExpectedDuration(ctx).Average (task.go:3519) */
  const int64_t* queue_basis_ns;   /* ActivatedTime if !IsZero, else IngestTime if !IsZero, else EVG_TIME_ZERO (planner.go:318-322) */
  const int64_t* wait_basis_ns;    /* later of ScheduledTime, DependenciesMetTime (scheduler.go:119-122); EVG_TIME_ZERO if both zero */
  const int32_t* num_dependents;   /* Task.NumDependents */
  const int32_t* task_group_order; /* Task.TaskGroupOrder */
  const int32_t* group_id;         /* distro-local dense id of Task.GetTaskGroupString() (task.go:417); -1 when TaskGroup == "" */
  const int32_t* version_id;       /* distro-local dense id of Task.Version */
  const uint32_t* flags;           /* EVG_TF_* */
  /* Task.DependsOn restricted to dependencies that are themselves in this
   * distro's queue (planner.go:449-456), CSR over tasks; NULL when n_edges==0 */
  const int64_t* dep_off;          /* n_tasks + 1 */
  const int32_t* dep_idx;          /* distro-local index of the dependency */
} evg_task_soa;

/* distro.PlannerSettings (model/distro/distro.go:286-300), raw: the <=0 -> 1
 * clamp of the factor getters (distro.go:353-408) happens on the device. */
typedef struct {
  int64_t patch_factor;
  int64_t patch_time_in_queue_factor;
  int64_t commit_queue_factor;
  int64_t mainline_time_in_queue_factor;
  int64_t expected_runtime_factor;
  int64_t generate_task_factor;
  int64_t stepback_task_factor;
  double num_dependents_factor;
  int64_t target_time_ns;        /* d.GetTargetTime() (distro.go:434-440), resolved by the shim */
  int32_t group_versions;        /* PlannerSettings.ShouldGroupVersions() */
  int32_t includes_dependencies; /* DispatcherSettings.Version == "revised-with-dependencies" (scheduler.go:28) */
  int32_t n_versions;            /* number of distinct version ids in this distro */
  int32_t _reserved;
} evg_distro_cfg;

typedef struct {
  int32_t n_distros;
  int32_t _reserved;
  const int64_t* task_off;        /* n_distros + 1 */
  const int64_t* group_off;       /* n_distros + 1 */
  const evg_distro_cfg* cfg;      /* n_distros */
  const int32_t* group_max_hosts; /* per group slot: Task.TaskGroupMaxHosts of the group (scheduler.go:87-90) */
} evg_distro_table;

/* model.TaskGroupInfo without the name (model/task_queue.go:22-47); the name
 * of slot group_off[d]+g is the shim's string for group id g. 72 B. */
typedef struct {
  int64_t count;
  int64_t count_free;      /* written by the allocator (allocator.go:107-110) */
  int64_t count_required;  /* written by the allocator */
  int64_t max_hosts;
  int64_t expected_duration;
  int64_t count_duration_over_threshold;
  int64_t count_wait_over_threshold;
  int64_t count_dep_filled_merge_queue_tasks;
  int64_t duration_over_threshold;
} evg_group_info;

/* model.DistroQueueInfo (model/task_queue.go:49-75).  `ungrouped` is the
 * TaskGroupInfo named "" (standalone tasks); it exists in TaskGroupInfos only
 * when has_ungrouped != 0. */
typedef struct {
  int64_t length;
  int64_t length_with_dependencies_met;
  int64_t count_dep_filled_merge_queue_tasks;
  int64_t expected_duration;
  int64_t max_duration_threshold;
  int64_t count_duration_over_threshold;
  int64_t duration_over_threshold;
  int64_t count_wait_over_threshold;
  int64_t secondary_queue; /* any task.DistroId != distro (scheduler.go:75-77); callers overwrite it (scheduler.go:44) */
  int64_t has_ungrouped;
  evg_group_info ungrouped;
} evg_queue_info;

/* task.SortingValueBreakdown flattened to 13 int64 (model/task/task.go:3990-4038) */
enum {
  EVG_BD_TASK_GROUP_LENGTH = 0, EVG_BD_TOTAL_VALUE,
  EVG_BD_P_INITIAL, EVG_BD_P_TASK_GROUP, EVG_BD_P_GENERATOR, EVG_BD_P_COMMIT_QUEUE,
  EVG_BD_R_COMMIT_QUEUE, EVG_BD_R_NUM_DEPENDENTS, EVG_BD_R_ESTIMATED_RUNTIME,
  EVG_BD_R_MAINLINE_WAIT, EVG_BD_R_STEPBACK, EVG_BD_R_PATCH, EVG_BD_R_PATCH_WAIT,
  EVG_BD_N
};

/* Planner outputs (replaces the []task.Task PrioritizeTasks returns,
 * scheduler.go:27, and the DistroQueueInfo of scheduler.go:43). */
typedef struct {
  int32_t* order;             /* [n_tasks] slot task_off[d]+r = distro-local index of the task ranked r (TaskPlan.Export, planner.go:462-481) */
  int64_t* total_value;       /* [n_tasks] SortingValueBreakdown.TotalValue of the unit the task was emitted from, rank order */
  int64_t* breakdown;         /* [n_tasks * EVG_BD_N] full breakdown in rank order, or NULL */
  evg_queue_info* info;       /* [n_distros] */
  evg_group_info* group_info; /* [group_off[n_distros]] */
} evg_plan_out;

/* evg_host_soa.flags */
#define EVG_HF_RUNNING 0x1u    /* Host.RunningTask != "" */
#define EVG_HF_TEARDOWN 0x2u   /* !Host.TaskGroupTeardownStartTime.IsZero() (host.go:219-221) */
#define EVG_HF_RT_FOUND 0x4u   /* the running task was returned by task.Find(ByIds) (allocator.go:337) */

/* host bucket codes for evg_host_soa.group_id (groupByTaskGroup, allocator.go:223-260) */
#define EVG_HG_NONE (-1)       /* name "" : no running task or no running task group */
#define EVG_HG_UNQUEUED (-2)   /* a named group with no TaskGroupInfo in the queue */

/* Existing hosts, SoA (replaces HostAllocatorData.ExistingHosts []host.Host,
 * host_allocator.go:17-23, model/host/host.go:79-88).  32 B per host. */
typedef struct {
  int64_t n_hosts;
  const uint32_t* flags;      /* EVG_HF_* */
  const int32_t* group_id;    /* EVG_HG_* or the distro-local task-group id of Host.GetTaskGroupString() (host.go:663) */
  const int64_t* expected_ns; /* running task FetchExpectedDuration().Average (allocator.go:357-358) */
  const int64_t* std_ns;      /* ... .StdDev (allocator.go:359) */
  const int64_t* start_ns;    /* running task StartTime (allocator.go:360), EVG_TIME_ZERO if unset */
} evg_host_soa;

enum { EVG_PROVIDER_STATIC = 0, /* not in evergreen.ProviderSpawnable (globals.go:723-728) */
       EVG_PROVIDER_EPHEMERAL = 1, /* ec2-ondemand, ec2-fleet, mock */
       EVG_PROVIDER_DOCKER = 2 };

/* distro.HostAllocatorSettings + the rest of HostAllocatorData that is not
 * hosts or queue info (model/distro/distro.go:267-280, host_allocator.go:17-23) */
typedef struct {
  double future_host_fraction;
  int32_t provider;                   /* EVG_PROVIDER_* */
  int32_t disabled;                   /* Distro.Disabled */
  int32_t minimum_hosts;
  int32_t maximum_hosts;
  int32_t round_up;                   /* RoundingRule == "round-up" (allocator.go:174-177) */
  int32_t waits_over_thresh_feedback; /* FeedbackRule == "waits-over-thresh-feedback" (allocator.go:179-182) */
  int32_t has_pool;                   /* HostAllocatorData.ContainerPool != nil */
  int32_t pool_max_containers;        /* ContainerPool.MaxContainers */
  int32_t parent_found;               /* distro.FindOneId(pool.Distro) succeeded (allocator.go:151-158) */
  int32_t parent_maximum_hosts;       /* parent HostAllocatorSettings.MaximumHosts (allocator.go:159) */
} evg_alloc_cfg;

/* Allocator outputs (replaces the (int, int, error) of HostAllocator,
 * host_allocator.go:15).  `result` is the same data packed for the
 * multi-GPU all-gather: 16 B per distro. */
typedef struct {
  int32_t new_hosts;   /* numNewHostsToRequest */
  int32_t free_hosts;  /* numFreeApprox (or len(freeHosts) on the early returns) */
  int64_t deficit_ns;  /* auxiliary: max(0, expected_duration - free_hosts*threshold), host-time the free pool cannot absorb */
} evg_alloc_result;

typedef struct {
  evg_alloc_result* result; /* [n_distros] */
  int32_t* status;          /* [n_distros] EVG_ALLOC_* */
} evg_alloc_out;

/* option bits */
#define EVG_OPT_BREAKDOWN 0x1u /* materialise evg_plan_out.breakdown */

typedef struct evg_ctx evg_ctx;

/* ---- lifecycle ---------------------------------------------------------- */

/* Bind a context to CUDA device `device`.  `stream` is a cudaStream_t the
 * kernels are launched on (e.g. the caller's torch stream) or NULL for a
 * private stream.  Replaces nothing in the reference (process bootstrap). */
int evg_init(int device, void* stream, evg_ctx** out);
void evg_shutdown(evg_ctx* ctx);
/* thread-local message for the last failing call on this thread */
const char* evg_last_error(void);
int evg_abi_version(void);

/* Pinned host buffers for the SoA columns (the Go shim fills C-allocated
 * memory so no Go pointer is retained across the call). */
void* evg_host_alloc(uint64_t bytes);
void evg_host_free(void* p);

/* ---- one-shot batch entry points: HOST pointers, H2D + kernels + D2H ---- */

/* Tunable planner + queue info for every distro of the tick.
 * Replaces: scheduler.PrioritizeTasks / runTunablePlanner minus persistence
 * (scheduler/scheduler.go:27-51): PrepareTasksForPlanning(...).Export
 * (planner.go:431-481) and GetDistroQueueInfo (scheduler.go:56-159). */
int evg_plan_batch(evg_ctx* ctx, const evg_task_soa* tasks, const evg_distro_table* distros,
                   int64_t now_ns, uint32_t opts, evg_plan_out* out);

/* Utilization host allocator for every distro, from queue infos the caller
 * already has (the reference reads them back from MongoDB,
 * units/host_allocator.go:152).  `groups` is in/out: count_free and
 * count_required are written like the reference mutates TaskGroupInfos.
 * Replaces: scheduler.UtilizationBasedHostAllocator
 * (scheduler/utilization_based_host_allocator.go:26-130) behind the
 * HostAllocator plug point (scheduler/host_allocator.go:15,25-32). */
int evg_alloc_batch(evg_ctx* ctx, const evg_host_soa* hosts, const int64_t* host_off,
                    const evg_alloc_cfg* cfg, const evg_queue_info* info, evg_group_info* groups,
                    const int64_t* group_off, int32_t n_distros, int64_t now_ns, evg_alloc_out* out);

/* Fused planner + allocator: the queue info never leaves the device.
 * Replaces: distroSchedulerJob.Run + hostAllocatorJob.Run for all distros of
 * one tick (units/scheduler.go:57-87, units/host_allocator.go:76-196). */
int evg_plan_and_alloc_batch(evg_ctx* ctx, const evg_task_soa* tasks, const evg_distro_table* distros,
                             const evg_host_soa* hosts, const int64_t* host_off,
                             const evg_alloc_cfg* acfg, int64_t now_ns, uint32_t opts,
                             evg_plan_out* plan_out, evg_alloc_out* alloc_out);

/* ---- resident API: inputs stay in HBM between ticks --------------------- */

/* Copy a tick's inputs into context-owned device buffers (hosts/host_off/acfg
 * may be NULL for planner-only use). */
int evg_upload(evg_ctx* ctx, const evg_task_soa* tasks, const evg_distro_table* distros,
               const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* acfg);
/* Tick-to-tick update of the resident task table: row rows[i] (a task slot of the last evg_upload, 0 <= rows[i] <
 * n_tasks) gets priority, num_dependents, task_group_order, flags, expected_ns, queue_basis_ns and wait_basis_ns of row i
 * of `values` (values->n_tasks == n_rows; its group / version / dependency columns are not read: a task keeps its
 * distro, its task group, its version and its in-queue dependency edges -- a tick that adds or removes tasks uploads
 * again).  48 bytes cross PCIe per changed row instead of the whole table.  Not available after evg_upload_device (the
 * caller owns those columns and edits them in place).  Replaces nothing in the reference: there the scheduler re-reads
 * every task document each tick (scheduler/task_finder.go:40-197). */
int evg_update_tasks(evg_ctx* ctx, int64_t n_rows, const int64_t* rows, const evg_task_soa* values);

/* Like evg_upload, but the task columns already live in DEVICE memory (the finder's output, a generator kernel, a
 * previous tick edited in place): `tasks` holds device pointers, which the context borrows until the next upload or
 * evg_shutdown -- nothing is copied.  Every column must be 16-byte aligned and readable 8 elements past its last
 * row (the kernels read whole 128-bit vectors / TMA tiles).  `distros`, `hosts`, `host_off`, `acfg` are host
 * pointers as in evg_upload.  Replaces nothing in the reference (there the tasks are already in the process). */
int evg_upload_device(evg_ctx* ctx, const evg_task_soa* device_tasks, const evg_distro_table* distros,
                      const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* acfg);
/* Launch the fused path on the resident inputs; asynchronous on the context
 * stream.  Safe to call repeatedly (each call recomputes from the inputs). */
int evg_run_resident(evg_ctx* ctx, int64_t now_ns, uint32_t opts);
/* Wait for the stream and copy results out; either pointer may be NULL. */
int evg_download(evg_ctx* ctx, evg_plan_out* plan_out, evg_alloc_out* alloc_out);
/* ---- the persisted queue (SURVEY.md §8 f.4) ---- */

#define EVG_QI_DEPS_MET 0x1u /* TaskQueueItem.DependenciesMet = Task.HasDependenciesMet() after GetDistroQueueInfo
                                stamped the task (scheduler.go:98,137; model/task/task.go:653,3393) */
/* The numeric half of model.TaskQueueItem (model/task_queue.go:131-153) for one persisted rank; the string half
 * (Id, DisplayName, BuildVariant, Requester, Revision, Project, Group, Version, ActivatedBy, Dependencies) is read by
 * the shim from its own []task.Task at index `task`.  40 B. */
typedef struct {
  int32_t task;            /* distro-local index of the task at this rank */
  int32_t group_index;     /* GroupIndex = Task.TaskGroupOrder */
  int32_t group_max_hosts; /* GroupMaxHosts = Task.TaskGroupMaxHosts (0 outside task groups) */
  uint32_t flags;          /* EVG_QI_* */
  int64_t priority;        /* Priority */
  int64_t expected_ns;     /* FetchExpectedDuration().Average: the ExpectedDuration GetDistroQueueInfo writes on every task it
                              counts (scheduler.go:98); under IncludesDependencies a task without EVG_QI_DEPS_MET keeps its own */
  int64_t total_value;     /* SortingValueBreakdown.TotalValue of the unit the task was emitted from (planner.go:475) */
} evg_queue_item;
#define EVG_PERSISTED_QUEUE_CAP 10000 /* TaskQueue.Save keeps the first 10 000 items (model/task_queue.go:216-219) */

/* After evg_run_resident: project the head of every distro's ranked queue -- the first min(length, cap) ranks, cap = 0
 * meaning EVG_PERSISTED_QUEUE_CAP -- into TaskQueueItem rows on the device and copy only those to the host.
 * item_off (n_distros + 1) receives the offsets of each distro's rows in `items`; `items_capacity` rows must be
 * available (sum over distros of min(length, cap); -EVG_ERR_INVALID with the needed count in evg_last_error otherwise).
 * Replaces: the TaskQueueItem projection and truncation of PersistTaskQueue / TaskQueue.Save
 * (scheduler/task_queue_persister.go:14-42, model/task_queue.go:216-219).  The upsert stays with the caller. */
int evg_download_queue(evg_ctx* ctx, int32_t cap, int64_t* item_off, evg_queue_item* items, int64_t items_capacity);

/* Like evg_run_resident, but only the first min(length, cap) ranks of every distro are ordered: what
 * PersistTaskQueue / TaskQueue.Save keep (scheduler/task_queue_persister.go:14-55, model/task_queue.go:216-219), and
 * all a PlanDistro caller reads of the plan besides len(plan) (scheduler/wrapper.go:107-127).  Distros above the
 * on-chip capacity select their cap smallest keys instead of sorting every task (when the longest of them exceeds twice
 * the cap; below that the full sort is faster and its first cap ranks are the head).
 * cap: 0 means EVG_PERSISTED_QUEUE_CAP; otherwise 1 <= cap <= EVG_PERSISTED_QUEUE_CAP, else -EVG_ERR_INVALID.
 * Queue info, group info and allocator results are the same as after evg_run_resident, and so is every rank below
 * the cap.  opts: EVG_OPT_BREAKDOWN is honoured for those ranks only.  Afterwards evg_download with a non-NULL order,
 * total_value or breakdown is -EVG_ERR_STATE (those rows are not defined past the cut), and so are evg_download_queue /
 * evg_download_queue_bd with a cap above this one (cap 0 included when this one is below EVG_PERSISTED_QUEUE_CAP).
 * The next evg_run_resident restores the full contract.  evg_general_timing_ms's sort_ms spans select, compaction and
 * head sort. */
int evg_run_resident_head(evg_ctx* ctx, int64_t now_ns, uint32_t opts, int32_t cap);

/* evg_download_queue plus breakdown[rows * EVG_BD_N]: the full SortingValueBreakdown of each row, in the same order
 * (the TaskQueueItem.SortingValueBreakdown PersistTaskQueue copies, task_queue_persister.go:33).  Works after either
 * kind of run that set EVG_OPT_BREAKDOWN; -EVG_ERR_STATE otherwise. */
int evg_download_queue_bd(evg_ctx* ctx, int32_t cap, int64_t* item_off, evg_queue_item* items,
                          int64_t* breakdown, int64_t items_capacity);

/* Device pointer to the resident evg_alloc_result[n_distros] vector, the
 * send buffer of the per-distro all-gather (SURVEY.md §8e). */
void* evg_device_result_ptr(evg_ctx* ctx);
/* Make the allocator kernel write its evg_alloc_result[] rows straight into a
 * caller-owned DEVICE buffer (e.g. the NCCL send buffer of the all-gather),
 * `capacity` rows long; NULL restores the context-owned buffer. */
int evg_bind_result_buffer(evg_ctx* ctx, void* device_ptr, int64_t capacity);
/* Number of kernel launches issued by the last evg_run_resident. */
int64_t evg_last_launch_count(evg_ctx* ctx);
/* Device time in ms of the last evg_run_resident, from CUDA events on the context
 * stream (valid after a sync / download): total_ms spans the whole tick; sort_ms is
 * the general path's segmented radix sort when the tick had a distro above 12288
 * tasks, otherwise the k_plan_smem<1024,12> launch (see evg_kernel_timing_ms). */
int evg_last_timing_ms(evg_ctx* ctx, float* total_ms, float* sort_ms);

/* Device time in ms of the dominant kernel of on-chip ticks -- k_plan_cta<512,10240>, the on-chip planner of distros
 * with 5121..10240 tasks (or k_plan_smem<1024,12> when the tick has none) -- for each of the last `n`
 * evg_run_resident calls that launched it (n <= 128), from CUDA events recorded around that launch on its stream. */
int evg_kernel_timing_ms(evg_ctx* ctx, float* out_ms, int32_t n);

/* The general path's two big stages in the last evg_run_resident (ms, CUDA events on its stream): the per-task
 * pass k_gtask (reads every input column once) and the segmented radix sort (all passes); after
 * evg_run_resident_head, the select, compaction and head sort that replace it. */
int evg_general_timing_ms(evg_ctx* ctx, float* task_pass_ms, float* sort_ms);

/* ---- dependency filter (SURVEY.md §8f.1: the next row after the planner/allocator path) ---- */

/* evg_deps_in.dep_kind */
#define EVG_DEP_IN_QUEUE 0  /* dep_ref = index (in this call's task table) of the dependency; its state is task_state[dep_ref] */
#define EVG_DEP_EXTERNAL 1  /* dep_ref indexes ext_state[] (the dependency was fetched from the tasks collection) */
#define EVG_DEP_MISSING 2   /* lookup failed: never met (checkDependenciesMet, scheduler/scheduler.go:161-168) */
/* evg_deps_in.dep_want: Dependency.Status */
#define EVG_WANT_SUCCESS 0  /* "success" or "" (model/task/task.go:533-534) */
#define EVG_WANT_FAILED 1   /* "failed" */
#define EVG_WANT_ANY 2      /* "*" AllStatuses: failed, succeeded or blocked (task.go:537-538) */
#define EVG_WANT_OTHER 3    /* any other string: never satisfied */
/* task_state / ext_state bits */
#define EVG_TS_STATUS_MASK 0x3u /* 0 "success", 1 "failed", 2 anything else */
#define EVG_TS_BLOCKED 0x4u     /* Task.Blocked() (task.go:3649-3660) */
/* task_pre bits: Task.HasDependenciesMet short-circuits (task.go:3393-3395) */
#define EVG_TP_OVERRIDE 0x1u    /* OverrideDependencies */
#define EVG_TP_MET_TIME 0x2u    /* !utility.IsZeroTime(DependenciesMetTime) */

/* All DIRECT dependencies of every task, CSR over tasks. */
typedef struct {
  int64_t n_tasks;
  int64_t n_deps;
  const int64_t* dep_off;   /* n_tasks + 1 */
  const uint8_t* dep_kind;  /* EVG_DEP_* */
  const int32_t* dep_ref;
  const uint8_t* dep_want;  /* EVG_WANT_* of the FIRST of the task's Dependencies naming the same task: SatisfiesDependency
                              judges every edge to a task by that one (model/task/task.go:529-543) */
  const uint8_t* task_state;/* n_tasks, EVG_TS_* of the in-queue tasks themselves */
  const uint8_t* task_pre;  /* n_tasks, EVG_TP_* */
  const uint8_t* ext_state; /* n_ext, EVG_TS_* */
  int64_t n_ext;
} evg_deps_in;

/* met[t] = Task.DependenciesMet(ctx, depCache) for every task (model/task/task.go:632-671 with
 * SatisfiesDependency :529-543): the bit evg_task_soa.flags carries as EVG_TF_DEPS_MET and the predicate the
 * task finders filter on (scheduler/task_finder.go:40-197).  Host pointers in and out. */
int evg_deps_met_batch(evg_ctx* ctx, const evg_deps_in* in, uint8_t* met);

/* evg_upload with the dependency predicate evaluated ON THE DEVICE and wired into the planner's inputs: after the
 * copy, Task.DependenciesMet runs for every task (same tables as evg_deps_met_batch, over the same n_tasks tasks) and
 *   - the EVG_TF_DEPS_MET bit of the resident flags column is set from its verdict (the caller's bit is ignored);
 *   - a task whose dependencies were evaluated afresh and found met is stamped like Task.setDependenciesMetTime does
 *     (model/task/task.go:653,673-684): the latest non-zero dep_finished_ns[] (Dependency.FinishedAt, per dependency,
 *     NULL = unknown) of its dependencies, else now_ns; its resident wait basis becomes the later of the caller's
 *     wait_basis_ns (ScheduledTime) and that stamp (scheduler.go:119-122).
 * Neither the bit nor the stamp visits the host; evg_download_deps returns them for the write-back the reference does
 * (UpdateOne of DependenciesMetTime, task.go:659-666).
 * Replaces: checkDependenciesMet inside GetDistroQueueInfo (scheduler/scheduler.go:82-98,161-168). */
int evg_upload_with_deps(evg_ctx* ctx, const evg_task_soa* tasks, const evg_distro_table* distros,
                         const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* acfg,
                         const evg_deps_in* deps, const int64_t* dep_finished_ns, int64_t now_ns);
/* met[t] = Task.DependenciesMet; met_time_ns[t] = the stamp (EVG_TIME_ZERO when nothing was stamped).  Either may be NULL. */
int evg_download_deps(evg_ctx* ctx, uint8_t* met, int64_t* met_time_ns);

/* ---- runnable-task filter: the task finders (SURVEY.md §8f.1) ------------- */

/* evg_runnable_in.sched: what schedulableHostTasksQuery (model/task/db.go:671-689) and ProjectCanDispatchTask read of a task */
#define EVG_SQ_ACTIVATED 0x01u      /* Activated */
#define EVG_SQ_UNDISPATCHED 0x02u   /* Status == "undispatched" */
#define EVG_SQ_PRIORITY_OK 0x04u    /* Priority > DisabledTaskPriority (-1) */
#define EVG_SQ_HOST_PLATFORM 0x08u  /* ByExecutionPlatform(host): field absent or "host" (db.go:647-663) */
#define EVG_SQ_UNATTAINABLE 0x10u   /* UnattainableDependency */
#define EVG_SQ_OVERRIDE_DEPS 0x20u  /* OverrideDependencies */
#define EVG_SQ_GITHUB_PR 0x40u      /* Requester == "github_pull_request" */
#define EVG_SQ_PATCH_REQUEST 0x80u  /* Task.IsPatchRequest() (model/task/task.go:545-547) */
/* evg_runnable_in.project_flags: ProjectRef fields ProjectCanDispatchTask reads (model/project_ref.go:3441-3462) */
#define EVG_PF_ENABLED 0x1u
#define EVG_PF_HIDDEN 0x2u
#define EVG_PF_DISPATCHING_DISABLED 0x4u
#define EVG_PF_PATCHING_DISABLED 0x8u
/* evg_runnable_in.finder, per distro */
#define EVG_FINDER_NO_DEPS 0    /* DispatcherSettings.Version == "revised-with-dependencies": dependencies are not filtered (task_finder.go:85) */
#define EVG_FINDER_LEGACY 1     /* LegacyFindRunnableTasks: Task.DependenciesMet, with the HasDependenciesMet short-circuit */
#define EVG_FINDER_ALTERNATE 2  /* AlternateTaskFinder / ParallelTaskFinder: Task.AllDependenciesSatisfied (task.go:795-821), no short-circuit */

/* Every candidate task of every distro (the rows task.FindHostSchedulable would be asked about), concatenated. */
typedef struct {
  int64_t n_tasks;
  int32_t n_distros;
  int32_t n_projects;
  const int64_t* task_off;      /* n_distros + 1 */
  const uint8_t* sched;         /* n_tasks, EVG_SQ_* */
  const int32_t* project;       /* n_tasks: row of project_flags, or -1 when the project-ref cache has no such project */
  const uint8_t* project_flags; /* n_projects, EVG_PF_* */
  const int64_t* valid_off;     /* n_distros + 1: CSR of Distro.ValidProjects as project rows (-1 = a name no ref has) */
  const int32_t* valid_idx;
  const uint8_t* finder;        /* n_distros, EVG_FINDER_* */
  const evg_deps_in* deps;      /* direct dependencies of the same n_tasks tasks; NULL when every finder is NO_DEPS */
} evg_runnable_in;

/* LegacyFindRunnableTasks / AlternateTaskFinder / ParallelTaskFinder (scheduler/task_finder.go:40-317) over all
 * distros at once: runnable[task_off[d] .. task_off[d] + count[d]) holds the distro-local indices of the tasks
 * the finder returns for distro d, in input order (the reference appends in query order); the rest of the
 * distro's slots are -1.  Host pointers. */
int evg_find_runnable_batch(evg_ctx* ctx, const evg_runnable_in* in, int32_t* runnable, int64_t* count);

/* The finder's output feeds the planner without leaving the device.  `in` describes every CANDIDATE task of every
 * distro as for evg_find_runnable_batch (in->deps is required: the planner's EVG_TF_DEPS_MET bit comes from it);
 * `candidates` holds the same rows' planner columns (flags without EVG_TF_DEPS_MET, wait_basis_ns = ScheduledTime,
 * in-queue dependency edges between candidates as distro-local candidate indices); `distros` is the distro table over
 * the candidates (task_off == in->task_off; group / version ids may name groups no kept task is in).  On the device:
 * k_deps_met (both predicates, DependenciesMetTime stamps from dep_finished_ns, as evg_upload_with_deps) -> the finders
 * -> a stable compaction of the nine planner columns (EVG_TF_DEPS_MET and the stamped wait basis applied on the way)
 * -> the dependency edges whose two ends were kept, re-indexed.  The compacted table becomes the context's resident
 * tick: call evg_run_resident / evg_download next; ranks refer to the compacted queues, and `runnable` (n_tasks, may be
 * NULL) / `count` (n_distros) map them back exactly as evg_find_runnable_batch reports them.  Group slot k of distro d
 * in the resident tick -- its evg_group_info row and a queue item's group_max_hosts -- is the k-th candidate group of d,
 * in id order, that kept at least one task; a group the finder emptied has no slot and no TaskGroupInfo, as in the
 * reference, which builds them from the planned tasks (scheduler.go:60-143).  hosts->group_id names candidate groups;
 * a host running a task of an emptied group counts as EVG_HG_UNQUEUED.  The only values the host reads in between are
 * the n_distros counts and one byte per candidate group (the routing needs queue lengths and group counts).
 * Replaces: the finder + checkDependenciesMet + PrioritizeTasks hand-over inside scheduler.PlanDistro
 * (scheduler/wrapper.go:60-118, scheduler/scheduler.go:56-168), where the filtered []task.Task is rebuilt on the host. */
int evg_plan_from_finder(evg_ctx* ctx, const evg_runnable_in* in, const evg_task_soa* candidates, const evg_distro_table* distros,
                         const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* acfg,
                         const int64_t* dep_finished_ns, int64_t now_ns, int32_t* runnable, int64_t* count);

/* ---- host-side string interning for the marshaller ------------------------ */

/* A column of n strings: bytes[off[i] .. off[i+1]) is string i (not NUL-terminated). */
typedef struct {
  const char* bytes;
  const int64_t* off; /* n + 1 */
} evg_str_col;

/* The strings of a tick's tasks, concatenated distro by distro like evg_task_soa. */
typedef struct {
  int64_t n_tasks;
  int32_t n_distros;
  const int64_t* task_off;          /* n_distros + 1 */
  evg_str_col id;                   /* Task.Id */
  evg_str_col version;              /* Task.Version */
  evg_str_col group_key;            /* Task.GetTaskGroupString() (model/task/task.go:417-419); "" when Task.TaskGroup == "" */
  const int32_t* group_max_hosts;   /* Task.TaskGroupMaxHosts, n_tasks */
  const int64_t* dep_off;           /* n_tasks + 1: CSR over Task.DependsOn */
  evg_str_col dep_id;               /* Dependency.TaskId, dep_off[n_tasks] strings */
} evg_string_cols;

/* What the planner's columns need of those strings; every array is caller-allocated. */
typedef struct {
  int32_t* group_id;        /* n_tasks: dense per distro in first-appearance order, -1 without a task group */
  int32_t* version_id;      /* n_tasks: dense per distro in first-appearance order */
  int64_t* group_off;       /* n_distros + 1 */
  int32_t* n_versions;      /* n_distros */
  int32_t* group_max_hosts; /* capacity n_tasks: one per group slot, group_off[n_distros] used */
  int64_t* group_first;     /* capacity n_tasks: row of each group's first member (its name is group_key there) */
  int64_t* dep_off;         /* n_tasks + 1: in-queue dependency edges (planner.go:449-456) */
  int32_t* dep_idx;         /* capacity dep_off_in[n_tasks]: distro-local index of the dependency; targets outside the queue are dropped */
} evg_intern_out;

/* String work of marshalling a tick (scheduler.PrioritizeTasks builds the same maps while it walks a queue:
 * planner.go:431-456 files units under exactly these strings): group keys and versions to dense ids, dependency ids
 * to queue indices, per distro, `threads` distros at a time (<= 0: hardware concurrency).  Host only: no context.
 * EVG_ERR_INVALID when members of one task group disagree on TaskGroupMaxHosts (evg_last_error names the row). */
int evg_intern_columns(const evg_string_cols* in, evg_intern_out* out, int32_t threads);

/* ---- expected-duration statistics (SURVEY.md §8f.2) ----------------------- */

/* evg_duration_rows.flags */
#define EVG_DR_COMPLETED 0x1u  /* Status in evergreen.TaskCompletedStatuses (expected_duration.go:41-43) */
#define EVG_DR_TIMED_OUT 0x2u  /* Details.TimedOut == true (excluded, :44-46) */

/* Finished tasks (one row each) of any number of (project, build variant) windows at once; `key` interns the
 * group-by key -- (project, build variant, display name) -- so one call replaces one aggregation per pair. */
typedef struct {
  int64_t n_rows;
  int32_t n_keys;
  int32_t _reserved;
  const int32_t* key;            /* n_rows: 0 .. n_keys-1 */
  const int64_t* time_taken_ns;  /* n_rows: Task.TimeTaken */
  const int64_t* start_ns;       /* n_rows: Task.StartTime (UnixNano) */
  const int64_t* finish_ns;      /* n_rows: Task.FinishTime */
  const uint8_t* flags;          /* n_rows: EVG_DR_* */
  int64_t window_start_ns;       /* $match: StartTime > window_start && FinishTime <= window_end (:47-52) */
  int64_t window_end_ns;
} evg_duration_rows;

/* One group of the $group stage (expected_duration.go:66-76): {$avg, $stdDevPop} of TimeTaken.  count == 0 means the
 * aggregation returns no document for the key.  mean_ns = double(sum) / double(count); stddev_ns = sqrt(variance)
 * with the variance accumulated EXACTLY in integers around floor(mean) and rounded once at the end (MongoDB's
 * streaming Welford update differs from it in the last few ulps; the reference's own test allows 0.01 minutes). */
typedef struct {
  int64_t count;
  double mean_ns;
  double stddev_ns;
} evg_duration_stat;

/* getExpectedDurationsForWindow (model/task/expected_duration.go:36-96) for every key at once.  Host pointers. */
int evg_expected_durations_batch(evg_ctx* ctx, const evg_duration_rows* in, evg_duration_stat* out);

/* ---- legacy comparator prioritiser (SURVEY.md §8 row L) ---------------------- */

/* evg_legacy_soa.flags */
#define EVG_LF_REQ_MASK 0x3u
#define EVG_LF_REQ_SYSTEM 0u              /* Requester in evergreen.SystemVersionRequesterTypes (globals.go:766-772): repotracker list, "commit build" */
#define EVG_LF_REQ_PATCH 1u               /* evergreen.IsPatchRequester (globals.go:1179-1185): patch list */
#define EVG_LF_REQ_OTHER 2u               /* anything else: logged and dropped (task_prioritizer.go:232-240) */
#define EVG_LF_GENERATE 0x4u              /* Task.GenerateTask */
#define EVG_LF_MERGE_QUEUE_VERSION 0x8u   /* versions[Task.Version].Requester == github_merge_request (byCommitQueue) */
/* byAge (task_priority_cmp.go:73-95) of one list, decided by the shim when it marshals the list */
#define EVG_LEGACY_MODE_INGEST 0    /* no two commit builds of the list share a project: IngestTime ascending */
#define EVG_LEGACY_MODE_REVISION 1  /* every non-group task is a commit build of ONE project: RevisionOrderNumber descending */
#define EVG_LEGACY_MODE_LITERAL 2   /* neither (or zero and non-zero expected durations mixed, or two (TaskGroup, BuildId)
                                       pairs format to one string): the chain is not a strict weak order on this list */
/* per-distro status */
#define EVG_LEGACY_OK 0
#define EVG_LEGACY_NOT_DECOMPOSABLE 1 /* some list was EVG_LEGACY_MODE_LITERAL: no order is common to all stable sorts there;
                                         the list was sorted by the nearest transitive key (byAge by IngestTime only),
                                         which need not be the order Go's sort.Stable produces */

/* What CmpBasedTaskPrioritizer reads of []task.Task and map[string]model.Version, SoA over the concatenated distros
 * (scheduler/task_prioritizer.go:80-278, task_priority_cmp.go:25-208, setup_funcs.go:72-87).  Strings are interned
 * by the shim; ranks are per distro. */
typedef struct {
  int64_t n_tasks;
  const int64_t* priority;         /* Task.Priority (int64: the > MaxTaskPriority split and byPriority) */
  const int64_t* ingest_ns;        /* Task.IngestTime */
  const int64_t* expected_ns;      /* Task.FetchExpectedDuration(ctx).Average */
  const int32_t* num_dependents;
  const int32_t* revision_order;   /* Task.RevisionOrderNumber */
  const int32_t* project_id;       /* interned Task.Project */
  const int32_t* tg_rank;          /* rank of "BuildId-TaskGroup" among the distro's distinct such strings, ascending byte order; -1 when TaskGroup == "" */
  const int32_t* tg_pair_id;       /* dense id of the (TaskGroup, BuildId) pair; -1 when TaskGroup == "" */
  const int32_t* task_group_order;
  const int32_t* presort_rank;     /* position of "BuildId-TaskGroup-Id" in DESCENDING byte order inside the distro (groupTaskGroups) */
  const uint32_t* flags;           /* EVG_LF_* */
} evg_legacy_soa;

/* CmpBasedTaskPrioritizer.PrioritizeTasks for every distro of the tick.  list_mode[3*d + {0,1,2}] is the
 * EVG_LEGACY_MODE_* of distro d's high-priority / patch / repotracker list.  order[task_off[d] .. +count[d]) receives
 * the distro-local indices of the prioritised tasks (dropped tasks leave -1 in the remaining slots).  Host pointers.
 * Replaces: the TaskPrioritizer interface (scheduler/task_prioritizer.go:20-25) minus the orderingLogic reasons. */
int evg_prioritize_legacy_batch(evg_ctx* ctx, const evg_legacy_soa* tasks, const int64_t* task_off, const uint8_t* list_mode,
                                int32_t n_distros, int32_t* order, int64_t* count, int32_t* status);

/* ---- DAG dispatcher rebuild (SURVEY.md §8 f.3) ------------------------------ */

/* The persisted queues of a batch of distros, concatenated in queue order (item k of distro d has queueIndex k). */
typedef struct {
  int64_t n_items;
  int64_t n_deps;
  const int64_t* dep_off;      /* n_items + 1: CSR of TaskQueueItem.Dependencies */
  const int32_t* dep_item;     /* n_deps: distro-local index of the item with that id, -1 when it is not in this queue */
  const int32_t* group_id;     /* n_items: distro-local dense id of compositeGroupID(Group, BuildVariant, Project, Version), -1 when Group == "" */
  const int32_t* group_index;  /* n_items: TaskQueueItem.GroupIndex */
} evg_dag_in;

/* basicCachedDAGDispatcherImpl.rebuild for every distro (model/task_queue_service_dependency.go:153-252).
 * sorted[item_off[d] .. + n_sorted[d]) = d.sorted as distro-local item indices: topo.SortStabilized over the edges
 *   dependency -> item with ties in queue order; -1 stands for the nil gonum leaves for a dependency cycle (one per
 *   cyclic component, n_cycles[d] of them); the rest of the distro's slots are -2.
 * unit_items[item_off[d] ..] = the items that have a group, bucketed by group id and stably sorted by GroupIndex inside
 *   each bucket (d.taskGroups[...].tasks); group g of distro d is unit_items[item_off[d] + unit_off[u + g] ..
 *   item_off[d] + unit_off[u + g + 1]) with u = group_off[d] + d (each distro has one closing entry).  A declared
 *   group no item is in is the empty range that starts where the next group starts.
 * Host pointers.  group_off (n_distros + 1) counts the groups of each distro; unit_off holds group_off[n_distros] +
 * n_distros entries.  Every group_id must be -1 or below its distro's group count: -EVG_ERR_INVALID otherwise, checked
 * on the host before anything is copied or launched. */
int evg_dag_rebuild_batch(evg_ctx* ctx, const evg_dag_in* in, const int64_t* item_off, const int64_t* group_off, int32_t n_distros,
                          int32_t* sorted, int32_t* n_sorted, int32_t* n_cycles, int32_t* unit_items, int32_t* unit_off);

/* ---- single-distro wrappers: the per-job drop-in ------------------------- */

/* One distro: PrioritizeTasks for `d` (scheduler/scheduler.go:27). */
int evg_plan_distro(evg_ctx* ctx, const evg_task_soa* tasks, const evg_distro_cfg* cfg,
                    int32_t n_groups, const int32_t* group_max_hosts, int64_t now_ns, uint32_t opts,
                    evg_plan_out* out);
/* One distro: UtilizationBasedHostAllocator(ctx, &HostAllocatorData{...})
 * (scheduler/utilization_based_host_allocator.go:26). */
int evg_alloc_distro(evg_ctx* ctx, const evg_host_soa* hosts, const evg_alloc_cfg* cfg,
                     const evg_queue_info* info, evg_group_info* groups, int32_t n_groups,
                     int64_t now_ns, evg_alloc_result* result, int32_t* status);

#ifdef __cplusplus
}
#endif
#endif /* EVG_SCHED_H */

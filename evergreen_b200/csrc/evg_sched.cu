// evg_sched.cu -- libevgsched.so: CUDA kernels (sm_100a) + the C-ABI of
// include/evg_sched.h.  See DESIGN.md for the data layout and the kernel list.
//
// Distros are routed by size and shape on the host:
//   <= 32 tasks      k_plan_warp (evg_plan_warp.cuh): one warp plans the distro
//   <= 10240 tasks, no GroupVersions, no in-queue dependency edges
//                    k_plan_cta<THREADS,CAP> (evg_plan_cta.cuh): one CTA plans the distro on-chip, several CTAs per
//                    SM, TMA-staged columns, u32 keys; distros it cannot hold (values beyond 32 bits, ...) are
//                    handed back ("punted") to k_plan_smem on the device
//   <= 12288 tasks   k_plan_smem<THREADS,ITEMS> (evg_plan_smem.cuh): one CTA per distro, any unit structure
//   larger           the general path (evg_plan_general.cuh), any size up to 2^21-1 tasks:
//     k_gmark/k_gtask/k_gunit/k_gbest  dependents, per-task pass, multi-member units
//     k_gsum/k_gscan/k_gplace*     canonical pre-arrangement by counting
//     k_ghist/k_gdscan/k_gscatter  segmented stable LSD radix sort of 32-bit keys
//     k_gemit                      ranked queue + TotalValue
//     k_finalize_info              DistroQueueInfo / TaskGroupInfo scalars (scheduler.go:144-158)
// Both:
//   k_breakdown           the 13-field SortingValueBreakdown per ranked task (EVG_OPT_BREAKDOWN)
//   k_alloc<TPD>          utilization host allocator, a warp or a block per distro (utilization_based_host_allocator.go:26-409)
//   k_validate            range check of the distro-local ids the planners index with
// The rows either side of the path (SURVEY.md §8f):
//   k_deps_met            Task.DependenciesMet / AllDependenciesSatisfied (model/task/task.go:632-671,795-821)
//   k_runnable            the task finders' filter + stable compaction (scheduler/task_finder.go:40-317)
//   k_dur_sum/dev/final   expected-duration statistics (model/task/expected_duration.go:36-96)
// No CPU fallback exists in this file: without a device every entry point fails.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <type_traits>
#include <cstdlib>
#include <mutex>
#include <string>
#include <vector>

#include "evg_score.cuh"
#include "evg_intern.h"

using namespace evg;

// --------------------------------------------------------------------------
// host-side helpers
// --------------------------------------------------------------------------
namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(e_ == cudaErrorMemoryAllocation ? EVG_ERR_NOMEM : EVG_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e_), __FILE__, __LINE__);                                \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool owned = true;  // false: p is caller-owned device memory (evg_upload_device)
  void adopt(void* q) {
    if (owned && p) cudaFree(p);
    p = q; cap = 0; owned = false;
  }
  cudaError_t ensure(size_t bytes) {
    if (!owned) { p = nullptr; cap = 0; owned = true; }
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) return e;
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p && owned) cudaFree(p);
    p = nullptr;
    cap = 0;
    owned = true;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// on-chip planner classes <THREADS, ITEMS>: capacity = THREADS*ITEMS tasks per distro
#ifndef EVG_C_THREADS  // shape of the largest on-chip class (threads x tasks per thread = 12288 tasks in 218 KB)
#define EVG_C_THREADS 1024
#define EVG_C_ITEMS 12
#endif
constexpr int kCapA = 128 * 8, kCapB = 256 * 16, kCapC = EVG_C_THREADS * EVG_C_ITEMS;
constexpr int64_t kWideAllocGroups = 1024;  // k_alloc<128> (a block per distro) once some distro has more task groups
constexpr int kCapW = 32;  // k_plan_warp: one warp per distro
constexpr int64_t kGrouplessHosts = 64;  // k_alloc_groupless walks a distro's hosts with one thread: only short walks
constexpr int64_t kBigUnitTasks = 128;  // GroupVersions distros above this size in k_plan_smem's smallest class count as a class of their own
constexpr int64_t kSparseClass = 64;  // a k_plan_smem class of 1025+ task distros with fewer members than this goes to the general path
// second-generation on-chip planner classes <THREADS, CAP, CTAs per SM> (evg_plan_cta.cuh)
constexpr int kNT_A = 128, kNCapA = 1280, kNOccA = 8;
// the smallest k_plan_cta class: a launch list's distros of at most 384 tasks (and few task groups) take 64-thread CTAs,
// sixteen per SM -- twice the distros in flight (configs[3] "total": 10 000 distros of 100 tasks)
constexpr int kNT_S = 64, kNCapS = 384, kNOccS = 16;
constexpr int kNT_B = 256, kNCapB = 5120, kNOccB = 4;
constexpr int kNT_C = 512, kNCapC = 10240, kNOccC = 2;
constexpr uint32_t kInactive = 0xFFFFFFFFu;  // next[]: pair not linked / head[]: empty list
constexpr uint32_t kEnd = 0xFFFFFFFEu;       // next[]: end of list
constexpr uint32_t kNoAnchor = 0xFFFFFFFFu;

}  // namespace

// --------------------------------------------------------------------------
// device-side views
// --------------------------------------------------------------------------
struct DTasks {
  int64_t n, n_edges;
  const int32_t* priority;
  const int64_t* expected;
  const int64_t* qbasis;
  const int64_t* wbasis;
  const int32_t* numdep;
  const int32_t* tgo;
  const int32_t* gid;
  const int32_t* vid;
  const uint32_t* flags;
  const int64_t* dep_off;
  const int32_t* dep_idx;
};

struct DDistros {
  int32_t n;
  const int64_t* task_off;
  const int64_t* group_off;
  const evg_distro_cfg* cfg;
  const int32_t* gmax;
  const int64_t* unit_base;  // n+1: first unit slot of each distro
};

struct SortBuf {
  uint64_t* key_v;  // [T] k_plan_smem: Vmax - V of a distro whose value range exceeds 32 bits
};

struct DWork {
  uint8_t* has_dep;      // [T]
  uint32_t* head;        // [unit slots]
  uint32_t* next;        // [2T+E]
  uint32_t* pair_slot;   // [2T+E]
  uint32_t* edge_task;   // [E]
  uint8_t* edge_live;    // [E] on-chip path: 1 = edge pair linked (not a duplicate membership)
  const uint8_t* route;  // [D] 1 = distro planned by k_plan_smem (general kernels skip it)
  int* err;              // [1] set by k_validate when a distro-local id is out of range; planners then do nothing
  int64_t* unit_v;       // [unit slots] on-chip path: TotalValue of the unit
  uint32_t* unit_a;      // [unit slots] anchor
  uint32_t* unit_n;      // [unit slots] member count
  unsigned long long* unit_mask;  // [unit slots] ranks emitted from the unit (units of <= 64 members)
  uint32_t* best_pair;   // [T]
  SortBuf buf[1];
  evg_queue_info* qinfo; // [D]
  evg_group_info* ginfo; // [G]
};

struct DHosts {
  int64_t n;
  const uint32_t* flags;
  const int32_t* gid;
  const int64_t* expected;
  const int64_t* stddev;
  const int64_t* start;
  const int64_t* host_off;
  const evg_alloc_cfg* cfg;
};

// --------------------------------------------------------------------------
// device helpers
// --------------------------------------------------------------------------
__device__ __forceinline__ int find_distro(const int64_t* __restrict__ off, int lo, int hi, int64_t t) {
  // largest d in [lo, hi] with off[d] <= t  (off[lo] <= t guaranteed)
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (__ldg(off + mid) <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Block-cooperative distro lookup: thread 0 / last thread bracket the block's
// range, then each thread searches only inside the bracket.
__device__ __forceinline__ int block_find_distro(const int64_t* __restrict__ off, int n_distros, int64_t t,
                                                 int64_t n_items) {
  __shared__ int s_lo, s_hi;
  int64_t first = int64_t(blockIdx.x) * blockDim.x;
  if (threadIdx.x == 0) s_lo = find_distro(off, 0, n_distros - 1, first);
  if (threadIdx.x == blockDim.x - 1) {
    int64_t last = first + blockDim.x - 1;
    if (last >= n_items) last = n_items - 1;
    s_hi = find_distro(off, 0, n_distros - 1, last);
  }
  __syncthreads();
  if (t >= n_items) return -1;
  return find_distro(off, s_lo, s_hi, t);
}

__device__ __forceinline__ int64_t warp_sum64(int64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ uint64_t warp_or64(uint64_t v) {
  uint32_t lo = __reduce_or_sync(0xffffffffu, uint32_t(v));
  uint32_t hi = __reduce_or_sync(0xffffffffu, uint32_t(v >> 32));
  return (uint64_t(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t warp_and64(uint64_t v) {
  uint32_t lo = __reduce_and_sync(0xffffffffu, uint32_t(v));
  uint32_t hi = __reduce_and_sync(0xffffffffu, uint32_t(v >> 32));
  return (uint64_t(hi) << 32) | lo;
}
__device__ __forceinline__ void atomic_add64(int64_t* p, int64_t v) {
  if (v != 0) atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)v);
}

// unit slot (distro-local) a task is filed under by its id key (planner.go:434-445)
__device__ __forceinline__ uint32_t own_slot_local(int32_t gid, int32_t vid, uint32_t local_idx, uint32_t n_groups,
                                                   bool group_versions) {
  if (gid >= 0) return uint32_t(gid);
  return n_groups + (group_versions ? uint32_t(vid) : local_idx);
}

__device__ __forceinline__ void link_pair(DWork& W, uint32_t pair, uint32_t slot) {
  W.pair_slot[pair] = slot;
  uint32_t prev = atomicExch(W.head + slot, pair);
  W.next[pair] = (prev == kInactive) ? kEnd : prev;
}

__device__ __forceinline__ uint32_t pair_task(const DTasks& T, const DWork& W, uint32_t p) {
  if (p < uint32_t(T.n)) return p;
  if (p < uint32_t(2 * T.n)) return p - uint32_t(T.n);
  return W.edge_task[p - uint32_t(2 * T.n)];
}

#include "evg_plan_smem.cuh"
#include "evg_plan_warp.cuh"
#include "evg_plan_cta.cuh"
#include "evg_plan_general.cuh"
#include "evg_legacy.cuh"
#include "evg_dag.cuh"

// --------------------------------------------------------------------------
// kernels (general path: any distro size)
// --------------------------------------------------------------------------

// Distro-local ids index device tables directly, so they are range-checked once per upload:
// group_id in [-1, n_groups), version_id in [0, n_versions), dep_idx in [0, tasks of the distro).
__global__ void __launch_bounds__(256) k_validate(DTasks T, DDistros D, DWork W, int64_t t_begin, int64_t t_end) {
  const int64_t t = t_begin + int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= t_end) return;
  const int d = find_distro(D.task_off, 0, D.n - 1, t);
  const int64_t tn = D.task_off[d + 1] - D.task_off[d];
  const int64_t ng = D.group_off[d + 1] - D.group_off[d];
  const int32_t gid = T.gid[t], vid = T.vid[t];
  bool bad = gid < -1 || gid >= ng || vid < 0 || vid >= D.cfg[d].n_versions;
  if (T.n_edges > 0) {
    const int64_t e0 = T.dep_off[t], e1 = T.dep_off[t + 1];
    bad = bad || e1 < e0 || e0 < 0 || e1 > T.n_edges;
    if (!bad)
      for (int64_t e = e0; e < e1; e++) bad = bad || T.dep_idx[e] < 0 || T.dep_idx[e] >= tn;
  }
  if (bad) atomicOr(W.err, 1);
}

// Task.DependenciesMet over direct dependencies (model/task/task.go:529-543,632-671).
struct DDeps {
  int64_t n_tasks;
  const int64_t* dep_off;
  const uint8_t* dep_kind;
  const int32_t* dep_ref;
  const uint8_t* dep_want;
  const uint8_t* task_state;
  const uint8_t* task_pre;
  const uint8_t* ext_state;
  int64_t n_ext;
};
// met[t] bit 0: Task.DependenciesMet (with the HasDependenciesMet short-circuit); with `both`, bit 1:
// Task.AllDependenciesSatisfied (task.go:795-821: the same walk without the short-circuit).
__global__ void __launch_bounds__(256) k_deps_met(DDeps X, uint8_t* met, int* err, int both, const int64_t* __restrict__ dep_fin,
                                                  int64_t now, int64_t* __restrict__ met_time) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= X.n_tasks) return;
  const int64_t e0 = X.dep_off[t], e1 = X.dep_off[t + 1];
  bool ok = true;
  const bool shortcut = (X.task_pre[t] & (EVG_TP_OVERRIDE | EVG_TP_MET_TIME)) != 0;  // HasDependenciesMet task.go:3393
  if (e1 > e0 && (both || !shortcut)) {
    for (int64_t e = e0; e < e1 && ok; e++) {
      const uint8_t kind = X.dep_kind[e];
      const int32_t ref = X.dep_ref[e];
      uint8_t st;
      if (kind == EVG_DEP_IN_QUEUE) {
        if (ref < 0 || ref >= X.n_tasks) { atomicOr(err, 1); ok = false; break; }
        st = X.task_state[ref];
      } else if (kind == EVG_DEP_EXTERNAL) {
        if (ref < 0 || ref >= X.n_ext) { atomicOr(err, 1); ok = false; break; }
        st = X.ext_state[ref];
      } else {
        ok = false;  // lookup error -> false (scheduler.go:161-168)
        break;
      }
      const uint32_t status = st & EVG_TS_STATUS_MASK;
      switch (X.dep_want[e]) {  // SatisfiesDependency task.go:529-543
        case EVG_WANT_SUCCESS: ok = status == 0; break;
        case EVG_WANT_FAILED: ok = status == 1; break;
        case EVG_WANT_ANY: ok = status < 2 || (st & EVG_TS_BLOCKED); break;
        default: ok = false;
      }
    }
  }
  met[t] = uint8_t(((ok || shortcut) ? 1 : 0) | ((both && ok) ? 2 : 0));
  if (met_time) {
    // a fresh evaluation that comes out met stamps DependenciesMetTime (setDependenciesMetTime, task.go:653,673-684):
    // the latest non-zero FinishedAt of the dependencies (utility.IsZeroTime: Go's zero time or the Unix epoch), else now
    int64_t stamp = EVG_TIME_ZERO;
    if (ok && !shortcut && e1 > e0) {
      if (dep_fin)
        for (int64_t e = e0; e < e1; e++) {
          const int64_t f = dep_fin[e];
          if (f != EVG_TIME_ZERO && f != 0 && f > stamp) stamp = f;
        }
      if (stamp == EVG_TIME_ZERO || stamp == 0) stamp = now;
    }
    met_time[t] = stamp;
  }
}

// The resident planner inputs take the device's own verdict: the EVG_TF_DEPS_MET bit of every task, and for freshly
// stamped tasks the later of the wait basis the caller gave (ScheduledTime) and the stamp (scheduler.go:119-122).
__global__ void __launch_bounds__(256) k_apply_deps(int64_t n, const uint8_t* __restrict__ met, const int64_t* __restrict__ met_time,
                                                    uint32_t* __restrict__ flags, int64_t* __restrict__ wbasis) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n) return;
  flags[t] = (flags[t] & ~EVG_TF_DEPS_MET) | ((met[t] & 1) ? EVG_TF_DEPS_MET : 0u);
  const int64_t s = met_time[t];
  if (s != EVG_TIME_ZERO && s > wbasis[t]) wbasis[t] = s;
}

// The task finders' filter (task_finder.go:40-197) with a stable per-distro compaction: one block per distro,
// 256 tasks per step, ballot + warp totals for the positions.
struct DRunnable {
  int64_t n_tasks;
  int32_t n_distros, n_projects;
  const int64_t* task_off;
  const uint8_t* sched;
  const int32_t* project;
  const uint8_t* project_flags;
  const int64_t* valid_off;
  const int32_t* valid_idx;
  const uint8_t* finder;
  const uint8_t* met;  // k_deps_met(both) output, or nullptr
};
__global__ void __launch_bounds__(256) k_runnable(DRunnable R, int32_t* __restrict__ out, int64_t* __restrict__ count, int* err) {
  constexpr int ITEMS = 4;  // candidates per thread and step: their loads are in flight together, one barrier pair per 1024
  const int d = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned full = 0xffffffffu;
  const int64_t base = R.task_off[d], end = R.task_off[d + 1];
  const int64_t v0 = R.valid_off[d], v1 = R.valid_off[d + 1];
  const uint32_t finder = R.finder[d];
  const uint32_t met_bit = finder == EVG_FINDER_LEGACY ? 1u : 2u;
  __shared__ uint32_t s_cnt[ITEMS * 8];  // survivors of (item j, warp w), in output order j-major
  int64_t running = 0;  // kept identically by every thread
  for (int64_t c0 = base; c0 < end; c0 += 256 * ITEMS) {
    uint32_t sq[ITEMS], mt[ITEMS];
    int32_t pj[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
      const int64_t t = c0 + j * 256 + threadIdx.x;
      const bool in = t < end;
      sq[j] = in ? R.sched[t] : 0u;
      pj[j] = in ? R.project[t] : -1;
      mt[j] = (in && finder != EVG_FINDER_NO_DEPS) ? R.met[t] : 3u;
    }
    bool keep[ITEMS];
    unsigned m[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
      const uint32_t q = sq[j];
      // schedulableHostTasksQuery (model/task/db.go:671-689)
      bool k = (q & EVG_SQ_ACTIVATED) && (q & EVG_SQ_UNDISPATCHED) && (q & EVG_SQ_PRIORITY_OK) && (q & EVG_SQ_HOST_PLATFORM) &&
               (!(q & EVG_SQ_UNATTAINABLE) || (q & EVG_SQ_OVERRIDE_DEPS));
      const int32_t p = pj[j];
      if (p >= R.n_projects) { atomicOr(err, 1); k = false; }
      else if (p < 0) k = false;  // "could not find project for task" (task_finder.go:57-67)
      else if (k) {
        const uint32_t pf = R.project_flags[p];
        // ProjectCanDispatchTask (model/project_ref.go:3441-3462)
        if (!(pf & EVG_PF_ENABLED) && !((q & EVG_SQ_GITHUB_PR) && (pf & EVG_PF_HIDDEN))) k = false;
        if (pf & EVG_PF_DISPATCHING_DISABLED) k = false;
        if ((q & EVG_SQ_PATCH_REQUEST) && (pf & EVG_PF_PATCHING_DISABLED)) k = false;
        if (k && v1 > v0) {  // len(d.ValidProjects) > 0 && !contains(ref.Id) (task_finder.go:74-84)
          bool found = false;
          for (int64_t x = v0; x < v1 && !found; x++) found = R.valid_idx[x] == p;
          k = found;
        }
        if (k) k = (mt[j] & met_bit) != 0;  // the finder's dependency predicate (NO_DEPS reads 3: always met)
      }
      keep[j] = k;
      m[j] = __ballot_sync(full, k);
      if (lane == 0) s_cnt[j * 8 + warp] = __popc(m[j]);
    }
    __syncthreads();
    uint32_t total = 0, before[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
#pragma unroll
      for (int w = 0; w < 8; w++) {
        if (w == warp) before[j] = total;
        total += s_cnt[j * 8 + w];
      }
    }
#pragma unroll
    for (int j = 0; j < ITEMS; j++)
      if (keep[j]) out[base + running + before[j] + __popc(m[j] & ((1u << lane) - 1u))] = int32_t(c0 + j * 256 + threadIdx.x - base);
    running += total;
    __syncthreads();
  }
  for (int64_t i = base + running + threadIdx.x; i < end; i += 256) out[i] = -1;  // unused tail of the distro's slots
  if (threadIdx.x == 0) count[d] = running;
}

// Expected-duration statistics (model/task/expected_duration.go:36-96): the $match, then per key count / sum, then
// the squared deviations from floor(mean) as an exact 128-bit integer, then one rounding per output.
struct DDur {
  int64_t n_rows;
  int32_t n_keys;
  const int32_t* key;
  const int64_t* taken;
  const int64_t* start;
  const int64_t* finish;
  const uint8_t* flags;
  int64_t w0, w1;
  unsigned long long* cnt;  // [n_keys]
  unsigned long long* sum;  // [n_keys] two's complement
  unsigned long long* sq_lo;
  unsigned long long* sq_hi;
};
__device__ __forceinline__ bool dur_row_matches(const DDur& X, int64_t r) {
  const uint32_t f = X.flags[r];
  return (f & EVG_DR_COMPLETED) && !(f & EVG_DR_TIMED_OUT) && X.start[r] > X.w0 && X.finish[r] <= X.w1;
}
__global__ void __launch_bounds__(256) k_dur_sum(DDur X, int* err) {
  const int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= X.n_rows) return;
  const int32_t k = X.key[r];
  if (k < 0 || k >= X.n_keys) { atomicOr(err, 1); return; }
  if (!dur_row_matches(X, r)) return;
  atomicAdd(X.cnt + k, 1ull);
  atomicAdd(X.sum + k, (unsigned long long)X.taken[r]);
}
__global__ void __launch_bounds__(256) k_dur_dev(DDur X) {
  const int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= X.n_rows) return;
  const int32_t k = X.key[r];
  if (k < 0 || k >= X.n_keys || !dur_row_matches(X, r)) return;
  const int64_t n = int64_t(X.cnt[k]), s = int64_t(X.sum[k]);
  int64_t m0 = s / n;
  if ((s % n) < 0) m0 -= 1;  // floor
  const int64_t dv = X.taken[r] - m0;
  const unsigned long long a = dv < 0 ? (unsigned long long)(-dv) : (unsigned long long)dv;
  const unsigned long long lo = a * a, hi = __umul64hi(a, a);
  const unsigned long long old = atomicAdd(X.sq_lo + k, lo);
  const unsigned long long carry = (old + lo < old) ? 1ull : 0ull;
  if (hi + carry) atomicAdd(X.sq_hi + k, hi + carry);
}
__global__ void __launch_bounds__(256) k_dur_final(DDur X, evg_duration_stat* out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= X.n_keys) return;
  evg_duration_stat st;
  st.count = int64_t(X.cnt[k]);
  st.mean_ns = 0.0;
  st.stddev_ns = 0.0;
  if (st.count > 0) {
    const int64_t n = st.count, s = int64_t(X.sum[k]);
    int64_t m0 = s / n, rem = s % n;
    if (rem < 0) { m0 -= 1; rem += n; }
    const double dn = __ll2double_rn(n);
    st.mean_ns = __ddiv_rn(__ll2double_rn(s), dn);
    // variance = S2/n - (rem/n)^2 with S2 = sum (x - floor(mean))^2 held exactly in 128 bits
    const double s2 = __dadd_rn(__dmul_rn(__ull2double_rn(X.sq_hi[k]), 18446744073709551616.0), __ull2double_rn(X.sq_lo[k]));
    const double fr = __ddiv_rn(__ll2double_rn(rem), dn);
    double var = __dadd_rn(__ddiv_rn(s2, dn), -__dmul_rn(fr, fr));
    if (var < 0.0) var = 0.0;
    st.stddev_ns = __dsqrt_rn(var);
  }
  out[k] = st;
}

// The 13-field SortingValueBreakdown of the unit each ranked task was emitted
// from (planner.go:472-476, model/task/task.go:3990-4038); both paths.  Row j of `breakdown` is rank j - row_off[d]
// of the distro d with row_off[d] <= j < row_off[d + 1]: row_off = task_off gives every rank, the head offsets of
// evg_run_resident_head the first min(length, cap).
__global__ void __launch_bounds__(256) k_breakdown(DTasks T, DDistros D, DWork W, const URec* rec, int64_t now, int any_complex,
                                                   const int32_t* order, const int64_t* row_off, int64_t n_rows, int64_t* breakdown) {
  if (*W.err) return;
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int d = block_find_distro(row_off, D.n, t, n_rows);
  if (d < 0) return;
  const int64_t base = D.task_off[d];
  const int64_t g = base + order[base + t - row_off[d]];
  UnitAcc a;
  acc_init(a);
  const uint32_t bp = any_complex ? W.best_pair[g] : kInactive;
  if (bp == kInactive) {
    acc_add(a, now, T.priority[g], T.expected[g], T.qbasis[g], T.numdep[g], T.gid[g], T.flags[g]);
  } else if (W.route[d]) {  // on-chip planners leave member lists (breakdown mode only)
    for (uint32_t q = W.head[W.pair_slot[bp]]; q < kEnd; q = W.next[q]) {
      const uint32_t tq = pair_task(T, W, q);
      acc_add(a, now, T.priority[tq], T.expected[tq], T.qbasis[tq], T.numdep[tq], T.gid[tq], T.flags[tq]);
    }
  } else {  // general path: the unit table
    const uint32_t slot = W.pair_slot[bp];
    const URec* run = rec + W.head[slot];
    const uint32_t cnt = W.unit_n[slot];
    for (uint32_t i = 0; i < cnt; i++) rec_acc(a, now, rec_load(run + i));
  }
  int64_t bd[EVG_BD_N];
  unit_value(a, D.cfg[d], bd);
  for (int k = 0; k < EVG_BD_N; k++) breakdown[t * EVG_BD_N + k] = bd[k];
}

// scheduler.go:144-158: scalars of DistroQueueInfo / TaskGroupInfo that are not sums.
__global__ void k_finalize_info(DDistros D, DWork W, int32_t d_begin, int32_t d_end, int64_t g_begin, int64_t g_end) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t di = d_begin + i;
  if (di < d_end && !W.route[di]) {  // on-chip planners write their rows whole (and may be doing so right now on another stream)
    evg_queue_info* q = W.qinfo + di;
    q->length = D.task_off[di + 1] - D.task_off[di];
    q->max_duration_threshold = D.cfg[di].target_time_ns;
    q->secondary_queue = q->secondary_queue != 0;
    q->has_ungrouped = q->has_ungrouped != 0;
  }
  // group rows between the first and the last general-path distro; an on-chip distro in between stores the same value
  if (g_begin + i < g_end) W.ginfo[g_begin + i].max_hosts = D.gmax[g_begin + i];
}

// UtilizationBasedHostAllocator (utilization_based_host_allocator.go:26-130 and
// the helpers it calls).  FP64 sums run in host-index order (the canonical
// order; the reference's channel order is nondeterministic, allocator.go:381-391).
struct GroupScratch {
  int32_t n_hosts;
  int32_t n_free;
  double soon;
};

__device__ int eval_group(const evg_alloc_cfg& c, const evg_group_info& info, int64_t threshold, int64_t max_hosts,
                          int64_t n_hosts, int64_t n_free, double soon, int64_t* out_new, int64_t* out_free) {
  // evalHostUtilization allocator.go:135-220
  *out_new = 0;
  *out_free = 0;
  if (c.provider == EVG_PROVIDER_STATIC) return EVG_ALLOC_OK;
  if (c.has_pool) {
    if (!c.parent_found) return EVG_ALLOC_ERR_PARENT_MISSING;
    max_hosts = int64_t(c.parent_maximum_hosts) * int64_t(c.pool_max_containers);
  }
  if (c.future_host_fraction > 1.0) return EVG_ALLOC_ERR_FUTURE_FRACTION;
  const int64_t exp_free = n_free + d2i_floor(soon);  // allocator.go:317
  const int64_t overdue = c.waits_over_thresh_feedback ? info.count_wait_over_threshold : 0;
  const int64_t short_ns = wsub(info.expected_duration, info.duration_over_threshold);
  int64_t n = calc_new_hosts_needed(short_ns, threshold, exp_free, info.count_duration_over_threshold, overdue,
                                    info.count_dep_filled_merge_queue_tasks, !c.round_up);
  if (n > info.count) n = info.count;
  if (is_max_hosts_capacity(max_hosts, c.has_pool != 0, c.pool_max_containers, n, n_hosts)) n = max_hosts - n_hosts;
  if (n < 0) n = 0;
  if (max_hosts < 1) return EVG_ALLOC_ERR_POOL_SIZE;
  *out_new = n;
  *out_free = exp_free;
  return EVG_ALLOC_OK;
}

// TPD threads per distro: a warp (four distros per block) when task groups are few, the whole 128-thread block
// when some distro has thousands of them (a distro of a million tasks has tens of thousands).  The first warp
// of the team walks the hosts in index order; the lane that owns a bucket (lane 0 for "", lane g%32 for group
// g) does that bucket's updates, so every bucket's FP64 sum is accumulated in host order while buckets proceed
// in parallel.  The team then evaluates the task groups; per-group results are integers, so the reduction is exact.
template <int TPD>
__global__ void __launch_bounds__(128, TPD == 32 ? 6 : 4) k_alloc(DHosts H, int32_t d_begin, int32_t n_distros, const int64_t* group_off,
                                               const evg_queue_info* qinfo, evg_group_info* ginfo, GroupScratch* gs,
                                               int64_t now, evg_alloc_result* result, int32_t* status, int skip_groupless,
                                               const int32_t* list, int32_t n_list) {
  constexpr int TEAMS = 128 / TPD, TW = TPD / 32;  // teams per block, warps per team
  const int team = threadIdx.x / TPD, tt = threadIdx.x % TPD;
  const int ti = int(blockIdx.x) * TEAMS + team;
  if (list && ti >= n_list) return;  // team-uniform; a team never shares a barrier with another
  const int d = list ? list[ti] : d_begin + ti;  // `list`: the distros k_alloc_groupless does not take (built at upload)
  const int lane = threadIdx.x & 31, warp = tt >> 5;
  const unsigned full = 0xffffffffu;
  if (d >= n_distros) return;  // team-uniform (n_distros = end of the range)
  auto team_sync = [&]() { if (TPD == 128) __syncthreads(); else __syncwarp(); };
  __shared__ long long sh_nfree[TEAMS], sh_uhosts[TEAMS], sh_ufree[TEAMS], sh_req[TEAMS][TW], sh_fre[TEAMS][TW];
  __shared__ double sh_usoon[TEAMS];
  __shared__ int sh_st[TEAMS][TW];
  long long& s_nfree = sh_nfree[team]; long long& s_uhosts = sh_uhosts[team]; long long& s_ufree = sh_ufree[team];
  double& s_usoon = sh_usoon[team];
  long long* s_req = sh_req[team]; long long* s_fre = sh_fre[team];
  int* s_st = sh_st[team];
  const int64_t g0 = group_off[d], g1 = group_off[d + 1];
  const int64_t h0 = H.host_off[d], h1 = H.host_off[d + 1];
  if (skip_groupless && g1 == g0 && h1 - h0 <= kGrouplessHosts) return;  // team-uniform: k_alloc_groupless plans it, one thread instead of a warp
  const evg_alloc_cfg c = H.cfg[d];
  const evg_queue_info qi = qinfo[d];
  const int64_t threshold = qi.max_duration_threshold;
  const int64_t n_existing = h1 - h0;
  // IsFree count (allocator.go:33-37), bucket sizes (groupByTaskGroup :223-260), soon-to-be-free sums (:324-394).
  // The buckets of kCache task groups at a time live in SHARED memory while the hosts are walked (a distro with more
  // groups walks its hosts once per stretch of kCache): a bucket update used to be a load-add-store on global scratch,
  // an L2 round trip per host in a serial loop.
  constexpr int kCache = TPD == 32 ? 128 : 512;
  __shared__ GroupScratch sh_gs[TEAMS][kCache];
  GroupScratch* sg = sh_gs[team];
  if (warp == 0) {
    int64_t n_free_all = 0, u_hosts = 0, u_free = 0;
    double u_soon = 0.0;
    const int64_t ng = g1 - g0;
    for (int64_t gb = 0; gb == 0 || gb < ng; gb += kCache) {
      const bool first = gb == 0;  // the "" bucket and the free count are taken on the first walk only
      const int64_t ge = ng - gb < kCache ? ng - gb : kCache;  // groups of this stretch: [gb, gb + ge)
      for (int64_t i = lane; i < ge; i += 32) { sg[i].n_hosts = 0; sg[i].n_free = 0; sg[i].soon = 0.0; }
      __syncwarp();
      // 32 hosts per trip: lane L loads host hc + L (coalesced) and evaluates ITS host's soon-to-be-free term
      // (allocator.go:357-378: an FP64 division and a dozen overflow-checked integer steps, independent of the bucket).
      // Everything that is a COUNT is order-free and taken in parallel (lane-local counters, shared-memory atomics on the
      // bucket); only the FP64 sums need host order, so only the RUNNING hosts of this stretch are replayed in index
      // order through shuffles, the bucket's owner lane adding the term.
      for (int64_t hc = h0; hc < h1; hc += 32) {
        const int64_t hm = hc + lane;
        const bool in = hm < h1;
        const uint32_t my_f = in ? H.flags[hm] : 0u;
        const int32_t my_g = in ? H.gid[hm] : -2;
        const bool my_free = in && !(my_f & EVG_HF_RUNNING) && !(my_f & EVG_HF_TEARDOWN);
        const bool my_run = in && (my_f & EVG_HF_RUNNING) && (my_f & EVG_HF_RT_FOUND);
        const bool my_none = in && my_g == EVG_HG_NONE;
        const bool my_here = in && my_g >= gb && my_g < gb + ge;  // a bucket of this stretch
        const double my_term = my_run ? soon_free_term(now, H.expected[hm], H.stddev[hm], H.start[hm], threshold, c.future_host_fraction) : 0.0;
        if (first) {
          n_free_all += my_free;
          u_hosts += my_none;
          u_free += my_none && my_free;
        }
        if (my_here) {
          atomicAdd(&sg[my_g - gb].n_hosts, 1);
          if (my_free) atomicAdd(&sg[my_g - gb].n_free, 1);
        }
        unsigned todo = __ballot_sync(full, my_run && (my_here || (first && my_none)));
        while (todo) {  // warp-uniform
          const int j = __ffs(todo) - 1;
          todo &= todo - 1u;
          const int32_t g = __shfl_sync(full, my_g, j);
          const double term = __shfl_sync(full, my_term, j);
          if (g == EVG_HG_NONE) { if (lane == 0) u_soon = fadd64(u_soon, term); }
          else if (((g - int32_t(gb)) & 31) == lane) sg[g - gb].soon = fadd64(sg[g - gb].soon, term);
        }
      }
      __syncwarp();
      for (int64_t i = lane; i < ge; i += 32) gs[g0 + gb + i] = sg[i];
    }
    n_free_all = warp_sum64(n_free_all); u_hosts = warp_sum64(u_hosts); u_free = warp_sum64(u_free);  // lane-local counts
    if (lane == 0) { s_nfree = n_free_all; s_uhosts = u_hosts; s_ufree = u_free; s_usoon = u_soon; }
  }
  team_sync();
  const int64_t n_free_all = s_nfree;
  int32_t st = EVG_ALLOC_OK;
  int64_t n_new = 0, n_free_out = n_free_all;
  if (c.provider != EVG_PROVIDER_DOCKER && n_existing >= c.maximum_hosts) {
    n_new = 0;  // allocator.go:39-48
  } else if (c.disabled) {
    n_new = int64_t(c.minimum_hosts) - n_existing;  // allocator.go:51-66
    if (n_new < 0) n_new = 0;
  } else {  // team-uniform branch: c and the host count are per distro
    int64_t required = 0, free_approx = 0;
    // "" bucket exists when standalone tasks are queued or hosts are bucketed under ""
    if (tt == 0 && (qi.has_ungrouped || s_uhosts > 0)) {
      int64_t n, f;
      st = eval_group(c, qi.ungrouped, threshold, c.maximum_hosts, s_uhosts, s_ufree, s_usoon, &n, &f);
      required += n;
      free_approx += f;
    }
    for (int64_t g = g0 + tt; g < g1; g += TPD) {
      evg_group_info* gi = ginfo + g;
      if (gi->count == 0) continue;  // allocator.go:84-86
      int64_t n, f;
      const int e = eval_group(c, *gi, threshold, gi->max_hosts, gs[g].n_hosts, gs[g].n_free, gs[g].soon, &n, &f);
      if (e != EVG_ALLOC_OK) { st = max(st, e); continue; }
      required += n;
      free_approx += f;
      gi->count_free = f;  // allocator.go:107-110
      gi->count_required = n;
    }
    // a data error is distro-wide (fraction, parent) or the pool-size check of some group: any thread's error wins
    st = __reduce_max_sync(full, st);
    required = warp_sum64(required);
    free_approx = warp_sum64(free_approx);
    if (TW > 1) {
      if (lane == 0) { s_st[warp] = st; s_req[warp] = required; s_fre[warp] = free_approx; }
      team_sync();
      st = s_st[0]; required = s_req[0]; free_approx = s_fre[0];
#pragma unroll
      for (int w = 1; w < TW; w++) { st = max(st, s_st[w]); required += s_req[w]; free_approx += s_fre[w]; }
    }
    if (st == EVG_ALLOC_OK) {
      if (required + n_free_all > qi.length_with_dependencies_met) required = qi.length_with_dependencies_met - n_free_all;
      if (required < 0) required = 0;
      int64_t topup = 0;
      if (n_existing + required < c.minimum_hosts) topup = c.minimum_hosts - (n_existing + required);
      n_new = required + topup;
      n_free_out = free_approx;
    } else {
      n_new = 0;  // (0, len(freeHosts), err) allocator.go:99-101
      n_free_out = n_free_all;
    }
  }
  if (tt == 0) {
    int64_t deficit = wsub(qi.expected_duration, wmul(n_free_out, threshold));
    if (deficit < 0) deficit = 0;
    result[d].new_hosts = int32_t(n_new);
    result[d].free_hosts = int32_t(n_free_out);
    result[d].deficit_ns = deficit;
    status[d] = st;
  }
}

// Distros without task groups -- nearly all of a tick with 10^5 small queues -- have one bucket (""): the whole
// decision is a scalar chain over a handful of hosts, so ONE THREAD plans a distro (k_alloc<32> spent a warp, and its
// 13 us latency chain, on each).  Same arithmetic in the same order as k_alloc: hosts in index order, FP64 sum of the
// soon-to-be-free terms, eval_group on the "" bucket, the same tail.
__global__ void __launch_bounds__(128) k_alloc_groupless(DHosts H, int32_t d_begin, int32_t n_distros, const int64_t* group_off,
                                                         const evg_queue_info* qinfo, int64_t now, evg_alloc_result* result, int32_t* status) {
  const int d = d_begin + int(blockIdx.x * blockDim.x + threadIdx.x);
  if (d >= n_distros) return;
  const int64_t h0 = H.host_off[d], h1 = H.host_off[d + 1];
  if (group_off[d + 1] != group_off[d] || h1 - h0 > kGrouplessHosts) return;  // k_alloc's
  const evg_alloc_cfg c = H.cfg[d];
  const evg_queue_info qi = qinfo[d];
  const int64_t threshold = qi.max_duration_threshold;
  const int64_t n_existing = h1 - h0;
  int64_t n_free_all = 0, u_hosts = 0, u_free = 0;
  double u_soon = 0.0;
  for (int64_t h = h0; h < h1; h++) {
    const uint32_t f = H.flags[h];
    const bool is_free = !(f & EVG_HF_RUNNING) && !(f & EVG_HF_TEARDOWN);
    n_free_all += is_free;
    if (H.gid[h] == EVG_HG_NONE) {  // a host bucketed under a group name the queue does not have joins no bucket (allocator.go:223-260)
      const bool running = (f & EVG_HF_RUNNING) && (f & EVG_HF_RT_FOUND);
      u_hosts++;
      u_free += is_free;
      if (running) u_soon = fadd64(u_soon, soon_free_term(now, H.expected[h], H.stddev[h], H.start[h], threshold, c.future_host_fraction));
    }
  }
  int32_t st = EVG_ALLOC_OK;
  int64_t n_new = 0, n_free_out = n_free_all;
  if (c.provider != EVG_PROVIDER_DOCKER && n_existing >= c.maximum_hosts) {
    n_new = 0;  // allocator.go:39-48
  } else if (c.disabled) {
    n_new = int64_t(c.minimum_hosts) - n_existing;  // allocator.go:51-66
    if (n_new < 0) n_new = 0;
  } else {
    int64_t required = 0, free_approx = 0;
    if (qi.has_ungrouped || u_hosts > 0) {
      int64_t n, f;
      st = eval_group(c, qi.ungrouped, threshold, c.maximum_hosts, u_hosts, u_free, u_soon, &n, &f);
      required += n;
      free_approx += f;
    }
    if (st == EVG_ALLOC_OK) {
      if (required + n_free_all > qi.length_with_dependencies_met) required = qi.length_with_dependencies_met - n_free_all;
      if (required < 0) required = 0;
      int64_t topup = 0;
      if (n_existing + required < c.minimum_hosts) topup = c.minimum_hosts - (n_existing + required);
      n_new = required + topup;
      n_free_out = free_approx;
    } else {
      n_new = 0;  // (0, len(freeHosts), err) allocator.go:99-101
      n_free_out = n_free_all;
    }
  }
  int64_t deficit = wsub(qi.expected_duration, wmul(n_free_out, threshold));
  if (deficit < 0) deficit = 0;
  result[d].new_hosts = int32_t(n_new);
  result[d].free_hosts = int32_t(n_free_out);
  result[d].deficit_ns = deficit;
  status[d] = st;
}

// --------------------------------------------------------------------------
// context
// --------------------------------------------------------------------------
struct evg_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  // Entry points may be called from any OS thread (cgo runs a call on whatever M the goroutine sits on): every
  // extern "C" function that takes a context holds this lock for its duration, so one context serialises its
  // callers and several contexts (one per worker) run side by side on their own streams.
  std::recursive_mutex mu;
  cudaEvent_t ev_begin = nullptr, ev_sort0 = nullptr, ev_sort1 = nullptr, ev_end = nullptr, ev_gt0 = nullptr, ev_gt1 = nullptr;
  bool general_timed = false;
  // ring of event pairs around the dominant kernel of a tick: per-run kernel time without syncing inside a timed loop
  static constexpr int kRing = 128;
  cudaEvent_t ring0[kRing] = {}, ring1[kRing] = {};
  int64_t runs = 0;
  int64_t max_groups = 0;  // most task groups in any distro: picks the allocator's team width
  int sort_slot = -1;      // ring slot of the last run's dominant-kernel pair
  // route streams: the size classes of one tick are independent until the allocator, so they run side by side
  static constexpr int kAux = 6;
  cudaStream_t s_aux[kAux] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kAux] = {};
  // resident inputs
  bool have_tasks = false, have_hosts = false;
  int64_t T = 0, E = 0, G = 0, H = 0, U = 0, NT = 0, t_pad = 0;
  int32_t Dn = 0;
  int any_complex = 0;
  int64_t launches = 0;
  bool timed = false;
  bool adopted = false;  // task columns are caller-owned device memory (evg_upload_device)
  bool deps_resident = false;  // evg_upload_with_deps left the verdicts and stamps of this tick on the device
  DevBuf b_prio, b_exp, b_qb, b_wb, b_nd, b_tgo, b_gid, b_vid, b_flags, b_depoff, b_depidx;
  DevBuf b_taskoff, b_groupoff, b_cfg, b_gmax, b_unitbase;
  DevBuf b_hasdep, b_head, b_next, b_pslot, b_etask, b_elive, b_ca, b_crk, b_bestpair;
  DevBuf b_rn0, b_rn1, b_rn2, b_rn3, b_rn4, b_rn5, b_rn6, b_rn7;
  DevBuf b_pf[39];  // evg_plan_from_finder: finder tables, candidate columns, compacted columns, edge scratch, group slots
  DevBuf b_err, b_dx0, b_dx1, b_dx2, b_dx3, b_dx4, b_dx5, b_dx6, b_dx7;
  DevBuf b_route, b_listW, b_listA, b_listB, b_listC, b_listG, b_listNA, b_listNB, b_listNC, b_unitv, b_unita, b_unitn, b_unitmask;
  DevBuf b_punt, b_puntcnt;
  int32_t nW = 0, nA = 0, nB = 0, nC = 0, nNA = 0, nNB = 0, nNC = 0, n_general = 0;  // distros per route
  int64_t max_cta_tasks = 0;  // largest distro routed to k_plan_cta: picks the fallback instance for what it hands back
  int32_t nNA_big = 0;  // leading entries of the largest-first NA list that need the 128-thread instance
  std::vector<int32_t> h_listW, h_listA, h_listB, h_listC, h_listNA, h_listNB, h_listNC;  // host copies (ascending distro ids)
  DevBuf b_alist;            // distros k_alloc plans itself (task groups, or more than kGrouplessHosts hosts), listed by upload_hosts
  int64_t n_alist = 0;
  bool alist_valid = false;
  DevBuf b_lptA, b_lptB, b_lptC, b_lptNA, b_lptNB, b_lptNC;  // the same lists, largest distro first: the resident tick's launch order
  std::vector<int64_t> h_taskoff, h_groupoff, h_unitbase, h_edgeoff, h_dtileoff;
  std::vector<int32_t> h_listG;
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  static constexpr int kMaxChunks = 16;
  cudaEvent_t ev_h[kMaxChunks] = {}, ev_c[kMaxChunks] = {};
  int general_complex = 0;
  int64_t Tgc = 0;  // tasks in general-path distros that can hold multi-member units (work-list capacity)
  int64_t max_general = 0;  // tasks in the longest general-path distro
  DevBuf b_kv, b_vmm, b_klo[2], b_khi[2], b_ix[2], b_e, b_tilesum, b_gmisc;
  DevBuf b_tiledistro, b_tilestart, b_dtileoff, b_tilehist, b_clist, b_rec, b_tie, b_hlist, b_usum, b_upd;
  DevBuf b_qinfo, b_ginfo, b_order, b_tv, b_bd;
  DevBuf b_hsel, b_hhist, b_heq, b_hoff;  // evg_run_resident_head: selection state, digit counts, tile counts, head row offsets
  int32_t head_cap = 0;                   // 0: the last run ranked every task; else only the first min(length, head_cap)
  std::vector<int64_t> h_headoff;         // [D+1] offsets of each distro's head rows (the breakdown rows of a head run)
  DevBuf b_hflags, b_hgid, b_hexp, b_hstd, b_hstart, b_hostoff, b_acfg, b_gs, b_result, b_status;
  bool bd_valid = false;
  evg_alloc_result* ext_result = nullptr;  // caller-owned send buffer (evg_bind_result_buffer)
  int64_t ext_capacity = 0;
  evg_alloc_result* result_ptr() const { return ext_result ? ext_result : b_result.as<evg_alloc_result>(); }
};

namespace {

DTasks dtasks(const evg_ctx* c);
DDistros ddistros(const evg_ctx* c);
DWork dwork(const evg_ctx* c);
DGen dgen(const evg_ctx* c);
inline unsigned grid_for(int64_t n, int block) { return unsigned((n + block - 1) / block); }

// Columns are padded so that 128-bit loads and TMA copies that start inside the table may run past its last row.
constexpr int64_t kColPad = 8;

// Route every distro of the tick, stage the small tables, size the work buffers.  Columns: copied from the host
// (copy_columns), left for the pipelined call to copy chunk by chunk, or adopted from caller-owned device memory.
// `edge_off` (D+1, host) is dep_off sampled at the distro boundaries; NULL when the host can read t->dep_off itself.
int upload_tasks(evg_ctx* c, const evg_task_soa* t, const evg_distro_table* dt, bool copy_columns = true, bool adopt = false,
                 const int64_t* edge_off = nullptr) {
  if (!t || !dt) return fail(EVG_ERR_INVALID, "null task table / distro table");
  const int64_t T = t->n_tasks, E = t->n_edges;
  const int32_t D = dt->n_distros;
  if (T < 0 || E < 0 || D < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (T >= (int64_t(1) << 31) - 2) return fail(EVG_ERR_INVALID, "n_tasks %lld exceeds 2^31-2 per call", (long long)T);
  if (2 * T + E >= int64_t(0xFFFFFFF0u)) return fail(EVG_ERR_INVALID, "2*n_tasks+n_edges exceeds the 32-bit pair id space");
  if (D > 0 && (!dt->task_off || !dt->group_off || !dt->cfg)) return fail(EVG_ERR_INVALID, "null distro arrays");
  if (T > 0 && (!t->priority || !t->expected_ns || !t->queue_basis_ns || !t->wait_basis_ns || !t->num_dependents ||
                !t->task_group_order || !t->group_id || !t->version_id || !t->flags))
    return fail(EVG_ERR_INVALID, "null task column");
  if (E > 0 && (!t->dep_off || !t->dep_idx)) return fail(EVG_ERR_INVALID, "n_edges > 0 but dep_off/dep_idx null");
  if (D == 0 && T != 0) return fail(EVG_ERR_INVALID, "tasks without distros");
  std::vector<int64_t> unit_base(size_t(D) + 1, 0), dtile_off(size_t(D) + 1, 0);
  std::vector<int32_t> tile_distro, listW, listA, listB, listC, listG, listNA, listNB, listNC;
  std::vector<int64_t> tile_start;
  std::vector<uint8_t> route(size_t(D) + 1, 0);
  int32_t n_general = 0;
  int64_t max_general = 0;
  int general_complex = 0;
  int any_complex = E > 0 ? 1 : 0;
  int64_t Tgc = 0, Prec = 0;
  constexpr int kGA = PlanCta<kNT_A, kNCapA>::kGroupCap, kGB = PlanCta<kNT_B, kNCapB>::kGroupCap, kGC = PlanCta<kNT_C, kNCapC>::kGroupCap;
  // Size class of distro d (no side effects): W warp, 1..3 k_plan_cta classes, 4..6 k_plan_smem classes, 7 general path.
  auto classify = [&](int32_t d) -> int {
    const int64_t a = dt->task_off[d], b = dt->task_off[d + 1];
    const int64_t n = b - a, g = dt->group_off[d + 1] - dt->group_off[d];
    const evg_distro_cfg& cf = dt->cfg[d];
    const int64_t de = (E > 0) ? (edge_off ? edge_off[d + 1] - edge_off[d] : t->dep_off[b] - t->dep_off[a]) : 0;
    const bool narrow = !cf.group_versions && de == 0;  // k_plan_cta: task groups are the only multi-member units it knows
    if (n <= kCapW) return 0;
    if (narrow && n <= kNCapA && g <= kGA) return 1;
    if (narrow && n <= kNCapB && g <= kGB) return 2;
    if (narrow && n <= kNCapC && g <= kGC) return 3;
    if (n <= kCapA) return (cf.group_versions && n > kBigUnitTasks) ? 8 : 4;  // 8: version units of dozens of tasks, walked member by member
    if (n <= kCapB) return 5;
    if (n <= kCapC) return 6;
    return 7;
  };
  // k_plan_smem walks the unit lists of GroupVersions / dependency distros with ONE CTA per distro: fine when a class
  // has enough distros to fill the GPU, a millisecond-long tail when it has a handful (configs[4]: ~20 distros of 1-6k
  // tasks held the whole tick, then ~50 GroupVersions distros of 129-1024 tasks whose version units are walked member by
  // member).  The general path spreads every distro over all SMs, so sparse classes go there.
  int64_t n_class[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int32_t d = 0; d < D; d++) {
    const int64_t a = dt->task_off[d], b = dt->task_off[d + 1];
    if (d == 0 && (a != 0 || dt->group_off[0] != 0)) return fail(EVG_ERR_INVALID, "offsets must start at 0");
    if (b < a || dt->group_off[d + 1] < dt->group_off[d]) return fail(EVG_ERR_INVALID, "offsets of distro %d decrease", d);
    if (b > T) return fail(EVG_ERR_INVALID, "task_off of distro %d exceeds n_tasks", d);
    n_class[classify(d)]++;
  }
  const char* sparse_env = getenv("EVG_SPARSE_CLASS");  // tests set 0 to keep every class on its own kernel
  const int64_t sparse = sparse_env ? atoll(sparse_env) : kSparseClass;
  const bool sparse_b = n_class[5] > 0 && n_class[5] < sparse, sparse_c = n_class[6] > 0 && n_class[6] < sparse;
  const bool sparse_v = n_class[8] > 0 && n_class[8] < sparse;
  for (int32_t d = 0; d < D; d++) {
    const int64_t a = dt->task_off[d], b = dt->task_off[d + 1];
    const int64_t ga = dt->group_off[d], gb = dt->group_off[d + 1];
    if (b - a > kMaxTasksPerDistro) return fail(EVG_ERR_INVALID, "distro %d holds %lld tasks (max %lld)", d, (long long)(b - a), (long long)kMaxTasksPerDistro);
    const evg_distro_cfg& cf = dt->cfg[d];
    if (cf.n_versions < 0) return fail(EVG_ERR_INVALID, "distro %d: negative n_versions", d);
    if (gb > ga || cf.group_versions) any_complex = 1;
    unit_base[d + 1] = unit_base[d] + (gb - ga) + (cf.group_versions ? int64_t(cf.n_versions) : (b - a));
    const int64_t n = b - a;
    const int64_t de = (E > 0) ? (edge_off ? edge_off[d + 1] - edge_off[d] : t->dep_off[b] - t->dep_off[a]) : 0;
    int cls = classify(d);
    if ((cls == 5 && sparse_b) || (cls == 6 && sparse_c)) cls = 7;
    if (cls == 8) cls = sparse_v ? 7 : 4;
    switch (cls) {
      case 0: listW.push_back(d); route[d] = 1; break;
      case 1: listNA.push_back(d); route[d] = 1; break;
      case 2: listNB.push_back(d); route[d] = 1; break;
      case 3: listNC.push_back(d); route[d] = 1; break;
      case 4: listA.push_back(d); route[d] = 1; break;
      case 5: listB.push_back(d); route[d] = 1; break;
      case 6: listC.push_back(d); route[d] = 1; break;
      default: {
        n_general++;
        max_general = std::max(max_general, n);
        listG.push_back(d);
        if (gb > ga || cf.group_versions || de > 0) {
          general_complex = 1;
          Tgc += n;
          Prec += n + ((cf.group_versions && gb > ga) ? n : 0) + de;  // own-key, version and dependency memberships at most
        }
        const int64_t a0 = a & ~int64_t(3);  // tiles start 16-byte aligned in every column
        for (int64_t s = a0; s < b; s += kGTile) { tile_distro.push_back(d); tile_start.push_back(s); }
      }
    }
    dtile_off[d + 1] = int64_t(tile_distro.size());
  }
  if (D > 0 && dt->task_off[D] != T) return fail(EVG_ERR_INVALID, "task_off[n_distros] != n_tasks");
  const int64_t G = D > 0 ? dt->group_off[D] : 0;
  if (G > 0 && !dt->group_max_hosts) return fail(EVG_ERR_INVALID, "null group_max_hosts");
  const int64_t U = unit_base[D];
  if (U >= int64_t(0xFFFFFFF0u)) return fail(EVG_ERR_INVALID, "unit slot space exceeds 32 bits");
  if (Prec >= int64_t(0xFFFFFFF0u)) return fail(EVG_ERR_INVALID, "unit table exceeds 32 bits");
  const int64_t NT = int64_t(tile_distro.size());
  const int64_t P = 2 * T + E;
  cudaStream_t s = c->stream;
#define UP(buf, ptr, count, type)                                                                     \
  do {                                                                                                \
    CK((buf).ensure(sizeof(type) * size_t((count) > 0 ? (count) : 1)));                               \
    if ((count) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count), cudaMemcpyHostToDevice, s)); \
  } while (0)
#define UPC(buf, ptr, count, type)                                                                    \
  do {                                                                                                \
    if (adopt) {                                                                                      \
      if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0) return fail(EVG_ERR_INVALID, "device column %s is not 16-byte aligned", #ptr); \
      (buf).adopt(const_cast<void*>(static_cast<const void*>(ptr)));                                  \
    } else {                                                                                          \
      CK((buf).ensure(sizeof(type) * size_t((count) + kColPad)));                                     \
      if (copy_columns && (count) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count), cudaMemcpyHostToDevice, s)); \
    }                                                                                                 \
  } while (0)
  UPC(c->b_prio, t->priority, T, int32_t);
  UPC(c->b_exp, t->expected_ns, T, int64_t);
  UPC(c->b_qb, t->queue_basis_ns, T, int64_t);
  UPC(c->b_wb, t->wait_basis_ns, T, int64_t);
  UPC(c->b_nd, t->num_dependents, T, int32_t);
  UPC(c->b_tgo, t->task_group_order, T, int32_t);
  UPC(c->b_gid, t->group_id, T, int32_t);
  UPC(c->b_vid, t->version_id, T, int32_t);
  UPC(c->b_flags, t->flags, T, uint32_t);
  if (E > 0) {
    UPC(c->b_depoff, t->dep_off, T + 1, int64_t);
    UPC(c->b_depidx, t->dep_idx, E, int32_t);
  }
#undef UPC
  UP(c->b_taskoff, dt->task_off, D + 1, int64_t);
  UP(c->b_groupoff, dt->group_off, D + 1, int64_t);
  UP(c->b_cfg, dt->cfg, D, evg_distro_cfg);
  UP(c->b_gmax, dt->group_max_hosts, G, int32_t);
  UP(c->b_unitbase, unit_base.data(), D + 1, int64_t);
  UP(c->b_tiledistro, tile_distro.data(), NT, int32_t);
  UP(c->b_tilestart, tile_start.data(), NT, int64_t);
  UP(c->b_dtileoff, dtile_off.data(), D + 1, int64_t);
  UP(c->b_route, route.data(), D + 1, uint8_t);
  UP(c->b_listW, listW.data(), int64_t(listW.size()), int32_t);
  UP(c->b_listG, listG.data(), int64_t(listG.size()), int32_t);
  UP(c->b_listA, listA.data(), int64_t(listA.size()), int32_t);
  UP(c->b_listB, listB.data(), int64_t(listB.size()), int32_t);
  UP(c->b_listC, listC.data(), int64_t(listC.size()), int32_t);
  UP(c->b_listNA, listNA.data(), int64_t(listNA.size()), int32_t);
  UP(c->b_listNB, listNB.data(), int64_t(listNB.size()), int32_t);
  UP(c->b_listNC, listNC.data(), int64_t(listNC.size()), int32_t);
  // One CTA per distro: with the largest first, the last (partial) wave of a launch holds the smallest distros and the
  // tail is short (configs[4]: 1371 distros of 33..1024 tasks on 1184 CTA slots).  The ascending lists stay: the
  // pipelined one-shot call cuts them by distro range.
  std::vector<int32_t> lptA(listA), lptB(listB), lptC(listC), lptNA(listNA), lptNB(listNB), lptNC(listNC);
  for (std::vector<int32_t>* v : {&lptA, &lptB, &lptC, &lptNA, &lptNB, &lptNC})
    std::stable_sort(v->begin(), v->end(), [&](int32_t x, int32_t y) {
      return dt->task_off[x + 1] - dt->task_off[x] > dt->task_off[y + 1] - dt->task_off[y];
    });
  // the tail of the smallest class that fits the 64-thread instance (size AND task groups) goes last, largest first
  constexpr int kGS = PlanCta<kNT_S, kNCapS>::kGroupCap;
  auto fits_s = [&](int32_t x) { return dt->task_off[x + 1] - dt->task_off[x] <= kNCapS && dt->group_off[x + 1] - dt->group_off[x] <= kGS; };
  std::stable_partition(lptNA.begin(), lptNA.end(), [&](int32_t x) { return !fits_s(x); });
  c->nNA_big = int32_t(std::count_if(lptNA.begin(), lptNA.end(), [&](int32_t x) { return !fits_s(x); }));
  c->max_cta_tasks = 0;
  for (const std::vector<int32_t>* v : {&listNA, &listNB, &listNC})
    for (int32_t x : *v) c->max_cta_tasks = std::max<int64_t>(c->max_cta_tasks, dt->task_off[x + 1] - dt->task_off[x]);
  UP(c->b_lptA, lptA.data(), int64_t(lptA.size()), int32_t);
  UP(c->b_lptB, lptB.data(), int64_t(lptB.size()), int32_t);
  UP(c->b_lptC, lptC.data(), int64_t(lptC.size()), int32_t);
  UP(c->b_lptNA, lptNA.data(), int64_t(lptNA.size()), int32_t);
  UP(c->b_lptNB, lptNB.data(), int64_t(lptNB.size()), int32_t);
  UP(c->b_lptNC, lptNC.data(), int64_t(lptNC.size()), int32_t);
  // the staging vectors above must outlive the async copies
  CK(cudaStreamSynchronize(s));
  // work buffers
  const bool on_chip_cta = !(listA.empty() && listB.empty() && listC.empty() && listNA.empty() && listNB.empty() && listNC.empty());
  if (any_complex) {
    CK(c->b_hasdep.ensure(size_t(T) + 16));
    CK(c->b_head.ensure(sizeof(uint32_t) * size_t(U + 1)));
    CK(c->b_next.ensure(sizeof(uint32_t) * size_t(P + 1)));
    CK(c->b_pslot.ensure(sizeof(uint32_t) * size_t(P + 1)));
    CK(c->b_etask.ensure(sizeof(uint32_t) * size_t(E + 1)));
    CK(c->b_elive.ensure(size_t(E) + 1));
    CK(c->b_unitv.ensure(sizeof(int64_t) * size_t(U + 1)));
    CK(c->b_unita.ensure(sizeof(uint32_t) * size_t(U + 1)));
    CK(c->b_unitn.ensure(sizeof(uint32_t) * size_t(U + 1)));
    CK(c->b_unitmask.ensure(sizeof(uint64_t) * size_t(U + 1)));
    CK(c->b_bestpair.ensure(sizeof(uint32_t) * size_t(T + 1)));
  }
  if (on_chip_cta) CK(c->b_kv.ensure(sizeof(uint64_t) * size_t(T + 1)));  // k_plan_smem's scratch for value ranges above 32 bits
  if (n_general > 0) {  // the general path's buffers exist only when a distro takes it
    for (int k = 0; k < 2; k++) {
      CK(c->b_klo[k].ensure(sizeof(uint32_t) * size_t(T + 1)));
      CK(c->b_khi[k].ensure(sizeof(uint32_t) * size_t(T + 1)));
      CK(c->b_ix[k].ensure(sizeof(uint32_t) * size_t(T + 1)));
    }
    CK(c->b_vmm.ensure(sizeof(uint64_t) * 2 * size_t(D + 1)));
    CK(c->b_gmisc.ensure(64));
    CK(c->b_tilesum.ensure(sizeof(uint32_t) * size_t(NT + 1)));
    CK(c->b_tilehist.ensure(sizeof(uint32_t) * 256 * size_t(NT + 1)));
    if (general_complex) {
      CK(c->b_e.ensure(sizeof(uint32_t) * size_t(T + kColPad)));
      CK(c->b_clist.ensure(sizeof(uint32_t) * 2 * size_t(Tgc + 1)));
      CK(c->b_rec.ensure(sizeof(URec) * size_t(Prec + 1)));
      CK(c->b_hlist.ensure(sizeof(uint2) * size_t(Prec + 1)));
      CK(c->b_usum.ensure(sizeof(uint4) * size_t(U + 1)));
      CK(c->b_tie.ensure(sizeof(uint4) * size_t(T + 1)));
    }
  }
  CK(c->b_punt.ensure(sizeof(int32_t) * size_t(D + 1)));
  CK(c->b_puntcnt.ensure(sizeof(int32_t) * (evg_ctx::kMaxChunks + 2)));
  CK(c->b_qinfo.ensure(sizeof(evg_queue_info) * size_t(D + 1)));
  CK(c->b_ginfo.ensure(sizeof(evg_group_info) * size_t(G + 1)));
  CK(c->b_order.ensure(sizeof(int32_t) * size_t(T + 1)));
  CK(c->b_tv.ensure(sizeof(int64_t) * size_t(T + kColPad)));
  c->T = T; c->E = E; c->G = G; c->U = U; c->NT = NT; c->Dn = D;
  c->t_pad = (T + 3) & ~int64_t(3);
  c->adopted = adopt;
  c->deps_resident = false;
  if (c->head_cap > 0) c->bd_valid = false;  // a head run's breakdown rows are laid out for the previous table
  c->head_cap = 0;
  c->Tgc = Tgc;
  c->max_groups = 0;
  for (int32_t d = 0; d < D; d++) c->max_groups = std::max(c->max_groups, dt->group_off[d + 1] - dt->group_off[d]);
  c->any_complex = any_complex;
  c->nW = int32_t(listW.size());
  c->nA = int32_t(listA.size()); c->nB = int32_t(listB.size()); c->nC = int32_t(listC.size());
  c->nNA = int32_t(listNA.size()); c->nNB = int32_t(listNB.size()); c->nNC = int32_t(listNC.size());
  c->n_general = n_general;
  c->max_general = max_general;
  c->general_complex = general_complex;
  CK(c->b_err.ensure(sizeof(int) * 4));
  CK(cudaMemsetAsync(c->b_err.p, 0, sizeof(int) * 4, s));
  c->h_listW.swap(listW);
  c->h_listA.swap(listA); c->h_listB.swap(listB); c->h_listC.swap(listC);
  c->h_listNA.swap(listNA); c->h_listNB.swap(listNB); c->h_listNC.swap(listNC);
  c->h_taskoff.assign(dt->task_off, dt->task_off + D + 1);
  c->h_groupoff.assign(dt->group_off, dt->group_off + D + 1);
  c->h_edgeoff.assign(size_t(D) + 1, 0);
  if (E > 0)
    for (int32_t d = 0; d <= D; d++) c->h_edgeoff[size_t(d)] = edge_off ? edge_off[d] : t->dep_off[dt->task_off[d]];
  c->h_unitbase.swap(unit_base);
  c->h_dtileoff.swap(dtile_off);
  c->h_listG.swap(listG);
  c->have_tasks = true;
  c->alist_valid = false;  // upload_hosts lists the allocator's distros against THIS table
  c->have_hosts = false;
  if ((copy_columns || adopt) && T > 0) {  // range-check the ids the kernels index with (the pipelined call checks chunk by chunk)
    DTasks dtv = dtasks(c);
    DDistros ddv = ddistros(c);
    DWork wv = dwork(c);
    k_validate<<<grid_for(T, 256), 256, 0, s>>>(dtv, ddv, wv, 0, T);
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, c->b_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (bad) { c->have_tasks = false; return fail(EVG_ERR_INVALID, "a group_id / version_id / dep_idx is out of range for its distro"); }
  }
  return EVG_OK;
}

int upload_hosts(evg_ctx* c, const evg_host_soa* h, const int64_t* host_off, const evg_alloc_cfg* acfg, int32_t D) {
  if (!h || (D > 0 && !acfg)) return fail(EVG_ERR_INVALID, "null host table / allocator config");
  const int64_t H = h->n_hosts;
  if (H < 0) return fail(EVG_ERR_INVALID, "negative n_hosts");
  if (D > 0 && !host_off) return fail(EVG_ERR_INVALID, "null host_off");
  if (D == 0 && H != 0) return fail(EVG_ERR_INVALID, "hosts without distros");
  for (int32_t d = 0; d < D; d++)
    if (host_off[d + 1] < host_off[d] || (d == 0 && host_off[0] != 0)) return fail(EVG_ERR_INVALID, "bad host_off at distro %d", d);
  if (D > 0 && host_off[D] != H) return fail(EVG_ERR_INVALID, "host_off[n_distros] != n_hosts");
  if (H > 0 && (!h->flags || !h->group_id || !h->expected_ns || !h->std_ns || !h->start_ns)) return fail(EVG_ERR_INVALID, "null host column");
  cudaStream_t s = c->stream;
  UP(c->b_hflags, h->flags, H, uint32_t);
  UP(c->b_hgid, h->group_id, H, int32_t);
  UP(c->b_hexp, h->expected_ns, H, int64_t);
  UP(c->b_hstd, h->std_ns, H, int64_t);
  UP(c->b_hstart, h->start_ns, H, int64_t);
  if (D > 0) UP(c->b_hostoff, host_off, D + 1, int64_t);
  UP(c->b_acfg, acfg, D, evg_alloc_cfg);
  c->alist_valid = false;
  std::vector<int32_t> alist;
  if (c->have_tasks && c->Dn == D && int64_t(c->h_groupoff.size()) == int64_t(D) + 1) {
    for (int32_t d = 0; d < D; d++)
      if (c->h_groupoff[d + 1] != c->h_groupoff[d] || host_off[d + 1] - host_off[d] > kGrouplessHosts) alist.push_back(d);
    UP(c->b_alist, alist.data(), int64_t(alist.size()), int32_t);
    CK(cudaStreamSynchronize(s));  // `alist` is a local
    c->n_alist = int64_t(alist.size());
    c->alist_valid = true;
  }
  CK(c->b_result.ensure(sizeof(evg_alloc_result) * size_t(D + 1)));
  CK(c->b_status.ensure(sizeof(int32_t) * size_t(D + 1)));
  c->H = H;
  c->have_hosts = true;
  return EVG_OK;
}
#undef UP

DTasks dtasks(const evg_ctx* c) {
  DTasks t;
  t.n = c->T; t.n_edges = c->E;
  t.priority = c->b_prio.as<int32_t>(); t.expected = c->b_exp.as<int64_t>();
  t.qbasis = c->b_qb.as<int64_t>(); t.wbasis = c->b_wb.as<int64_t>();
  t.numdep = c->b_nd.as<int32_t>(); t.tgo = c->b_tgo.as<int32_t>();
  t.gid = c->b_gid.as<int32_t>(); t.vid = c->b_vid.as<int32_t>(); t.flags = c->b_flags.as<uint32_t>();
  t.dep_off = c->b_depoff.as<int64_t>(); t.dep_idx = c->b_depidx.as<int32_t>();
  return t;
}
DDistros ddistros(const evg_ctx* c) {
  DDistros d;
  d.n = c->Dn; d.task_off = c->b_taskoff.as<int64_t>(); d.group_off = c->b_groupoff.as<int64_t>();
  d.cfg = c->b_cfg.as<evg_distro_cfg>(); d.gmax = c->b_gmax.as<int32_t>(); d.unit_base = c->b_unitbase.as<int64_t>();
  return d;
}
DWork dwork(const evg_ctx* c) {
  DWork w;
  w.has_dep = c->b_hasdep.as<uint8_t>(); w.head = c->b_head.as<uint32_t>(); w.next = c->b_next.as<uint32_t>();
  w.pair_slot = c->b_pslot.as<uint32_t>(); w.edge_task = c->b_etask.as<uint32_t>();
  w.edge_live = c->b_elive.as<uint8_t>(); w.route = c->b_route.as<uint8_t>();
  w.err = c->b_err.as<int>();
  w.unit_v = c->b_unitv.as<int64_t>(); w.unit_a = c->b_unita.as<uint32_t>(); w.unit_n = c->b_unitn.as<uint32_t>();
  w.unit_mask = c->b_unitmask.as<unsigned long long>();
  w.best_pair = c->b_bestpair.as<uint32_t>();
  w.buf[0].key_v = c->b_kv.as<uint64_t>();
  w.qinfo = c->b_qinfo.as<evg_queue_info>(); w.ginfo = c->b_ginfo.as<evg_group_info>();
  return w;
}
DGen dgen(const evg_ctx* c) {
  DGen g;
  g.n_tiles = c->NT;
  g.tile0 = 0;
  g.tile_distro = c->b_tiledistro.as<int32_t>(); g.tile_start = c->b_tilestart.as<int64_t>();
  g.dtile_off = c->b_dtileoff.as<int64_t>();
  g.vmm = c->b_vmm.as<unsigned long long>();
  for (int k = 0; k < 2; k++) {
    g.key_lo[k] = c->b_klo[k].as<uint32_t>(); g.key_hi[k] = c->b_khi[k].as<uint32_t>(); g.idx[k] = c->b_ix[k].as<uint32_t>();
  }
  g.e = c->b_e.as<uint32_t>(); g.tile_sum = c->b_tilesum.as<uint32_t>(); g.tile_hist = c->b_tilehist.as<uint32_t>();
  g.clist = c->b_clist.as<uint32_t>();
  g.clist_d = c->b_clist.as<int32_t>() + (c->Tgc + 1);
  g.ccount = c->b_gmisc.as<unsigned int>();
  g.maxpass = c->b_gmisc.as<int32_t>() + 1;
  g.rcount = c->b_gmisc.as<unsigned int>() + 2;
  g.hcount = c->b_gmisc.as<unsigned int>() + 3;
  g.hlist = c->b_hlist.as<uint2>();
  g.usum = c->b_usum.as<uint4>();
  g.rec = c->b_rec.as<URec>();
  g.tie = c->b_tie.as<uint4>();
  g.tv = c->b_tv.as<int64_t>();
  return g;
}

#define LOCK(c) std::lock_guard<std::recursive_mutex> lock_((c)->mu)
#define LAUNCH_ON(c, st, kernel, grid, block, ...)                           \
  do {                                                                       \
    if ((grid) > 0) {                                                        \
      kernel<<<(grid), (block), 0, (st)>>>(__VA_ARGS__);                     \
      (c)->launches++;                                                       \
    }                                                                        \
  } while (0)
#define LAUNCH(c, kernel, grid, block, ...) LAUNCH_ON(c, (c)->stream, kernel, grid, block, __VA_ARGS__)

int run_alloc_range(evg_ctx* c, int64_t now, int32_t d0, int32_t d1) {
  DHosts h;
  h.n = c->H; h.flags = c->b_hflags.as<uint32_t>(); h.gid = c->b_hgid.as<int32_t>();
  h.expected = c->b_hexp.as<int64_t>(); h.stddev = c->b_hstd.as<int64_t>(); h.start = c->b_hstart.as<int64_t>();
  h.host_off = c->b_hostoff.as<int64_t>(); h.cfg = c->b_acfg.as<evg_alloc_cfg>();
  if (c->ext_result && c->ext_capacity < c->Dn) return fail(EVG_ERR_INVALID, "bound result buffer holds %lld rows, need %d", (long long)c->ext_capacity, c->Dn);
  CK(c->b_gs.ensure(sizeof(GroupScratch) * size_t(c->G + 1)));
  // a warp per distro (four per block) unless some distro has thousands of task groups, then a block per distro
  // ... and a thread per distro for the distros that have no task groups, when there are enough distros for that to matter
  const int split = (d1 - d0) >= 4096 ? 1 : 0;
  // ... and only for the distros it has to take when the upload listed them (whole-table ranges)
  const bool listed = split && c->alist_valid && d0 == 0 && d1 == c->Dn;
  const int32_t* al = listed ? c->b_alist.as<int32_t>() : nullptr;
  const int64_t teams = listed ? c->n_alist : int64_t(d1 - d0);
  if (c->max_groups > kWideAllocGroups)
    LAUNCH(c, k_alloc<128>, unsigned(teams), 128, h, d0, d1, c->b_groupoff.as<int64_t>(), c->b_qinfo.as<evg_queue_info>(),
           c->b_ginfo.as<evg_group_info>(), c->b_gs.as<GroupScratch>(), now, c->result_ptr(), c->b_status.as<int32_t>(), split, al, int32_t(c->n_alist));
  else
    LAUNCH(c, k_alloc<32>, grid_for(teams, 4), 128, h, d0, d1, c->b_groupoff.as<int64_t>(), c->b_qinfo.as<evg_queue_info>(),
           c->b_ginfo.as<evg_group_info>(), c->b_gs.as<GroupScratch>(), now, c->result_ptr(), c->b_status.as<int32_t>(), split, al, int32_t(c->n_alist));
  if (split)
    LAUNCH(c, k_alloc_groupless, grid_for(d1 - d0, 128), 128, h, d0, d1, c->b_groupoff.as<int64_t>(), c->b_qinfo.as<evg_queue_info>(), now,
           c->result_ptr(), c->b_status.as<int32_t>());
  CK(cudaGetLastError());
  return EVG_OK;
}
int run_alloc(evg_ctx* c, int64_t now) { return run_alloc_range(c, now, 0, c->Dn); }

template <int THREADS, int ITEMS, int MIN_CTAS>
int launch_smem(evg_ctx* c, cudaStream_t st, const DTasks& dt, const DDistros& dd, const DWork& w, const int32_t* list, int32_t n,
                int64_t now, int lists_needed = 0, const int32_t* list_count = nullptr) {
  if (n <= 0) return EVG_OK;
  const size_t bytes = PlanSmem<THREADS, ITEMS>::kBytes;
  CK(cudaFuncSetAttribute(k_plan_smem<THREADS, ITEMS, MIN_CTAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)));
  k_plan_smem<THREADS, ITEMS, MIN_CTAS><<<unsigned(n), THREADS, bytes, st>>>(dt, dd, w, list, list_count, now, lists_needed,
                                                                          c->b_order.as<int32_t>(), c->b_tv.as<int64_t>());
  c->launches++;
  return EVG_OK;
}

// Second-generation on-chip planner for one class; distros it hands back land in punt_list[0 .. *punt_count).
template <int THREADS, int CAP, int OCC>
int launch_cta(evg_ctx* c, cudaStream_t st, const DTasks& dt, const DDistros& dd, const DWork& w, const int32_t* list, int32_t n,
               int64_t now, int32_t* punt_list, int32_t* punt_count) {
  if (n <= 0) return EVG_OK;
  const size_t bytes = PlanCta<THREADS, CAP>::kBytes;
  CK(cudaFuncSetAttribute(k_plan_cta<THREADS, CAP, OCC>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)));
  k_plan_cta<THREADS, CAP, OCC><<<unsigned(n), THREADS, bytes, st>>>(dt, dd, w, list, now, c->t_pad, c->b_order.as<int32_t>(),
                                                                  c->b_tv.as<int64_t>(), punt_list, punt_count);
  c->launches++;
  return EVG_OK;
}

// Distros of at most 32 tasks: one warp each (k_plan_warp).  Breakdown mode needs the unit lists, so it
// sends them through the smallest on-chip class instead.
int launch_tiny(evg_ctx* c, cudaStream_t st, const DTasks& dt, const DDistros& dd, const DWork& w, const int32_t* list, int32_t n,
                int64_t now, int lists_needed) {
  if (n <= 0) return EVG_OK;
  if (lists_needed) return launch_smem<128, 8, 8>(c, st, dt, dd, w, list, n, now, 1);
  k_plan_warp<<<grid_for(int64_t(n) * 32, 256), 256, 0, st>>>(dt, dd, w, list, n, now, c->b_order.as<int32_t>(), c->b_tv.as<int64_t>());
  c->launches++;
  return EVG_OK;
}

// Everything the general path accumulates into or links through starts from zero / "empty", for the distros
// [d0, d1) (first to last general-path distro of the tick, or of one chunk of the pipelined call).  On the resident
// path this runs on the context stream BEFORE the routes fork: an on-chip distro inside the span rewrites its own rows
// afterwards.
int prepare_general(evg_ctx* c, cudaStream_t s, int32_t d0, int32_t d1) {
  const int64_t t0 = c->h_taskoff[d0], t1 = c->h_taskoff[d1], u0 = c->h_unitbase[d0], u1 = c->h_unitbase[d1];
  const int64_t g0 = c->h_groupoff[d0], g1 = c->h_groupoff[d1], e0 = c->h_edgeoff[d0], e1 = c->h_edgeoff[d1];
  CK(cudaMemsetAsync(c->b_qinfo.as<evg_queue_info>() + d0, 0, sizeof(evg_queue_info) * size_t(d1 - d0), s));
  if (g1 > g0) CK(cudaMemsetAsync(c->b_ginfo.as<evg_group_info>() + g0, 0, sizeof(evg_group_info) * size_t(g1 - g0), s));
  if (c->general_complex) {
    const size_t nt = size_t(t1 - t0);
    CK(cudaMemsetAsync(c->b_hasdep.as<uint8_t>() + t0, 0, nt, s));
    CK(cudaMemsetAsync(c->b_unitn.as<uint32_t>() + u0, 0, sizeof(uint32_t) * size_t(u1 - u0), s));   // members drawn so far
  }
  return EVG_OK;
}

// The general path on stream `st` for the general-path distros listG[gfirst .. gfirst + gcount) (evg_plan_general.cuh).
int run_general(evg_ctx* c, cudaStream_t st, const DTasks& dt, const DDistros& dd, const DWork& w, int64_t now, int32_t gfirst,
                int32_t gcount, int32_t head_cap = 0) {
  if (gcount <= 0) return EVG_OK;
  DGen g = dgen(c);
  const int gc = c->general_complex;
  const int32_t d_first = c->h_listG[size_t(gfirst)], d_last = c->h_listG[size_t(gfirst + gcount - 1)];
  g.tile0 = c->h_dtileoff[size_t(d_first)];
  const unsigned nt = unsigned(c->h_dtileoff[size_t(d_last) + 1] - g.tile0);
  const int32_t* gl = c->b_listG.as<int32_t>() + gfirst;
  LAUNCH_ON(c, st, k_ginit, grid_for(gcount, 256), 256, g, gl, gcount);
  if (gc && c->E > 0) LAUNCH_ON(c, st, k_gmark, nt, 256, dt, dd, w, g);
  if (c->timed) CK(cudaEventRecord(c->ev_gt0, st));
  LAUNCH_ON(c, st, k_gtask, nt, 256, dt, dd, w, g, now, gc);
  if (c->timed) { CK(cudaEventRecord(c->ev_gt1, st)); c->general_timed = true; }
  const unsigned wl_grid = unsigned(std::min<int64_t>(std::max<int64_t>(1, (c->Tgc + 255) / 256), 148 * 16));
  if (gc) {
    LAUNCH_ON(c, st, k_glink, wl_grid, 256, dt, dd, w, g, now);
    LAUNCH_ON(c, st, k_galloc, wl_grid, 256, dt, dd, w, g);
    LAUNCH_ON(c, st, k_gfill, wl_grid, 256, dt, dd, w, g);
    LAUNCH_ON(c, st, k_gunit, wl_grid, 256, dd, w, g, now);
    LAUNCH_ON(c, st, k_gbest, wl_grid, 256, dt, dd, w, g, c->bd_valid ? 1 : 0);
  }
  LAUNCH_ON(c, st, k_gsched, grid_for(gcount, 128), 128, g, gl, gcount);
  if (gc) {
    LAUNCH_ON(c, st, k_gsum, nt, 256, dd, g);
    LAUNCH_ON(c, st, k_gscan, unsigned(gcount), 1024, g, gl);
  }
  LAUNCH_ON(c, st, k_gplace, nt, 256, dd, w, g, gc);
  if (gc) LAUNCH_ON(c, st, k_gplace_disp, wl_grid, 256, dt, dd, w, g);
  if (c->timed) CK(cudaEventRecord(c->ev_sort0, st));  // the general path's segmented sort
  // The select pays when it discards most of a distro.  When no general-path distro is longer than twice the cap, the
  // tile-parallel full sort (whose first cap ranks are the head) beats one CTA per distro sorting nearly all of it
  // (configs[4]: a 12 546-task distro and two dozen sparse-class ones).
  if (head_cap == 0 || c->max_general <= 2 * int64_t(head_cap)) {
    for (int j = 0; j < 8; j++) {  // passes beyond the tick's longest key exit at once (*maxpass is device-side)
      LAUNCH_ON(c, st, k_ghist, nt, 256, j, dd, g);
      LAUNCH_ON(c, st, k_gdscan, unsigned(gcount), 1024, j, gl, g);
      LAUNCH_ON(c, st, k_gscatter, nt, 256, j, dd, g);
    }
    if (c->timed) CK(cudaEventRecord(c->ev_sort1, st));
    LAUNCH_ON(c, st, k_gemit, nt, 256, dd, g, c->b_order.as<int32_t>(), c->b_tv.as<int64_t>());
  } else {  // select + compaction + head sort; TotalValue by task in b_tv was last read by k_gplace_disp
    DHead h;
    h.sel = c->b_hsel.as<HeadSel>(); h.hist = c->b_hhist.as<uint32_t>(); h.eq_sum = c->b_heq.as<uint32_t>(); h.cap = head_cap;
    LAUNCH_ON(c, st, k_hinit, unsigned(gcount), 256, dd, g, h, gl);
    for (int j = 0; j < 8; j++) {
      LAUNCH_ON(c, st, k_hhist, nt, 256, j, dd, g, h);
      LAUNCH_ON(c, st, k_hstep, unsigned(gcount), 256, j, gl, g, h);
    }
    LAUNCH_ON(c, st, k_hcount, nt, 256, dd, g, h);
    LAUNCH_ON(c, st, k_gscan, unsigned(gcount), 1024, g, gl);
    DGen ge = g;
    ge.tile_sum = h.eq_sum;
    LAUNCH_ON(c, st, k_gscan, unsigned(gcount), 1024, ge, gl);
    LAUNCH_ON(c, st, k_hplace, nt, 256, dd, g, h);
    constexpr size_t b0 = hsort_smem<false>(), b1 = hsort_smem<true>();
    CK(cudaFuncSetAttribute(k_hsort<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(b0)));
    CK(cudaFuncSetAttribute(k_hsort<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(b1)));
    k_hsort<false><<<unsigned(gcount), kHsThreads, b0, st>>>(gl, dd, g, h, c->b_order.as<int32_t>(), c->b_tv.as<int64_t>());
    k_hsort<true><<<unsigned(gcount), kHsThreads, b1, st>>>(gl, dd, g, h, c->b_order.as<int32_t>(), c->b_tv.as<int64_t>());
    c->launches += 2;
    if (c->timed) CK(cudaEventRecord(c->ev_sort1, st));
  }
  const int64_t g0 = c->h_groupoff[size_t(d_first)], g1 = c->h_groupoff[size_t(d_last) + 1];
  LAUNCH_ON(c, st, k_finalize_info, grid_for(std::max<int64_t>(d_last + 1 - d_first, g1 - g0), 256), 256, dd, w, d_first, d_last + 1, g0, g1);
  return EVG_OK;
}

int ensure_aux_streams(evg_ctx* c) {
  if (c->ev_fork) return EVG_OK;
  for (int k = 0; k < evg_ctx::kAux; k++) {
    CK(cudaStreamCreateWithFlags(&c->s_aux[k], cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&c->ev_join[k], cudaEventDisableTiming));
  }
  CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  return EVG_OK;
}

// head_cap > 0 (evg_run_resident_head): general-path distros rank only their first min(length, head_cap) tasks, and
// breakdown rows exist for those ranks only, at the offsets c->h_headoff / b_hoff.
int run_plan(evg_ctx* c, int64_t now, uint32_t opts, int32_t head_cap = 0) {
  const int64_t T = c->T;
  const int32_t D = c->Dn;
  cudaStream_t s = c->stream;
  DTasks dt = dtasks(c);
  DDistros dd = ddistros(c);
  DWork w = dwork(c);
  int64_t* bd = nullptr;
  c->bd_valid = false;
  c->head_cap = head_cap;
  const int64_t* bd_off = c->b_taskoff.as<int64_t>();
  int64_t bd_rows = T;
  if (head_cap > 0) {
    if (c->n_general > 0) {
      CK(c->b_hsel.ensure(sizeof(HeadSel) * size_t(D + 1)));
      CK(c->b_hhist.ensure(sizeof(uint32_t) * 256 * size_t(c->n_general)));
      CK(c->b_heq.ensure(sizeof(uint32_t) * size_t(c->NT + 1)));
    }
    if (opts & EVG_OPT_BREAKDOWN) {  // host work before the first launch: only when the rows are wanted
      c->h_headoff.assign(size_t(D) + 1, 0);
      for (int32_t d = 0; d < D; d++)
        c->h_headoff[size_t(d) + 1] = c->h_headoff[size_t(d)] + std::min<int64_t>(c->h_taskoff[size_t(d) + 1] - c->h_taskoff[size_t(d)], head_cap);
      bd_rows = c->h_headoff[size_t(D)];
      CK(c->b_hoff.ensure(sizeof(int64_t) * size_t(D + 1)));
      CK(cudaMemcpyAsync(c->b_hoff.p, c->h_headoff.data(), sizeof(int64_t) * size_t(D + 1), cudaMemcpyHostToDevice, s));
      bd_off = c->b_hoff.as<int64_t>();
    }
  }
  if (opts & EVG_OPT_BREAKDOWN) {
    CK(c->b_bd.ensure(sizeof(int64_t) * EVG_BD_N * size_t(bd_rows + 1)));
    bd = c->b_bd.as<int64_t>();
    c->bd_valid = true;
  }
  c->sort_slot = -1;
  if (D == 0) {
    if (c->timed) { CK(cudaEventRecord(c->ev_sort0, s)); CK(cudaEventRecord(c->ev_sort1, s)); }
    return EVG_OK;
  }
  const bool general = c->n_general > 0;
  // breakdown mode reads best_pair for every task: tasks emitted from their own single-task unit keep kInactive
  if (bd && c->any_complex) CK(cudaMemsetAsync(c->b_bestpair.p, 0xFF, sizeof(uint32_t) * size_t(T + 1), s));
  const int32_t n_new = bd ? 0 : c->nNA + c->nNB + c->nNC;
  if (n_new > 0) CK(cudaMemsetAsync(c->b_puntcnt.p, 0, sizeof(int32_t), s));
  if (general) { int rcg = prepare_general(c, s, c->h_listG.front(), c->h_listG.back() + 1); if (rcg != EVG_OK) return rcg; }
  // Routes run side by side when the tick has more than one: fork the aux streams off the context stream here, join
  // them before returning (the allocator and the caller's later work are ordered behind every planner kernel).
  struct Route { int id; int64_t weight; };
  const int64_t routes_present = (c->nW > 0) + (c->nA > 0) + (c->nB > 0) + (c->nC > 0) + (n_new > 0 || (bd && (c->nNA + c->nNB + c->nNC) > 0)) + (general ? 1 : 0);
  const bool fork = routes_present > 1;
  if (fork) {
    int rc0 = ensure_aux_streams(c);
    if (rc0 != EVG_OK) return rc0;
    CK(cudaEventRecord(c->ev_fork, s));
    for (int k = 0; k < evg_ctx::kAux; k++) CK(cudaStreamWaitEvent(c->s_aux[k], c->ev_fork, 0));
  }
  auto st = [&](int k) { return fork ? c->s_aux[k] : s; };
  int rc;
  const int slot = int(c->runs % evg_ctx::kRing);
  // --- stream 0: the second-generation on-chip planner (the dominant kernel of configs[1]-like ticks), then the
  //     distros it handed back
  if (bd) {  // breakdown needs the unit lists: every on-chip distro goes through k_plan_smem (its largest class holds them all)
    if ((rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, st(0), dt, dd, w, c->b_lptNC.as<int32_t>(), c->nNC, now, 1)) != EVG_OK) return rc;
    if ((rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, st(0), dt, dd, w, c->b_lptNB.as<int32_t>(), c->nNB, now, 1)) != EVG_OK) return rc;
    if ((rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, st(0), dt, dd, w, c->b_lptNA.as<int32_t>(), c->nNA, now, 1)) != EVG_OK) return rc;
  } else if (n_new > 0) {
    int32_t* pl = c->b_punt.as<int32_t>();
    int32_t* pc = c->b_puntcnt.as<int32_t>();
    const bool time_it = c->timed && !general && c->nNC > 0;
    if (time_it) CK(cudaEventRecord(c->ring0[slot], st(0)));
    if ((rc = launch_cta<kNT_C, kNCapC, kNOccC>(c, st(0), dt, dd, w, c->b_lptNC.as<int32_t>(), c->nNC, now, pl, pc)) != EVG_OK) return rc;
    if (time_it) { CK(cudaEventRecord(c->ring1[slot], st(0))); c->runs++; c->sort_slot = slot; }
    if ((rc = launch_cta<kNT_B, kNCapB, kNOccB>(c, st(0), dt, dd, w, c->b_lptNB.as<int32_t>(), c->nNB, now, pl, pc)) != EVG_OK) return rc;
    if ((rc = launch_cta<kNT_A, kNCapA, kNOccA>(c, st(0), dt, dd, w, c->b_lptNA.as<int32_t>(), c->nNA_big, now, pl, pc)) != EVG_OK) return rc;
    if ((rc = launch_cta<kNT_S, kNCapS, kNOccS>(c, st(0), dt, dd, w, c->b_lptNA.as<int32_t>() + c->nNA_big, c->nNA - c->nNA_big, now, pl, pc)) != EVG_OK) return rc;
    // the distros handed back: the smallest k_plan_smem instance that holds the largest of them (the launch has one CTA
    // per distro that COULD come back; CTAs beyond *pc exit at once, and 10^4 empty 1024-thread CTAs are not free)
    if (c->max_cta_tasks <= kCapA) rc = launch_smem<128, 8, 8>(c, st(0), dt, dd, w, pl, n_new, now, 0, pc);
    else if (c->max_cta_tasks <= kCapB) rc = launch_smem<256, 16, 3>(c, st(0), dt, dd, w, pl, n_new, now, 0, pc);
    else rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, st(0), dt, dd, w, pl, n_new, now, 0, pc);
    if (rc != EVG_OK) return rc;
  }
  // --- streams 1..3: first-generation classes (GroupVersions, in-queue dependency edges, very many task groups)
  {
    const bool time_it = c->timed && !general && c->sort_slot < 0 && c->nC > 0;
    if (time_it) CK(cudaEventRecord(c->ring0[slot], st(1)));
    if ((rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, st(1), dt, dd, w, c->b_lptC.as<int32_t>(), c->nC, now, bd ? 1 : 0)) != EVG_OK) return rc;
    if (time_it) { CK(cudaEventRecord(c->ring1[slot], st(1))); c->runs++; c->sort_slot = slot; }
  }
  if ((rc = launch_smem<256, 16, 3>(c, st(2), dt, dd, w, c->b_lptB.as<int32_t>(), c->nB, now, bd ? 1 : 0)) != EVG_OK) return rc;
  if ((rc = launch_smem<128, 8, 8>(c, st(3), dt, dd, w, c->b_lptA.as<int32_t>(), c->nA, now, bd ? 1 : 0)) != EVG_OK) return rc;
  // --- stream 4: one warp per tiny distro
  if ((rc = launch_tiny(c, st(4), dt, dd, w, c->b_listW.as<int32_t>(), c->nW, now, bd ? 1 : 0)) != EVG_OK) return rc;
  // --- stream 5: the general path
  if (general && (rc = run_general(c, st(5), dt, dd, w, now, 0, c->n_general, head_cap)) != EVG_OK) return rc;
  if (fork) {
    for (int k = 0; k < evg_ctx::kAux; k++) {
      CK(cudaEventRecord(c->ev_join[k], c->s_aux[k]));
      CK(cudaStreamWaitEvent(s, c->ev_join[k], 0));
    }
  }
  if (bd) LAUNCH(c, k_breakdown, grid_for(bd_rows, 256), 256, dt, dd, w, c->b_rec.as<URec>(), now, c->any_complex, c->b_order.as<int32_t>(),
                 bd_off, bd_rows, bd);
  CK(cudaGetLastError());
  return EVG_OK;
}

}  // namespace

// --------------------------------------------------------------------------
// C-ABI
// --------------------------------------------------------------------------
extern "C" {

const char* evg_last_error(void) { return g_err.c_str(); }
int evg_abi_version(void) { return EVG_ABI_VERSION; }

int evg_init(int device, void* stream, evg_ctx** out) {
  if (!out) return fail(EVG_ERR_INVALID, "evg_init: out is null");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) return fail(EVG_ERR_CUDA, "no CUDA device: %s (libevgsched has no CPU fallback)", cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(EVG_ERR_INVALID, "device %d out of range (%d devices)", device, n);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(EVG_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  evg_ctx* c = new evg_ctx();
  c->device = device;
  if (stream) { c->stream = reinterpret_cast<cudaStream_t>(stream); c->own_stream = false; }
  else { CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }
  CK(cudaEventCreate(&c->ev_begin)); CK(cudaEventCreate(&c->ev_sort0));
  CK(cudaEventCreate(&c->ev_sort1)); CK(cudaEventCreate(&c->ev_end));
  CK(cudaEventCreate(&c->ev_gt0)); CK(cudaEventCreate(&c->ev_gt1));
  for (int k = 0; k < evg_ctx::kRing; k++) { CK(cudaEventCreate(&c->ring0[k])); CK(cudaEventCreate(&c->ring1[k])); }
  *out = c;
  return EVG_OK;
}

void evg_shutdown(evg_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  DevBuf* all[] = {&c->b_prio, &c->b_exp, &c->b_qb, &c->b_wb, &c->b_nd, &c->b_tgo, &c->b_gid, &c->b_vid, &c->b_flags,
                   &c->b_depoff, &c->b_depidx, &c->b_taskoff, &c->b_groupoff, &c->b_cfg, &c->b_gmax, &c->b_unitbase,
                   &c->b_hasdep, &c->b_head, &c->b_next, &c->b_pslot, &c->b_etask, &c->b_elive, &c->b_unitv, &c->b_unita,
                   &c->b_unitn, &c->b_unitmask, &c->b_rn0, &c->b_rn1, &c->b_rn2, &c->b_rn3, &c->b_rn4, &c->b_rn5, &c->b_rn6,
                   &c->b_rn7, &c->b_err, &c->b_dx0, &c->b_dx1, &c->b_dx2, &c->b_dx3, &c->b_dx4, &c->b_dx5, &c->b_dx6, &c->b_dx7,
                   &c->b_route, &c->b_listW, &c->b_listA, &c->b_listB, &c->b_listC, &c->b_listG, &c->b_listNA, &c->b_listNB,
                   &c->b_listNC, &c->b_lptA, &c->b_lptB, &c->b_lptC, &c->b_lptNA, &c->b_lptNB, &c->b_lptNC, &c->b_punt, &c->b_puntcnt, &c->b_ca, &c->b_crk, &c->b_bestpair, &c->b_kv, &c->b_vmm,
                   &c->b_klo[0], &c->b_klo[1], &c->b_khi[0], &c->b_khi[1], &c->b_ix[0], &c->b_ix[1], &c->b_e, &c->b_tilesum,
                   &c->b_gmisc, &c->b_clist, &c->b_rec, &c->b_tie, &c->b_hlist, &c->b_usum, &c->b_upd, &c->b_tiledistro, &c->b_tilestart, &c->b_dtileoff, &c->b_tilehist,
                   &c->b_qinfo, &c->b_ginfo, &c->b_order, &c->b_tv, &c->b_bd,
                   &c->b_hsel, &c->b_hhist, &c->b_heq, &c->b_hoff, &c->b_hflags, &c->b_hgid, &c->b_hexp, &c->b_hstd,
                   &c->b_hstart, &c->b_hostoff, &c->b_acfg, &c->b_gs, &c->b_result, &c->b_status};
  for (DevBuf* b : all) b->release();
  for (DevBuf& b : c->b_pf) b.release();
  c->b_alist.release();
  for (int k = 0; k < evg_ctx::kRing; k++) { if (c->ring0[k]) cudaEventDestroy(c->ring0[k]); if (c->ring1[k]) cudaEventDestroy(c->ring1[k]); }
  cudaEventDestroy(c->ev_begin); cudaEventDestroy(c->ev_sort0); cudaEventDestroy(c->ev_sort1); cudaEventDestroy(c->ev_end);
  cudaEventDestroy(c->ev_gt0); cudaEventDestroy(c->ev_gt1);
  for (int k = 0; k < evg_ctx::kMaxChunks; k++) { if (c->ev_h[k]) cudaEventDestroy(c->ev_h[k]); if (c->ev_c[k]) cudaEventDestroy(c->ev_c[k]); }
  if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
  if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
  for (int k = 0; k < evg_ctx::kAux; k++) { if (c->s_aux[k]) cudaStreamDestroy(c->s_aux[k]); if (c->ev_join[k]) cudaEventDestroy(c->ev_join[k]); }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

int evg_upload(evg_ctx* c, const evg_task_soa* tasks, const evg_distro_table* distros, const evg_host_soa* hosts,
               const int64_t* host_off, const evg_alloc_cfg* acfg) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  CK(cudaSetDevice(c->device));
  int rc = upload_tasks(c, tasks, distros);
  if (rc != EVG_OK) return rc;
  if (hosts) {
    rc = upload_hosts(c, hosts, host_off, acfg, distros->n_distros);
    if (rc != EVG_OK) return rc;
    CK(cudaStreamSynchronize(c->stream));
  }
  return EVG_OK;
}

__global__ void k_gather_i64(const int64_t* __restrict__ src, const int64_t* __restrict__ at, int64_t* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = src[at[i]];
}

// evg_update_tasks: scatter changed rows into the resident columns.
__global__ void __launch_bounds__(256) k_update_rows(int64_t n, const int64_t* __restrict__ rows, int64_t T, int32_t* priority, int32_t* numdep,
                                                     int32_t* tgo, uint32_t* flags, int64_t* expected, int64_t* qbasis, int64_t* wbasis,
                                                     const int32_t* v_priority, const int32_t* v_numdep, const int32_t* v_tgo,
                                                     const uint32_t* v_flags, const int64_t* v_expected, const int64_t* v_qbasis,
                                                     const int64_t* v_wbasis, int* bad) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t r = rows[i];
  if (r < 0 || r >= T) { *bad = 1; return; }
  priority[r] = v_priority[i]; numdep[r] = v_numdep[i]; tgo[r] = v_tgo[i]; flags[r] = v_flags[i];
  expected[r] = v_expected[i]; qbasis[r] = v_qbasis[i]; wbasis[r] = v_wbasis[i];
}

int evg_update_tasks(evg_ctx* c, int64_t n_rows, const int64_t* rows, const evg_task_soa* v) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!c->have_tasks) return fail(EVG_ERR_STATE, "evg_update_tasks before evg_upload");
  if (c->adopted) return fail(EVG_ERR_STATE, "the resident columns are borrowed (evg_upload_device): edit them in place instead");
  if (n_rows < 0) return fail(EVG_ERR_INVALID, "negative row count");
  if (n_rows == 0) return EVG_OK;
  if (!rows || !v || v->n_tasks != n_rows || !v->priority || !v->num_dependents || !v->task_group_order || !v->flags || !v->expected_ns ||
      !v->queue_basis_ns || !v->wait_basis_ns)
    return fail(EVG_ERR_INVALID, "evg_update_tasks: rows and a %lld-row value table (priority, num_dependents, task_group_order, flags, "
                                 "expected_ns, queue_basis_ns, wait_basis_ns) are required", (long long)n_rows);
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const size_t n = size_t(n_rows);
  // staging: rows (8) + three 8-byte and four 4-byte columns = 48 B per changed row
  CK(c->b_upd.ensure(n * 48 + 64));
  unsigned char* base = c->b_upd.as<unsigned char>();
  int64_t* d_rows = reinterpret_cast<int64_t*>(base);
  int64_t* d_exp = d_rows + n; int64_t* d_qb = d_exp + n; int64_t* d_wb = d_qb + n;
  int32_t* d_prio = reinterpret_cast<int32_t*>(d_wb + n); int32_t* d_nd = d_prio + n; int32_t* d_tgo = d_nd + n;
  uint32_t* d_fl = reinterpret_cast<uint32_t*>(d_tgo + n);
  CK(cudaMemcpyAsync(d_rows, rows, n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_exp, v->expected_ns, n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_qb, v->queue_basis_ns, n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_wb, v->wait_basis_ns, n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_prio, v->priority, n * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_nd, v->num_dependents, n * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_tgo, v->task_group_order, n * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_fl, v->flags, n * 4, cudaMemcpyHostToDevice, s));
  int* bad = reinterpret_cast<int*>(base + n * 48);
  CK(cudaMemsetAsync(bad, 0, sizeof(int), s));
  k_update_rows<<<grid_for(n_rows, 256), 256, 0, s>>>(n_rows, d_rows, c->T, c->b_prio.as<int32_t>(), c->b_nd.as<int32_t>(), c->b_tgo.as<int32_t>(),
                                                      c->b_flags.as<uint32_t>(), c->b_exp.as<int64_t>(), c->b_qb.as<int64_t>(), c->b_wb.as<int64_t>(),
                                                      d_prio, d_nd, d_tgo, d_fl, d_exp, d_qb, d_wb, bad);
  CK(cudaGetLastError());
  int h_bad = 0;
  CK(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));  // the caller's staging arrays are free again
  if (h_bad) return fail(EVG_ERR_INVALID, "evg_update_tasks: a row index is outside [0, n_tasks)");
  c->deps_resident = false;  // flags / wait bases written by a device-side dependency evaluation may have been replaced
  return EVG_OK;
}

int evg_upload_device(evg_ctx* c, const evg_task_soa* tasks, const evg_distro_table* distros, const evg_host_soa* hosts,
                      const int64_t* host_off, const evg_alloc_cfg* acfg) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!tasks || !distros) return fail(EVG_ERR_INVALID, "null task table / distro table");
  CK(cudaSetDevice(c->device));
  std::vector<int64_t> edge_off;
  const int32_t D = distros->n_distros;
  if (tasks->n_edges > 0 && D > 0) {  // dep_off is device memory: sample it at the distro boundaries for the routing
    if (!tasks->dep_off || !distros->task_off) return fail(EVG_ERR_INVALID, "null dep_off / task_off");
    edge_off.resize(size_t(D) + 1);
    CK(c->b_rn0.ensure(sizeof(int64_t) * size_t(D + 1)));
    CK(c->b_rn1.ensure(sizeof(int64_t) * size_t(D + 1)));
    CK(cudaMemcpyAsync(c->b_rn0.p, distros->task_off, sizeof(int64_t) * size_t(D + 1), cudaMemcpyHostToDevice, c->stream));
    k_gather_i64<<<grid_for(D + 1, 256), 256, 0, c->stream>>>(tasks->dep_off, c->b_rn0.as<int64_t>(), c->b_rn1.as<int64_t>(), D + 1);
    CK(cudaMemcpyAsync(edge_off.data(), c->b_rn1.p, sizeof(int64_t) * size_t(D + 1), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  int rc = upload_tasks(c, tasks, distros, /*copy_columns=*/false, /*adopt=*/true, edge_off.empty() ? nullptr : edge_off.data());
  if (rc != EVG_OK) return rc;
  if (hosts) {
    rc = upload_hosts(c, hosts, host_off, acfg, distros->n_distros);
    if (rc != EVG_OK) return rc;
    CK(cudaStreamSynchronize(c->stream));
  }
  return EVG_OK;
}

int evg_run_resident(evg_ctx* c, int64_t now_ns, uint32_t opts) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!c->have_tasks) return fail(EVG_ERR_STATE, "evg_run_resident before evg_upload");
  CK(cudaSetDevice(c->device));
  c->launches = 0;
  c->timed = true;
  c->general_timed = false;
  CK(cudaEventRecord(c->ev_begin, c->stream));
  int rc = run_plan(c, now_ns, opts);
  if (rc != EVG_OK) return rc;
  if (c->have_hosts) {
    rc = run_alloc(c, now_ns);
    if (rc != EVG_OK) return rc;
  }
  CK(cudaEventRecord(c->ev_end, c->stream));
  return EVG_OK;
}

int evg_run_resident_head(evg_ctx* c, int64_t now_ns, uint32_t opts, int32_t cap) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (cap == 0) cap = EVG_PERSISTED_QUEUE_CAP;
  if (cap < 1 || cap > EVG_PERSISTED_QUEUE_CAP) return fail(EVG_ERR_INVALID, "evg_run_resident_head: cap %d outside [1, %d]", cap, EVG_PERSISTED_QUEUE_CAP);
  if (!c->have_tasks) return fail(EVG_ERR_STATE, "evg_run_resident_head before evg_upload");
  CK(cudaSetDevice(c->device));
  c->launches = 0;
  c->timed = true;
  c->general_timed = false;
  CK(cudaEventRecord(c->ev_begin, c->stream));
  int rc = run_plan(c, now_ns, opts, cap);
  if (rc != EVG_OK) return rc;
  if (c->have_hosts) {
    rc = run_alloc(c, now_ns);
    if (rc != EVG_OK) return rc;
  }
  CK(cudaEventRecord(c->ev_end, c->stream));
  return EVG_OK;
}

int evg_download(evg_ctx* c, evg_plan_out* po, evg_alloc_out* ao) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!c->have_tasks) return fail(EVG_ERR_STATE, "evg_download before evg_upload");
  if (po && c->head_cap > 0 && (po->order || po->total_value || po->breakdown))
    return fail(EVG_ERR_STATE, "the last run ordered only the first %d ranks of each distro: download them with evg_download_queue", c->head_cap);
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  if (po) {
    if (po->order && c->T) CK(cudaMemcpyAsync(po->order, c->b_order.p, sizeof(int32_t) * size_t(c->T), cudaMemcpyDeviceToHost, s));
    if (po->total_value && c->T) CK(cudaMemcpyAsync(po->total_value, c->b_tv.p, sizeof(int64_t) * size_t(c->T), cudaMemcpyDeviceToHost, s));
    if (po->breakdown && c->T) {
      if (!c->bd_valid) return fail(EVG_ERR_STATE, "breakdown requested but the run did not set EVG_OPT_BREAKDOWN");
      CK(cudaMemcpyAsync(po->breakdown, c->b_bd.p, sizeof(int64_t) * EVG_BD_N * size_t(c->T), cudaMemcpyDeviceToHost, s));
    }
    if (po->info && c->Dn) CK(cudaMemcpyAsync(po->info, c->b_qinfo.p, sizeof(evg_queue_info) * size_t(c->Dn), cudaMemcpyDeviceToHost, s));
    if (po->group_info && c->G) CK(cudaMemcpyAsync(po->group_info, c->b_ginfo.p, sizeof(evg_group_info) * size_t(c->G), cudaMemcpyDeviceToHost, s));
  }
  if (ao) {
    if (!c->have_hosts) return fail(EVG_ERR_STATE, "allocator results requested but no hosts were uploaded");
    if (ao->result && c->Dn) CK(cudaMemcpyAsync(ao->result, c->result_ptr(), sizeof(evg_alloc_result) * size_t(c->Dn), cudaMemcpyDeviceToHost, s));
    if (ao->status && c->Dn) CK(cudaMemcpyAsync(ao->status, c->b_status.p, sizeof(int32_t) * size_t(c->Dn), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return EVG_OK;
}

// TaskQueueItem rows of the persisted head of every queue (task_queue_persister.go:14-42): one thread per output row.
__global__ void __launch_bounds__(256) k_project_queue(DTasks T, DDistros D, const int64_t* __restrict__ item_off, int64_t n_items,
                                                       const int32_t* __restrict__ order, const int64_t* __restrict__ total_value,
                                                       evg_queue_item* __restrict__ items) {
  const int64_t j = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (j >= n_items) return;
  const int d = find_distro(item_off, 0, D.n - 1, j);
  const int64_t base = D.task_off[d];
  const int64_t r = j - item_off[d];
  const int32_t i = order[base + r];
  const int64_t t = base + i;
  const int32_t gid = T.gid[t];
  evg_queue_item q;
  q.task = i;
  q.group_index = T.tgo[t];
  q.group_max_hosts = gid >= 0 ? D.gmax[D.group_off[d] + gid] : 0;
  q.flags = (T.flags[t] & EVG_TF_DEPS_MET) ? EVG_QI_DEPS_MET : 0u;
  q.priority = T.priority[t];
  q.expected_ns = T.expected[t];
  q.total_value = total_value[base + r];
  items[j] = q;
}

// Row j of `out`: the breakdown row of the same rank as TaskQueueItem row j, read at bd_off[d] + rank.
__global__ void __launch_bounds__(256) k_project_breakdown(int32_t n_distros, const int64_t* __restrict__ item_off, int64_t n_items,
                                                           const int64_t* __restrict__ bd_off, const int64_t* __restrict__ bd,
                                                           int64_t* __restrict__ out) {
  const int64_t j = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (j >= n_items) return;
  const int d = find_distro(item_off, 0, n_distros - 1, j);
  const int64_t* src = bd + (bd_off[d] + j - item_off[d]) * EVG_BD_N;
#pragma unroll
  for (int k = 0; k < EVG_BD_N; k++) out[j * EVG_BD_N + k] = src[k];
}

namespace {
int download_queue(evg_ctx* c, int32_t cap, int64_t* item_off, evg_queue_item* items, int64_t* breakdown, int64_t items_capacity) {
  if (!c->have_tasks) return fail(EVG_ERR_STATE, "evg_download_queue before evg_upload");
  if (cap < 0 || !item_off) return fail(EVG_ERR_INVALID, "evg_download_queue: bad argument");
  if (cap == 0) cap = EVG_PERSISTED_QUEUE_CAP;
  if (c->head_cap > 0 && cap > c->head_cap)
    return fail(EVG_ERR_STATE, "evg_download_queue: cap %d exceeds the %d ranks the last run ordered", cap, c->head_cap);
  if (breakdown && !c->bd_valid) return fail(EVG_ERR_STATE, "evg_download_queue_bd: the last run did not set EVG_OPT_BREAKDOWN");
  const int32_t D = c->Dn;
  item_off[0] = 0;
  for (int32_t d = 0; d < D; d++) item_off[d + 1] = item_off[d] + std::min<int64_t>(c->h_taskoff[d + 1] - c->h_taskoff[d], cap);
  const int64_t n = item_off[D];
  if (n > items_capacity || (n > 0 && !items)) return fail(EVG_ERR_INVALID, "evg_download_queue: %lld rows needed, %lld available", (long long)n, (long long)items_capacity);
  if (n == 0) return EVG_OK;
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  CK(c->b_rn0.ensure(sizeof(int64_t) * size_t(D + 1)));
  CK(c->b_rn1.ensure(sizeof(evg_queue_item) * size_t(n)));
  CK(cudaMemcpyAsync(c->b_rn0.p, item_off, sizeof(int64_t) * size_t(D + 1), cudaMemcpyHostToDevice, s));
  k_project_queue<<<grid_for(n, 256), 256, 0, s>>>(dtasks(c), ddistros(c), c->b_rn0.as<int64_t>(), n, c->b_order.as<int32_t>(),
                                                 c->b_tv.as<int64_t>(), c->b_rn1.as<evg_queue_item>());
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(items, c->b_rn1.p, sizeof(evg_queue_item) * size_t(n), cudaMemcpyDeviceToHost, s));
  if (breakdown) {  // the breakdown rows of a head run sit at its head offsets, those of a full run at task_off
    const int64_t* bd_off = c->head_cap > 0 ? c->b_hoff.as<int64_t>() : c->b_taskoff.as<int64_t>();
    CK(c->b_rn2.ensure(sizeof(int64_t) * EVG_BD_N * size_t(n)));
    k_project_breakdown<<<grid_for(n, 256), 256, 0, s>>>(D, c->b_rn0.as<int64_t>(), n, bd_off, c->b_bd.as<int64_t>(), c->b_rn2.as<int64_t>());
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(breakdown, c->b_rn2.p, sizeof(int64_t) * EVG_BD_N * size_t(n), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return EVG_OK;
}
}  // namespace

int evg_download_queue(evg_ctx* c, int32_t cap, int64_t* item_off, evg_queue_item* items, int64_t items_capacity) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  return download_queue(c, cap, item_off, items, nullptr, items_capacity);
}

int evg_download_queue_bd(evg_ctx* c, int32_t cap, int64_t* item_off, evg_queue_item* items, int64_t* breakdown,
                          int64_t items_capacity) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!breakdown) return fail(EVG_ERR_INVALID, "evg_download_queue_bd: null breakdown");
  return download_queue(c, cap, item_off, items, breakdown, items_capacity);
}

void* evg_device_result_ptr(evg_ctx* c) { return c ? (void*)c->result_ptr() : nullptr; }
int evg_bind_result_buffer(evg_ctx* c, void* device_ptr, int64_t capacity) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (device_ptr && capacity < 0) return fail(EVG_ERR_INVALID, "negative capacity");
  c->ext_result = reinterpret_cast<evg_alloc_result*>(device_ptr);
  c->ext_capacity = device_ptr ? capacity : 0;
  return EVG_OK;
}
int64_t evg_last_launch_count(evg_ctx* c) { return c ? c->launches : 0; }

int evg_last_timing_ms(evg_ctx* c, float* total_ms, float* sort_ms) {
  if (!c || !c->timed) return fail(EVG_ERR_STATE, "no timed run");
  LOCK(c);
  CK(cudaSetDevice(c->device));
  CK(cudaEventSynchronize(c->ev_end));
  if (total_ms) CK(cudaEventElapsedTime(total_ms, c->ev_begin, c->ev_end));
  if (sort_ms) {
    if (c->sort_slot >= 0) CK(cudaEventElapsedTime(sort_ms, c->ring0[c->sort_slot], c->ring1[c->sort_slot]));
    else if (c->general_timed) CK(cudaEventElapsedTime(sort_ms, c->ev_sort0, c->ev_sort1));
    else *sort_ms = 0.0f;  // a tick of small distros only: no kernel of its own was bracketed
  }
  return EVG_OK;
}

int evg_general_timing_ms(evg_ctx* c, float* task_pass_ms, float* sort_ms) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!c->timed || !c->general_timed) return fail(EVG_ERR_STATE, "the last timed run had no general-path distro");
  CK(cudaSetDevice(c->device));
  CK(cudaEventSynchronize(c->ev_end));
  if (task_pass_ms) CK(cudaEventElapsedTime(task_pass_ms, c->ev_gt0, c->ev_gt1));
  if (sort_ms) CK(cudaEventElapsedTime(sort_ms, c->ev_sort0, c->ev_sort1));
  return EVG_OK;
}

int evg_kernel_timing_ms(evg_ctx* c, float* out_ms, int32_t n) {
  if (!c || !out_ms || n < 0) return fail(EVG_ERR_INVALID, "evg_kernel_timing_ms: bad argument");
  LOCK(c);
  if (n > evg_ctx::kRing || n > c->runs) return fail(EVG_ERR_STATE, "only %lld timed runs recorded (ring of %d)", (long long)c->runs, evg_ctx::kRing);
  CK(cudaSetDevice(c->device));
  for (int32_t k = 0; k < n; k++) {
    const int slot = int((c->runs - n + k) % evg_ctx::kRing);
    CK(cudaEventSynchronize(c->ring1[slot]));
    CK(cudaEventElapsedTime(out_ms + k, c->ring0[slot], c->ring1[slot]));
  }
  return EVG_OK;
}

int evg_plan_batch(evg_ctx* c, const evg_task_soa* tasks, const evg_distro_table* distros, int64_t now_ns, uint32_t opts,
                   evg_plan_out* out) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  int rc = evg_upload(c, tasks, distros, nullptr, nullptr, nullptr);
  if (rc != EVG_OK) return rc;
  rc = evg_run_resident(c, now_ns, opts);
  if (rc != EVG_OK) return rc;
  return evg_download(c, out, nullptr);
}

// The one-shot call as a three-stage pipeline over chunks of whole distros: H2D of chunk k+1, kernels of chunk k
// and D2H of chunk k-1 overlap on three streams, so the tick costs about max(H2D, D2H) instead of their sum.
// Used for ticks of at least 2^21 tasks when no breakdown is requested; a chunk's general-path distros run through the
// general path restricted to their tiles.
static int plan_and_alloc_pipelined(evg_ctx* c, const evg_task_soa* t, const evg_distro_table* dt, const evg_host_soa* hosts,
                                    const int64_t* host_off, const evg_alloc_cfg* acfg, int64_t now, evg_plan_out* po,
                                    evg_alloc_out* ao) {
  const int64_t T = c->T, E = c->E;
  const int32_t D = c->Dn;
  if (!c->s_h2d) {
    CK(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < evg_ctx::kMaxChunks; k++) {
      CK(cudaEventCreateWithFlags(&c->ev_h[k], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&c->ev_c[k], cudaEventDisableTiming));
    }
  }
  cudaStream_t s = c->stream;
  DTasks dtk = dtasks(c);
  DDistros dd = ddistros(c);
  DWork w = dwork(c);
  if (c->ext_result && c->ext_capacity < D) return fail(EVG_ERR_INVALID, "bound result buffer too small");
  CK(c->b_gs.ensure(sizeof(GroupScratch) * size_t(c->G + 1)));
  c->launches = 0;
  c->timed = false;
  c->bd_valid = false;
  c->head_cap = 0;
  CK(cudaMemsetAsync(c->b_puntcnt.p, 0, sizeof(int32_t) * (evg_ctx::kMaxChunks + 2), s));
  // chunk boundaries: whole distros, about equal task counts
  const int n_chunks = int(std::min<int64_t>(evg_ctx::kMaxChunks, std::max<int64_t>(1, T / (1 << 20))));
  std::vector<int32_t> cut(size_t(n_chunks) + 1, D);
  cut[0] = 0;
  {
    int32_t d = 0;
    for (int k = 1; k < n_chunks; k++) {
      const int64_t want = T * k / n_chunks;
      while (d < D && c->h_taskoff[d] < want) d++;
      cut[k] = d;
    }
  }
  auto sub = [](const std::vector<int32_t>& v, int32_t d0, int32_t d1, int32_t* first) {
    auto a = std::lower_bound(v.begin(), v.end(), d0), b = std::lower_bound(v.begin(), v.end(), d1);
    *first = int32_t(a - v.begin());
    return int32_t(b - a);
  };
#define H2D(buf, ptr, off, count, type)                                                                  \
  if ((count) > 0) CK(cudaMemcpyAsync((buf).as<type>() + (off), (ptr) + (off), sizeof(type) * size_t(count), cudaMemcpyHostToDevice, c->s_h2d))
#define D2H(dst, src, off, count, type)                                                                  \
  if ((dst) && (count) > 0) CK(cudaMemcpyAsync((dst) + (off), (src) + (off), sizeof(type) * size_t(count), cudaMemcpyDeviceToHost, c->s_d2h))
  int rc;
  for (int k = 0; k < n_chunks; k++) {
    const int32_t d0 = cut[k], d1 = cut[k + 1];
    if (d1 <= d0) continue;
    const int64_t t0 = c->h_taskoff[d0], n = c->h_taskoff[d1] - t0;
    const int64_t g0 = c->h_groupoff[d0], ng = c->h_groupoff[d1] - g0;
    H2D(c->b_prio, t->priority, t0, n, int32_t);
    H2D(c->b_exp, t->expected_ns, t0, n, int64_t);
    H2D(c->b_qb, t->queue_basis_ns, t0, n, int64_t);
    H2D(c->b_wb, t->wait_basis_ns, t0, n, int64_t);
    H2D(c->b_nd, t->num_dependents, t0, n, int32_t);
    H2D(c->b_tgo, t->task_group_order, t0, n, int32_t);
    H2D(c->b_gid, t->group_id, t0, n, int32_t);
    H2D(c->b_vid, t->version_id, t0, n, int32_t);
    H2D(c->b_flags, t->flags, t0, n, uint32_t);
    if (E > 0) {
      const int64_t e0 = t->dep_off[t0], ne = t->dep_off[t0 + n] - e0;
      H2D(c->b_depoff, t->dep_off, t0, n + 1, int64_t);
      H2D(c->b_depidx, t->dep_idx, e0, ne, int32_t);
    }
    CK(cudaEventRecord(c->ev_h[k], c->s_h2d));
    CK(cudaStreamWaitEvent(s, c->ev_h[k], 0));
    k_validate<<<grid_for(n, 256), 256, 0, s>>>(dtk, dd, w, t0, t0 + n);
    int32_t first, cnt;
    {  // second-generation on-chip classes; the distros they hand back are replanned by k_plan_smem right behind them
      int32_t fC, fB, fA;
      const int32_t nC = sub(c->h_listNC, d0, d1, &fC), nB = sub(c->h_listNB, d0, d1, &fB), nA = sub(c->h_listNA, d0, d1, &fA);
      int32_t* pl = c->b_punt.as<int32_t>() + d0;  // a chunk hands back at most its own d1 - d0 distros
      int32_t* pc = c->b_puntcnt.as<int32_t>() + 1 + k;
      if ((rc = launch_cta<kNT_C, kNCapC, kNOccC>(c, s, dtk, dd, w, c->b_listNC.as<int32_t>() + fC, nC, now, pl, pc)) != EVG_OK) return rc;
      if ((rc = launch_cta<kNT_B, kNCapB, kNOccB>(c, s, dtk, dd, w, c->b_listNB.as<int32_t>() + fB, nB, now, pl, pc)) != EVG_OK) return rc;
      if ((rc = launch_cta<kNT_A, kNCapA, kNOccA>(c, s, dtk, dd, w, c->b_listNA.as<int32_t>() + fA, nA, now, pl, pc)) != EVG_OK) return rc;
      if ((rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, s, dtk, dd, w, pl, nC + nB + nA, now, 0, pc)) != EVG_OK) return rc;
    }
    cnt = sub(c->h_listG, d0, d1, &first);
    if (cnt > 0) {  // the chunk's general-path distros: same kernels, restricted to their tiles
      if ((rc = prepare_general(c, s, c->h_listG[size_t(first)], c->h_listG[size_t(first + cnt - 1)] + 1)) != EVG_OK) return rc;
      if ((rc = run_general(c, s, dtk, dd, w, now, first, cnt)) != EVG_OK) return rc;
    }
    cnt = sub(c->h_listC, d0, d1, &first);
    if ((rc = launch_smem<EVG_C_THREADS, EVG_C_ITEMS, 1>(c, s, dtk, dd, w, c->b_listC.as<int32_t>() + first, cnt, now)) != EVG_OK) return rc;
    cnt = sub(c->h_listB, d0, d1, &first);
    if ((rc = launch_smem<256, 16, 3>(c, s, dtk, dd, w, c->b_listB.as<int32_t>() + first, cnt, now)) != EVG_OK) return rc;
    cnt = sub(c->h_listA, d0, d1, &first);
    if ((rc = launch_smem<128, 8, 8>(c, s, dtk, dd, w, c->b_listA.as<int32_t>() + first, cnt, now)) != EVG_OK) return rc;
    cnt = sub(c->h_listW, d0, d1, &first);
    if ((rc = launch_tiny(c, s, dtk, dd, w, c->b_listW.as<int32_t>() + first, cnt, now, 0)) != EVG_OK) return rc;
    if ((rc = run_alloc_range(c, now, d0, d1)) != EVG_OK) return rc;
    CK(cudaEventRecord(c->ev_c[k], s));
    CK(cudaStreamWaitEvent(c->s_d2h, c->ev_c[k], 0));
    if (po) {
      D2H(po->order, c->b_order.as<int32_t>(), t0, n, int32_t);
      D2H(po->total_value, c->b_tv.as<int64_t>(), t0, n, int64_t);
      D2H(po->info, c->b_qinfo.as<evg_queue_info>(), d0, d1 - d0, evg_queue_info);
      D2H(po->group_info, c->b_ginfo.as<evg_group_info>(), g0, ng, evg_group_info);
    }
    if (ao) {
      D2H(ao->result, c->result_ptr(), d0, d1 - d0, evg_alloc_result);
      D2H(ao->status, c->b_status.as<int32_t>(), d0, d1 - d0, int32_t);
    }
  }
#undef H2D
#undef D2H
  CK(cudaGetLastError());
  int bad = 0;
  CK(cudaMemcpyAsync(&bad, c->b_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(c->s_d2h));
  CK(cudaStreamSynchronize(s));
  if (bad) { c->have_tasks = false; return fail(EVG_ERR_INVALID, "a group_id / version_id / dep_idx is out of range for its distro"); }
  c->have_hosts = true;
  return EVG_OK;
}

int evg_plan_and_alloc_batch(evg_ctx* c, const evg_task_soa* tasks, const evg_distro_table* distros,
                             const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* acfg, int64_t now_ns,
                             uint32_t opts, evg_plan_out* plan_out, evg_alloc_out* alloc_out) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!hosts || (!acfg && distros && distros->n_distros > 0)) return fail(EVG_ERR_INVALID, "evg_plan_and_alloc_batch needs hosts and allocator config");
  if (!(opts & EVG_OPT_BREAKDOWN) && tasks && distros && tasks->n_tasks >= (int64_t(1) << 21)) {
    // large tick: stage the small tables, then pipeline the columns chunk by chunk
    CK(cudaSetDevice(c->device));
    int rc0 = upload_tasks(c, tasks, distros, /*copy_columns=*/false);
    if (rc0 != EVG_OK) return rc0;
    rc0 = upload_hosts(c, hosts, host_off, acfg, distros->n_distros);
    if (rc0 != EVG_OK) return rc0;
    CK(cudaStreamSynchronize(c->stream));
    return plan_and_alloc_pipelined(c, tasks, distros, hosts, host_off, acfg, now_ns, plan_out, alloc_out);
  }
  int rc = evg_upload(c, tasks, distros, hosts, host_off, acfg);
  if (rc != EVG_OK) return rc;
  rc = evg_run_resident(c, now_ns, opts);
  if (rc != EVG_OK) return rc;
  return evg_download(c, plan_out, alloc_out);
}

int evg_alloc_batch(evg_ctx* c, const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* cfg,
                    const evg_queue_info* info, evg_group_info* groups, const int64_t* group_off, int32_t n_distros,
                    int64_t now_ns, evg_alloc_out* out) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (n_distros < 0 || (n_distros > 0 && (!info || !group_off || !out))) return fail(EVG_ERR_INVALID, "evg_alloc_batch: null argument");
  CK(cudaSetDevice(c->device));
  const int64_t G = n_distros > 0 ? group_off[n_distros] : 0;
  if (G > 0 && !groups) return fail(EVG_ERR_INVALID, "evg_alloc_batch: groups is null");
  c->have_tasks = false;  // the resident planner inputs no longer match the tables of this call (and upload_hosts must not list distros from them)
  int rc = upload_hosts(c, hosts, host_off, cfg, n_distros);
  if (rc != EVG_OK) return rc;
  cudaStream_t s = c->stream;
  CK(c->b_groupoff.ensure(sizeof(int64_t) * size_t(n_distros + 1)));
  CK(c->b_qinfo.ensure(sizeof(evg_queue_info) * size_t(n_distros + 1)));
  CK(c->b_ginfo.ensure(sizeof(evg_group_info) * size_t(G + 1)));
  if (n_distros > 0) {
    CK(cudaMemcpyAsync(c->b_groupoff.p, group_off, sizeof(int64_t) * size_t(n_distros + 1), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->b_qinfo.p, info, sizeof(evg_queue_info) * size_t(n_distros), cudaMemcpyHostToDevice, s));
  }
  if (G > 0) CK(cudaMemcpyAsync(c->b_ginfo.p, groups, sizeof(evg_group_info) * size_t(G), cudaMemcpyHostToDevice, s));
  c->Dn = n_distros;
  c->G = G;
  c->max_groups = 0;
  for (int32_t d = 0; d < n_distros; d++) c->max_groups = std::max(c->max_groups, group_off[d + 1] - group_off[d]);
  c->have_tasks = false;  // the resident planner inputs no longer match these tables
  c->launches = 0;
  rc = run_alloc(c, now_ns);
  if (rc != EVG_OK) return rc;
  if (out->result && n_distros) CK(cudaMemcpyAsync(out->result, c->result_ptr(), sizeof(evg_alloc_result) * size_t(n_distros), cudaMemcpyDeviceToHost, s));
  if (out->status && n_distros) CK(cudaMemcpyAsync(out->status, c->b_status.p, sizeof(int32_t) * size_t(n_distros), cudaMemcpyDeviceToHost, s));
  if (G > 0) CK(cudaMemcpyAsync(groups, c->b_ginfo.p, sizeof(evg_group_info) * size_t(G), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return EVG_OK;
}

// Stage an evg_deps_in table and run k_deps_met into b_dx7 (left on the device); `both` adds the no-short-circuit bit.
static int deps_to_device(evg_ctx* c, const evg_deps_in* in, int both, const int64_t* dep_finished = nullptr, int64_t now = 0,
                          bool want_stamp = false) {
  const int64_t T = in->n_tasks, E = in->n_deps, X = in->n_ext;
  if (T < 0 || E < 0 || X < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (T == 0) return EVG_OK;
  if (!in->dep_off || !in->task_state || !in->task_pre) return fail(EVG_ERR_INVALID, "null task arrays");
  if (E > 0 && (!in->dep_kind || !in->dep_ref || !in->dep_want)) return fail(EVG_ERR_INVALID, "null dependency arrays");
  if (X > 0 && !in->ext_state) return fail(EVG_ERR_INVALID, "null ext_state");
  if (in->dep_off[0] != 0 || in->dep_off[T] != E) return fail(EVG_ERR_INVALID, "dep_off does not span n_deps");
  cudaStream_t s = c->stream;
#define UPD(buf, ptr, count, type)                                                                                 \
  do {                                                                                                             \
    CK((buf).ensure(sizeof(type) * size_t((count) > 0 ? (count) : 1)));                                            \
    if ((count) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count), cudaMemcpyHostToDevice, s)); \
  } while (0)
  UPD(c->b_dx0, in->dep_off, T + 1, int64_t);
  UPD(c->b_dx1, in->dep_kind, E, uint8_t);
  UPD(c->b_dx2, in->dep_ref, E, int32_t);
  UPD(c->b_dx3, in->dep_want, E, uint8_t);
  UPD(c->b_dx4, in->task_state, T, uint8_t);
  UPD(c->b_dx5, in->task_pre, T, uint8_t);
  UPD(c->b_dx6, in->ext_state, X, uint8_t);
#undef UPD
  CK(c->b_dx7.ensure(size_t(T)));
  int64_t* stamp = nullptr;
  const int64_t* fin = nullptr;
  if (want_stamp) {
    CK(c->b_rn7.ensure(sizeof(int64_t) * size_t(T)));
    stamp = c->b_rn7.as<int64_t>();
    if (dep_finished && E > 0) {
      CK(c->b_rn6.ensure(sizeof(int64_t) * size_t(E)));
      CK(cudaMemcpyAsync(c->b_rn6.p, dep_finished, sizeof(int64_t) * size_t(E), cudaMemcpyHostToDevice, s));
      fin = c->b_rn6.as<int64_t>();
    }
  }
  DDeps d;
  d.n_tasks = T; d.dep_off = c->b_dx0.as<int64_t>(); d.dep_kind = c->b_dx1.as<uint8_t>(); d.dep_ref = c->b_dx2.as<int32_t>();
  d.dep_want = c->b_dx3.as<uint8_t>(); d.task_state = c->b_dx4.as<uint8_t>(); d.task_pre = c->b_dx5.as<uint8_t>();
  d.ext_state = c->b_dx6.as<uint8_t>(); d.n_ext = X;
  k_deps_met<<<grid_for(T, 256), 256, 0, s>>>(d, c->b_dx7.as<uint8_t>(), c->b_err.as<int>(), both, fin, now, stamp);
  c->launches++;
  CK(cudaGetLastError());
  return EVG_OK;
}

int evg_deps_met_batch(evg_ctx* c, const evg_deps_in* in, uint8_t* met) {
  if (!c || !in || (in->n_tasks > 0 && !met)) return fail(EVG_ERR_INVALID, "evg_deps_met_batch: null argument");
  LOCK(c);
  if (in->n_tasks == 0) return EVG_OK;
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  CK(c->b_err.ensure(sizeof(int) * 4));
  CK(cudaMemsetAsync(c->b_err.p, 0, sizeof(int) * 4, s));
  c->launches = 0;
  int rc = deps_to_device(c, in, 0);
  if (rc != EVG_OK) return rc;
  int bad = 0;
  CK(cudaMemcpyAsync(met, c->b_dx7.p, size_t(in->n_tasks), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&bad, c->b_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bad) return fail(EVG_ERR_INVALID, "a dep_ref is out of range");
  return EVG_OK;
}

int evg_upload_with_deps(evg_ctx* c, const evg_task_soa* tasks, const evg_distro_table* distros, const evg_host_soa* hosts,
                         const int64_t* host_off, const evg_alloc_cfg* acfg, const evg_deps_in* deps, const int64_t* dep_finished_ns,
                         int64_t now_ns) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!tasks || !deps) return fail(EVG_ERR_INVALID, "evg_upload_with_deps: null argument");
  if (deps->n_tasks != tasks->n_tasks) return fail(EVG_ERR_INVALID, "deps covers %lld tasks, the task table %lld", (long long)deps->n_tasks, (long long)tasks->n_tasks);
  int rc = evg_upload(c, tasks, distros, hosts, host_off, acfg);
  if (rc != EVG_OK) return rc;
  const int64_t T = tasks->n_tasks;
  if (T == 0) return EVG_OK;
  cudaStream_t s = c->stream;
  rc = deps_to_device(c, deps, 0, dep_finished_ns, now_ns, /*want_stamp=*/true);
  if (rc != EVG_OK) { c->have_tasks = false; return rc; }
  k_apply_deps<<<grid_for(T, 256), 256, 0, s>>>(T, c->b_dx7.as<uint8_t>(), c->b_rn7.as<int64_t>(), c->b_flags.as<uint32_t>(), c->b_wb.as<int64_t>());
  c->launches++;
  int bad = 0;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(&bad, c->b_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bad) { c->have_tasks = false; return fail(EVG_ERR_INVALID, "a dep_ref is out of range"); }
  c->deps_resident = true;
  return EVG_OK;
}

int evg_download_deps(evg_ctx* c, uint8_t* met, int64_t* met_time_ns) {
  if (!c) return fail(EVG_ERR_INVALID, "null context");
  LOCK(c);
  if (!c->have_tasks) return fail(EVG_ERR_STATE, "evg_download_deps before evg_upload_with_deps");
  CK(cudaSetDevice(c->device));
  if (c->T == 0) return EVG_OK;
  if (!c->deps_resident) return fail(EVG_ERR_STATE, "the resident tick was not uploaded with evg_upload_with_deps");
  if (met) CK(cudaMemcpyAsync(met, c->b_dx7.p, size_t(c->T), cudaMemcpyDeviceToHost, c->stream));
  if (met_time_ns) CK(cudaMemcpyAsync(met_time_ns, c->b_rn7.p, sizeof(int64_t) * size_t(c->T), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return EVG_OK;
}

int evg_expected_durations_batch(evg_ctx* c, const evg_duration_rows* in, evg_duration_stat* out) {
  if (!c || !in) return fail(EVG_ERR_INVALID, "evg_expected_durations_batch: null argument");
  LOCK(c);
  const int64_t R = in->n_rows;
  const int32_t K = in->n_keys;
  if (R < 0 || K < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (K == 0) return R == 0 ? EVG_OK : fail(EVG_ERR_INVALID, "rows without keys");
  if (!out) return fail(EVG_ERR_INVALID, "null output");
  if (R > 0 && (!in->key || !in->time_taken_ns || !in->start_ns || !in->finish_ns || !in->flags)) return fail(EVG_ERR_INVALID, "null row column");
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  c->launches = 0;
  c->have_tasks = false;  // shares scratch buffers with the finder entry points
#define UPX(buf, ptr, count, type)                                                                                 \
  do {                                                                                                             \
    CK((buf).ensure(sizeof(type) * size_t((count) > 0 ? (count) : 1)));                                            \
    if ((count) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count), cudaMemcpyHostToDevice, s)); \
  } while (0)
  UPX(c->b_rn0, in->key, R, int32_t);
  UPX(c->b_rn1, in->time_taken_ns, R, int64_t);
  UPX(c->b_rn2, in->start_ns, R, int64_t);
  UPX(c->b_rn3, in->finish_ns, R, int64_t);
  UPX(c->b_rn4, in->flags, R, uint8_t);
#undef UPX
  CK(c->b_rn5.ensure(sizeof(unsigned long long) * 4 * size_t(K)));
  CK(c->b_rn6.ensure(sizeof(evg_duration_stat) * size_t(K)));
  CK(c->b_err.ensure(sizeof(int) * 4));
  CK(cudaMemsetAsync(c->b_err.p, 0, sizeof(int) * 4, s));
  CK(cudaMemsetAsync(c->b_rn5.p, 0, sizeof(unsigned long long) * 4 * size_t(K), s));
  DDur x;
  x.n_rows = R; x.n_keys = K; x.key = c->b_rn0.as<int32_t>(); x.taken = c->b_rn1.as<int64_t>(); x.start = c->b_rn2.as<int64_t>();
  x.finish = c->b_rn3.as<int64_t>(); x.flags = c->b_rn4.as<uint8_t>(); x.w0 = in->window_start_ns; x.w1 = in->window_end_ns;
  x.cnt = c->b_rn5.as<unsigned long long>(); x.sum = x.cnt + K; x.sq_lo = x.sum + K; x.sq_hi = x.sq_lo + K;
  if (R > 0) {
    k_dur_sum<<<grid_for(R, 256), 256, 0, s>>>(x, c->b_err.as<int>());
    k_dur_dev<<<grid_for(R, 256), 256, 0, s>>>(x);
    c->launches += 2;
  }
  k_dur_final<<<grid_for(K, 256), 256, 0, s>>>(x, c->b_rn6.as<evg_duration_stat>());
  c->launches++;
  CK(cudaGetLastError());
  int bad = 0;
  CK(cudaMemcpyAsync(out, c->b_rn6.p, sizeof(evg_duration_stat) * size_t(K), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&bad, c->b_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bad) return fail(EVG_ERR_INVALID, "a key is out of range");
  return EVG_OK;
}

int evg_find_runnable_batch(evg_ctx* c, const evg_runnable_in* in, int32_t* runnable, int64_t* count) {
  if (!c || !in) return fail(EVG_ERR_INVALID, "evg_find_runnable_batch: null argument");
  LOCK(c);
  const int64_t T = in->n_tasks;
  const int32_t D = in->n_distros, P = in->n_projects;
  if (T < 0 || D < 0 || P < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (D == 0) return T == 0 ? EVG_OK : fail(EVG_ERR_INVALID, "tasks without distros");
  if (!count || (T > 0 && !runnable)) return fail(EVG_ERR_INVALID, "null output");
  if (!in->task_off || !in->valid_off || !in->finder) return fail(EVG_ERR_INVALID, "null distro arrays");
  if (T > 0 && (!in->sched || !in->project)) return fail(EVG_ERR_INVALID, "null task column");
  if (P > 0 && !in->project_flags) return fail(EVG_ERR_INVALID, "null project_flags");
  if (in->task_off[0] != 0 || in->task_off[D] != T || in->valid_off[0] != 0) return fail(EVG_ERR_INVALID, "offsets do not span the tables");
  bool any_deps = false;
  for (int32_t d = 0; d < D; d++) {
    if (in->task_off[d + 1] < in->task_off[d] || in->valid_off[d + 1] < in->valid_off[d]) return fail(EVG_ERR_INVALID, "offsets of distro %d decrease", d);
    if (in->finder[d] > EVG_FINDER_ALTERNATE) return fail(EVG_ERR_INVALID, "distro %d: unknown finder %d", d, int(in->finder[d]));
    any_deps = any_deps || in->finder[d] != EVG_FINDER_NO_DEPS;
  }
  const int64_t V = in->valid_off[D];
  if (V > 0 && !in->valid_idx) return fail(EVG_ERR_INVALID, "null valid_idx");
  if (any_deps && T > 0 && (!in->deps || in->deps->n_tasks != T)) return fail(EVG_ERR_INVALID, "a finder checks dependencies but deps is null or of another size");
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  CK(c->b_err.ensure(sizeof(int) * 4));
  CK(cudaMemsetAsync(c->b_err.p, 0, sizeof(int) * 4, s));
  c->launches = 0;
  c->have_tasks = false;  // the scratch columns below are shared with nothing resident, but the order buffer is reused
  if (any_deps && T > 0) {
    int rc = deps_to_device(c, in->deps, 1);
    if (rc != EVG_OK) return rc;
  }
#define UPR(buf, ptr, count, type)                                                                                 \
  do {                                                                                                             \
    CK((buf).ensure(sizeof(type) * size_t((count) > 0 ? (count) : 1)));                                            \
    if ((count) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count), cudaMemcpyHostToDevice, s)); \
  } while (0)
  UPR(c->b_rn0, in->task_off, D + 1, int64_t);
  UPR(c->b_rn1, in->sched, T, uint8_t);
  UPR(c->b_rn2, in->project, T, int32_t);
  UPR(c->b_rn3, in->project_flags, P, uint8_t);
  UPR(c->b_rn4, in->valid_off, D + 1, int64_t);
  UPR(c->b_rn5, in->valid_idx, V, int32_t);
  UPR(c->b_rn6, in->finder, D, uint8_t);
#undef UPR
  CK(c->b_order.ensure(sizeof(int32_t) * size_t(T + 1)));
  CK(c->b_rn7.ensure(sizeof(int64_t) * size_t(D)));
  DRunnable r;
  r.n_tasks = T; r.n_distros = D; r.n_projects = P;
  r.task_off = c->b_rn0.as<int64_t>(); r.sched = c->b_rn1.as<uint8_t>(); r.project = c->b_rn2.as<int32_t>();
  r.project_flags = c->b_rn3.as<uint8_t>(); r.valid_off = c->b_rn4.as<int64_t>(); r.valid_idx = c->b_rn5.as<int32_t>();
  r.finder = c->b_rn6.as<uint8_t>(); r.met = (any_deps && T > 0) ? c->b_dx7.as<uint8_t>() : nullptr;
  k_runnable<<<unsigned(D), 256, 0, s>>>(r, c->b_order.as<int32_t>(), c->b_rn7.as<int64_t>(), c->b_err.as<int>());
  c->launches++;
  CK(cudaGetLastError());
  int bad = 0;
  if (T > 0) CK(cudaMemcpyAsync(runnable, c->b_order.p, sizeof(int32_t) * size_t(T), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(count, c->b_rn7.p, sizeof(int64_t) * size_t(D), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&bad, c->b_err.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bad) return fail(EVG_ERR_INVALID, "a project row or dep_ref is out of range");
  return EVG_OK;
}

// --------------------------------------------------------------------------
// evg_plan_from_finder: finder -> dependency predicate -> compaction -> resident planner inputs, all on the device
// --------------------------------------------------------------------------
struct PfCols {  // nine planner columns, candidate table (src) and compacted table (dst)
  const int32_t *priority, *numdep, *tgo, *gid, *vid;
  const uint32_t* flags;
  const int64_t *expected, *qbasis, *wbasis;
  int32_t *o_priority, *o_numdep, *o_tgo, *o_gid, *o_vid;
  uint32_t* o_flags;
  int64_t *o_expected, *o_qbasis, *o_wbasis;
  const int64_t* group_off;  // candidate group table (n_distros + 1); nullptr when no distro has a group
  const int32_t* group_remap;  // [group_off[d] + g] = distro-local slot of candidate group g among the kept groups
};
// used[group_off[d] + g] = 1 for every candidate group g of distro d that kept at least one task; a group id outside
// [-1, groups of the distro) raises err[1] instead of indexing anything.
__global__ void __launch_bounds__(256) k_pf_mark_groups(int64_t n_cand, int32_t D, const int64_t* __restrict__ cand_off,
                                                        const int32_t* __restrict__ kept, const int64_t* __restrict__ count,
                                                        const int32_t* __restrict__ gid, const int64_t* __restrict__ group_off,
                                                        uint8_t* __restrict__ used, int* err) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int d = block_find_distro(cand_off, D, i, n_cand);
  if (d < 0 || i - cand_off[d] >= count[d]) return;
  const int32_t g = gid[cand_off[d] + kept[i]];
  if (g < -1 || g >= group_off[d + 1] - group_off[d]) atomicOr(err + 1, 1);
  else if (g >= 0) used[group_off[d] + g] = 1;
}
// One thread per KEPT task: its row of the candidate table moves to its place in the compacted table; the
// EVG_TF_DEPS_MET bit and the stamped wait basis come from the device's own evaluation (k_deps_met), like
// evg_upload_with_deps; the group id becomes the group's slot among the groups that kept a task.
// new_idx[candidate row] = distro-local index in the compacted queue (memset to -1 before).
__global__ void __launch_bounds__(256) k_pf_gather(int64_t n_new, int32_t D, const int64_t* __restrict__ new_off, const int64_t* __restrict__ cand_off,
                                                   const int32_t* __restrict__ kept, PfCols C, const uint8_t* __restrict__ met,
                                                   const int64_t* __restrict__ met_time, int32_t* __restrict__ new_idx, int64_t* __restrict__ src_row) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int d = block_find_distro(new_off, D, i, n_new);
  if (d < 0) return;
  const int64_t k = i - new_off[d];
  const int64_t src = cand_off[d] + kept[cand_off[d] + k];
  const int32_t g = C.gid[src];
  C.o_priority[i] = C.priority[src]; C.o_numdep[i] = C.numdep[src]; C.o_tgo[i] = C.tgo[src]; C.o_vid[i] = C.vid[src];
  C.o_gid[i] = (g >= 0 && C.group_remap) ? C.group_remap[C.group_off[d] + g] : g;
  C.o_expected[i] = C.expected[src]; C.o_qbasis[i] = C.qbasis[src];
  C.o_flags[i] = (C.flags[src] & ~EVG_TF_DEPS_MET) | ((met[src] & 1) ? EVG_TF_DEPS_MET : 0u);
  const int64_t wb = C.wbasis[src], st = met_time[src];
  C.o_wbasis[i] = (st != EVG_TIME_ZERO && st > wb) ? st : wb;
  new_idx[src] = int32_t(k);
  src_row[i] = src;
}
// in-queue dependency edges that survive: both ends kept
__global__ void __launch_bounds__(256) k_pf_edge_count(int64_t n_new, int32_t D, const int64_t* __restrict__ new_off, const int64_t* __restrict__ cand_off,
                                                       const int64_t* __restrict__ src_row, const int64_t* __restrict__ dep_off,
                                                       const int32_t* __restrict__ dep_idx, const int32_t* __restrict__ new_idx, int32_t* __restrict__ cnt) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int d = block_find_distro(new_off, D, i, n_new);
  if (d < 0) return;
  const int64_t src = src_row[i], cb = cand_off[d];
  int32_t n = 0;
  for (int64_t e = dep_off[src]; e < dep_off[src + 1]; e++) n += new_idx[cb + dep_idx[e]] >= 0;
  cnt[i] = n;
}
__global__ void __launch_bounds__(256) k_pf_edge_write(int64_t n_new, int32_t D, const int64_t* __restrict__ new_off, const int64_t* __restrict__ cand_off,
                                                       const int64_t* __restrict__ src_row, const int64_t* __restrict__ dep_off,
                                                       const int32_t* __restrict__ dep_idx, const int32_t* __restrict__ new_idx,
                                                       const int64_t* __restrict__ o_dep_off, int32_t* __restrict__ o_dep_idx) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int d = block_find_distro(new_off, D, i, n_new);
  if (d < 0) return;
  const int64_t src = src_row[i], cb = cand_off[d];
  int64_t w = o_dep_off[i];
  for (int64_t e = dep_off[src]; e < dep_off[src + 1]; e++) {
    const int32_t j = new_idx[cb + dep_idx[e]];
    if (j >= 0) o_dep_idx[w++] = j;
  }
}
// exclusive scan of int32 counts into int64 offsets (n + 1 entries), three launches
__global__ void __launch_bounds__(1024) k_scan_blocks(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out, int64_t* __restrict__ block_sum) {
  __shared__ int64_t sw[32];
  const int64_t i = int64_t(blockIdx.x) * 1024 + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t v = i < n ? in[i] : 0;
  int64_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int64_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
  if (lane == 31) sw[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int64_t w = sw[lane];
    int64_t winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int64_t y = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += y; }
    sw[lane] = winc - w;
    if (lane == 31) block_sum[blockIdx.x] = winc;
  }
  __syncthreads();
  if (i < n) out[i] = sw[warp] + inc - v;
}
__global__ void __launch_bounds__(1024) k_scan_sums(int64_t* __restrict__ block_sum, int64_t nb) {  // one block
  __shared__ int64_t sw[32];
  __shared__ int64_t carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t c0 = 0; c0 < nb; c0 += 1024) {
    const int64_t i = c0 + threadIdx.x;
    const int64_t v = i < nb ? block_sum[i] : 0;
    int64_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int64_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) sw[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const int64_t w = sw[lane];
      int64_t winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int64_t y = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += y; }
      sw[lane] = winc - w;
    }
    __syncthreads();
    const int64_t ex = carry + sw[warp] + inc - v;
    if (i < nb) block_sum[i] = ex;
    __syncthreads();
    if (threadIdx.x == 1023) carry = ex + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) block_sum[nb] = carry;  // the grand total
}
__global__ void __launch_bounds__(1024) k_scan_add(int64_t* __restrict__ out, int64_t n, const int64_t* __restrict__ block_sum, int64_t nb) {
  const int64_t i = int64_t(blockIdx.x) * 1024 + threadIdx.x;
  if (i < n) out[i] += block_sum[blockIdx.x];
  if (i == 0) out[n] = block_sum[nb];
}

int evg_plan_from_finder(evg_ctx* c, const evg_runnable_in* in, const evg_task_soa* cand, const evg_distro_table* distros,
                         const evg_host_soa* hosts, const int64_t* host_off, const evg_alloc_cfg* acfg, const int64_t* dep_finished_ns,
                         int64_t now_ns, int32_t* runnable, int64_t* count) {
  if (!c || !in || !cand || !distros) return fail(EVG_ERR_INVALID, "evg_plan_from_finder: null argument");
  LOCK(c);
  const int64_t T = in->n_tasks, E = cand->n_edges;
  const int32_t D = in->n_distros, P = in->n_projects;
  if (T < 0 || D < 0 || P < 0 || E < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (cand->n_tasks != T || distros->n_distros != D) return fail(EVG_ERR_INVALID, "the candidate table, the finder table and the distro table disagree on their sizes");
  if (D == 0) return T == 0 ? evg_upload(c, cand, distros, hosts, host_off, acfg) : fail(EVG_ERR_INVALID, "tasks without distros");
  if (!count) return fail(EVG_ERR_INVALID, "null count");
  if (!in->task_off || !in->valid_off || !in->finder || !distros->task_off) return fail(EVG_ERR_INVALID, "null distro arrays");
  if (T > 0 && (!in->sched || !in->project)) return fail(EVG_ERR_INVALID, "null task column");
  if (P > 0 && !in->project_flags) return fail(EVG_ERR_INVALID, "null project_flags");
  if (in->task_off[0] != 0 || in->task_off[D] != T || in->valid_off[0] != 0) return fail(EVG_ERR_INVALID, "offsets do not span the tables");
  for (int32_t d = 0; d <= D; d++)
    if (in->task_off[d] != distros->task_off[d]) return fail(EVG_ERR_INVALID, "the finder table and the distro table cut the candidates differently at distro %d", d);
  for (int32_t d = 0; d < D; d++) {
    if (in->task_off[d + 1] < in->task_off[d] || in->valid_off[d + 1] < in->valid_off[d]) return fail(EVG_ERR_INVALID, "offsets of distro %d decrease", d);
    if (in->finder[d] > EVG_FINDER_ALTERNATE) return fail(EVG_ERR_INVALID, "distro %d: unknown finder %d", d, int(in->finder[d]));
  }
  const int64_t V = in->valid_off[D];
  if (V > 0 && !in->valid_idx) return fail(EVG_ERR_INVALID, "null valid_idx");
  if (T > 0 && (!in->deps || in->deps->n_tasks != T)) return fail(EVG_ERR_INVALID, "evg_plan_from_finder needs the candidates' dependency table (the planner's EVG_TF_DEPS_MET comes from it)");
  if (T > 0 && (!cand->priority || !cand->expected_ns || !cand->queue_basis_ns || !cand->wait_basis_ns || !cand->num_dependents ||
                !cand->task_group_order || !cand->group_id || !cand->version_id || !cand->flags))
    return fail(EVG_ERR_INVALID, "null candidate column");
  if (E > 0 && (!cand->dep_off || !cand->dep_idx)) return fail(EVG_ERR_INVALID, "null candidate dependency edges");
  if (!distros->group_off || distros->group_off[0] != 0) return fail(EVG_ERR_INVALID, "null or misplaced group_off");
  for (int32_t d = 0; d < D; d++)
    if (distros->group_off[d + 1] < distros->group_off[d]) return fail(EVG_ERR_INVALID, "group offsets of distro %d decrease", d);
  const int64_t Gc = distros->group_off[D];
  if (Gc > 0 && !distros->group_max_hosts) return fail(EVG_ERR_INVALID, "null group_max_hosts");
  // Group slots of the resident tick are the candidate groups that kept a task, in id order (include/evg_sched.h): a
  // group the finder emptied must not come back as a TaskGroupInfo, the reference builds those from the plan's tasks
  // alone (scheduler.go:60-143).  remap[group_off[d] + g] = new slot of candidate group g, -1 when it kept nothing.
  std::vector<int64_t> kgroup_off(size_t(D) + 1, 0);
  std::vector<int32_t> kgroup_max, remap(size_t(Gc), -1), host_gid;
  evg_host_soa hosts_k;
  const evg_host_soa* hosts_in = hosts;
  auto keep_groups = [&](const std::vector<uint8_t>& used) {
    for (int32_t d = 0; d < D; d++) {
      int32_t k = 0;
      for (int64_t g = distros->group_off[d]; g < distros->group_off[d + 1]; g++)
        if (used[size_t(g)]) { remap[size_t(g)] = k++; kgroup_max.push_back(distros->group_max_hosts[g]); }
      kgroup_off[size_t(d) + 1] = kgroup_off[size_t(d)] + k;
    }
    // hosts name groups by candidate slot; a host running a task of an emptied group is in no queued group
    // (groupByTaskGroup gives its bucket no TaskGroupInfo, utilization_based_host_allocator.go:223-260).  Malformed host
    // tables are left for upload_hosts to reject.
    if (!hosts || Gc == 0 || hosts->n_hosts <= 0 || !hosts->group_id || !host_off || host_off[0] != 0 || host_off[D] != hosts->n_hosts) return;
    for (int32_t d = 0; d < D; d++)
      if (host_off[d + 1] < host_off[d]) return;
    host_gid.assign(hosts->group_id, hosts->group_id + hosts->n_hosts);
    for (int32_t d = 0; d < D; d++) {
      const int64_t g0 = distros->group_off[d], ng = distros->group_off[d + 1] - g0;
      for (int64_t h = host_off[d]; h < host_off[d + 1]; h++) {
        const int32_t g = host_gid[size_t(h)];
        if (g >= 0 && g < ng) host_gid[size_t(h)] = remap[size_t(g0 + g)] >= 0 ? remap[size_t(g0 + g)] : EVG_HG_UNQUEUED;
      }
    }
    hosts_k = *hosts;
    hosts_k.group_id = host_gid.data();
    hosts_in = &hosts_k;
  };
  auto kept_table = [&]() {
    evg_distro_table dn = *distros;
    dn.group_off = kgroup_off.data();
    dn.group_max_hosts = kgroup_max.empty() ? nullptr : kgroup_max.data();
    return dn;
  };
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  CK(c->b_err.ensure(sizeof(int) * 4));
  CK(cudaMemsetAsync(c->b_err.p, 0, sizeof(int) * 4, s));
  c->launches = 0;
  c->have_tasks = false;
  if (T == 0) {
    for (int32_t d = 0; d < D; d++) count[d] = 0;
    keep_groups(std::vector<uint8_t>(size_t(Gc), 0));
    const evg_distro_table dn = kept_table();
    return evg_upload(c, cand, &dn, hosts_in, host_off, acfg);
  }
  // 1. Task.DependenciesMet / AllDependenciesSatisfied of every candidate, with the DependenciesMetTime stamps
  int rc = deps_to_device(c, in->deps, 1, dep_finished_ns, now_ns, /*want_stamp=*/true);
  if (rc != EVG_OK) return rc;
  // 2. the finders (buffers of their own: deps_to_device holds b_rn6 / b_rn7)
#define UPF(buf, ptr, cnt_, type)                                                                                  \
  do {                                                                                                             \
    CK((buf).ensure(sizeof(type) * size_t((cnt_) > 0 ? (cnt_) : 1)));                                              \
    if ((cnt_) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(cnt_), cudaMemcpyHostToDevice, s));   \
  } while (0)
  UPF(c->b_pf[0], in->task_off, D + 1, int64_t);
  UPF(c->b_pf[1], in->sched, T, uint8_t);
  UPF(c->b_pf[2], in->project, T, int32_t);
  UPF(c->b_pf[3], in->project_flags, P, uint8_t);
  UPF(c->b_pf[4], in->valid_off, D + 1, int64_t);
  UPF(c->b_pf[5], in->valid_idx, V, int32_t);
  UPF(c->b_pf[6], in->finder, D, uint8_t);
  CK(c->b_pf[7].ensure(sizeof(int32_t) * size_t(T + 1)));  // kept lists
  CK(c->b_pf[8].ensure(sizeof(int64_t) * size_t(D + 1)));  // counts
  DRunnable r;
  r.n_tasks = T; r.n_distros = D; r.n_projects = P;
  r.task_off = c->b_pf[0].as<int64_t>(); r.sched = c->b_pf[1].as<uint8_t>(); r.project = c->b_pf[2].as<int32_t>();
  r.project_flags = c->b_pf[3].as<uint8_t>(); r.valid_off = c->b_pf[4].as<int64_t>(); r.valid_idx = c->b_pf[5].as<int32_t>();
  r.finder = c->b_pf[6].as<uint8_t>(); r.met = c->b_dx7.as<uint8_t>();
  k_runnable<<<unsigned(D), 256, 0, s>>>(r, c->b_pf[7].as<int32_t>(), c->b_pf[8].as<int64_t>(), c->b_err.as<int>());
  c->launches++;
  UPF(c->b_pf[12], cand->group_id, T, int32_t);
  std::vector<uint8_t> used(size_t(Gc), 0);
  if (Gc > 0) {  // which candidate groups kept a task
    UPF(c->b_pf[36], distros->group_off, D + 1, int64_t);
    CK(c->b_pf[37].ensure(size_t(Gc)));
    CK(cudaMemsetAsync(c->b_pf[37].p, 0, size_t(Gc), s));
    k_pf_mark_groups<<<grid_for(T, 256), 256, 0, s>>>(T, D, c->b_pf[0].as<int64_t>(), c->b_pf[7].as<int32_t>(), c->b_pf[8].as<int64_t>(),
                                                      c->b_pf[12].as<int32_t>(), c->b_pf[36].as<int64_t>(), c->b_pf[37].as<uint8_t>(),
                                                      c->b_err.as<int>());
    c->launches++;
  }
  CK(cudaGetLastError());
  // 3. the only things the host needs before the planner can be routed: how many tasks each distro kept, and which groups
  int bad[2] = {0, 0};
  CK(cudaMemcpyAsync(count, c->b_pf[8].p, sizeof(int64_t) * size_t(D), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(bad, c->b_err.p, sizeof(bad), cudaMemcpyDeviceToHost, s));
  if (Gc > 0) CK(cudaMemcpyAsync(used.data(), c->b_pf[37].p, size_t(Gc), cudaMemcpyDeviceToHost, s));
  if (runnable) CK(cudaMemcpyAsync(runnable, c->b_pf[7].p, sizeof(int32_t) * size_t(T), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (bad[0]) return fail(EVG_ERR_INVALID, "a project row or dep_ref is out of range");
  if (bad[1]) return fail(EVG_ERR_INVALID, "a kept candidate's group_id is out of range for its distro");
  std::vector<int64_t> new_off(size_t(D) + 1, 0);
  for (int32_t d = 0; d < D; d++) {
    if (count[d] < 0 || count[d] > in->task_off[d + 1] - in->task_off[d]) return fail(EVG_ERR_CUDA, "finder count out of range");
    new_off[size_t(d) + 1] = new_off[size_t(d)] + count[d];
  }
  const int64_t Tn = new_off[size_t(D)];
  keep_groups(used);
  // 4. candidate columns to the device, compaction into the context's own buffers
  UPF(c->b_pf[9], cand->priority, T, int32_t);
  UPF(c->b_pf[10], cand->num_dependents, T, int32_t);
  UPF(c->b_pf[11], cand->task_group_order, T, int32_t);
  UPF(c->b_pf[13], cand->version_id, T, int32_t);
  UPF(c->b_pf[14], cand->flags, T, uint32_t);
  UPF(c->b_pf[15], cand->expected_ns, T, int64_t);
  UPF(c->b_pf[16], cand->queue_basis_ns, T, int64_t);
  UPF(c->b_pf[17], cand->wait_basis_ns, T, int64_t);
  UPF(c->b_pf[18], new_off.data(), D + 1, int64_t);
  const size_t np = size_t(Tn + kColPad);
  for (int k = 19; k <= 23; k++) { CK(c->b_pf[k].ensure(sizeof(int32_t) * np)); CK(cudaMemsetAsync(c->b_pf[k].p, 0, sizeof(int32_t) * np, s)); }
  CK(c->b_pf[24].ensure(sizeof(uint32_t) * np)); CK(cudaMemsetAsync(c->b_pf[24].p, 0, sizeof(uint32_t) * np, s));
  for (int k = 25; k <= 27; k++) { CK(c->b_pf[k].ensure(sizeof(int64_t) * np)); CK(cudaMemsetAsync(c->b_pf[k].p, 0, sizeof(int64_t) * np, s)); }
  CK(c->b_pf[28].ensure(sizeof(int32_t) * size_t(T + 1)));   // new_idx
  CK(cudaMemsetAsync(c->b_pf[28].p, 0xFF, sizeof(int32_t) * size_t(T + 1), s));
  CK(c->b_pf[29].ensure(sizeof(int64_t) * size_t(Tn + 1)));  // src_row
  PfCols pc;
  pc.priority = c->b_pf[9].as<int32_t>(); pc.numdep = c->b_pf[10].as<int32_t>(); pc.tgo = c->b_pf[11].as<int32_t>();
  pc.gid = c->b_pf[12].as<int32_t>(); pc.vid = c->b_pf[13].as<int32_t>(); pc.flags = c->b_pf[14].as<uint32_t>();
  pc.expected = c->b_pf[15].as<int64_t>(); pc.qbasis = c->b_pf[16].as<int64_t>(); pc.wbasis = c->b_pf[17].as<int64_t>();
  pc.o_priority = c->b_pf[19].as<int32_t>(); pc.o_numdep = c->b_pf[20].as<int32_t>(); pc.o_tgo = c->b_pf[21].as<int32_t>();
  pc.o_gid = c->b_pf[22].as<int32_t>(); pc.o_vid = c->b_pf[23].as<int32_t>(); pc.o_flags = c->b_pf[24].as<uint32_t>();
  pc.o_expected = c->b_pf[25].as<int64_t>(); pc.o_qbasis = c->b_pf[26].as<int64_t>(); pc.o_wbasis = c->b_pf[27].as<int64_t>();
  pc.group_off = nullptr; pc.group_remap = nullptr;
  if (Gc > 0) {
    UPF(c->b_pf[38], remap.data(), Gc, int32_t);
    pc.group_off = c->b_pf[36].as<int64_t>(); pc.group_remap = c->b_pf[38].as<int32_t>();
  }
  const int64_t* d_new_off = c->b_pf[18].as<int64_t>();
  const int64_t* d_cand_off = c->b_pf[0].as<int64_t>();
  if (Tn > 0) {
    k_pf_gather<<<grid_for(Tn, 256), 256, 0, s>>>(Tn, D, d_new_off, d_cand_off, c->b_pf[7].as<int32_t>(), pc, c->b_dx7.as<uint8_t>(),
                                                  c->b_rn7.as<int64_t>(), c->b_pf[28].as<int32_t>(), c->b_pf[29].as<int64_t>());
    c->launches++;
  }
  // 5. in-queue dependency edges between kept tasks
  int64_t En = 0;
  std::vector<int64_t> edge_off;
  if (E > 0 && Tn > 0) {
    UPF(c->b_pf[30], cand->dep_off, T + 1, int64_t);
    UPF(c->b_pf[31], cand->dep_idx, E, int32_t);
    CK(c->b_pf[32].ensure(sizeof(int32_t) * size_t(Tn + 1)));                 // surviving edges per kept task
    CK(c->b_pf[33].ensure(sizeof(int64_t) * size_t(Tn + 1 + kColPad)));       // new dep_off
    const int64_t nb = (Tn + 1023) / 1024;
    CK(c->b_pf[34].ensure(sizeof(int64_t) * size_t(nb + 1)));
    k_pf_edge_count<<<grid_for(Tn, 256), 256, 0, s>>>(Tn, D, d_new_off, d_cand_off, c->b_pf[29].as<int64_t>(), c->b_pf[30].as<int64_t>(),
                                                      c->b_pf[31].as<int32_t>(), c->b_pf[28].as<int32_t>(), c->b_pf[32].as<int32_t>());
    k_scan_blocks<<<unsigned(nb), 1024, 0, s>>>(c->b_pf[32].as<int32_t>(), Tn, c->b_pf[33].as<int64_t>(), c->b_pf[34].as<int64_t>());
    k_scan_sums<<<1, 1024, 0, s>>>(c->b_pf[34].as<int64_t>(), nb);
    k_scan_add<<<unsigned(nb), 1024, 0, s>>>(c->b_pf[33].as<int64_t>(), Tn, c->b_pf[34].as<int64_t>(), nb);
    c->launches += 4;
    CK(cudaMemcpyAsync(&En, c->b_pf[33].as<int64_t>() + Tn, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    // dep_off sampled at the distro boundaries: what the routing needs of the edges
    edge_off.resize(size_t(D) + 1);
    CK(c->b_rn0.ensure(sizeof(int64_t) * size_t(D + 1)));
    k_gather_i64<<<grid_for(D + 1, 256), 256, 0, s>>>(c->b_pf[33].as<int64_t>(), d_new_off, c->b_rn0.as<int64_t>(), D + 1);
    CK(cudaMemcpyAsync(edge_off.data(), c->b_rn0.p, sizeof(int64_t) * size_t(D + 1), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(c->b_pf[35].ensure(sizeof(int32_t) * size_t(En + 1)));
    if (En > 0) {
      k_pf_edge_write<<<grid_for(Tn, 256), 256, 0, s>>>(Tn, D, d_new_off, d_cand_off, c->b_pf[29].as<int64_t>(), c->b_pf[30].as<int64_t>(),
                                                        c->b_pf[31].as<int32_t>(), c->b_pf[28].as<int32_t>(), c->b_pf[33].as<int64_t>(),
                                                        c->b_pf[35].as<int32_t>());
      c->launches++;
    }
  }
#undef UPF
  CK(cudaGetLastError());
  // 6. the compacted table becomes the resident tick (columns stay where they are: context-owned device memory)
  evg_task_soa ts;
  memset(&ts, 0, sizeof(ts));
  ts.n_tasks = Tn; ts.n_edges = En;
  ts.priority = pc.o_priority; ts.num_dependents = pc.o_numdep; ts.task_group_order = pc.o_tgo; ts.group_id = pc.o_gid; ts.version_id = pc.o_vid;
  ts.flags = pc.o_flags; ts.expected_ns = pc.o_expected; ts.queue_basis_ns = pc.o_qbasis; ts.wait_basis_ns = pc.o_wbasis;
  if (En > 0) { ts.dep_off = c->b_pf[33].as<int64_t>(); ts.dep_idx = c->b_pf[35].as<int32_t>(); }
  evg_distro_table dn = kept_table();
  dn.task_off = new_off.data();
  rc = upload_tasks(c, &ts, &dn, /*copy_columns=*/false, /*adopt=*/true, (En > 0) ? edge_off.data() : nullptr);
  if (rc != EVG_OK) return rc;
  if (hosts) {
    rc = upload_hosts(c, hosts_in, host_off, acfg, D);
    if (rc != EVG_OK) return rc;
  }
  CK(cudaStreamSynchronize(s));
  return EVG_OK;
}

// --------------------------------------------------------------------------
// evg_intern_columns: host-side string interning (evg_intern.h)
// --------------------------------------------------------------------------
int evg_intern_columns(const evg_string_cols* in, evg_intern_out* out, int32_t threads) {
  using namespace evg_intern;
  if (!in || !out) return fail(EVG_ERR_INVALID, "evg_intern_columns: null argument");
  const int64_t T = in->n_tasks;
  const int32_t D = in->n_distros;
  if (T < 0 || D < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (!out->group_off || (D > 0 && (!in->task_off || !out->n_versions))) return fail(EVG_ERR_INVALID, "null distro arrays");
  if (D == 0) { out->group_off[0] = 0; return T == 0 ? EVG_OK : fail(EVG_ERR_INVALID, "tasks without distros"); }
  if (in->task_off[0] != 0 || in->task_off[D] != T) return fail(EVG_ERR_INVALID, "task_off does not span n_tasks");
  if (T > 0 && (!in->id.off || !in->version.off || !in->group_key.off || !in->group_max_hosts || !in->dep_off || !out->group_id ||
                !out->version_id || !out->group_max_hosts || !out->group_first || !out->dep_off))
    return fail(EVG_ERR_INVALID, "null column");
  const int64_t E = T > 0 ? in->dep_off[T] : 0;
  if (E > 0 && (!in->dep_id.off || !out->dep_idx)) return fail(EVG_ERR_INVALID, "null dependency columns");
  // per distro: groups found, surviving edges (phase 1 counts into per-distro scratch, phase 2 writes at the scanned offsets)
  std::vector<int64_t> n_groups(size_t(D), 0), n_edges(size_t(D), 0);
  std::vector<std::vector<int32_t>> grp_max_by_distro(static_cast<size_t>(D));
  std::vector<std::vector<int64_t>> grp_first_by_distro(static_cast<size_t>(D));
  std::vector<std::vector<int32_t>> edge_by_distro(static_cast<size_t>(D));
  std::atomic<int32_t> next{0};
  std::atomic<int64_t> bad_row{-1};
  int nt = threads > 0 ? threads : int(std::thread::hardware_concurrency());
  nt = std::max(1, std::min(nt, int(D)));
  auto work = [&]() {
    Table groups, versions, ids;
    for (;;) {
      const int32_t d = next.fetch_add(1);
      if (d >= D) return;
      const int64_t a = in->task_off[d], b = in->task_off[d + 1];
      if (b < a) { bad_row.store(a); return; }
      const int64_t n = b - a;
      groups.reset(n); versions.reset(n); ids.reset(n);
      int32_t ng = 0, nv = 0;
      bool ins;
      for (int64_t t = a; t < b; t++) {
        ids.get_or_put(str_at(in->id.bytes, in->id.off, t), in->id.bytes, in->id.off, t, int32_t(t - a), &ins);  // a repeated id keeps its first index
        const Str gk = str_at(in->group_key.bytes, in->group_key.off, t);
        int32_t gid = -1;
        if (gk.n > 0) {
          gid = groups.get_or_put(gk, in->group_key.bytes, in->group_key.off, t, ng, &ins);
          if (ins) { ng++; grp_max_by_distro[size_t(d)].push_back(in->group_max_hosts[t]); grp_first_by_distro[size_t(d)].push_back(t); }
          else if (grp_max_by_distro[size_t(d)][size_t(gid)] != in->group_max_hosts[t]) { int64_t none = -1; bad_row.compare_exchange_strong(none, t); }
        }
        out->group_id[t] = gid;
        const int32_t vid = versions.get_or_put(str_at(in->version.bytes, in->version.off, t), in->version.bytes, in->version.off, t, nv, &ins);
        if (ins) nv++;
        out->version_id[t] = vid;
      }
      out->n_versions[d] = nv;
      n_groups[size_t(d)] = ng;
      std::vector<int32_t>& ed = edge_by_distro[size_t(d)];
      for (int64_t t = a; t < b; t++) {
        int64_t kept = 0;
        for (int64_t e = in->dep_off[t]; e < in->dep_off[t + 1]; e++) {
          const int32_t j = ids.find(str_at(in->dep_id.bytes, in->dep_id.off, e), in->id.bytes, in->id.off);
          if (j >= 0) { ed.push_back(j); kept++; }
        }
        out->dep_off[t + 1] = kept;  // counts for now; scanned below
      }
      n_edges[size_t(d)] = int64_t(ed.size());
    }
  };
  std::vector<std::thread> pool;
  for (int k = 1; k < nt; k++) pool.emplace_back(work);
  work();
  for (std::thread& th : pool) th.join();
  if (bad_row.load() >= 0) return fail(EVG_ERR_INVALID, "task group of row %lld: TaskGroupMaxHosts differs between members (or offsets decrease)", (long long)bad_row.load());
  // offsets, then the per-distro pieces move to their places
  out->group_off[0] = 0;
  for (int32_t d = 0; d < D; d++) out->group_off[d + 1] = out->group_off[d] + n_groups[size_t(d)];
  if (T > 0) {
    out->dep_off[0] = 0;
    for (int64_t t = 0; t < T; t++) out->dep_off[t + 1] += out->dep_off[t];
  }
  for (int32_t d = 0; d < D; d++) {
    const int64_t g0 = out->group_off[d];
    for (size_t k = 0; k < grp_max_by_distro[size_t(d)].size(); k++) { out->group_max_hosts[g0 + int64_t(k)] = grp_max_by_distro[size_t(d)][k]; out->group_first[g0 + int64_t(k)] = grp_first_by_distro[size_t(d)][k]; }
    if (!edge_by_distro[size_t(d)].empty()) memcpy(out->dep_idx + out->dep_off[in->task_off[d]], edge_by_distro[size_t(d)].data(), sizeof(int32_t) * edge_by_distro[size_t(d)].size());
  }
  return EVG_OK;
}

int evg_prioritize_legacy_batch(evg_ctx* c, const evg_legacy_soa* in, const int64_t* task_off, const uint8_t* list_mode,
                                int32_t n_distros, int32_t* order, int64_t* count, int32_t* status) {
  if (!c || !in) return fail(EVG_ERR_INVALID, "evg_prioritize_legacy_batch: null argument");
  LOCK(c);
  const int64_t T = in->n_tasks;
  const int32_t D = n_distros;
  if (T < 0 || D < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (D == 0) return T == 0 ? EVG_OK : fail(EVG_ERR_INVALID, "tasks without distros");
  if (!task_off || !list_mode || !count || !status || (T > 0 && !order)) return fail(EVG_ERR_INVALID, "null argument");
  if (T > 0 && (!in->priority || !in->ingest_ns || !in->expected_ns || !in->num_dependents || !in->revision_order || !in->project_id ||
                !in->tg_rank || !in->tg_pair_id || !in->task_group_order || !in->presort_rank || !in->flags))
    return fail(EVG_ERR_INVALID, "null task column");
  if (task_off[0] != 0 || task_off[D] != T) return fail(EVG_ERR_INVALID, "task_off does not span n_tasks");
  int64_t max_n = 0;
  for (int32_t d = 0; d < D; d++) {
    if (task_off[d + 1] < task_off[d]) return fail(EVG_ERR_INVALID, "offsets of distro %d decrease", d);
    max_n = std::max(max_n, task_off[d + 1] - task_off[d]);
  }
  for (int64_t k = 0; k < 3 * int64_t(D); k++)
    if (list_mode[k] > EVG_LEGACY_MODE_LITERAL) return fail(EVG_ERR_INVALID, "unknown list mode %d", int(list_mode[k]));
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  c->launches = 0;
  c->have_tasks = false;  // shares scratch buffers with the other entry points
#define UPL(buf, ptr, count_, type)                                                                                \
  do {                                                                                                             \
    CK((buf).ensure(sizeof(type) * size_t((count_) > 0 ? (count_) : 1)));                                          \
    if ((count_) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count_), cudaMemcpyHostToDevice, s)); \
  } while (0)
  UPL(c->b_exp, in->priority, T, int64_t);
  UPL(c->b_qb, in->ingest_ns, T, int64_t);
  UPL(c->b_wb, in->expected_ns, T, int64_t);
  UPL(c->b_nd, in->num_dependents, T, int32_t);
  UPL(c->b_prio, in->revision_order, T, int32_t);
  UPL(c->b_vid, in->project_id, T, int32_t);
  UPL(c->b_gid, in->tg_rank, T, int32_t);
  UPL(c->b_rn0, in->tg_pair_id, T, int32_t);
  UPL(c->b_tgo, in->task_group_order, T, int32_t);
  UPL(c->b_rn1, in->presort_rank, T, int32_t);
  UPL(c->b_flags, in->flags, T, uint32_t);
  UPL(c->b_rn2, list_mode, 3 * int64_t(D), uint8_t);
  UPL(c->b_taskoff, task_off, D + 1, int64_t);
#undef UPL
  CK(c->b_order.ensure(sizeof(int32_t) * size_t(T + 1)));
  CK(c->b_rn3.ensure(sizeof(int32_t) * size_t(T + 1)));
  CK(c->b_rn4.ensure(sizeof(int32_t) * size_t(T + 1)));
  CK(c->b_rn5.ensure(sizeof(unsigned int) * 4 * size_t(D)));
  CK(c->b_rn6.ensure(sizeof(int64_t) * size_t(D)));
  CK(c->b_status.ensure(sizeof(int32_t) * size_t(D + 1)));
  CK(cudaMemsetAsync(c->b_rn5.p, 0, sizeof(unsigned int) * 4 * size_t(D), s));
  DLegacy x;
  x.n = T; x.priority = c->b_exp.as<int64_t>(); x.ingest = c->b_qb.as<int64_t>(); x.expected = c->b_wb.as<int64_t>();
  x.numdep = c->b_nd.as<int32_t>(); x.revision = c->b_prio.as<int32_t>(); x.project = c->b_vid.as<int32_t>();
  x.tg_rank = c->b_gid.as<int32_t>(); x.tg_pair = c->b_rn0.as<int32_t>(); x.tgo = c->b_tgo.as<int32_t>();
  x.presort = c->b_rn1.as<int32_t>(); x.flags = c->b_flags.as<uint32_t>(); x.list_mode = c->b_rn2.as<uint8_t>();
  x.task_off = c->b_taskoff.as<int64_t>(); x.n_distros = D;
  int32_t* buf[2] = {c->b_rn3.as<int32_t>(), c->b_rn4.as<int32_t>()};
  int cur = 0;
  if (T > 0) {
    LAUNCH(c, k_legacy_init, grid_for(T, 256), 256, x, buf[0], c->b_rn5.as<unsigned int>());
    for (int64_t L = 1; L < max_n; L <<= 1) {
      LAUNCH(c, k_legacy_merge_pass, grid_for(T, 256), 256, x, buf[cur], buf[cur ^ 1], L);
      cur ^= 1;
    }
    LAUNCH(c, k_legacy_interleave, grid_for(T, 256), 256, x, buf[cur], c->b_rn5.as<unsigned int>(), c->b_order.as<int32_t>(),
           c->b_rn6.as<int64_t>(), c->b_status.as<int32_t>());
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(order, c->b_order.p, sizeof(int32_t) * size_t(T), cudaMemcpyDeviceToHost, s));
  }
  // distros without tasks never reach k_legacy_interleave's q == 0 thread
  std::vector<int64_t> cnt(size_t(D), 0);
  std::vector<int32_t> st(size_t(D), EVG_LEGACY_OK);
  if (T > 0) {
    CK(cudaMemcpyAsync(cnt.data(), c->b_rn6.p, sizeof(int64_t) * size_t(D), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(st.data(), c->b_status.p, sizeof(int32_t) * size_t(D), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  for (int32_t d = 0; d < D; d++) {
    const bool empty = task_off[d + 1] == task_off[d];
    count[d] = empty ? 0 : cnt[d];
    status[d] = empty ? EVG_LEGACY_OK : st[d];
  }
  return EVG_OK;
}

int evg_dag_rebuild_batch(evg_ctx* c, const evg_dag_in* in, const int64_t* item_off, const int64_t* group_off, int32_t n_distros,
                          int32_t* sorted, int32_t* n_sorted, int32_t* n_cycles, int32_t* unit_items, int32_t* unit_off) {
  if (!c || !in) return fail(EVG_ERR_INVALID, "evg_dag_rebuild_batch: null argument");
  LOCK(c);
  const int64_t N = in->n_items, E = in->n_deps;
  const int32_t D = n_distros;
  if (N < 0 || E < 0 || D < 0) return fail(EVG_ERR_INVALID, "negative sizes");
  if (D == 0) return N == 0 ? EVG_OK : fail(EVG_ERR_INVALID, "items without distros");
  if (!item_off || !group_off || !n_sorted || !n_cycles || !unit_off || (N > 0 && (!sorted || !unit_items))) return fail(EVG_ERR_INVALID, "null argument");
  if (N > 0 && (!in->dep_off || !in->group_id || !in->group_index)) return fail(EVG_ERR_INVALID, "null item column");
  if (E > 0 && !in->dep_item) return fail(EVG_ERR_INVALID, "null dep_item");
  if (item_off[0] != 0 || item_off[D] != N || group_off[0] != 0) return fail(EVG_ERR_INVALID, "offsets do not span the tables");
  if (N > 0 && (in->dep_off[0] != 0 || in->dep_off[N] != E)) return fail(EVG_ERR_INVALID, "dep_off does not span n_deps");
  int64_t max_n = 0;
  for (int32_t d = 0; d < D; d++) {
    if (item_off[d + 1] < item_off[d] || group_off[d + 1] < group_off[d]) return fail(EVG_ERR_INVALID, "offsets of distro %d decrease", d);
    max_n = std::max(max_n, item_off[d + 1] - item_off[d]);
  }
  if (max_n >= (int64_t(1) << 31) - 1) return fail(EVG_ERR_INVALID, "a queue exceeds 2^31 items");
  // k_dag_units writes unit_off[group_off[d] + d + group_id]: every id must name one of its distro's groups
  for (int32_t d = 0; d < D; d++) {
    const int64_t ng = group_off[d + 1] - group_off[d];
    for (int64_t i = item_off[d]; i < item_off[d + 1]; i++)
      if (in->group_id[i] < -1 || in->group_id[i] >= ng)
        return fail(EVG_ERR_INVALID, "item %lld: group_id %d outside [-1, %lld) of distro %d", (long long)i, int(in->group_id[i]), (long long)ng, d);
  }
  const int64_t G = group_off[D];
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  c->launches = 0;
  c->have_tasks = false;  // shares scratch buffers with the planner's resident inputs
#define UPG(buf, ptr, count_, type)                                                                                \
  do {                                                                                                             \
    CK((buf).ensure(sizeof(type) * size_t((count_) > 0 ? (count_) : 1)));                                          \
    if ((count_) > 0) CK(cudaMemcpyAsync((buf).p, (ptr), sizeof(type) * size_t(count_), cudaMemcpyHostToDevice, s)); \
  } while (0)
  UPG(c->b_taskoff, item_off, D + 1, int64_t);
  UPG(c->b_groupoff, group_off, D + 1, int64_t);
  UPG(c->b_depoff, in->dep_off, N + 1, int64_t);
  UPG(c->b_depidx, in->dep_item, E, int32_t);
  UPG(c->b_gid, in->group_id, N, int32_t);
  UPG(c->b_tgo, in->group_index, N, int32_t);
#undef UPG
  DevBuf* scratch[] = {&c->b_prio, &c->b_nd, &c->b_vid, &c->b_flags, &c->b_rn0, &c->b_rn1, &c->b_rn2, &c->b_rn3, &c->b_rn4};
  for (DevBuf* b : scratch) CK(b->ensure(sizeof(int32_t) * size_t(N + D + 1)));
  CK(c->b_rn5.ensure(sizeof(int32_t) * size_t(E + 1)));
  CK(c->b_hasdep.ensure(size_t(N) + 16));
  CK(c->b_order.ensure(sizeof(int32_t) * size_t(N + 1)));
  CK(c->b_rn6.ensure(sizeof(int32_t) * 3 * size_t(D + 1)));
  CK(c->b_rn7.ensure(sizeof(int32_t) * size_t(G + D + 1)));
  DDag x;
  x.n = N; x.n_deps = E; x.n_distros = D;
  x.item_off = c->b_taskoff.as<int64_t>(); x.dep_off = c->b_depoff.as<int64_t>(); x.dep_item = c->b_depidx.as<int32_t>();
  x.group_id = c->b_gid.as<int32_t>(); x.group_index = c->b_tgo.as<int32_t>();
  x.succ_off = c->b_prio.as<int32_t>(); x.succ = c->b_rn5.as<int32_t>(); x.index = c->b_nd.as<int32_t>(); x.low = c->b_vid.as<int32_t>();
  x.stack = c->b_flags.as<int32_t>(); x.cs_node = c->b_rn0.as<int32_t>(); x.cs_pos = c->b_rn1.as<int32_t>(); x.emit = c->b_rn2.as<int32_t>();
  x.on_stack = c->b_hasdep.as<uint8_t>();
  int32_t* d_nsorted = c->b_rn6.as<int32_t>();
  int32_t* d_ncycles = d_nsorted + (D + 1);
  int32_t* d_grouped = d_ncycles + (D + 1);
  LAUNCH(c, k_dag_topo, grid_for(int64_t(D) * 32, 64), 64, x, c->b_order.as<int32_t>(), d_nsorted, d_ncycles);
  std::vector<int32_t> grouped(size_t(D), 0);
  int32_t* buf[2] = {c->b_rn3.as<int32_t>(), c->b_rn4.as<int32_t>()};
  int cur = 0;
  if (N > 0) {
    CK(cudaMemcpyAsync(sorted, c->b_order.p, sizeof(int32_t) * size_t(N), cudaMemcpyDeviceToHost, s));
    // every item has a group or not: "no ungrouped item" leaves grouped[d] at the distro's length
    for (int32_t d = 0; d < D; d++) grouped[size_t(d)] = int32_t(item_off[d + 1] - item_off[d]);
    CK(cudaMemcpyAsync(d_grouped, grouped.data(), sizeof(int32_t) * size_t(D), cudaMemcpyHostToDevice, s));
    LAUNCH(c, k_dag_group_init, grid_for(N, 256), 256, x, buf[0]);
    for (int64_t L = 1; L < max_n; L <<= 1) {
      LAUNCH(c, k_dag_group_pass, grid_for(N, 256), 256, x, buf[cur], buf[cur ^ 1], L);
      cur ^= 1;
    }
    CK(cudaMemsetAsync(c->b_rn7.p, 0xFF, sizeof(int32_t) * size_t(G + D), s));  // -1: a group no item is in
    LAUNCH(c, k_dag_units, grid_for(N, 256), 256, x, buf[cur], c->b_groupoff.as<int64_t>(), c->b_rn7.as<int32_t>(), d_grouped);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(unit_items, buf[cur], sizeof(int32_t) * size_t(N), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(unit_off, c->b_rn7.p, sizeof(int32_t) * size_t(G + D), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(grouped.data(), d_grouped, sizeof(int32_t) * size_t(D), cudaMemcpyDeviceToHost, s));
  }
  CK(cudaMemcpyAsync(n_sorted, d_nsorted, sizeof(int32_t) * size_t(D), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(n_cycles, d_ncycles, sizeof(int32_t) * size_t(D), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (N == 0) std::fill(unit_off, unit_off + (G + D), -1);
  for (int32_t d = 0; d < D; d++) {
    int32_t* u = unit_off + group_off[d] + d;
    const int64_t ng = group_off[d + 1] - group_off[d];
    u[ng] = grouped[size_t(d)];  // the closing entry of each distro
    // a group without items is the empty range that starts where the next group starts
    for (int64_t g = ng - 1; g >= 0; g--)
      if (u[g] < 0) u[g] = u[g + 1];
  }
  return EVG_OK;
}

int evg_plan_distro(evg_ctx* c, const evg_task_soa* tasks, const evg_distro_cfg* cfg, int32_t n_groups,
                    const int32_t* group_max_hosts, int64_t now_ns, uint32_t opts, evg_plan_out* out) {
  if (!tasks || !cfg) return fail(EVG_ERR_INVALID, "evg_plan_distro: null argument");
  int64_t task_off[2] = {0, tasks->n_tasks};
  int64_t group_off[2] = {0, n_groups};
  evg_distro_table dt;
  dt.n_distros = 1; dt._reserved = 0; dt.task_off = task_off; dt.group_off = group_off; dt.cfg = cfg;
  dt.group_max_hosts = group_max_hosts;
  return evg_plan_batch(c, tasks, &dt, now_ns, opts, out);
}

int evg_alloc_distro(evg_ctx* c, const evg_host_soa* hosts, const evg_alloc_cfg* cfg, const evg_queue_info* info,
                     evg_group_info* groups, int32_t n_groups, int64_t now_ns, evg_alloc_result* result, int32_t* status) {
  if (!hosts || !cfg || !info) return fail(EVG_ERR_INVALID, "evg_alloc_distro: null argument");
  int64_t host_off[2] = {0, hosts->n_hosts};
  int64_t group_off[2] = {0, n_groups};
  evg_alloc_out ao;
  ao.result = result; ao.status = status;
  return evg_alloc_batch(c, hosts, host_off, cfg, info, groups, group_off, 1, now_ns, &ao);
}

void* evg_host_alloc(uint64_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    g_err = "cudaHostAlloc failed";
    return nullptr;
  }
  return p;
}
void evg_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"

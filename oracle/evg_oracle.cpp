// evg_oracle.cpp -- CPU ORACLE (test infrastructure, NOT product code).
// See evg_oracle.h for the contract and the parity status.  This is a
// restatement of the reference algorithm (string-keyed maps, Go time/Duration
// semantics, FP64 intermediates), written from the behaviour of the cited
// reference lines; it shares no code with the CUDA product path.
#include "evg_oracle.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace {

constexpr int64_t kSecond = 1000000000LL;
constexpr int64_t kMinute = 60 * kSecond;
constexpr int64_t kHour = 60 * kMinute;
constexpr int64_t kMaxDurationPerDistroHost = 30 * kMinute;               // globals.go:267
constexpr int64_t kMaxDurationPerDistroHostWithContainers = 2 * kMinute;  // globals.go:268
constexpr int64_t kDefaultTaskDuration = 10 * kMinute;                    // model/task/task.go:64
constexpr int64_t kPredictionTTL = 8 * kHour;                             // model/task/task.go:67

inline std::string_view sv(const evo_strcol& c, int64_t i) {
  if (!c.buf || !c.off) return std::string_view();
  return std::string_view(c.buf + c.off[i], size_t(c.off[i + 1] - c.off[i]));
}

// Go: time.Duration arithmetic wraps (two's complement); do it unsigned.
inline int64_t wadd(int64_t a, int64_t b) { return int64_t(uint64_t(a) + uint64_t(b)); }
inline int64_t wmul(int64_t a, int64_t b) { return int64_t(uint64_t(a) * uint64_t(b)); }

// Go time.Time.Sub / time.Since: saturating (time/time.go Sub).
inline int64_t since(int64_t now, int64_t t) {
  if (t == EVO_TIME_ZERO) return INT64_MAX;  // now - year 1 overflows -> maxDuration
  __int128 d = (__int128)now - (__int128)t;
  if (d > INT64_MAX) return INT64_MAX;
  if (d < INT64_MIN) return INT64_MIN;
  return int64_t(d);
}
inline bool go_is_zero(int64_t t) { return t == EVO_TIME_ZERO; }               // time.Time.IsZero
inline bool util_is_zero_time(int64_t t) { return t == EVO_TIME_ZERO || t == 0; }  // utility.IsZeroTime
// time.Time.After with the year-1 sentinel ordered before everything.
inline bool after(int64_t a, int64_t b) {
  if (a == EVO_TIME_ZERO) return false;
  if (b == EVO_TIME_ZERO) return true;
  return a > b;
}

// time.Duration.Minutes()/Hours() (Go stdlib time/time.go).
inline double dur_minutes(int64_t d) { return double(d / kMinute) + double(d % kMinute) / (60.0 * 1e9); }
inline double dur_hours(int64_t d) { return double(d / kHour) + double(d % kHour) / (60.0 * 60.0 * 1e9); }

// model/distro/distro.go:353-408 factor getters: <= 0 -> 1.
inline int64_t F(int64_t x) { return x <= 0 ? 1 : x; }
inline double Fd(double x) { return x <= 0 ? 1.0 : x; }

// globals.go:1179-1197
inline bool is_merge_queue(std::string_view r) { return r == "github_merge_request"; }
inline bool is_patch(std::string_view r) {
  return r == "patch_request" || r == "github_pull_request" || r == "github_merge_request";
}

struct View {
  const evo_tasks* t;
  int64_t base, n;
  int64_t g(int64_t i) const { return base + i; }
};

std::string task_group_string(const View& v, int64_t i) {  // model/task/task.go:417-419
  std::string s;
  s.append(sv(v.t->task_group, v.g(i))).append("_").append(sv(v.t->build_variant, v.g(i)));
  s.append("_").append(sv(v.t->project, v.g(i))).append("_").append(sv(v.t->version, v.g(i)));
  return s;
}

// ---- Unit.info + unitInfo.value: scheduler/planner.go:209-337 ----
void unit_value(const View& v, const std::vector<int64_t>& members, const evo_planner_settings& s,
                int64_t now, int64_t bd[EVO_BD_N]) {
  const evo_tasks& t = *v.t;
  bool mq = false, pat = false, nongroup = false, gen = false, stepback = false;
  int64_t tiq = 0, max_prio = 0, runtime = 0, max_deps = 0;
  for (int64_t m : members) {
    int64_t i = v.g(m);
    std::string_view req = sv(t.requester, i);
    if (is_merge_queue(req)) mq = true;            // planner.go:308
    else if (is_patch(req)) pat = true;            // planner.go:310
    nongroup = nongroup || sv(t.task_group, i).empty();
    gen = gen || (t.generate_task && t.generate_task[i]);
    stepback = stepback || sv(t.activated_by, i) == "stepback";  // globals.go:219
    if (!go_is_zero(t.activated_time[i])) tiq = wadd(tiq, since(now, t.activated_time[i]));
    else if (!go_is_zero(t.ingest_time[i])) tiq = wadd(tiq, since(now, t.ingest_time[i]));
    if (t.priority[i] > max_prio) max_prio = t.priority[i];
    runtime = wadd(runtime, t.expected_ns[i]);
    if (int64_t(t.num_dependents[i]) > max_deps) max_deps = t.num_dependents[i];
  }
  for (int k = 0; k < EVO_BD_N; k++) bd[k] = 0;
  const int64_t len = int64_t(members.size());
  bd[EVO_BD_TASK_GROUP_LENGTH] = len;
  // computePriority planner.go:271-300
  int64_t prio = wadd(1, max_prio);
  bd[EVO_BD_P_INITIAL] = prio;
  if (!nongroup) {
    bd[EVO_BD_P_TASK_GROUP] = len;
    prio = wadd(prio, len);
  }
  if (gen) {
    int64_t prev = prio;
    prio = wmul(prio, F(s.generate_task_factor));
    bd[EVO_BD_P_GENERATOR] = wadd(prio, -prev);
    if (!nongroup) {
      bd[EVO_BD_P_TASK_GROUP] = wmul(bd[EVO_BD_P_TASK_GROUP], F(s.generate_task_factor));
      bd[EVO_BD_P_GENERATOR] = wadd(bd[EVO_BD_P_GENERATOR], -wmul(len, F(s.generate_task_factor)));
    }
  }
  if (mq) {
    bd[EVO_BD_P_COMMIT_QUEUE] = 200;
    prio = wadd(prio, 200);
  }
  // computeRankValue planner.go:223-265
  if (pat) {
    bd[EVO_BD_R_PATCH] = F(s.patch_factor);
    bd[EVO_BD_R_PATCH_WAIT] =
        wmul(F(s.patch_time_in_queue_factor), int64_t(std::floor(dur_minutes(tiq) / double(len))));
  } else if (mq) {
    bd[EVO_BD_R_COMMIT_QUEUE] = F(s.commit_queue_factor);
  } else {
    int64_t avg = tiq / len;
    if (avg < 7 * 24 * kHour)
      bd[EVO_BD_R_MAINLINE_WAIT] =
          wmul(F(s.mainline_time_in_queue_factor), int64_t(dur_hours(7 * 24 * kHour - avg)));
    if (stepback) bd[EVO_BD_R_STEPBACK] = F(s.stepback_task_factor);
  }
  bd[EVO_BD_R_NUM_DEPENDENTS] = int64_t(Fd(s.num_dependents_factor) * double(max_deps));
  bd[EVO_BD_R_ESTIMATED_RUNTIME] =
      wmul(F(s.expected_runtime_factor), int64_t(std::floor(dur_minutes(runtime) / double(len))));
  int64_t rank = 1;
  rank = wadd(rank, bd[EVO_BD_R_PATCH]);
  rank = wadd(rank, bd[EVO_BD_R_PATCH_WAIT]);
  rank = wadd(rank, bd[EVO_BD_R_MAINLINE_WAIT]);
  rank = wadd(rank, bd[EVO_BD_R_COMMIT_QUEUE]);
  rank = wadd(rank, bd[EVO_BD_R_STEPBACK]);
  rank = wadd(rank, bd[EVO_BD_R_NUM_DEPENDENTS]);
  rank = wadd(rank, bd[EVO_BD_R_ESTIMATED_RUNTIME]);
  bd[EVO_BD_TOTAL_VALUE] = wadd(wmul(prio, rank), len);  // planner.go:215
}

// ---- UnitCache / PrepareTasksForPlanning: scheduler/planner.go:23-89,431-459 ----
struct Unit {
  std::map<std::string, int64_t> tasks;  // Unit.tasks keyed by task id (planner.go:131)
  bool has_distro = false;
  int64_t anchor = INT64_MAX;  // smallest input index of a task that SetDistro'd this unit (canonical tie-break)
};
using UnitPtr = std::shared_ptr<Unit>;
struct UnitCache {
  std::unordered_map<std::string, UnitPtr> m;
  std::vector<std::string> key_order;  // deterministic iteration (Go's is random; order is unobservable after canonical sort)
  UnitPtr create(const std::string& key, const std::string& id, int64_t idx) {  // planner.go:61-70
    auto it = m.find(key);
    if (it != m.end()) { it->second->tasks[id] = idx; return it->second; }
    auto u = std::make_shared<Unit>();
    u->tasks[id] = idx;
    m.emplace(key, u);
    key_order.push_back(key);
    return u;
  }
  void add_new(const std::string& key, const UnitPtr& unit) {  // planner.go:42-52
    auto it = m.find(key);
    if (it != m.end()) {
      if (it->second != unit) for (auto& kv : unit->tasks) it->second->tasks[kv.first] = kv.second;
      return;
    }
    m.emplace(key, unit);
    key_order.push_back(key);
  }
  void add_when(bool cond, const std::string& key, const std::string& id, int64_t idx) {  // planner.go:26-37
    if (!cond) return;
    create(key, id, idx);
  }
};

struct PlannedUnit {
  std::vector<int64_t> members;  // sorted ascending input index
  int64_t bd[EVO_BD_N];
  int64_t min_member, anchor;
};

struct PlanResult {
  std::vector<int64_t> order;
  std::vector<int64_t> unit_of_rank;  // index into units for each emitted task
  std::vector<PlannedUnit> units;
};

PlanResult plan(const View& v, const evo_planner_settings& s, int64_t now) {
  const evo_tasks& t = *v.t;
  UnitCache cache;
  std::vector<std::string> ids(v.n);
  for (int64_t i = 0; i < v.n; i++) ids[i] = std::string(sv(t.id, v.g(i)));
  // pass 1 planner.go:434-447
  for (int64_t i = 0; i < v.n; i++) {
    UnitPtr unit;
    std::string version(sv(t.version, v.g(i)));
    if (!sv(t.task_group, v.g(i)).empty()) {
      unit = cache.create(task_group_string(v, i), ids[i], i);
      cache.add_new(ids[i], unit);
      cache.add_when(s.group_versions != 0, version, ids[i], i);
    } else if (s.group_versions) {
      unit = cache.create(version, ids[i], i);
      cache.add_new(ids[i], unit);
    } else {
      unit = cache.create(ids[i], ids[i], i);
    }
    unit->has_distro = true;
    unit->anchor = std::min(unit->anchor, i);
  }
  // pass 2 planner.go:449-456
  for (int64_t i = 0; i < v.n; i++) {
    for (int64_t e = t.dep_off ? t.dep_off[v.g(i)] : 0; t.dep_off && e < t.dep_off[v.g(i) + 1]; e++) {
      std::string dep(sv(t.dep_task_id, e));
      auto it = cache.m.find(dep);
      if (it != cache.m.end()) it->second->tasks[ids[i]] = i;
    }
  }
  // Export planner.go:73-89: distinct units (by sorted member ids) with a distro.
  PlanResult r;
  std::map<std::vector<int64_t>, size_t> seen;  // member-index set -> slot (ids are unique => same identity as Unit.ID)
  std::unordered_set<Unit*> visited;
  for (auto& key : cache.key_order) {
    UnitPtr u = cache.m[key];
    if (!visited.insert(u.get()).second) continue;
    if (!u->has_distro) continue;
    std::vector<int64_t> mem;
    mem.reserve(u->tasks.size());
    for (auto& kv : u->tasks) mem.push_back(kv.second);
    std::sort(mem.begin(), mem.end());
    auto it = seen.find(mem);
    if (it != seen.end()) {  // duplicate member set: keep the smaller anchor (canonical)
      r.units[it->second].anchor = std::min(r.units[it->second].anchor, u->anchor);
      continue;
    }
    PlannedUnit pu;
    pu.members = mem;
    pu.min_member = mem.front();
    pu.anchor = u->anchor;
    unit_value(v, mem, s, now, pu.bd);
    seen.emplace(mem, r.units.size());
    r.units.push_back(std::move(pu));
  }
  // TaskPlan.Export planner.go:462-481 with the canonical tie policy:
  // units: TotalValue desc, then anchor asc (anchor = smallest input index among the
  // tasks that SetDistro'd the unit; every task anchors exactly one unit, so this is total).
  std::vector<size_t> uo(r.units.size());
  for (size_t k = 0; k < uo.size(); k++) uo[k] = k;
  std::sort(uo.begin(), uo.end(), [&](size_t a, size_t b) {
    const PlannedUnit &A = r.units[a], &B = r.units[b];
    if (A.bd[EVO_BD_TOTAL_VALUE] != B.bd[EVO_BD_TOTAL_VALUE])
      return A.bd[EVO_BD_TOTAL_VALUE] > B.bd[EVO_BD_TOTAL_VALUE];
    return A.anchor < B.anchor;
  });
  std::vector<uint8_t> emitted(v.n, 0);
  for (size_t k : uo) {
    std::vector<int64_t> mem = r.units[k].members;
    // TaskList.Less planner.go:387-405, ties by input index.
    std::sort(mem.begin(), mem.end(), [&](int64_t a, int64_t b) {
      int64_t ga = v.g(a), gb = v.g(b);
      if (t.task_group_order[ga] != t.task_group_order[gb]) return t.task_group_order[ga] < t.task_group_order[gb];
      if (t.num_dependents[ga] != t.num_dependents[gb]) return t.num_dependents[ga] > t.num_dependents[gb];
      if (t.priority[ga] != t.priority[gb]) return t.priority[ga] > t.priority[gb];
      if (t.expected_ns[ga] != t.expected_ns[gb]) return t.expected_ns[ga] > t.expected_ns[gb];
      return a < b;
    });
    for (int64_t m : mem) {
      if (emitted[m]) continue;  // seen.Visit planner.go:472
      emitted[m] = 1;
      r.order.push_back(m);
      r.unit_of_rank.push_back(int64_t(k));
    }
  }
  return r;
}

// ---- Task.DependenciesMet: model/task/task.go:529-543,632-671,3393-3395 ----
// bit 0: Task.DependenciesMet; bit 1: the dependencies were evaluated afresh (no HasDependenciesMet short-circuit),
// which is when the reference also runs setDependenciesMetTime on the task (task.go:653).
std::vector<uint8_t> deps_met(const View& v) {
  const evo_tasks& t = *v.t;
  std::unordered_map<std::string_view, int64_t> cache;  // depCache scheduler.go:61-64
  for (int64_t i = 0; i < v.n; i++) cache[sv(t.id, v.g(i))] = i;
  std::vector<uint8_t> met(v.n, 0);
  for (int64_t i = 0; i < v.n; i++) {
    int64_t gi = v.g(i);
    int64_t e0 = t.dep_off ? t.dep_off[gi] : 0, e1 = t.dep_off ? t.dep_off[gi + 1] : 0;
    if (e1 == e0 || (t.override_dependencies && t.override_dependencies[gi]) ||
        !util_is_zero_time(t.dependencies_met_time[gi])) {  // HasDependenciesMet task.go:3393: nothing is stamped
      met[i] = 1;
      continue;
    }
    bool ok = true;
    for (int64_t e = e0; e < e1 && ok; e++) {
      std::string_view dep_id = sv(t.dep_task_id, e);
      std::string_view dep_status, want = sv(t.dep_status, e);
      for (int64_t f = e0; f < e; f++)  // SatisfiesDependency reads the FIRST Dependency naming the task (task.go:529-543)
        if (sv(t.dep_task_id, f) == dep_id) { want = sv(t.dep_status, f); break; }
      bool dep_blocked = false;
      auto it = cache.find(dep_id);
      if (it != cache.end()) {
        dep_status = sv(t.status, v.g(it->second));
        dep_blocked = t.blocked && t.blocked[v.g(it->second)];
      } else if (t.dep_found && t.dep_found[e]) {
        dep_status = sv(t.dep_task_status, e);
        dep_blocked = t.dep_task_blocked && t.dep_task_blocked[e];
      } else {
        ok = false;  // lookup error -> checkDependenciesMet returns false (scheduler.go:161-168)
        break;
      }
      // SatisfiesDependency task.go:529-543
      if (want == "success" || want.empty()) ok = dep_status == "success";
      else if (want == "failed") ok = dep_status == "failed";
      else if (want == "*") ok = dep_status == "failed" || dep_status == "success" || dep_blocked;
      else ok = false;
    }
    met[i] = ok ? 3 : 0;
  }
  return met;
}

// Task.setDependenciesMetTime (model/task/task.go:673-684): the latest non-zero FinishedAt of the dependencies, else now.
int64_t fresh_dependencies_met_time(const View& v, int64_t i, int64_t now) {
  const evo_tasks& t = *v.t;
  const int64_t gi = v.g(i);
  int64_t best = EVO_TIME_ZERO;  // utility.ZeroTime
  if (t.dep_off && t.dep_finished_at)
    for (int64_t e = t.dep_off[gi]; e < t.dep_off[gi + 1]; e++) {
      const int64_t f = t.dep_finished_at[e];
      if (!util_is_zero_time(f) && after(f, best)) best = f;
    }
  return util_is_zero_time(best) ? now : best;
}

int64_t target_time(const evo_planner_settings& s) {  // model/distro/distro.go:422-440
  if (s.target_time_ns != 0) return s.target_time_ns;
  return s.has_container_pool ? kMaxDurationPerDistroHostWithContainers : kMaxDurationPerDistroHost;
}

// ---- GetDistroQueueInfo: scheduler/scheduler.go:56-159 ----
struct QueueInfo {
  evo_queue_info info;
  std::vector<evo_group_info> groups;
  std::vector<std::string> names;
};

QueueInfo queue_info(const View& v, const int64_t* order, int64_t n_order, std::string_view distro_id,
                     int64_t threshold, bool includes_deps, int64_t now) {
  const evo_tasks& t = *v.t;
  std::vector<uint8_t> met = deps_met(v);
  QueueInfo q;
  std::memset(&q.info, 0, sizeof(q.info));
  std::unordered_map<std::string, size_t> gmap;
  for (int64_t r = 0; r < n_order; r++) {
    int64_t i = order[r], gi = v.g(i);
    std::string name;
    if (!sv(t.task_group, gi).empty()) name = task_group_string(v, i);
    int64_t duration = t.expected_ns[gi];
    if (sv(t.distro_id, gi) != distro_id) q.info.secondary_queue = 1;
    bool dm = (met[i] & 1) != 0;
    bool counted = !includes_deps || dm;
    auto it = gmap.find(name);
    size_t gidx;
    if (it == gmap.end()) {
      evo_group_info g;
      std::memset(&g, 0, sizeof(g));
      g.name_task = name.empty() ? -1 : i;
      g.max_hosts = t.task_group_max_hosts[gi];
      gidx = q.groups.size();
      q.groups.push_back(g);
      q.names.push_back(name);
      gmap.emplace(name, gidx);
    } else {
      gidx = it->second;
    }
    evo_group_info& g = q.groups[gidx];
    if (counted) { g.count++; g.expected_duration = wadd(g.expected_duration, duration); }
    if (dm) {
      q.info.length_with_dependencies_met++;
      if (is_merge_queue(sv(t.requester, gi))) {
        q.info.count_dep_filled_merge_queue_tasks++;
        g.count_dep_filled_merge_queue_tasks++;
      }
    }
    if (counted) {
      q.info.expected_duration = wadd(q.info.expected_duration, duration);
      if (duration > threshold) {
        g.count_duration_over_threshold++;
        g.duration_over_threshold = wadd(g.duration_over_threshold, duration);
        q.info.count_duration_over_threshold++;
        q.info.duration_over_threshold = wadd(q.info.duration_over_threshold, duration);
      }
      if (dm) {
        // checkDependenciesMet ran on the loop's copy of the task first (scheduler.go:82-98): a fresh evaluation has
        // already stamped DependenciesMetTime on it (task.go:653) when the wait is measured (scheduler.go:119-123)
        const int64_t met_time = (met[i] & 2) ? fresh_dependencies_met_time(v, i, now) : t.dependencies_met_time[gi];
        int64_t start = t.scheduled_time[gi];
        if (after(met_time, start)) start = met_time;
        int64_t wait = since(now, start);
        if (wait > threshold) { g.count_wait_over_threshold++; q.info.count_wait_over_threshold++; }
      }
    }
  }
  q.info.length = n_order;
  q.info.max_duration_threshold = threshold;
  q.info.n_groups = int64_t(q.groups.size());
  return q;
}

// ---- allocator: scheduler/utilization_based_host_allocator.go ----
struct HView {
  const evo_hosts* h;
  int64_t base, n;
  int64_t g(int64_t i) const { return base + i; }
};

bool host_is_free(const HView& hv, int64_t i) {  // model/host/host.go:214-221
  return sv(hv.h->running_task, hv.g(i)).empty() && go_is_zero(hv.h->teardown_start_time[hv.g(i)]);
}
std::string host_group_name(const HView& hv, int64_t i) {  // allocator.go:226-229, host.go:663-665
  const evo_hosts& h = *hv.h;
  int64_t gi = hv.g(i);
  if (sv(h.running_task, gi).empty() || sv(h.running_task_group, gi).empty()) return std::string();
  std::string s;
  s.append(sv(h.running_task_group, gi)).append("_").append(sv(h.running_task_bv, gi)).append("_");
  s.append(sv(h.running_task_project, gi)).append("_").append(sv(h.running_task_version, gi));
  return s;
}

int64_t calc_new_hosts_needed(int64_t short_ns, int64_t threshold, int64_t exp_free, int64_t n_long,
                              int64_t n_overdue, int64_t n_mq, bool round_down) {  // :268-296
  double turn = double(short_ns) / double(threshold);
  double x = turn - double(exp_free) + double(n_long) + double(n_overdue) + double(n_mq);
  if (exp_free < 1 && x > 0 && x < 1) return 1;
  int64_t n = round_down ? int64_t(std::floor(x)) : int64_t(std::ceil(x));
  return n < 0 ? 0 : n;
}

// getSoonToBeFreeHosts :324-394, canonical FP64 summation order = host order.
double soon_to_be_free(const HView& hv, const std::vector<int64_t>& hosts, double frac, int64_t threshold, int64_t now) {
  const evo_hosts& h = *hv.h;
  double sum = 0.0;
  for (int64_t i : hosts) {
    int64_t gi = hv.g(i);
    if (sv(h.running_task, gi).empty()) continue;
    if (!(h.rt_found && h.rt_found[gi])) continue;  // task.Find returned no document for it
    int64_t expected = h.rt_expected_ns[gi], stddev = h.rt_std_ns[gi];
    int64_t elapsed = since(now, h.rt_start_time[gi]);
    int64_t left = wadd(expected, -elapsed);
    double f;
    if (elapsed > kMaxDurationPerDistroHost && stddev > 0 && elapsed > wadd(expected, wmul(3, stddev))) f = 0;
    else f = double(wadd(threshold, -left)) / double(threshold);
    if (f < 0) f = 0;
    if (f > 1) f = 1;
    sum += frac * f;
  }
  return sum;
}

int32_t calc_existing_free_hosts(const HView& hv, const std::vector<int64_t>& hosts, double frac,
                                 int64_t threshold, int64_t now, int64_t* out) {  // :300-318
  *out = 0;
  if (frac > 1) return EVO_ERR_FUTURE_FRACTION;
  int64_t n_free = 0;
  for (int64_t i : hosts) if (host_is_free(hv, i)) n_free++;
  *out = n_free + int64_t(std::floor(soon_to_be_free(hv, hosts, frac, threshold, now)));
  return EVO_OK;
}

bool is_max_hosts_capacity(int64_t max_hosts, bool pool, int64_t pool_max, int64_t n_new, int64_t n_existing) {  // :397-409
  if (pool && n_new > max_hosts * pool_max - n_existing) return true;
  return n_new + n_existing > max_hosts;
}

bool is_ephemeral(const char* provider) {  // globals.go:723-728, distro.go:478-480
  std::string_view p(provider ? provider : "");
  return p == "ec2-ondemand" || p == "ec2-fleet" || p == "mock" || p == "docker";
}

int32_t eval_host_utilization(const HView& hv, const evo_alloc_settings& a, const std::vector<int64_t>& hosts,
                              const evo_group_info& info, int64_t threshold, int64_t max_hosts, int64_t now,
                              int64_t* out_new, int64_t* out_free) {  // :135-220
  *out_new = 0; *out_free = 0;
  if (!is_ephemeral(a.provider)) return EVO_OK;
  if (a.has_pool) {
    if (!a.parent_found) return EVO_ERR_PARENT_MISSING;
    max_hosts = int64_t(a.parent_maximum_hosts) * a.pool_max_containers;
  }
  int64_t exp_free = 0;
  int32_t st = calc_existing_free_hosts(hv, hosts, a.future_host_fraction, threshold, now, &exp_free);
  if (st != EVO_OK) { *out_free = exp_free; return st; }
  bool round_down = std::string_view(a.rounding_rule ? a.rounding_rule : "") != "round-up";
  int64_t overdue = std::string_view(a.feedback_rule ? a.feedback_rule : "") == "waits-over-thresh-feedback"
                        ? info.count_wait_over_threshold : 0;
  int64_t short_ns = wadd(info.expected_duration, -info.duration_over_threshold);
  int64_t n = calc_new_hosts_needed(short_ns, threshold, exp_free, info.count_duration_over_threshold, overdue,
                                    info.count_dep_filled_merge_queue_tasks, round_down);
  if (n > info.count) n = info.count;
  if (is_max_hosts_capacity(max_hosts, a.has_pool != 0, a.pool_max_containers, n, int64_t(hosts.size())))
    n = max_hosts - int64_t(hosts.size());
  if (n < 0) n = 0;
  if (max_hosts < 1) return EVO_ERR_POOL_SIZE;
  *out_new = n; *out_free = exp_free;
  return EVO_OK;
}

int32_t allocate(const HView& hv, const evo_alloc_settings& a, const evo_queue_info& info, evo_group_info* groups,
                 const std::vector<std::string>& names, int64_t now, int64_t* out_new, int64_t* out_free) {  // :26-130
  const int64_t n_existing = hv.n;
  int64_t n_free = 0;
  for (int64_t i = 0; i < hv.n; i++) if (host_is_free(hv, i)) n_free++;
  *out_new = 0; *out_free = n_free;
  if (std::string_view(a.provider ? a.provider : "") != "docker" && n_existing >= a.maximum_hosts) return EVO_OK;
  if (a.disabled) {
    int64_t need = a.minimum_hosts - n_existing;
    *out_new = need > 0 ? need : 0;
    return EVO_OK;
  }
  // groupByTaskGroup :223-260
  struct Data { std::vector<int64_t> hosts; int64_t info = -1; };
  std::map<std::string, Data> datas;
  for (int64_t i = 0; i < hv.n; i++) datas[host_group_name(hv, i)].hosts.push_back(i);
  std::map<std::string, int64_t> info_by_name;  // later duplicates overwrite, like the Go map
  for (size_t g = 0; g < names.size(); g++) info_by_name[names[g]] = int64_t(g);
  for (auto& kv : info_by_name) datas[kv.first].info = kv.second;
  int64_t required = 0, free_approx = 0;
  evo_group_info empty;
  std::memset(&empty, 0, sizeof(empty));
  for (auto& kv : datas) {
    const std::string& name = kv.first;
    const evo_group_info& gi = kv.second.info >= 0 ? groups[kv.second.info] : empty;
    int64_t max_hosts;
    if (name.empty()) max_hosts = a.maximum_hosts;
    else {
      if (gi.count == 0) continue;
      max_hosts = gi.max_hosts;
    }
    int64_t n = 0, f = 0;
    int32_t st = eval_host_utilization(hv, a, kv.second.hosts, gi, info.max_duration_threshold, max_hosts, now, &n, &f);
    if (st != EVO_OK) { *out_new = 0; *out_free = n_free; return st; }
    required += n;
    free_approx += f;
    if (!name.empty()) {
      groups[info_by_name[name]].count_free = f;
      groups[info_by_name[name]].count_required = n;
    }
  }
  if (required + n_free > info.length_with_dependencies_met) required = info.length_with_dependencies_met - n_free;
  if (required < 0) required = 0;
  int64_t topup = 0;
  if (n_existing + required < a.minimum_hosts) topup = a.minimum_hosts - (n_existing + required);
  *out_new = required + topup;
  *out_free = free_approx;
  return EVO_OK;
}

}  // namespace

extern "C" {

void evo_unit_value(const evo_tasks* t, const int64_t* members, int64_t n_members,
                    const evo_planner_settings* s, int64_t now, int64_t out_bd[EVO_BD_N]) {
  View v{t, 0, t->n};
  std::vector<int64_t> m(members, members + n_members);
  unit_value(v, m, *s, now, out_bd);
}

int64_t evo_plan(const evo_tasks* t, const evo_planner_settings* s, int64_t now, int64_t* out_order,
                 int64_t* out_bd, int64_t* out_n_units) {
  View v{t, 0, t->n};
  PlanResult r = plan(v, *s, now);
  for (size_t k = 0; k < r.order.size(); k++) {
    out_order[k] = r.order[k];
    if (out_bd) std::memcpy(out_bd + k * EVO_BD_N, r.units[r.unit_of_rank[k]].bd, sizeof(int64_t) * EVO_BD_N);
  }
  if (out_n_units) *out_n_units = int64_t(r.units.size());
  return int64_t(r.order.size());
}

void evo_deps_met(const evo_tasks* t, uint8_t* out_met) {
  View v{t, 0, t->n};
  std::vector<uint8_t> m = deps_met(v);
  for (size_t k = 0; k < m.size(); k++) out_met[k] = m[k] & 1;
}

int64_t evo_get_distro_queue_info(const evo_tasks* t, const int64_t* order, int64_t n_order, const char* distro_id,
                       int64_t threshold_ns, int32_t includes_dependencies, int64_t now,
                       evo_queue_info* out_info, evo_group_info* out_groups) {
  View v{t, 0, t->n};
  QueueInfo q = queue_info(v, order, n_order, distro_id ? distro_id : "", threshold_ns, includes_dependencies != 0, now);
  *out_info = q.info;
  for (size_t g = 0; g < q.groups.size(); g++) out_groups[g] = q.groups[g];
  return int64_t(q.groups.size());
}

int64_t evo_target_time(const evo_planner_settings* s) { return target_time(*s); }

int64_t evo_calc_new_hosts_needed(int64_t short_ns, int64_t threshold_ns, int64_t expected_free, int64_t n_long,
                                  int64_t n_overdue, int64_t n_merge_queue, int32_t round_down) {
  return calc_new_hosts_needed(short_ns, threshold_ns, expected_free, n_long, n_overdue, n_merge_queue, round_down != 0);
}

int32_t evo_calc_existing_free_hosts(const evo_hosts* h, double future_host_fraction, int64_t threshold_ns,
                                     int64_t now, int64_t* out_free) {
  HView hv{h, 0, h->n};
  std::vector<int64_t> all(h->n);
  for (int64_t i = 0; i < h->n; i++) all[i] = i;
  return calc_existing_free_hosts(hv, all, future_host_fraction, threshold_ns, now, out_free);
}

int32_t evo_allocate(const evo_hosts* h, const evo_alloc_settings* a, const evo_queue_info* info,
                     evo_group_info* groups, const evo_strcol* group_names, int64_t now,
                     int64_t* out_new_hosts, int64_t* out_free_hosts) {
  HView hv{h, 0, h->n};
  std::vector<std::string> names;
  for (int64_t g = 0; g < info->n_groups; g++) names.emplace_back(sv(*group_names, g));
  return allocate(hv, *a, *info, groups, names, now, out_new_hosts, out_free_hosts);
}

int64_t evo_group_by_task_group(const evo_hosts* h, const evo_strcol* group_names, int64_t n_groups,
                                int64_t* out_host_bucket) {
  HView hv{h, 0, h->n};
  std::map<std::string, int64_t> code;
  for (int64_t g = 0; g < n_groups; g++) {
    std::string nm(sv(*group_names, g));
    code[nm] = nm.empty() ? -1 : g;
  }
  int64_t next_unknown = -2;
  for (int64_t i = 0; i < h->n; i++) {
    std::string nm = host_group_name(hv, i);
    auto it = code.find(nm);
    if (it == code.end()) it = code.emplace(nm, nm.empty() ? -1 : next_unknown--).first;
    out_host_bucket[i] = it->second;
  }
  return int64_t(code.size());
}

void evo_fetch_expected_duration(int64_t pred_value, int64_t pred_std, int64_t pred_ttl, int64_t pred_collected_at,
                                 int64_t expected_duration, int64_t expected_std, int64_t now, int32_t hist_found,
                                 int64_t hist_avg, int64_t hist_std, int64_t* out_avg, int64_t* out_std) {
  if (pred_ttl == 0) pred_ttl = kPredictionTTL;  // task.go:3520-3522 (jitter not modelled)
  if (pred_value == 0 && expected_duration != 0) {  // backfill task.go:3524-3539
    *out_avg = expected_duration; *out_std = expected_std;
    return;
  }
  if (since(now, pred_collected_at) < pred_ttl) {  // cached_value.go:127-129
    *out_avg = pred_value; *out_std = pred_std;
    return;
  }
  // refresher task.go:3541-3570
  if (!hist_found) {
    if (pred_value == 0) { *out_avg = kDefaultTaskDuration; *out_std = 0; }
    else { *out_avg = pred_value; *out_std = pred_std; }
    return;
  }
  if (hist_avg == 0) { *out_avg = kDefaultTaskDuration; *out_std = 0; return; }
  *out_avg = hist_avg; *out_std = hist_std;
}

void evo_job_batch(const evo_tasks* t, const int64_t* task_off, const evo_hosts* h, const int64_t* host_off,
                   const evo_planner_settings* ps, const evo_alloc_settings* as, const char* const* distro_ids,
                   int64_t n_distros, int64_t now, int32_t n_threads, int32_t* out_order, int64_t* out_total_value,
                   evo_queue_info* out_info, int64_t* out_new, int64_t* out_free, int32_t* out_status,
                   evo_group_info* out_groups, int64_t* out_bd) {
  std::atomic<int64_t> next{0};
  auto worker = [&]() {
    for (;;) {
      int64_t d = next.fetch_add(1);
      if (d >= n_distros) break;
      View v{t, task_off[d], task_off[d + 1] - task_off[d]};
      PlanResult r = plan(v, ps[d], now);
      for (size_t k = 0; k < r.order.size(); k++) {
        out_order[task_off[d] + k] = int32_t(r.order[k]);
        out_total_value[task_off[d] + k] = r.units[r.unit_of_rank[k]].bd[EVO_BD_TOTAL_VALUE];
        if (out_bd) std::memcpy(out_bd + (task_off[d] + int64_t(k)) * EVO_BD_N, r.units[r.unit_of_rank[k]].bd, sizeof(int64_t) * EVO_BD_N);
      }
      QueueInfo q = queue_info(v, r.order.data(), int64_t(r.order.size()), distro_ids ? distro_ids[d] : "",
                               target_time(ps[d]), ps[d].includes_dependencies != 0, now);
      out_info[d] = q.info;
      if (h && as) {
        HView hv{h, host_off[d], host_off[d + 1] - host_off[d]};
        out_status[d] = allocate(hv, as[d], q.info, q.groups.data(), q.names, now, &out_new[d], &out_free[d]);
      }
      if (out_groups)  // distro d's groups start at slot task_off[d] + d (at most n_tasks + 1 of them)
        for (size_t g = 0; g < q.groups.size(); g++) out_groups[task_off[d] + d + int64_t(g)] = q.groups[g];
    }
  };
  if (n_threads <= 1) { worker(); return; }
  std::vector<std::thread> th;
  for (int i = 0; i < n_threads; i++) th.emplace_back(worker);
  for (auto& x : th) x.join();
}

}  // extern "C"

// evg_plan_general.cuh -- the general path: distros too large for one CTA (any size up to 2^21-1 tasks).
//
// Second generation.  The first one sorted a 64-bit value word plus a 42-bit tie word per task with a 16-pass
// segmented LSD radix sort (20 B/task each way per pass).  This one:
//   k_gtask        per 2048-task tile: 128-bit column loads, 32-bit scoring (single_task_value32) where the
//                  distro allows it, queue-info sums folded per tile, TotalValue of single-task units, per-distro
//                  value range; tasks of multi-member units are linked and compacted into a work list
//   k_gunit/k_gbest  per work-list task: the member at the head of a unit's list computes Unit.info / value / anchor once;
//                  then every task makes its first-occurrence choice (planner.go:467-477) and walks the chosen unit
//                  for its rank; anchor histogram e[]
//   k_gsum/k_gscan/k_gplace(+_disp)
//                  canonical pre-arrangement by COUNTING instead of sorting tie bytes: an exclusive scan of e[] over
//                  the distro gives every anchor's run start; tasks are written to (key, index) buffers in
//                  (anchor, rank-in-unit) order.  Distros without multi-member units skip the scan (identity).
//   k_ghist/k_gdscan/k_gscatter
//                  stable LSD radix sort on key = Vmax - V only: 32-bit keys, ceil(bits(Vmax-Vmin)/8) passes (3 for
//                  a 20-bit range), 8 B/task each way per pass; a distro whose range exceeds 32 bits carries a
//                  second key word and up to 8 passes (per-distro branch, same kernels)
//   k_gemit        ranked queue + TotalValue
// TotalValue per task is parked in the total_value OUTPUT buffer between k_gtask and k_gplace (no 8 B/task scratch).
//
// Reference: scheduler/planner.go:209-481, scheduler/scheduler.go:56-159.
#pragma once

// minimum resident blocks of the work-list kernels (latency-bound: one thread per task or unit, scattered sectors)
#ifndef EVG_OCC_GLINK
#define EVG_OCC_GLINK 4
#endif
#ifndef EVG_OCC_GALLOC
#define EVG_OCC_GALLOC 4
#endif
#ifndef EVG_OCC_GFILL
#define EVG_OCC_GFILL 4
#endif
#ifndef EVG_OCC_GUNIT
#define EVG_OCC_GUNIT 4
#endif
#ifndef EVG_OCC_GBEST
#define EVG_OCC_GBEST 4
#endif
#ifndef EVG_GTASK_OCC
#define EVG_GTASK_OCC 3
#endif
constexpr int kGTile = 2048;  // tasks per tile; tiles start at multiples of 4 tasks (16-byte aligned vector loads)

struct DGen {
  // tiles of the general-path distros, in distro order
  int64_t n_tiles;
  int64_t tile0;               // first tile this launch covers (a chunk of the pipelined one-shot call); grids are relative to it
  const int32_t* tile_distro;  // [NT]
  const int64_t* tile_start;   // [NT] first task slot of the tile: (base & ~3) + k*kGTile, may precede the distro by <= 3
  const int64_t* dtile_off;    // [D+1]
  unsigned long long* vmm;     // [D*2] ord(Vmax), ord(Vmin)
  uint32_t* key_lo[2];         // [T] low word of Vmax - V, in sort position
  uint32_t* key_hi[2];         // [T] high word (distros with a range above 32 bits only)
  uint32_t* idx[2];            // [T] distro-local task index, in sort position
  uint32_t* e;                 // [T] anchor histogram, then exclusive positions
  uint32_t* tile_sum;          // [NT] sum of e over the tile, then the tile's exclusive offset inside its distro
  uint32_t* tile_hist;         // [NT*256]
  uint32_t* clist;             // work list: global task index of every task that touches a multi-member unit
  int32_t* clist_d;            // its distro
  unsigned int* ccount;        // [1]
  uint4* tie;                  // [T] work-list tasks: x = anchor of the unit the task is emitted from, y = rank inside it,
                               //     z = that unit's slot (kInactive: its own single-task unit)
  int32_t* maxpass;            // [1]
  struct URec* rec;            // unit table: the members of every multi-member unit, one contiguous run per unit
  unsigned int* rcount;        // [1] records reserved
  uint4* usum;                 // [unit slots] what k_gbest asks of a candidate unit, in one 16-byte load: x|y<<32 = TotalValue, z = anchor
                               //     (kNoAnchor: never exported), w = members
  uint2* hlist;                // multi-member units of the tick: x = slot, y = distro (k_galloc lists them, k_gunit folds them)
  unsigned int* hcount;        // [1]
  int64_t* tv;                 // [T] TotalValue by task (the output buffer, reused)
};

__device__ __forceinline__ int gen_bits(const DGen& G, int d) {  // significant bits of Vmax - Vmin
  const unsigned long long r = G.vmm[2 * d] - G.vmm[2 * d + 1];
  return r == 0 ? 0 : 64 - __clzll((long long)r);
}
__device__ __forceinline__ int gen_npass(int bits) { return (bits + 7) >> 3; }

__global__ void k_ginit(DGen G, const int32_t* __restrict__ general_list, int n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) { *G.ccount = 0u; *G.maxpass = 0; *G.rcount = 0u; *G.hcount = 0u; }
  if (k >= n) return;
  const int d = general_list[k];
  G.vmm[2 * d] = 0ull;
  G.vmm[2 * d + 1] = ~0ull;
}

// planner.go:449-456 (pass 2): mark every task some in-queue task depends on (general-path distros only).
__global__ void __launch_bounds__(256) k_gmark(DTasks T, DDistros D, DWork W, DGen G) {
  if (*W.err) return;
  const int tile = int(blockIdx.x + G.tile0);
  const int d = G.tile_distro[tile];
  const int64_t base = D.task_off[d], end = D.task_off[d + 1];
  const int64_t lo = max(G.tile_start[tile], base), hi = min(G.tile_start[tile] + kGTile, end);
  for (int64_t t = lo + threadIdx.x; t < hi; t += 256)
    for (int64_t e = T.dep_off[t]; e < T.dep_off[t + 1]; e++) W.has_dep[base + T.dep_idx[e]] = 1;
}

struct TileFold {  // queue-info partials of one tile (scheduler.go:66-138)
  unsigned int c[10];
  unsigned long long s[4];
  unsigned long long vmax, vmin;
};

// Per tile: queue info, single-task scores, unit links.  256 threads x 8 tasks: thread q of group u owns the four
// consecutive task slots tile_start + 4*(u*256 + q) .. +3, so every column is read with 128-bit loads.
__global__ void __launch_bounds__(256, EVG_GTASK_OCC) k_gtask(DTasks T, DDistros D, DWork W, DGen G, int64_t now, int any_complex) {
  if (*W.err) return;
  __shared__ TileFold F;
  __shared__ evg_distro_cfg s_cfg;
  __shared__ uint32_t s_nd[kNdTable];  // int64(NumDependentsFactor * n), n < kNdTable: fractional factors stay on the 32-bit scorer
  const int tile = int(blockIdx.x + G.tile0);
  const int d = G.tile_distro[tile];
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned full = 0xffffffffu;
  if (tid == 0) {
    for (int k = 0; k < 10; k++) F.c[k] = 0;
    for (int k = 0; k < 4; k++) F.s[k] = 0;
    F.vmax = 0ull; F.vmin = ~0ull;
    s_cfg = D.cfg[d];
  }
  __syncthreads();
  const evg_distro_cfg& cfg = s_cfg;
  const int64_t base = D.task_off[d], end = D.task_off[d + 1];
  const int64_t ts = G.tile_start[tile];
  const uint32_t ng = uint32_t(D.group_off[d + 1] - D.group_off[d]);
  const bool gv = cfg.group_versions != 0;
  const int64_t threshold = cfg.target_time_ns;
  const PlannerFactors pf = clamp_factors(cfg);
  const Factors32 f32 = factors32(pf, now);
  const bool sane_clock = threshold >= 0 && now >= threshold;
  const int64_t wait_cutoff = wsub(now, threshold);
  const bool fast_clock = now >= 0 && pf.nd_int != 0;
  const bool incl = cfg.includes_dependencies != 0;
  if (tid < kNdTable) {
    const int64_t e = nd_table_entry(pf, tid);
    s_nd[tid] = (e >= 0 && e < int64_t(kNdTermLimit)) ? uint32_t(e) : 0xFFFFFFFFu;
  }
  __syncthreads();
  const bool dcomplex = any_complex && (ng > 0 || gv || (T.n_edges > 0 && T.dep_off[end] > T.dep_off[base]));

  unsigned int c_dm = 0, c_mq = 0, c_over = 0, c_wait = 0, c_sec = 0, c_ung = 0, c_ucnt = 0, c_uover = 0, c_uwait = 0, c_umq = 0;
  int64_t s_exp = 0, s_over = 0, s_uexp = 0, s_uover = 0;
  unsigned long long kmax = 0ull, kmin = ~0ull;
  uint32_t cmask = 0;  // bit 4*u + m: task ts + 4*(u*256 + tid) + m goes on the work list

#pragma unroll 1
  for (int u = 0; u < 2; u++) {
    const int64_t t4 = ts + 4 * int64_t(u * 256 + tid);  // multiple of 4: 16-byte aligned in every column
    const bool live = t4 < end;  // the columns are readable 8 slots past the last task (upload pads them)
    int4 prio4 = make_int4(0, 0, 0, 0), nd4 = prio4, gid4 = make_int4(-1, -1, -1, -1);
    uint4 fl4 = make_uint4(0, 0, 0, 0);
    longlong2 ex01 = make_longlong2(0, 0), ex23 = ex01, qb01 = ex01, qb23 = ex01, wb01 = ex01, wb23 = ex01;
    if (live) {
      prio4 = *reinterpret_cast<const int4*>(T.priority + t4);
      nd4 = *reinterpret_cast<const int4*>(T.numdep + t4);
      gid4 = *reinterpret_cast<const int4*>(T.gid + t4);
      fl4 = *reinterpret_cast<const uint4*>(T.flags + t4);
      ex01 = *reinterpret_cast<const longlong2*>(T.expected + t4); ex23 = *reinterpret_cast<const longlong2*>(T.expected + t4 + 2);
      qb01 = *reinterpret_cast<const longlong2*>(T.qbasis + t4); qb23 = *reinterpret_cast<const longlong2*>(T.qbasis + t4 + 2);
      wb01 = *reinterpret_cast<const longlong2*>(T.wbasis + t4); wb23 = *reinterpret_cast<const longlong2*>(T.wbasis + t4 + 2);
    }
    // dependency offsets of the four tasks (five consecutive entries) and their "has dependents" bytes, as vectors too
    int64_t doff[5] = {0, 0, 0, 0, 0};
    uint32_t hd4 = 0;
    if (live && dcomplex) {
      if (T.n_edges > 0) {
        const longlong2 d01 = *reinterpret_cast<const longlong2*>(T.dep_off + t4), d23 = *reinterpret_cast<const longlong2*>(T.dep_off + t4 + 2);
        doff[0] = d01.x; doff[1] = d01.y; doff[2] = d23.x; doff[3] = d23.y; doff[4] = T.dep_off[t4 + 4];
      }
      hd4 = *reinterpret_cast<const uint32_t*>(W.has_dep + t4);
    }
    const int32_t prio_[4] = {prio4.x, prio4.y, prio4.z, prio4.w}, nd_[4] = {nd4.x, nd4.y, nd4.z, nd4.w};
    const int32_t gid_[4] = {gid4.x, gid4.y, gid4.z, gid4.w};
    const uint32_t fl_[4] = {fl4.x, fl4.y, fl4.z, fl4.w};
    const int64_t ex_[4] = {ex01.x, ex01.y, ex23.x, ex23.y}, qb_[4] = {qb01.x, qb01.y, qb23.x, qb23.y};
    const int64_t wb_[4] = {wb01.x, wb01.y, wb23.x, wb23.y};
    int64_t vout[4];
    uint32_t eout[4], nd_term[4];
    bool wr_v[4], solo[4];
    bool dom = true;
#pragma unroll
    for (int m = 0; m < 4; m++) {
      const int64_t t = t4 + m;
      const bool valid = live & (t >= base) & (t < end);
      const int32_t prio = prio_[m], nd = nd_[m], gid = gid_[m];
      const uint32_t fl = fl_[m];
      const int64_t exp_ns = ex_[m], qb = qb_[m], wb = wb_[m];
      // straight-line (bitwise bool operators, selects): the short-circuit forms cost a branch per operator
      const bool dm = valid & ((fl & EVG_TF_DEPS_MET) != 0);
      const bool counted = valid & (!incl | dm);
      const bool over = counted & (exp_ns > threshold);
      const bool waited = sane_clock ? (wb < wait_cutoff) : (since(now, wb) > threshold);  // sane_clock is block-uniform
      const bool wait_over = counted & dm & waited;
      const bool mq_dm = dm & ((fl & EVG_TF_REQ_MASK) == EVG_TF_REQ_MERGE_QUEUE);
      const bool ung = valid & (gid < 0);
      c_dm += dm; c_mq += mq_dm; c_over += over; c_wait += wait_over; c_sec += valid & ((fl & EVG_TF_OTHER_DISTRO) != 0);
      s_exp += counted ? exp_ns : 0;
      s_over += over ? exp_ns : 0;
      c_ung += ung; c_ucnt += ung & counted; c_uover += ung & over; c_uwait += ung & wait_over; c_umq += ung & mq_dm;
      s_uexp += (ung & counted) ? exp_ns : 0;
      s_uover += (ung & over) ? exp_ns : 0;
      // membership links, dependency edges and the TaskGroupInfo sums of multi-member-unit tasks are k_glink's job:
      // pointer chasing with a few active lanes per warp would stall this streaming pass
      const bool own_complex = valid & dcomplex & ((gid >= 0) | gv | (((hd4 >> (8 * m)) & 0xFFu) != 0));
      const bool complex_task = own_complex | (valid & dcomplex & (doff[m + 1] > doff[m]));
      const bool scores = valid & !own_complex;  // the unit filed under this task's own key is {this task}
      const uint32_t ndc = uint32_t(nd > 0 ? nd : 0);
      const uint32_t tab = s_nd[ndc < uint32_t(kNdTable) ? ndc : 0u];
      const uint32_t mul = (f32.ok & (ndc < kTask32Limit)) ? f32.nd * ndc : 0xFFFFFFFFu;
      nd_term[m] = ndc < uint32_t(kNdTable) ? tab : mul;
      dom = dom & (!scores | (score32_bad(now, prio, exp_ns, qb, nd_term[m]) == 0u));
      wr_v[m] = scores;
      solo[m] = scores & !complex_task;  // final: the task is emitted from its own unit
      eout[m] = (valid & !complex_task) ? 1u : 0u;
      cmask |= (complex_task ? 1u : 0u) << (4 * u + m);
    }
    if (f32.ok_base && __all_sync(full, dom)) {  // one warp vote per four tasks; the 64-bit scorers stay out of line
#pragma unroll
      for (int m = 0; m < 4; m++) vout[m] = int64_t(single_task_value32_nd(f32, now, prio_[m], ex_[m], qb_[m], nd_term[m], fl_[m]));
    } else {
#pragma unroll
      for (int m = 0; m < 4; m++) vout[m] = int64_t(score_slow(pf, fast_clock, wr_v[m], now, prio_[m], ex_[m], qb_[m], nd_[m], fl_[m]));
    }
#pragma unroll
    for (int m = 0; m < 4; m++) {
      const unsigned long long k = ord_i64(vout[m]);
      kmax = solo[m] ? max(kmax, k) : kmax;
      kmin = solo[m] ? min(kmin, k) : kmin;
    }
    // TotalValue of single-task units (also the own-unit candidate of a task that only joins other units by edges)
    if (!live) {
    } else if (t4 >= base && t4 + 3 < end) {  // whole sectors even when some of the four are multi-member-unit tasks: k_gbest rewrites theirs
      *reinterpret_cast<longlong2*>(G.tv + t4) = make_longlong2(vout[0], vout[1]);
      *reinterpret_cast<longlong2*>(G.tv + t4 + 2) = make_longlong2(vout[2], vout[3]);
    } else {
#pragma unroll
      for (int m = 0; m < 4; m++)
        if (wr_v[m]) G.tv[t4 + m] = vout[m];
    }
    if (dcomplex && live) {
      if (t4 >= base && t4 + 3 < end) *reinterpret_cast<uint4*>(G.e + t4) = make_uint4(eout[0], eout[1], eout[2], eout[3]);
      else {
#pragma unroll
        for (int m = 0; m < 4; m++)
          if (t4 + m >= base && t4 + m < end) G.e[t4 + m] = eout[m];
      }
    }
  }
  // Work list: ONE global atomic per tile (a block scan of the per-thread counts gives every entry its place) -- an
  // atomic per warp and task slot serialised every tile of the tick on one L2 address.
  if (dcomplex) {
    __shared__ uint32_t s_wsum[8];
    __shared__ uint32_t s_lbase;
    const uint32_t mine = __popc(cmask);
    uint32_t inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(full, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) s_wsum[tid >> 5] = inc;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) { const uint32_t x = s_wsum[w]; before += w < (tid >> 5) ? x : 0u; total += x; }
    if (total) {  // block-uniform
      if (tid == 0) s_lbase = atomicAdd(G.ccount, total);
      __syncthreads();
      uint32_t pos = s_lbase + before + inc - mine;
      for (uint32_t b = cmask; b; b &= b - 1u) {
        const int bit = __ffs(b) - 1;
        G.clist[pos] = uint32_t(ts + 4 * int64_t((bit >> 2) * 256 + tid) + (bit & 3));
        G.clist_d[pos] = d;
        pos++;
      }
    }
  }
  // fold: warp, then block (shared atomics), then one set of global atomics per tile
  {
    unsigned int cs[10] = {c_dm, c_mq, c_over, c_wait, c_sec, c_ung, c_ucnt, c_uover, c_uwait, c_umq};
#pragma unroll
    for (int k = 0; k < 10; k++) cs[k] = __reduce_add_sync(full, cs[k]);
    int64_t ss[4] = {s_exp, s_over, s_uexp, s_uover};
#pragma unroll
    for (int k = 0; k < 4; k++) ss[k] = warp_sum64(ss[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      kmax = max(kmax, __shfl_xor_sync(full, kmax, o));
      kmin = min(kmin, __shfl_xor_sync(full, kmin, o));
    }
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < 10; k++) if (cs[k]) atomicAdd(&F.c[k], cs[k]);
#pragma unroll
      for (int k = 0; k < 4; k++) if (ss[k]) atomicAdd(&F.s[k], (unsigned long long)ss[k]);
      atomicMax(&F.vmax, kmax); atomicMin(&F.vmin, kmin);
    }
  }
  __syncthreads();
  if (tid < 16) {
    evg_queue_info* q = W.qinfo + d;
    switch (tid) {
      case 0: atomic_add64(&q->length_with_dependencies_met, F.c[0]); break;
      case 1: atomic_add64(&q->count_dep_filled_merge_queue_tasks, F.c[1]); break;
      case 2: atomic_add64(&q->count_duration_over_threshold, F.c[2]); break;
      case 3: atomic_add64(&q->count_wait_over_threshold, F.c[3]); break;
      case 4: atomic_add64(&q->secondary_queue, F.c[4]); break;
      case 5: atomic_add64(&q->has_ungrouped, F.c[5]); break;
      case 6: atomic_add64(&q->ungrouped.count, F.c[6]); break;
      case 7: atomic_add64(&q->ungrouped.count_duration_over_threshold, F.c[7]); break;
      case 8: atomic_add64(&q->ungrouped.count_wait_over_threshold, F.c[8]); break;
      case 9: atomic_add64(&q->ungrouped.count_dep_filled_merge_queue_tasks, F.c[9]); break;
      case 10: atomic_add64(&q->expected_duration, int64_t(F.s[0])); break;
      case 11: atomic_add64(&q->duration_over_threshold, int64_t(F.s[1])); break;
      case 12: atomic_add64(&q->ungrouped.expected_duration, int64_t(F.s[2])); break;
      case 13: atomic_add64(&q->ungrouped.duration_over_threshold, int64_t(F.s[3])); break;
      case 14: if (F.vmax > __ldcg(G.vmm + 2 * d)) atomicMax(G.vmm + 2 * d, F.vmax); break;
      case 15: if (F.vmin < __ldcg(G.vmm + 2 * d + 1)) atomicMin(G.vmm + 2 * d + 1, F.vmin); break;
    }
  }
}

// ---- multi-member units: the unit table ----
// A membership ("pair": a task filed under a unit slot by its own key, by its version, or by one of its in-queue
// dependencies' keys; planner.go:431-456) used to be a node of a linked list per slot, and every walk a chain of
// dependent scattered loads through six task columns.  Now the members of a unit are one contiguous run of packed
// 32-byte records:
//   k_glink   per pair: k = atomicAdd(unit_n[slot], 1) -- its place in the run (any order: everything computed from a
//             run is order-free); TaskGroupInfo sums of task-group tasks
//   k_galloc  the pair that drew k == 0 reserves unit_n[slot] records: head[slot] = start of the run
//   k_gfill   every pair writes its task's record at head[slot] + k
//   k_gunit   the k == 0 pair folds the run into Unit.info (planner.go:302-337), value (planner.go:209-300), anchor
//   k_gbest   per task: the first unit it is emitted from among its memberships (TaskPlan.Export, planner.go:467-477),
//             then its rank inside it (TaskList.Less, planner.go:387-405) by one pass over the run
// pair ids: own-key pair of task t = t, version pair = T.n + t, pair of dependency edge e = 2*T.n + e.
struct __align__(16) URec {
  int32_t prio, nd;
  int64_t exp_ns, qb;
  int32_t tgo;
  uint32_t lif;  // bits 0..20 distro-local task index, 21 own-key pair, 22 group_id >= 0, 24..29 task flags
};
static_assert(sizeof(URec) == 32, "one L2 sector per member");
constexpr uint32_t kRecOwn = 1u << 21, kRecGrouped = 1u << 22;
__device__ __forceinline__ uint32_t rec_li(const URec& r) { return r.lif & 0x1FFFFFu; }
__device__ __forceinline__ URec rec_load(const URec* p) {  // two 128-bit loads
  const uint4 a = reinterpret_cast<const uint4*>(p)[0], b = reinterpret_cast<const uint4*>(p)[1];
  URec r;
  r.prio = int32_t(a.x); r.nd = int32_t(a.y); r.exp_ns = int64_t((unsigned long long)a.z | ((unsigned long long)a.w << 32));
  r.qb = int64_t((unsigned long long)b.x | ((unsigned long long)b.y << 32)); r.tgo = int32_t(b.z); r.lif = b.w;
  return r;
}
__device__ __forceinline__ void rec_store(URec* p, const URec& r) {
  reinterpret_cast<uint4*>(p)[0] = make_uint4(uint32_t(r.prio), uint32_t(r.nd), uint32_t(uint64_t(r.exp_ns)), uint32_t(uint64_t(r.exp_ns) >> 32));
  reinterpret_cast<uint4*>(p)[1] = make_uint4(uint32_t(uint64_t(r.qb)), uint32_t(uint64_t(r.qb) >> 32), uint32_t(r.tgo), r.lif);
}

// what a work-list task is filed under (the same answers in every kernel below)
struct WlTask {
  uint32_t t; int d; int64_t base; uint32_t li, ub, ng; int32_t gid, vid; bool gv, own_complex; uint32_t s_own, s_ver;
};
__device__ __forceinline__ WlTask wl_task(const DTasks& T, const DDistros& D, const DWork& W, const DGen& G, unsigned int k) {
  WlTask x;
  x.t = G.clist[k]; x.d = G.clist_d[k];
  x.base = D.task_off[x.d];
  x.gid = T.gid[x.t]; x.vid = T.vid[x.t];
  x.ng = uint32_t(D.group_off[x.d + 1] - D.group_off[x.d]);
  x.ub = uint32_t(D.unit_base[x.d]);
  x.gv = D.cfg[x.d].group_versions != 0;
  x.li = uint32_t(int64_t(x.t) - x.base);
  x.own_complex = x.gid >= 0 || x.gv || (W.has_dep[x.t] & 1) != 0;
  x.s_own = own_slot_local(x.gid, x.vid, x.li, x.ng, x.gv);
  x.s_ver = (x.gid >= 0 && x.gv) ? x.ng + uint32_t(x.vid) : kInactive;
  return x;
}
// f(pair, slot) for every membership of the task (after k_glink: pair_slot / edge_live are final)
template <typename F>
__device__ __forceinline__ void wl_pairs(const DTasks& T, const DWork& W, const WlTask& x, F&& f) {
  if (x.own_complex) f(x.t, x.ub + x.s_own);
  if (x.s_ver != kInactive) f(uint32_t(T.n + x.t), x.ub + x.s_ver);
  if (T.n_edges > 0)
    for (int64_t e = T.dep_off[x.t]; e < T.dep_off[x.t + 1]; e++)
      if (W.edge_live[e]) f(uint32_t(2 * T.n + e), W.pair_slot[2 * T.n + e]);
}

__global__ void __launch_bounds__(256, EVG_OCC_GLINK) k_glink(DTasks T, DDistros D, DWork W, DGen G, int64_t now) {
  if (*W.err) return;
  const unsigned int n = *G.ccount;
  for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const WlTask x = wl_task(T, D, W, G, k);
    const uint32_t t = x.t;
    const int d = x.d;
    if (x.gid >= 0) {
      const evg_distro_cfg* cf = D.cfg + d;
      const uint32_t fl = T.flags[t];
      const int64_t exp_ns = T.expected[t], threshold = cf->target_time_ns;
      const bool dm = (fl & EVG_TF_DEPS_MET) != 0;
      const bool counted = !cf->includes_dependencies || dm;
      const bool over = counted && exp_ns > threshold;
      const bool wait_over = counted && dm && since(now, T.wbasis[t]) > threshold;
      const bool mq_dm = dm && (fl & EVG_TF_REQ_MASK) == EVG_TF_REQ_MERGE_QUEUE;
      evg_group_info* g = W.ginfo + D.group_off[d] + x.gid;
      atomic_add64(&g->count, counted);
      atomic_add64(&g->expected_duration, counted ? exp_ns : 0);
      atomic_add64(&g->count_duration_over_threshold, over);
      atomic_add64(&g->duration_over_threshold, over ? exp_ns : 0);
      atomic_add64(&g->count_wait_over_threshold, wait_over);
      atomic_add64(&g->count_dep_filled_merge_queue_tasks, mq_dm);
    }
    auto join = [&](uint32_t pair, uint32_t slot) {
      W.pair_slot[pair] = slot;
      W.next[pair] = atomicAdd(W.unit_n + slot, 1u);  // the pair's place in the unit's run
    };
    if (x.own_complex) join(t, x.ub + x.s_own);
    if (x.s_ver != kInactive) join(uint32_t(T.n + t), x.ub + x.s_ver);  // planner.go:439
    if (T.n_edges > 0) {
      const int64_t e0 = T.dep_off[t], e1 = T.dep_off[t + 1];
      for (int64_t e = e0; e < e1; e++) {
        const uint32_t dl = uint32_t(T.dep_idx[e]);
        const uint32_t sl = own_slot_local(T.gid[x.base + dl], T.vid[x.base + dl], dl, x.ng, x.gv);
        bool dup = (sl == x.s_own) || (sl == x.s_ver);  // Unit.Add is keyed by task id (planner.go:131): join each unit once
        for (int64_t f = e0; f < e && !dup; f++) {
          const uint32_t fl2 = uint32_t(T.dep_idx[f]);
          dup = own_slot_local(T.gid[x.base + fl2], T.vid[x.base + fl2], fl2, x.ng, x.gv) == sl;
        }
        W.edge_task[e] = t;
        W.edge_live[e] = dup ? 0 : 1;
        if (!dup) join(uint32_t(2 * T.n + e), x.ub + sl);
      }
    }
  }
}

// Runs are reserved block by block: a block scan of the records its threads need, ONE atomic on the bump counter per
// block and trip (an atomic per unit serialised ~10^5 units of a tick on one L2 address: 340 us of a 1.4 ms tick).
__global__ void __launch_bounds__(256, EVG_OCC_GALLOC) k_galloc(DTasks T, DDistros D, DWork W, DGen G) {
  if (*W.err) return;
  __shared__ uint32_t s_wsum[8], s_wcnt[8];
  __shared__ uint32_t s_base, s_hbase;
  const unsigned int n = *G.ccount;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (unsigned int k0 = blockIdx.x * blockDim.x; k0 < n; k0 += gridDim.x * blockDim.x) {  // block-uniform trip count
    const unsigned int k = k0 + threadIdx.x;
    WlTask x;
    uint32_t need = 0, heads = 0;  // records / units this thread's k == 0 pairs stand for
    if (k < n) {
      x = wl_task(T, D, W, G, k);
      wl_pairs(T, W, x, [&](uint32_t pair, uint32_t slot) { if (W.next[pair] == 0u) { need += W.unit_n[slot]; heads++; } });
    }
    uint32_t inc = need, hinc = heads;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o), z = __shfl_up_sync(0xffffffffu, hinc, o);
      if (lane >= o) { inc += y; hinc += z; }
    }
    if (lane == 31) { s_wsum[warp] = inc; s_wcnt[warp] = hinc; }
    __syncthreads();
    uint32_t before = 0, total = 0, hbefore = 0, htotal = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) {
      const uint32_t y = s_wsum[w], z = s_wcnt[w];
      before += w < warp ? y : 0u; total += y; hbefore += w < warp ? z : 0u; htotal += z;
    }
    if (threadIdx.x == 0 && htotal) { s_base = atomicAdd(G.rcount, total); s_hbase = atomicAdd(G.hcount, htotal); }
    __syncthreads();
    if (heads) {
      uint32_t pos = s_base + before + inc - need, hp = s_hbase + hbefore + hinc - heads;
      wl_pairs(T, W, x, [&](uint32_t pair, uint32_t slot) {
        if (W.next[pair] == 0u) { W.head[slot] = pos; pos += W.unit_n[slot]; G.hlist[hp++] = make_uint2(slot, uint32_t(x.d)); }
      });
    }
    __syncthreads();  // the shared scratch is rewritten by the next trip
  }
}

__global__ void __launch_bounds__(256, EVG_OCC_GFILL) k_gfill(DTasks T, DDistros D, DWork W, DGen G) {
  if (*W.err) return;
  const unsigned int n = *G.ccount;
  for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const WlTask x = wl_task(T, D, W, G, k);
    URec r;
    r.prio = T.priority[x.t]; r.nd = T.numdep[x.t]; r.exp_ns = T.expected[x.t]; r.qb = T.qbasis[x.t]; r.tgo = T.tgo[x.t];
    r.lif = x.li | (x.gid >= 0 ? kRecGrouped : 0u) | ((T.flags[x.t] & 0x3Fu) << 24);
    wl_pairs(T, W, x, [&](uint32_t pair, uint32_t slot) {
      URec q = r;
      if (pair < uint32_t(T.n)) q.lif |= kRecOwn;  // own-key pairs are the SetDistro members (planner.go:446)
      rec_store(G.rec + W.head[slot] + W.next[pair], q);
    });
  }
}

__device__ __forceinline__ void rec_acc(UnitAcc& a, int64_t now, const URec& r) {
  acc_add(a, now, r.prio, r.exp_ns, r.qb, r.nd, (r.lif & kRecGrouped) ? 0 : -1, (r.lif >> 24) & 0x3Fu);
}

// One thread per multi-member unit (dense warps: the unit list, not the work list).
__global__ void __launch_bounds__(256, EVG_OCC_GUNIT) k_gunit(DDistros D, DWork W, DGen G, int64_t now) {
  if (*W.err) return;
  const unsigned int n = *G.hcount;
  for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {  // the host cannot know n: fixed grid
    const uint2 u = G.hlist[k];
    const uint32_t cnt = W.unit_n[u.x];
    const URec* run = G.rec + W.head[u.x];
    UnitAcc a;
    acc_init(a);
    uint32_t anchor = kNoAnchor;
    for (uint32_t i = 0; i < cnt; i++) {
      const URec r = rec_load(run + i);
      rec_acc(a, now, r);
      if (r.lif & kRecOwn) anchor = min(anchor, rec_li(r));
    }
    const unsigned long long v = (unsigned long long)unit_value(a, D.cfg[u.y], nullptr);
    G.usum[u.x] = make_uint4(uint32_t(v), uint32_t(v >> 32), anchor, cnt);  // kNoAnchor: the unit never got a distro -> not exported (planner.go:81-83)
    W.unit_mask[u.x] = 0ull;  // k_gbest ORs the emitted ranks in (cleared here, unit by unit, instead of a slot-wide memset)
  }
}

__global__ void __launch_bounds__(256, EVG_OCC_GBEST) k_gbest(DTasks T, DDistros D, DWork W, DGen G, int want_best_pair) {
  if (*W.err) return;
  const unsigned int n = *G.ccount;
  for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const WlTask x = wl_task(T, D, W, G, k);
    const uint32_t t = x.t, li = x.li;
    const int d = x.d;
    bool have = false;
    int64_t bv = 0;
    uint32_t ba = 0, brk = 0, bp = kInactive, bslot = kInactive, bn = 1, bkx = 0;
    if (!x.own_complex) { have = true; bv = G.tv[t]; ba = li; }  // its own single-task unit, scored by k_gtask
    wl_pairs(T, W, x, [&](uint32_t pair, uint32_t slot) {
      const uint4 u = G.usum[slot];
      const uint32_t kx = W.next[pair];  // this task's place in that unit's run (requested together with the summary)
      const uint32_t a = u.z;
      if (a == kNoAnchor) return;
      const int64_t v = int64_t((unsigned long long)u.x | ((unsigned long long)u.y << 32));
      if (!have || v > bv || (v == bv && a < ba)) { have = true; bv = v; ba = a; bp = pair; bslot = slot; bn = u.w; bkx = kx; }
    });
    if (bp != kInactive) {  // rank among ALL members of the chosen unit; the task's own fields are its record in the run
      const URec* run = G.rec + W.head[bslot];
      const URec me = rec_load(run + bkx);
      for (uint32_t i = 0; i < bn; i++) {
        const URec r = rec_load(run + i);
        if (in_unit_less(r.tgo, r.nd, r.prio, r.exp_ns, rec_li(r), me.tgo, me.nd, me.prio, me.exp_ns, li)) brk++;
      }
      if (bn <= 64) atomicOr(&W.unit_mask[bslot], 1ull << brk);  // ranks emitted from the unit: k_gplace_disp counts below its own
    }
    G.tv[t] = bv;
    G.tie[t] = make_uint4(ba, brk, bslot, 0u);
    if (want_best_pair) W.best_pair[t] = bp;  // k_breakdown's way back to the unit
    const bool displaced = !(ba == li && brk == 0);
    if (displaced) W.has_dep[t] |= 2;  // only this thread touches the byte now (k_gmark and k_gtask are done)
    atomicAdd(G.e + x.base + ba, 1u);
    // The distro's value range.  The work list is in task order, so a warp nearly always sits inside one distro: its 32
    // values are folded with shuffles and ONE lane looks at the distro's pair (every thread polling the same two L2 lines
    // was a third of this kernel's stall samples).
    const unsigned long long kk = ord_i64(bv);
    const unsigned act = __activemask();
    const int d0 = __shfl_sync(act, d, __ffs(act) - 1);
    if (__all_sync(act, d == d0)) {
      unsigned long long hi = kk, lo = kk;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long h2 = __shfl_xor_sync(act, hi, o), l2 = __shfl_xor_sync(act, lo, o);
        const bool other = (act >> ((threadIdx.x & 31) ^ o)) & 1u;  // an exited lane's register is not a value
        hi = (other && h2 > hi) ? h2 : hi;
        lo = (other && l2 < lo) ? l2 : lo;
      }
      if ((threadIdx.x & 31) == __ffs(act) - 1) {
        if (hi > __ldcg(G.vmm + 2 * d)) atomicMax(G.vmm + 2 * d, hi);
        if (lo < __ldcg(G.vmm + 2 * d + 1)) atomicMin(G.vmm + 2 * d + 1, lo);
      }
    } else {
      if (kk > __ldcg(G.vmm + 2 * d)) atomicMax(G.vmm + 2 * d, kk);
      if (kk < __ldcg(G.vmm + 2 * d + 1)) atomicMin(G.vmm + 2 * d + 1, kk);
    }
  }
}

// radix pass count of the tick (the host launches that many pass triples... it cannot know: it launches 8, the
// kernels of passes beyond *maxpass exit at once)
__global__ void k_gsched(DGen G, const int32_t* __restrict__ general_list, int n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int np = gen_npass(gen_bits(G, general_list[k]));
  if (np > 0) atomicMax(G.maxpass, np);
}

// sum of e[] over each tile
__global__ void __launch_bounds__(256) k_gsum(DDistros D, DGen G) {
  const int tile = int(blockIdx.x + G.tile0);
  const int d = G.tile_distro[tile];
  const int64_t base = D.task_off[d], end = D.task_off[d + 1];
  const int64_t lo = max(G.tile_start[tile], base), hi = min(G.tile_start[tile] + kGTile, end);
  uint32_t sum = 0;
  for (int64_t t = lo + threadIdx.x; t < hi; t += 256) sum += G.e[t];
  sum = __reduce_add_sync(0xffffffffu, sum);
  __shared__ uint32_t sw[8];
  if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) G.tile_sum[tile] = sw[0] + sw[1] + sw[2] + sw[3] + sw[4] + sw[5] + sw[6] + sw[7];
}

// exclusive scan of the tile sums of one distro (<= 1025 tiles), one block per general-path distro
__global__ void __launch_bounds__(1024) k_gscan(DGen G, const int32_t* __restrict__ general_list) {
  const int d = general_list[blockIdx.x];
  const int64_t t0 = G.dtile_off[d], nt = G.dtile_off[d + 1] - t0;
  __shared__ uint32_t sw[32];
  __shared__ uint32_t carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t c0 = 0; c0 < nt; c0 += 1024) {
    const int64_t i = c0 + threadIdx.x;
    const uint32_t v = i < nt ? G.tile_sum[t0 + i] : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) sw[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const uint32_t w = sw[lane];
      uint32_t winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += x; }
      sw[lane] = winc - w;
    }
    __syncthreads();
    const uint32_t ex = carry + sw[warp] + inc - v;
    if (i < nt) G.tile_sum[t0 + i] = ex;
    __syncthreads();
    if (threadIdx.x == 1023) carry = ex + v;
    __syncthreads();
  }
}

__device__ __forceinline__ void gen_put(const DGen& G, int64_t base, uint32_t pos, unsigned long long vmax_ord, bool wide,
                                        int64_t v, uint32_t li) {
  const unsigned long long key = vmax_ord - ord_i64(v);
  G.key_lo[0][base + pos] = uint32_t(key);
  if (wide) G.key_hi[0][base + pos] = uint32_t(key >> 32);
  G.idx[0][base + pos] = li;
}

// Per tile: exclusive scan of e[] (thread q owns 8 consecutive slots) on top of the tile's offset = the run start of
// every anchor; tasks that keep their own anchor with rank 0 are written to their sort position.  use_e == 0 (no
// multi-member unit in any general-path distro): positions are the input order.
__global__ void __launch_bounds__(256) k_gplace(DDistros D, DWork W, DGen G, int use_e) {
  const int tile = int(blockIdx.x + G.tile0);
  const int d = G.tile_distro[tile];
  const int64_t base = D.task_off[d], end = D.task_off[d + 1];
  const int64_t ts = G.tile_start[tile];
  const unsigned long long vmax_ord = G.vmm[2 * d];
  const bool wide = gen_bits(G, d) > 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t t8 = ts + 8 * int64_t(tid);  // multiple of 4
  const bool interior = t8 >= base && t8 + 7 < end;  // the common case: 128-bit loads
  uint32_t ev[8];
  uint32_t sum = 0;
  if (use_e) {
    if (interior) {
      const uint4 a = *reinterpret_cast<const uint4*>(G.e + t8), b = *reinterpret_cast<const uint4*>(G.e + t8 + 4);
      ev[0] = a.x; ev[1] = a.y; ev[2] = a.z; ev[3] = a.w; ev[4] = b.x; ev[5] = b.y; ev[6] = b.z; ev[7] = b.w;
    } else {
#pragma unroll
      for (int m = 0; m < 8; m++) { const int64_t t = t8 + m; ev[m] = (t >= base && t < end) ? G.e[t] : 0u; }
    }
#pragma unroll
    for (int m = 0; m < 8; m++) sum += ev[m];
  }
  uint32_t run = 0;
  if (use_e) {
    __shared__ uint32_t sw[8];
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
    if (lane == 31) sw[warp] = inc;
    __syncthreads();
    uint32_t before = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) if (w < warp) before += sw[w];
    run = G.tile_sum[tile] + before + inc - sum;
  }
  int64_t vv[8];
  uint32_t dsp = 0;  // bit m: task t8+m leaves its own anchor's first slot (placed by k_gplace_disp)
  if (interior) {
#pragma unroll
    for (int m = 0; m < 8; m += 2) {
      const longlong2 x = *reinterpret_cast<const longlong2*>(G.tv + t8 + m);
      vv[m] = x.x; vv[m + 1] = x.y;
    }
    if (use_e) {
      const uint32_t h0 = *reinterpret_cast<const uint32_t*>(W.has_dep + t8), h1 = *reinterpret_cast<const uint32_t*>(W.has_dep + t8 + 4);
#pragma unroll
      for (int m = 0; m < 4; m++) dsp |= (((h0 >> (8 * m + 1)) & 1u) << m) | (((h1 >> (8 * m + 1)) & 1u) << (m + 4));
    }
  } else {
#pragma unroll
    for (int m = 0; m < 8; m++) {
      const int64_t t = t8 + m;
      const bool in = t >= base && t < end;
      vv[m] = in ? G.tv[t] : 0;
      if (use_e && in && (W.has_dep[t] & 2)) dsp |= 1u << m;
    }
  }
  if (use_e) {
    // The tile's own-anchor tasks land in ONE contiguous stretch of the distro's segment, [tile_sum[tile], + sum of e over
    // the tile), with holes where displaced tasks will be put by k_gplace_disp.  They are staged in shared memory and
    // the stretch is written out whole (holes included: k_gplace_disp runs later and fills them): 4-byte stores
    // straight from registers cost a sector each (8.6 M sectors for 1.2 M sectors of payload).
    constexpr int kStage = 3072;
    __shared__ uint32_t st_lo[kStage], st_ix[kStage], st_hi[kStage];
    __shared__ uint32_t s_total;
    const uint32_t p_tile = G.tile_sum[tile];
    if (tid == 255) s_total = run + sum - p_tile;  // `run` is this thread's exclusive offset: the last thread knows the tile's total
    uint32_t ps[8];
#pragma unroll
    for (int m = 0; m < 8; m++) { ps[m] = run; run += ev[m]; }
    if (interior) {
      *reinterpret_cast<uint4*>(G.e + t8) = make_uint4(ps[0], ps[1], ps[2], ps[3]);
      *reinterpret_cast<uint4*>(G.e + t8 + 4) = make_uint4(ps[4], ps[5], ps[6], ps[7]);
    } else {
#pragma unroll
      for (int m = 0; m < 8; m++) { const int64_t t = t8 + m; if (t >= base && t < end) G.e[t] = ps[m]; }
    }
    __syncthreads();
    const uint32_t total = s_total;
    const bool staged = total <= uint32_t(kStage);  // block-uniform
#pragma unroll
    for (int m = 0; m < 8; m++) {
      const int64_t t = t8 + m;
      if (t >= base && t < end && !((dsp >> m) & 1u)) {
        if (staged) {
          const unsigned long long key = vmax_ord - ord_i64(vv[m]);
          const uint32_t q = ps[m] - p_tile;
          st_lo[q] = uint32_t(key); st_ix[q] = uint32_t(t - base);
          if (wide) st_hi[q] = uint32_t(key >> 32);
        } else {
          gen_put(G, base, ps[m], vmax_ord, wide, vv[m], uint32_t(t - base));
        }
      }
    }
    if (staged) {
      __syncthreads();
      uint32_t* dlo = G.key_lo[0] + base + p_tile;
      uint32_t* dix = G.idx[0] + base + p_tile;
      uint32_t* dhi = G.key_hi[0] + base + p_tile;
      for (uint32_t q = tid; q < total; q += 256) {
        dlo[q] = st_lo[q]; dix[q] = st_ix[q];
        if (wide) dhi[q] = st_hi[q];
      }
    }
  } else if (interior) {  // identity placement: position base + (t - base) = t, and t8 is a multiple of four -> 128-bit stores
    uint32_t kl[8], kh[8];
#pragma unroll
    for (int m = 0; m < 8; m++) {
      const unsigned long long key = vmax_ord - ord_i64(vv[m]);
      kl[m] = uint32_t(key); kh[m] = uint32_t(key >> 32);
    }
    const uint32_t p0 = uint32_t(t8 - base);
    *reinterpret_cast<uint4*>(G.key_lo[0] + t8) = make_uint4(kl[0], kl[1], kl[2], kl[3]);
    *reinterpret_cast<uint4*>(G.key_lo[0] + t8 + 4) = make_uint4(kl[4], kl[5], kl[6], kl[7]);
    *reinterpret_cast<uint4*>(G.idx[0] + t8) = make_uint4(p0, p0 + 1, p0 + 2, p0 + 3);
    *reinterpret_cast<uint4*>(G.idx[0] + t8 + 4) = make_uint4(p0 + 4, p0 + 5, p0 + 6, p0 + 7);
    if (wide) {
      *reinterpret_cast<uint4*>(G.key_hi[0] + t8) = make_uint4(kh[0], kh[1], kh[2], kh[3]);
      *reinterpret_cast<uint4*>(G.key_hi[0] + t8 + 4) = make_uint4(kh[4], kh[5], kh[6], kh[7]);
    }
  } else {
#pragma unroll
    for (int m = 0; m < 8; m++) {
      const int64_t t = t8 + m;
      if (t >= base && t < end) gen_put(G, base, uint32_t(t - base), vmax_ord, wide, vv[m], uint32_t(t - base));
    }
  }
}

// Displaced work-list tasks: position = run start of the anchor + number of tasks emitted from the same unit with a smaller rank.
__global__ void __launch_bounds__(256) k_gplace_disp(DTasks T, DDistros D, DWork W, DGen G) {
  const unsigned int n = *G.ccount;
  for (unsigned int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
  const uint32_t t = G.clist[k];
  if (!(W.has_dep[t] & 2)) continue;
  const int d = G.clist_d[k];
  const int64_t base = D.task_off[d];
  const uint4 tie = G.tie[t];
  const uint32_t a = tie.x, myrk = tie.y, slot = tie.z;
  uint32_t pos = G.e[base + a];
  const uint32_t cnt = W.unit_n[slot];
  if (cnt <= 64) {
    pos += __popcll(W.unit_mask[slot] & ((1ull << myrk) - 1ull));
  } else {
    const URec* run = G.rec + W.head[slot];
    for (uint32_t i = 0; i < cnt; i++) {
      const uint4 tq = G.tie[base + rec_li(rec_load(run + i))];
      if (tq.z == slot && tq.y < myrk) pos++;
    }
  }
  gen_put(G, base, pos, G.vmm[2 * d], gen_bits(G, d) > 32, G.tv[t], uint32_t(int64_t(t) - base));
  }
}

__device__ __forceinline__ bool gen_tile(const DDistros& D, const DGen& G, int tile, int j, int* d_out, int64_t* seg, int64_t* lo,
                                         int* cnt, bool* wide) {
  const int d = G.tile_distro[tile];
  const int bits = gen_bits(G, d);
  if (j >= gen_npass(bits)) return false;
  const int64_t base = D.task_off[d], end = D.task_off[d + 1];
  const int64_t a = max(G.tile_start[tile], base), b = min(G.tile_start[tile] + kGTile, end);
  *d_out = d; *seg = base; *lo = a; *cnt = int(b - a); *wide = bits > 32;
  return true;
}

__global__ void __launch_bounds__(256) k_ghist(int j, DDistros D, DGen G) {
  if (j >= *G.maxpass) return;
  int d, cnt; int64_t seg, lo; bool wide;
  const int tile = int(blockIdx.x + G.tile0);
  if (!gen_tile(D, G, tile, j, &d, &seg, &lo, &cnt, &wide)) return;
  const uint32_t* src = (j < 4 ? G.key_lo[j & 1] : G.key_hi[j & 1]) + lo;
  const int shift = 8 * (j & 3);
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < cnt; i += 256) atomicAdd(&h[(src[i] >> shift) & 255u], 1u);
  __syncthreads();
  G.tile_hist[int64_t(tile) * 256 + threadIdx.x] = h[threadIdx.x];
}

// Offsets of every (tile, digit) counter of one distro: exclusive over the tiles of a digit, then over the digits
// (four thread groups split the tiles, eight independent loads in flight per thread).
__global__ void __launch_bounds__(1024) k_gdscan(int j, const int32_t* __restrict__ general_list, DGen G) {
  if (j >= *G.maxpass) return;
  const int d = general_list[blockIdx.x];
  if (j >= gen_npass(gen_bits(G, d))) return;
  const int dg = threadIdx.x & 255, grp = threadIdx.x >> 8;
  const int64_t t0 = G.dtile_off[d], nt = G.dtile_off[d + 1] - t0;
  const int64_t per = (nt + 3) / 4;
  const int64_t a = t0 + (grp * per < nt ? grp * per : nt), b = t0 + ((grp + 1) * per < nt ? (grp + 1) * per : nt);
  uint32_t* h = G.tile_hist + dg;
  uint32_t sum = 0;
  int64_t tile = a;
  for (; tile + 8 <= b; tile += 8) {
    uint32_t x[8];
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = h[(tile + k) * 256];
#pragma unroll
    for (int k = 0; k < 8; k++) sum += x[k];
  }
  for (; tile < b; tile++) sum += h[tile * 256];
  __shared__ uint32_t part[4][256];
  __shared__ uint32_t s[256];
  part[grp][dg] = sum;
  __syncthreads();
  const uint32_t total = part[0][dg] + part[1][dg] + part[2][dg] + part[3][dg];
  if (grp == 0) s[dg] = total;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    uint32_t v = 0;
    if (grp == 0 && dg >= o) v = s[dg - o];
    __syncthreads();
    if (grp == 0) s[dg] += v;
    __syncthreads();
  }
  uint32_t run = s[dg] - total;
  for (int g = 0; g < grp; g++) run += part[g][dg];
  tile = a;
  for (; tile + 8 <= b; tile += 8) {
    uint32_t x[8];
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = h[(tile + k) * 256];
#pragma unroll
    for (int k = 0; k < 8; k++) { h[(tile + k) * 256] = run; run += x[k]; }
  }
  for (; tile < b; tile++) { const uint32_t x = h[tile * 256]; h[tile * 256] = run; run += x; }
}

// Warp w ranks chunks 8w .. 8w+7 of the tile in order (stability): one MATCH.ANY per chunk, the group's first lane adds
// the group size to the warp's digit counter and gets back the count of equal digits in the warp's earlier chunks (as in
// k_plan_cta).  The tile is then sorted by digit IN SHARED MEMORY and written out in that order: consecutive threads
// write consecutive addresses inside a digit's run, so a run costs its sectors once -- scattering straight from
// registers put nearly every 4-byte store in a sector of its own (8.1 M sectors for 9.6 M stores, L2-write bound).
template <bool WIDE>
__device__ __forceinline__ void gscatter_tile(int j, const DGen& G, int tile, int64_t seg, int64_t lo, int cnt, uint32_t (*wcnt)[256],
                                              uint32_t* s_lo, uint32_t* s_ix, uint32_t* s_hi, int32_t* s_delta, uint32_t* s_wsum) {
  constexpr bool wide = WIDE;
  const int sb = j & 1, db = sb ^ 1;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int w = 0; w < 8; w++) wcnt[w][tid] = 0u;
  __syncthreads();
  const unsigned lt = (1u << lane) - 1u;
  const int shift = 8 * (j & 3);
  const bool use_hi = j >= 4;
  const uint32_t* src_lo = G.key_lo[sb] + lo;
  const uint32_t* src_hi = G.key_hi[sb] + lo;
  const uint32_t* src_ix = G.idx[sb] + lo;
  uint32_t kl[8], kh[8], ix[8], dg[8], rk[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {  // all loads first
    const int i = (warp * 8 + k) * 32 + lane;
    const bool ok = i < cnt;
    kl[k] = ok ? src_lo[i] : 0u;
    kh[k] = (ok && wide) ? src_hi[i] : 0u;
    ix[k] = ok ? src_ix[i] : 0u;
  }
  // all eight MATCHes, then the eight leader atomics back to back (one warp's shared-memory atomics execute in issue
  // order: chunk k+1's returned count includes chunk k's add), then the shuffles: the atomic round trips overlap
  unsigned peers[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const int i = (warp * 8 + k) * 32 + lane;
    dg[k] = i < cnt ? (((use_hi ? kh[k] : kl[k]) >> shift) & 255u) : 256u;
    peers[k] = __match_any_sync(0xffffffffu, dg[k]);
  }
#pragma unroll
  for (int k = 0; k < 8; k++) {
    rk[k] = 0;
    if (dg[k] < 256u && (peers[k] & lt) == 0u) rk[k] = atomicAdd(&wcnt[warp][dg[k]], uint32_t(__popc(peers[k])));
  }
#pragma unroll
  for (int k = 0; k < 8; k++) rk[k] = __shfl_sync(0xffffffffu, rk[k], __ffs(peers[k]) - 1) + uint32_t(__popc(peers[k] & lt));
  __syncthreads();
  {  // thread = digit: the eight warp counters become offsets inside the digit; the digit totals are scanned over the block
    uint32_t x[8], tot = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) { x[w] = wcnt[w][tid]; tot += x[w]; }
    uint32_t inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) s_wsum[warp] = inc;
    __syncthreads();
    uint32_t before = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) before += w < warp ? s_wsum[w] : 0u;
    const uint32_t lbase = before + inc - tot;  // where digit `tid` starts in the sorted tile
    s_delta[tid] = int32_t(G.tile_hist[int64_t(tile) * 256 + tid]) - int32_t(lbase);
    uint32_t run = lbase;
#pragma unroll
    for (int w = 0; w < 8; w++) { wcnt[w][tid] = run; run += x[w]; }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 8; k++) {
    if (dg[k] < 256u) {
      const uint32_t lp = wcnt[warp][dg[k]] + rk[k];
      s_lo[lp] = kl[k];
      s_ix[lp] = ix[k];
      if (wide) s_hi[lp] = kh[k];
    }
  }
  __syncthreads();
  uint32_t* dst_lo = G.key_lo[db] + seg;
  uint32_t* dst_hi = G.key_hi[db] + seg;
  uint32_t* dst_ix = G.idx[db] + seg;
  for (int i = tid; i < cnt; i += 256) {
    const uint32_t a = s_lo[i], h = wide ? s_hi[i] : 0u;
    const uint32_t dgt = ((use_hi ? h : a) >> shift) & 255u;
    const int64_t pos = int64_t(s_delta[dgt]) + i;
    dst_lo[pos] = a;
    dst_ix[pos] = s_ix[i];
    if (wide) dst_hi[pos] = h;
  }
}

// The key's high word travels only for distros whose value range exceeds 32 bits (a handful of registers and 8 KB of
// shared memory the common case does not pay for).
__global__ void __launch_bounds__(256, 4) k_gscatter(int j, DDistros D, DGen G) {
  if (j >= *G.maxpass) return;
  int d, cnt; int64_t seg, lo; bool wide;
  const int tile = int(blockIdx.x + G.tile0);
  if (!gen_tile(D, G, tile, j, &d, &seg, &lo, &cnt, &wide)) return;
  __shared__ uint32_t wcnt[8][256];   // per-warp digit counters, then local positions
  __shared__ uint32_t s_lo[kGTile], s_ix[kGTile], s_hi[kGTile];
  __shared__ int32_t s_delta[256];    // digit -> (offset of the digit's run in the distro) - (its offset in the sorted tile)
  __shared__ uint32_t s_wsum[8];
  if (wide) gscatter_tile<true>(j, G, tile, seg, lo, cnt, wcnt, s_lo, s_ix, s_hi, s_delta, s_wsum);
  else gscatter_tile<false>(j, G, tile, seg, lo, cnt, wcnt, s_lo, s_ix, s_hi, s_delta, s_wsum);
}

// Ranked queue out: order[] and TotalValue per rank (planner.go:467-477).
__global__ void __launch_bounds__(256) k_gemit(DDistros D, DGen G, int32_t* __restrict__ order, int64_t* __restrict__ total_value) {
  const int tile = int(blockIdx.x + G.tile0);
  const int d = G.tile_distro[tile];
  const int64_t base = D.task_off[d], end = D.task_off[d + 1];
  const int64_t lo = max(G.tile_start[tile], base), hi = min(G.tile_start[tile] + kGTile, end);
  const int bits = gen_bits(G, d);
  const int fin = gen_npass(bits) & 1;
  const bool wide = bits > 32;
  const unsigned long long vmax_ord = G.vmm[2 * d];
  for (int64_t p = lo + threadIdx.x; p < hi; p += 256) {
    unsigned long long key = G.key_lo[fin][p];
    if (wide) key |= (unsigned long long)G.key_hi[fin][p] << 32;
    order[p] = int32_t(G.idx[fin][p]);
    total_value[p] = unord_i64(vmax_ord - key);
  }
}

// ---- the persisted head (evg_run_resident_head): only the first min(length, cap) ranks of every general-path distro ----
// After k_gplace the (key, index) pairs of a distro sit in key_lo[0] / key_hi[0] / idx[0] in canonical tie order, so the
// first cap ranks of the stable sort are the pairs with the cap smallest keys, ties broken by buffer position:
//   k_hinit/k_hhist/k_hstep  segmented radix SELECT, most significant digit first: the threshold key theta, the count of
//                            keys below it and m, the number of keys equal to theta that are taken
//   k_hcount/k_gscan x2/k_hplace
//                            stable compaction of those pairs into key_lo[1] / key_hi[1] / idx[1] (the LSD sort's second
//                            buffer, unused here), at the distro's own offset
//   k_hsort<WIDE>            one CTA per distro: stable LSD radix sort of its head over the key range [0, theta], then the
//                            ranked queue + TotalValue of ranks [0, min(length, cap))
struct HeadSel {
  unsigned long long prefix;  // digits of theta fixed so far (theta after the last pass)
  uint32_t need;              // ranks still to place among the keys that match the prefix (m after the last pass)
  uint32_t below;             // keys below the prefix's range (the keys < theta after the last pass)
  int32_t gpos;               // the distro's place in the general list: its row of `hist`
  uint32_t all;               // 1: length <= cap, the head is the whole distro (theta = its largest key, no select pass)
};
struct DHead {
  HeadSel* sel;      // [D]
  uint32_t* hist;    // [general distros * 256] digit counts of the current pass
  uint32_t* eq_sum;  // [NT] keys == theta per tile, then the tile's exclusive offset (G.tile_sum does the same for keys < theta)
  int32_t cap;
};
constexpr int kHeadCap = EVG_PERSISTED_QUEUE_CAP;
constexpr int kHsThreads = 1024, kHsWarps = kHsThreads / 32;
constexpr int kHsChunks = (kHeadCap + kHsThreads - 1) / kHsThreads;  // 32-item chunks per warp
static_assert(kHeadCap < 65536, "head positions are 16-bit");

__device__ __forceinline__ unsigned long long gen_key(const DGen& G, int b, int64_t p, bool wide) {
  unsigned long long k = G.key_lo[b][p];
  if (wide) k |= (unsigned long long)G.key_hi[b][p] << 32;
  return k;
}

__global__ void __launch_bounds__(256) k_hinit(DDistros D, DGen G, DHead H, const int32_t* __restrict__ general_list) {
  H.hist[blockIdx.x * 256 + threadIdx.x] = 0u;
  if (threadIdx.x == 0) {
    const int d = general_list[blockIdx.x];
    const int64_t n = D.task_off[d + 1] - D.task_off[d];
    HeadSel s;
    s.all = n <= H.cap ? 1u : 0u;
    s.prefix = s.all ? G.vmm[2 * d] - G.vmm[2 * d + 1] : 0ull;
    s.need = uint32_t(min(n, int64_t(H.cap))); s.below = 0u; s.gpos = int32_t(blockIdx.x);
    H.sel[d] = s;
  }
}

// The eight keys of slots t8 .. t8+7 (t8 a multiple of four: 128-bit loads inside [lo, hi)); bit m of the result: slot
// t8+m holds a key of the distro.
__device__ __forceinline__ uint32_t head_keys8(const DGen& G, int64_t t8, int64_t lo, int64_t hi, bool wide, unsigned long long key[8]) {
  if (t8 >= lo && t8 + 7 < hi) {
    const uint4 a = *reinterpret_cast<const uint4*>(G.key_lo[0] + t8), b = *reinterpret_cast<const uint4*>(G.key_lo[0] + t8 + 4);
    const uint32_t l[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t u[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (wide) {
      const uint4 c = *reinterpret_cast<const uint4*>(G.key_hi[0] + t8), e = *reinterpret_cast<const uint4*>(G.key_hi[0] + t8 + 4);
      u[0] = c.x; u[1] = c.y; u[2] = c.z; u[3] = c.w; u[4] = e.x; u[5] = e.y; u[6] = e.z; u[7] = e.w;
    }
#pragma unroll
    for (int m = 0; m < 8; m++) key[m] = l[m] | ((unsigned long long)u[m] << 32);
    return 0xFFu;
  }
  uint32_t ok = 0;
#pragma unroll
  for (int m = 0; m < 8; m++) {
    const int64_t p = t8 + m;
    const bool in = p >= lo && p < hi;
    key[m] = in ? gen_key(G, 0, p, wide) : 0ull;
    ok |= uint32_t(in) << m;
  }
  return ok;
}

// Pass j (most significant digit first): per tile, the digits of the keys that match the prefix fixed so far.  Thread q
// counts its 8 consecutive keys run by run: skewed values put most keys of a tile in a handful of top digits, and one
// shared atomic per key would serialise on those few counters.
__global__ void __launch_bounds__(256) k_hhist(int j, DDistros D, DGen G, DHead H) {
  if (j >= *G.maxpass) return;
  int d, cnt; int64_t seg, lo; bool wide;
  const int tile = int(blockIdx.x + G.tile0);
  if (!gen_tile(D, G, tile, j, &d, &seg, &lo, &cnt, &wide)) return;
  const int shift = 8 * (gen_npass(gen_bits(G, d)) - 1 - j);
  const HeadSel s = H.sel[d];
  if (s.all) return;
  const unsigned long long want = j == 0 ? 0ull : s.prefix >> (shift + 8);
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long key[8];
  const uint32_t ok = head_keys8(G, G.tile_start[tile] + 8 * int64_t(threadIdx.x), lo, lo + cnt, wide, key);
  uint32_t run_dg = 256u, run_n = 0;
#pragma unroll
  for (int m = 0; m < 8; m++) {
    const bool take = ((ok >> m) & 1u) && (j == 0 || (key[m] >> (shift + 8)) == want);
    const uint32_t dg = take ? uint32_t(key[m] >> shift) & 255u : 256u;
    if (dg != run_dg && dg < 256u) {
      if (run_n) atomicAdd(&h[run_dg], run_n);
      run_dg = dg; run_n = 0;
    }
    run_n += take;
  }
  if (run_n) atomicAdd(&h[run_dg], run_n);
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&H.hist[s.gpos * 256 + threadIdx.x], h[threadIdx.x]);
}

// Pass j, one block per distro, thread = digit: the digit at which the running count reaches `need` extends the prefix.
__global__ void __launch_bounds__(256) k_hstep(int j, const int32_t* __restrict__ general_list, DGen G, DHead H) {
  if (j >= *G.maxpass) return;
  const int d = general_list[blockIdx.x];
  const int np = gen_npass(gen_bits(G, d));
  if (j >= np || H.sel[d].all) return;
  const int shift = 8 * (np - 1 - j);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t* h = H.hist + blockIdx.x * 256;
  const uint32_t c = h[tid];
  h[tid] = 0u;  // ready for the next pass
  const uint32_t need = H.sel[d].need;
  __shared__ uint32_t sw[8];
  uint32_t inc = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
  if (lane == 31) sw[warp] = inc;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 8; w++) inc += w < warp ? sw[w] : 0u;
  const uint32_t excl = inc - c;
  if (excl < need && need <= inc) {  // exactly one digit: the keys matching the prefix number at least `need`
    HeadSel& s = H.sel[d];
    s.prefix |= (unsigned long long)tid << shift;
    s.below += excl;
    s.need = need - excl;
  }
}

__device__ __forceinline__ bool head_tile(const DDistros& D, const DGen& G, int tile, int* d, int64_t* base, int64_t* lo, int64_t* hi) {
  *d = G.tile_distro[tile];
  *base = D.task_off[*d];
  *lo = max(G.tile_start[tile], *base);
  *hi = min(G.tile_start[tile] + kGTile, D.task_off[*d + 1]);
  return gen_bits(G, *d) > 32;
}

// Per tile: keys < theta into G.tile_sum, keys == theta into H.eq_sum (k_gscan turns both into offsets).
__global__ void __launch_bounds__(256) k_hcount(DDistros D, DGen G, DHead H) {
  const int tile = int(blockIdx.x + G.tile0);
  int d; int64_t base, lo, hi;
  const bool wide = head_tile(D, G, tile, &d, &base, &lo, &hi);
  const unsigned long long theta = H.sel[d].prefix;
  uint32_t lt = 0, eq = 0;
  for (int64_t p = lo + threadIdx.x; p < hi; p += 256) {
    const unsigned long long key = gen_key(G, 0, p, wide);
    lt += key < theta;
    eq += key == theta;
  }
  lt = __reduce_add_sync(0xffffffffu, lt);
  eq = __reduce_add_sync(0xffffffffu, eq);
  __shared__ uint32_t sl[8], se[8];
  if ((threadIdx.x & 31) == 0) { sl[threadIdx.x >> 5] = lt; se[threadIdx.x >> 5] = eq; }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t a = 0, b = 0;
    for (int w = 0; w < 8; w++) { a += sl[w]; b += se[w]; }
    G.tile_sum[tile] = a;
    H.eq_sum[tile] = b;
  }
}

// Per tile, thread q owns 8 consecutive slots (buffer order = thread order): a pair is taken when its key is below theta
// or it is one of the first m keys equal to theta; its head position is the number of taken pairs before it.
__global__ void __launch_bounds__(256) k_hplace(DDistros D, DGen G, DHead H) {
  const int tile = int(blockIdx.x + G.tile0);
  int d; int64_t base, lo, hi;
  const bool wide = head_tile(D, G, tile, &d, &base, &lo, &hi);
  const HeadSel s = H.sel[d];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t t8 = G.tile_start[tile] + 8 * int64_t(tid);
  unsigned long long key[8];
  const uint32_t ok = head_keys8(G, t8, lo, hi, wide, key);
  uint32_t n_lt = 0, n_eq = 0;
#pragma unroll
  for (int m = 0; m < 8; m++) {
    n_lt += ((ok >> m) & 1u) && key[m] < s.prefix;
    n_eq += ((ok >> m) & 1u) && key[m] == s.prefix;
  }
  const uint32_t mine = n_lt | (n_eq << 16);  // at most 2048 of each per tile
  uint32_t inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += x; }
  __shared__ uint32_t sw[8];
  if (lane == 31) sw[warp] = inc;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 8; w++) inc += w < warp ? sw[w] : 0u;
  const uint32_t ex = inc - mine;
  uint32_t plt = G.tile_sum[tile] + (ex & 0xFFFFu), peq = H.eq_sum[tile] + (ex >> 16);
#pragma unroll
  for (int m = 0; m < 8; m++) {
    const int64_t p = t8 + m;
    if (!((ok >> m) & 1u)) continue;
    uint32_t pos;
    if (key[m] < s.prefix) pos = plt++ + min(peq, s.need);
    else if (key[m] == s.prefix && peq < s.need) pos = plt + peq++;
    else continue;
    G.key_lo[1][base + pos] = uint32_t(key[m]);
    if (wide) G.key_hi[1][base + pos] = uint32_t(key[m] >> 32);
    G.idx[1][base + pos] = G.idx[0][p];
  }
}

// One CTA per general-path distro whose head keys need (WIDE) or do not need a second word.  The head's positions are
// sorted, not the pairs: per pass, warp w ranks its contiguous slice of the current permutation chunk by chunk (MATCH
// on the digit, the group's first lane bumps the warp's digit counter), thread = digit turns the warp counters into
// offsets, and the positions are scattered into the other permutation.
template <bool WIDE>
__global__ void __launch_bounds__(kHsThreads, 1) k_hsort(const int32_t* __restrict__ general_list, DDistros D, DGen G, DHead H,
                                                     int32_t* __restrict__ order, int64_t* __restrict__ total_value) {
  const int d = general_list[blockIdx.x];
  const HeadSel s = H.sel[d];
  const int bits = s.prefix == 0ull ? 0 : 64 - __clzll((long long)s.prefix);  // head keys lie in [0, theta]
  if ((bits > 32) != WIDE) return;
  const int np = (bits + 7) >> 3;
  const uint32_t k = s.below + s.need;
  const int64_t base = D.task_off[d];
  extern __shared__ __align__(16) unsigned char hs_smem[];
  uint32_t (*wcnt)[256] = reinterpret_cast<uint32_t (*)[256]>(hs_smem);
  uint32_t* s_lo = reinterpret_cast<uint32_t*>(hs_smem + sizeof(uint32_t) * kHsWarps * 256);
  uint32_t* s_hi = s_lo + kHeadCap;  // WIDE only
  uint16_t* perm0 = reinterpret_cast<uint16_t*>(s_lo + (WIDE ? 2 : 1) * kHeadCap);
  uint16_t* perm1 = perm0 + kHeadCap;
  __shared__ uint32_t s_wsum[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint32_t i = tid; i < k; i += kHsThreads) {
    s_lo[i] = G.key_lo[1][base + i];
    if (WIDE) s_hi[i] = G.key_hi[1][base + i];
    perm0[i] = uint16_t(i);
  }
  const unsigned lt = (1u << lane) - 1u;
  uint16_t* cur = perm0;
  uint16_t* nxt = perm1;
  for (int pass = 0; pass < np; pass++) {
    const int sh = (8 * pass) & 31;
    const uint32_t* src = (WIDE && pass >= 4) ? s_hi : s_lo;
    for (int q = tid; q < kHsWarps * 256; q += kHsThreads) wcnt[q >> 8][q & 255] = 0u;
    __syncthreads();
    uint32_t dr[kHsChunks];  // digit (256 = no item) | rank inside the warp's slice << 9
#pragma unroll
    for (int c = 0; c < kHsChunks; c++) {
      const uint32_t i = uint32_t((warp * kHsChunks + c) * 32 + lane);
      const uint32_t dg = i < k ? (src[cur[i]] >> sh) & 255u : 256u;
      const unsigned peers = __match_any_sync(0xffffffffu, dg);
      const int lead = __ffs(peers) - 1;
      uint32_t b = 0;
      if (lane == lead && dg < 256u) { b = wcnt[warp][dg]; wcnt[warp][dg] = b + uint32_t(__popc(peers)); }
      b = __shfl_sync(0xffffffffu, b, lead) + uint32_t(__popc(peers & lt));
      dr[c] = dg | (b << 9);
      __syncwarp();
    }
    __syncthreads();
    uint32_t tot = 0;
    if (tid < 256) {
#pragma unroll
      for (int w = 0; w < kHsWarps; w++) tot += wcnt[w][tid];
      uint32_t inc = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
      if (lane == 31) s_wsum[warp] = inc;
      tot = inc - tot;  // exclusive inside the warp
    }
    __syncthreads();
    if (tid < 256) {
      uint32_t run = tot;
      for (int w = 0; w < warp; w++) run += s_wsum[w];
#pragma unroll
      for (int w = 0; w < kHsWarps; w++) { const uint32_t y = wcnt[w][tid]; wcnt[w][tid] = run; run += y; }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < kHsChunks; c++) {
      const uint32_t dg = dr[c] & 511u;
      if (dg < 256u) nxt[wcnt[warp][dg] + (dr[c] >> 9)] = cur[(warp * kHsChunks + c) * 32 + lane];
    }
    __syncthreads();
    uint16_t* t = cur; cur = nxt; nxt = t;
  }
  __syncthreads();
  const unsigned long long vmax_ord = G.vmm[2 * d];
  for (uint32_t r = tid; r < k; r += kHsThreads) {
    const uint32_t p = cur[r];
    unsigned long long key = s_lo[p];
    if (WIDE) key |= (unsigned long long)s_hi[p] << 32;
    order[base + r] = int32_t(G.idx[1][base + p]);
    total_value[base + r] = unord_i64(vmax_ord - key);
  }
}
template <bool WIDE>
constexpr size_t hsort_smem() { return sizeof(uint32_t) * kHsWarps * 256 + sizeof(uint32_t) * kHeadCap * (WIDE ? 2 : 1) + sizeof(uint16_t) * 2 * kHeadCap; }

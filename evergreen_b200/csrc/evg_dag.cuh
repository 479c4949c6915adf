// evg_dag.cuh -- the DAG dispatcher's rebuild (SURVEY.md §8 f.3): what consumes the persisted queue.
//
// Reference: basicCachedDAGDispatcherImpl.rebuild (model/task_queue_service_dependency.go:153-252): one node per
// TaskQueueItem (queueIndex = queue position), an edge dependency -> item for every dependency that is itself in the
// queue, topo.SortStabilized with ties ordered by queueIndex, and the task groups bucketed by composite id with each
// bucket stably sorted by GroupIndex.
//
// topo.SortStabilized (gonum v0.17.0, not vendored; restated in oracle/oracle_dag.py) is Tarjan's algorithm over
// nodes and successors taken in DESCENDING queueIndex, its emission order reversed: for a DAG, the reverse
// post-order of that depth-first search.  A lexicographic DFS order is inherently sequential (the problem is
// P-complete), and a persisted queue holds at most 10 000 items, so one THREAD (lane 0 of a warp of its own) walks one distro's graph -- successor
// lists built by a counting pass, an explicit call stack, everything in that distro's slice of global scratch -- and
// the batch's parallelism is across distros.  The task-group buckets are a segmented stable merge sort by
// (group id, GroupIndex): one thread per item and pass.
#pragma once

struct DDag {
  int64_t n, n_deps;
  int32_t n_distros;
  const int64_t* item_off;     // [D+1]
  const int64_t* dep_off;      // [n+1]
  const int32_t* dep_item;     // [n_deps] distro-local item of the dependency, -1 = not in the queue
  const int32_t* group_id;     // [n] distro-local dense composite group id, -1 = no group
  const int32_t* group_index;  // [n]
  int32_t* succ_off;           // [n + D] per distro n_d + 1 entries at item_off[d] + d
  int32_t* succ;               // [n_deps]
  int32_t* index;              // [n]
  int32_t* low;                // [n]
  int32_t* stack;              // [n] Tarjan's node stack
  int32_t* cs_node;            // [n] call stack: node ...
  int32_t* cs_pos;             // [n] ... and its next successor cursor
  int32_t* emit;               // [n] components in emission order
  uint8_t* on_stack;           // [n]
};

__global__ void __launch_bounds__(64) k_dag_topo(DDag X, int32_t* __restrict__ sorted, int32_t* __restrict__ n_sorted,
                                                 int32_t* __restrict__ n_cycles) {
  // one WARP per queue, its first lane walking: 32 walks in one warp diverge at every step and run one after the other
  // (measured: 200 queues of 10 000 items 216 ms with a thread per queue)
  const int d = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (d >= X.n_distros || (threadIdx.x & 31) != 0) return;
  const int64_t base = X.item_off[d];
  const int n = int(X.item_off[d + 1] - base);
  const int64_t ebase = n > 0 ? X.dep_off[base] : 0;
  int32_t* so = X.succ_off + base + d;
  int32_t* succ = X.succ + ebase;
  int32_t* index = X.index + base; int32_t* low = X.low + base; int32_t* stack = X.stack + base;
  int32_t* cs_node = X.cs_node + base; int32_t* cs_pos = X.cs_pos + base; int32_t* emit = X.emit + base;
  uint8_t* on_stack = X.on_stack + base;
  // successor lists: count, prefix, fill in ascending item order (so every list is ascending)
  for (int i = 0; i <= n; i++) so[i] = 0;
  for (int k = 0; k < n; k++)
    for (int64_t e = X.dep_off[base + k]; e < X.dep_off[base + k + 1]; e++) {
      const int32_t j = X.dep_item[e];
      if (j >= 0 && j < n) so[j + 1]++;  // "the depend_on task is not in the DAG so we don't need an edge" (:123-126)
    }
  for (int i = 0; i < n; i++) { so[i + 1] += so[i]; low[i] = so[i]; index[i] = 0; on_stack[i] = 0; }
  for (int k = 0; k < n; k++)
    for (int64_t e = X.dep_off[base + k]; e < X.dep_off[base + k + 1]; e++) {
      const int32_t j = X.dep_item[e];
      if (j >= 0 && j < n) succ[low[j]++] = k;
    }
  // Tarjan, nodes and successors in descending queueIndex (tarjanSCCstabilized: order, then reverse)
  int counter = 0, sp = 0, tsp = 0, n_emit = 0, cycles = 0;
  for (int root = n - 1; root >= 0; root--) {
    if (index[root] != 0) continue;
    index[root] = low[root] = ++counter; stack[tsp++] = root; on_stack[root] = 1;
    cs_node[sp] = root; cs_pos[sp] = so[root + 1] - 1; sp++;
    while (sp > 0) {
      const int v = cs_node[sp - 1];
      const int p = cs_pos[sp - 1];
      if (p >= so[v]) {
        const int w = succ[p];
        cs_pos[sp - 1] = p - 1;
        if (p + 1 < so[v + 1] && succ[p + 1] == w) continue;  // a parallel line: From() yields the neighbour once
        if (index[w] == 0) {
          index[w] = low[w] = ++counter; stack[tsp++] = w; on_stack[w] = 1;
          cs_node[sp] = w; cs_pos[sp] = so[w + 1] - 1; sp++;
        } else if (on_stack[w]) {
          low[v] = min(low[v], index[w]);
        }
      } else {
        if (low[v] == index[v]) {  // v roots a component: pop it
          int cnt = 0, w;
          do { w = stack[--tsp]; on_stack[w] = 0; cnt++; } while (w != v);
          if (cnt == 1) emit[n_emit++] = v;
          else { emit[n_emit++] = -1; cycles++; }  // sortedFrom: one nil per cyclic component
        }
        sp--;
        if (sp > 0) { const int u = cs_node[sp - 1]; low[u] = min(low[u], low[v]); }
      }
    }
  }
  for (int i = 0; i < n_emit; i++) sorted[base + i] = emit[n_emit - 1 - i];  // ordered.Reverse
  for (int i = n_emit; i < n; i++) sorted[base + i] = -2;                    // unused tail (members of cycles)
  n_sorted[d] = n_emit;
  n_cycles[d] = cycles;
}

// key of an item for the task-group buckets: (group id, GroupIndex); items without a group sort last
__device__ __forceinline__ unsigned long long dag_group_key(const DDag& X, int64_t g) {
  const int32_t gid = X.group_id[g];
  if (gid < 0) return ~0ull;
  return ((unsigned long long)uint32_t(gid) << 32) | (unsigned long long)(uint32_t(X.group_index[g]) ^ 0x80000000u);
}
__global__ void __launch_bounds__(256) k_dag_group_init(DDag X, int32_t* __restrict__ idx) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= X.n) return;
  const int d = find_distro(X.item_off, 0, X.n_distros - 1, p);
  idx[p] = int32_t(p - X.item_off[d]);
}
// one pass of a segmented STABLE merge sort (runs of length L inside each distro's items)
__global__ void __launch_bounds__(256) k_dag_group_pass(DDag X, const int32_t* __restrict__ src, int32_t* __restrict__ dst, int64_t L) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= X.n) return;
  const int d = find_distro(X.item_off, 0, X.n_distros - 1, p);
  const int64_t base = X.item_off[d], n = X.item_off[d + 1] - base;
  const int64_t q = p - base;
  const int32_t me = src[p];
  if (L >= n) { dst[p] = me; return; }
  const int64_t r = q / L, own0 = r * L;
  int64_t s0, s1;
  if ((r & 1) == 0) { s0 = own0 + L; s1 = min(s0 + L, n); } else { s0 = own0 - L; s1 = own0; }
  if (s0 >= n) { dst[p] = me; return; }
  const unsigned long long km = dag_group_key(X, base + me);
  int64_t lo = s0, hi = s1;
  if ((r & 1) == 0) {  // left run: sibling elements strictly smaller go first
    while (lo < hi) { const int64_t m = (lo + hi) >> 1; if (dag_group_key(X, base + src[base + m]) < km) lo = m + 1; else hi = m; }
    dst[base + own0 + (q - own0) + (lo - s0)] = me;
  } else {             // right run: sibling elements smaller or equal go first (stability)
    while (lo < hi) { const int64_t m = (lo + hi) >> 1; if (dag_group_key(X, base + src[base + m]) <= km) lo = m + 1; else hi = m; }
    dst[base + s0 + (lo - s0) + (q - own0)] = me;
  }
}
// bucket boundaries: unit_off[group_off[d] + g] = first position (distro-local) of group g in the sorted items;
// the entry after a distro's last group is written by the host from grouped[d] (items that have a group); the entries of
// groups no item is in keep the -1 they were set to, and the host gives them the start of the next group
__global__ void __launch_bounds__(256) k_dag_units(DDag X, const int32_t* __restrict__ order, const int64_t* __restrict__ group_off,
                                                   int32_t* __restrict__ unit_off, int32_t* __restrict__ grouped) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= X.n) return;
  const int d = find_distro(X.item_off, 0, X.n_distros - 1, p);
  const int64_t base = X.item_off[d];
  const int32_t g = X.group_id[base + order[p]];
  const int32_t gprev = p > base ? X.group_id[base + order[p - 1]] : -2;
  if (g >= 0 && g != gprev) unit_off[group_off[d] + d + g] = int32_t(p - base);
  if (g < 0 && (p == base || gprev >= 0)) grouped[d] = int32_t(p - base);  // first ungrouped item
}

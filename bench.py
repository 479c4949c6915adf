#!/usr/bin/env python3
"""bench.py -- the scheduler hot path on synthetic ticks of BASELINE.json's shapes.

  python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU algorithm on the host cores)
  python bench.py ... --dump-outputs DIR                   (also writes the last timed tick's outputs, see dump_outputs)

A "step" is one scheduler tick: tunable planner + DistroQueueInfo + utilization host allocator over every distro of
the workload.  Headline workload (per GPU): configs[2] read per distro -- distro queues of 100 000 tasks each, Zipf
priorities, 5 % of tasks with an unmet dependency on another queued task (DispatcherSettings "revised-with-
dependencies"), 10 % in task groups -- as many of the 10 000 distros as fit HBM next to the work buffers
(--distros, default 4000 = 4e8 tasks, 24 GB of columns).  A block of --block distros comes from evergreen_b200.synth
(splitmix64, the same generator the tests use) and is tiled on the device with a per-tile clock shift, so no two
tiles are equal and nothing is re-read from L2.
`value` = tasks ranked per second with the tick's inputs resident in HBM (evg_upload_device + evg_run_resident);
`e2e`   = the same tick shape through the one-shot C-ABI call (evg_plan_and_alloc_batch: pinned HOST columns in, host
          results out, H2D and D2H inside the timed region) on --e2e-distros distros;
`shapes`= the other BASELINE configs through the resident tick in the same process, each with its own roofline
          figures (configs[1] carries the on-chip planner's kernel-level numbers);
`cpu_baseline` / --impl reference = oracle/evg_oracle.cpp (C++ restatement of the Go path, "port": the image has
          no Go toolchain) on the usable host cores over the first --ref-sample distros of the same block.
N > 1: one process per GPU (torchrun), distros sharded whole by LPT, one NCCL all-gather of the per-distro result
vector per step on a second stream, max-over-ranks timing; weak scaling (each GPU owns --distros distros).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tasks scheduled/sec over N distros; host-allocator decisions/sec at 1/2/4/8 GPU"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


HEADLINE = "configs[2] per-distro reading"


def headline_block(rank: int, n_block: int, per: int):
    """The generated block: n_block distros x `per` tasks in configs[2]'s mix (synth.config(3, each=True)'s arguments)."""
    from evergreen_b200 import synth
    return synth.make(np.full(n_block, per, dtype=np.int64), synth.SEED_BASE + 3 + 1000 * rank,
                      name=f"C3 block: {n_block} distros x {per} tasks, Zipf priorities, 5% unmet deps",
                      zipf_priority=True, unmet_dep_frac=0.05, met_dep_frac=0.02, includes_dependencies=True, n_hosts=2 * n_block)


def tile_tables(w, reps: int):
    """Distro / host tables of `reps` copies of block `w` (host arrays; the task columns are tiled by tile_host /
    tile_device)."""
    from evergreen_b200.soa import DistroTable, HostSoA
    Db, Tb, Gb = w.distros.n_distros, w.n_tasks, w.distros.n_groups
    task_off = np.concatenate([[0], (w.distros.task_off[1:][None, :] + Tb * np.arange(reps)[:, None]).ravel()]).astype(np.int64)
    group_off = np.concatenate([[0], (w.distros.group_off[1:][None, :] + Gb * np.arange(reps)[:, None]).ravel()]).astype(np.int64)
    distros = DistroTable(task_off, group_off, np.tile(w.distros.cfg, reps), np.tile(w.distros.group_max_hosts, reps)).normalize()
    h = w.hosts
    Hb = h.n_hosts
    host_off = np.concatenate([[0], (h.host_off[1:][None, :] + Hb * np.arange(reps)[:, None]).ravel()]).astype(np.int64)
    hosts = HostSoA(np.tile(h.flags, reps), np.tile(h.group_id, reps), np.tile(h.expected_ns, reps), np.tile(h.std_ns, reps),
                    np.tile(h.start_ns, reps), host_off, np.tile(h.cfg, reps)).normalize()
    assert distros.n_distros == Db * reps
    return distros, hosts


SHIFT_QB, SHIFT_EXP = 10 ** 9, 10 ** 6  # tile r: activated r seconds earlier, expected r ms longer


def tile_host(w, reps: int):
    """`reps` shifted copies of block `w` as a host Workload (the e2e leg's input)."""
    from evergreen_b200 import synth
    from evergreen_b200.soa import TaskSoA
    t = w.tasks
    r = np.repeat(np.arange(reps, dtype=np.int64), w.n_tasks)
    cols = {name: np.tile(getattr(t, name), reps) for name, _ in t.COLUMNS}
    cols["queue_basis_ns"] = cols["queue_basis_ns"] - r * SHIFT_QB
    cols["expected_ns"] = cols["expected_ns"] + r * SHIFT_EXP
    dep_off = dep_idx = None
    if t.n_edges:
        dep_off = np.concatenate([(t.dep_off[:-1][None, :] + t.n_edges * np.arange(reps)[:, None]).ravel(), [t.n_edges * reps]])
        dep_idx = np.tile(t.dep_idx, reps)
    tasks = TaskSoA(*[cols[name] for name, _ in t.COLUMNS], dep_off, dep_idx).normalize()
    distros, hosts = tile_tables(w, reps)
    return synth.Workload(f"{w.name} x{reps}", w.now, tasks, distros, hosts)


def tile_device(torch, dev, w, reps: int):
    """`reps` shifted copies of block `w`'s task columns in device memory (8 padding rows each, as evg_upload_device
    asks).  Returns ({column: address}, tensors to keep alive, n_tasks, n_edges)."""
    t = w.tasks
    Tb, Eb = w.n_tasks, t.n_edges
    keep, cols = [], {}
    rr = torch.arange(reps, device=dev, dtype=torch.int64)[:, None]
    for name, _ in t.COLUMNS:
        a = getattr(t, name)
        blk = torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).to(dev)
        big = torch.zeros(reps * Tb + 8, dtype=blk.dtype, device=dev)
        v = big[: reps * Tb].view(reps, Tb)
        v.copy_(blk[None, :])
        if name == "queue_basis_ns":
            v.sub_(rr * SHIFT_QB)
        elif name == "expected_ns":
            v.add_(rr * SHIFT_EXP)
        keep.append(big)
        cols[name] = big.data_ptr()
        del blk
    if Eb:
        blk = torch.from_numpy(t.dep_off[:-1]).to(dev)
        big = torch.zeros(reps * Tb + 1 + 8, dtype=torch.int64, device=dev)
        v = big[: reps * Tb].view(reps, Tb)
        v.copy_(blk[None, :])
        v.add_(rr * Eb)
        big[reps * Tb] = reps * Eb
        keep.append(big)
        cols["dep_off"] = big.data_ptr()
        blk = torch.from_numpy(t.dep_idx).to(dev)
        big = torch.zeros(reps * Eb + 8, dtype=torch.int32, device=dev)
        big[: reps * Eb].view(reps, Eb).copy_(blk[None, :])
        keep.append(big)
        cols["dep_idx"] = big.data_ptr()
    return cols, keep, reps * Tb, reps * Eb


def alg_bytes(T, E, H, G, D):
    """SURVEY.md §8d: 60*T + 4*E + 28*H + 96*G + 16*D (compulsory traffic only)."""
    return 60 * T + 4 * E + 28 * H + 96 * G + 16 * D


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(n_tasks: int):
    """DRAM bytes of one launch of the roofline kernel: profiles/traffic.json holds dram__bytes_read + dram__bytes_write
    per task from one `ncu --set full` capture of that kernel (named there); scaled to this run's task count."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))
        return {"bytes_per_launch": int(float(t["dram_bytes_per_task"]) * n_tasks), "bytes_per_task": float(t["dram_bytes_per_task"]),
                "kernel": t.get("kernel"), "source": t.get("source")}
    except Exception:  # noqa: BLE001
        return None


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.idx = device_index
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(device_index), "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def bind_to_gpu_node(torch, local_rank: int):
    """Run this rank on the CPUs next to its GPU (NVML's affinity mask for the device with the same PCI bus id), so
    pinned host buffers are first-touched on the NUMA node the GPU's PCIe link hangs off.  Returns the previous
    affinity set (to restore for the host-core baseline leg) or None when anything about it is unavailable."""
    try:
        import pynvml
        prev = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        n = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = {i for i in range(n) if (int(mask[i // 64]) >> (i % 64)) & 1} & prev
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return prev
    except Exception:
        return None


def usable_cores():
    """Host cores this process may actually burn: the affinity mask capped by the cgroup CPU quota (the GPU boxes
    show 128 logical CPUs under a 16-CPU quota; 128 runnable threads there only add throttling)."""
    import math
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]  # cgroup v2
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())  # cgroup v1
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(math.ceil(quota))))
    return n, (os.cpu_count() or n), quota


def cores_note():
    n, logical, quota = usable_cores()
    return f"{n} threads = usable host cores ({logical} logical CPUs" + (f", cgroup CPU quota {quota:g}" if quota else "") + ")"


def cpu_baseline(w, n_distros: int, threads: int):
    """Time the oracle (C++ port of the reference algorithm) on a bounded sample: the first n distros."""
    from oracle import oracle as O
    sel = list(range(min(n_distros, w.distros.n_distros)))
    job = O.SoAJob(w.tasks, w.distros, w.hosts, sel)
    n_tasks = int(job.tasks.n)
    job.run(w.now, threads)  # warm-up pass (page faults, thread pool)
    passes, t0 = 0, time.perf_counter()
    while passes < 3 or time.perf_counter() - t0 < 10.0:  # about 10 s of CPU work
        job.run(w.now, threads)
        passes += 1
    dt = (time.perf_counter() - t0) / passes
    return {"value": n_tasks / dt, "unit": "tasks/s", "cores": threads, "kind": "port",
            "sample": f"first {len(sel)} distros ({n_tasks} tasks) of the workload, {passes} passes after one warm-up, "
                      f"{dt:.2f} s each, {cores_note()}; oracle/evg_oracle.cpp (C++17 restatement of the Go path; "
                      f"no Go toolchain in the image)",
            "decisions_per_s": len(sel) / dt}, job


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    w = headline_block(0, args.block, args.tasks_per_distro)
    threads = usable_cores()[0]
    from oracle import oracle as O
    O.build()
    sel = list(range(min(args.ref_sample, w.distros.n_distros)))
    job = O.SoAJob(w.tasks, w.distros, w.hosts, sel)
    n_tasks = int(job.tasks.n)
    for _ in range(min(args.warmup, 1)):
        job.run(w.now, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        job.run(w.now, threads)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    val = n_tasks / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "tasks/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"{HEADLINE}: distro queues of {args.tasks_per_distro} tasks, Zipf priorities, 5% unmet deps; "
                               f"each step plans the first {len(sel)} distros of the generated block ({n_tasks} tasks)",
                   "tasks_per_distro": args.tasks_per_distro, "sample_distros": len(sel),
                   "parallelism": f"{threads} host threads, one distro per work item"},
        "decisions_per_s": len(sel) / dt,
        "cpu_baseline": {"value": val, "unit": "tasks/s", "cores": threads, "kind": "port",
                         "sample": f"each step = first {len(sel)} distros ({n_tasks} tasks) of the workload's block; {cores_note()}; "
                                   "oracle/evg_oracle.cpp, C++17 restatement of the Go reference (Go toolchain absent)"},
        "e2e": {"value": val, "unit": "tasks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def time_resident(torch, eng, now, steps, warmup, stream):
    """ms per resident tick: `warmup` untimed ticks, then `steps` ticks between two events on the engine's stream."""
    for _ in range(warmup):
        eng.run(now)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        eng.run(now)
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


DUMP_TASK_ROWS, DUMP_GROUP_ROWS, DUMP_DISTRO_ROWS = 1 << 20, 1 << 18, 1 << 16  # at most ~48 MB of float64 in all


def dump_outputs(out_dir, po, ao):
    """Write what Engine.download() returned for the last timed tick as DIR/<name>.npy (float64): the per-task order
    and total value, every field of the per-distro queue info, per-group info and allocator result.  An output longer
    than its row cap is cut to a fixed seeded sample of rows (the same rows on every run with the same arguments), so
    two builds can be compared file for file.  Nanosecond sums above 2**53 are rounded to the nearest float64."""
    os.makedirs(out_dir, exist_ok=True)

    def rows(n, cap, seed):
        return slice(None) if n <= cap else np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))

    def save(name, a):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))

    def save_fields(prefix, a):
        for f in a.dtype.names:
            (save_fields if a.dtype[f].names else save)(f"{prefix}.{f}", a[f])

    t = rows(po.order.shape[0], DUMP_TASK_ROWS, 1)
    save("order", po.order[t])
    save("total_value", po.total_value[t])
    d = rows(po.info.shape[0], DUMP_DISTRO_ROWS, 2)
    save_fields("queue_info", po.info[d])
    save_fields("group_info", po.group_info[rows(po.group_info.shape[0], DUMP_GROUP_ROWS, 3)])
    if ao is not None:
        save_fields("alloc_result", ao.result[d])
        save("alloc_status", ao.status[d])


def measure_shapes(torch, eng, stream, peak, steps):
    """The other BASELINE shapes through the resident tick (same process, same engine)."""
    from evergreen_b200 import synth
    out = []
    specs = [
        ("configs[1]: 1k distros x 10k tasks each, uniform expected durations", lambda: synth.config(2)),
        ("configs[2] total reading: 10k distros, 100k tasks in total (Zipf, 5% unmet deps)", lambda: synth.config(3)),
        ("configs[3] total reading: 10k distros, 1M tasks in total, 50k hosts", lambda: synth.config(4)),
        ("configs[3] per-distro reading: 8 distros x 1M tasks each, 40 hosts", lambda: synth.config(4, 0.0008, each=True)),
        ("configs[4]: 100k distros, power-law queue sizes 1..1M, mixed providers", lambda: synth.config(5)),
    ]
    for name, make in specs:
        w = make()
        eng.upload(w.tasks, w.distros, w.hosts)
        ms = time_resident(torch, eng, w.now, steps, 3, stream)
        b = w.algorithmic_bytes()
        row = {"workload": name, "distros": w.distros.n_distros, "tasks": w.n_tasks, "ms_per_step": ms,
               "value": w.n_tasks / (ms * 1e-3), "unit": "tasks/s", "decisions_per_s": w.distros.n_distros / (ms * 1e-3),
               "gpu_launches_per_step": eng.last_launch_count(),
               "roofline_whole_tick": {"achieved": b / (ms * 1e-3) / 1e9, "frac": b / (ms * 1e-3) / 1e9 / peak,
                                       "algorithmic_bytes_per_step": int(b)}}
        if name.startswith("configs[1]"):
            try:
                k = eng.kernel_timing_ms(min(steps, 128))
                kb = 60 * w.tasks.n_tasks + 4 * w.tasks.n_edges + 96 * w.distros.n_groups
                ks = float(np.mean(k)) * 1e-3
                row["roofline_kernel"] = {"kernel": "k_plan_cta<512,10240,2> (on-chip planner: TMA-staged columns, u32 keys, "
                                                    "two CTAs per SM)", "kernel_ms": ks * 1e3, "algorithmic_bytes_per_launch": int(kb),
                                          "achieved": kb / ks / 1e9, "frac": kb / ks / 1e9 / peak,
                                          "kernel_share_of_step": ks / (ms * 1e-3)}
            except Exception as e:  # noqa: BLE001
                row["roofline_kernel"] = {"error": str(e)}
        out.append(row)
        del w
    return out


def measure_sharded_shapes(torch, dist, edist, eng, stream, dev, rank, world, steps):
    """N > 1: fixed ticks (strong scaling) sharded by whole distros with LPT -- configs[3] (hosts on) and configs[4]
    (power-law sizes, so the imbalance LPT leaves is visible).  Every rank plans its shard and all-gathers the allocator
    results (16 B/distro); per tick the max over ranks counts.  Returns rows with the per-rank load."""
    from evergreen_b200 import synth
    out = []
    for name, make in (("configs[3] total reading: 10k distros, 1M tasks, 50k hosts", lambda: synth.config(4)),
                       ("configs[4]: 100k distros, power-law queue sizes, mixed providers", lambda: synth.config(5))):
        w = make()
        weight = np.diff(w.distros.task_off) + np.diff(w.hosts.host_off)
        shards = edist.lpt_partition(weight, world)
        mine = synth.take_distros(w, shards.members[rank])
        gather = edist.ResultGather(shards, dev)
        eng.bind_result_buffer(gather.send.data_ptr(), shards.max_shard)
        eng.upload(mine.tasks, mine.distros, mine.hosts)
        for _ in range(3):
            eng.run(w.now); gather.gather()
        dist.barrier(); torch.cuda.synchronize(dev)
        e0, e1, g0, g1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record(stream)
        for _ in range(steps):
            eng.run(w.now)
            gather.gather()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        g0.record(stream)
        for _ in range(steps):
            gather.gather()
        g1.record(stream)
        torch.cuda.synchronize(dev)
        mine_ms = e0.elapsed_time(e1) / steps
        t = torch.tensor([mine_ms, g0.elapsed_time(g1) / steps, float(mine.n_tasks), float(mine.distros.n_distros)], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allr, t)
        per = [[float(x) for x in a.tolist()] for a in allr]
        ms = max(p[0] for p in per)
        out.append({"workload": name, "scaling": "strong", "distros": w.distros.n_distros, "tasks": w.n_tasks, "ms_per_step": ms,
                    "value": w.n_tasks / (ms * 1e-3), "unit": "tasks/s", "decisions_per_s": w.distros.n_distros / (ms * 1e-3),
                    "all_gather_ms": max(p[1] for p in per),
                    "per_rank": [{"rank": r, "ms_per_step": p[0], "tasks": int(p[2]), "distros": int(p[3]), "lpt_load": int(shards.load[r])}
                                 for r, p in enumerate(per)]})
        eng.bind_result_buffer(0, 0)
        del w, mine, gather
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--distros", type=int, default=4000, help="distros per GPU (configs[2] names 10000; see the docstring)")
    ap.add_argument("--block", type=int, default=40, help="distros generated on the host; tiled on the device up to --distros")
    ap.add_argument("--tasks-per-distro", type=int, default=100_000)
    ap.add_argument("--e2e-distros", type=int, default=400)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--shape-steps", type=int, default=10)
    ap.add_argument("--ref-sample", type=int, default=30, help="distros per reference/cpu_baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shapes", action="store_true")
    ap.add_argument("--no-delta", action="store_true", help="skip the resident-delta leg of the e2e object")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed tick as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.block = max(1, min(args.block, args.distros))
    reps = max(1, args.distros // args.block)
    args.distros = reps * args.block

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    from evergreen_b200 import dist as edist
    from evergreen_b200 import scheduler

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; evergreen_b200 has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    prev_affinity = bind_to_gpu_node(torch, local_rank)
    # NCCL / torchrun may write banners to fd 1; keep stdout clean for the single JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    blk = headline_block(rank, args.block, args.tasks_per_distro)
    distros, hosts = tile_tables(blk, reps)
    cols, keep, T, E = tile_device(torch, dev, blk, reps)
    D_local = distros.n_distros
    D_total = world * D_local
    sizes = np.full(D_total, args.tasks_per_distro, dtype=np.int64)
    shards = edist.lpt_partition(sizes, world)
    # a dedicated (non-default) stream: kernels, NCCL and the timing events all live on it
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng = scheduler.Engine(local_rank, stream.cuda_stream)
    # allocator results go straight into the all-gather send buffer
    # N > 1: two buffer sets, the all-gather of tick k on its own stream under tick k+1's planner
    pg = edist.PipelinedGather(shards, dev)
    gather = pg.slots[0]
    send = gather.send
    eng.bind_result_buffer(send.data_ptr(), shards.max_shard)
    torch.cuda.synchronize()
    eng.upload_device(cols, T, distros, hosts, n_edges=E)
    now = blk.now
    tick = [0]

    def step():
        k = tick[0]
        tick[0] += 1
        if world == 1:
            eng.run(now)
            return
        pg.before_tick(k, stream)
        eng.bind_result_buffer(pg.send(k).data_ptr(), shards.max_shard)
        eng.run(now)
        pg.launch(k, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    barrier()
    launches_per_step = eng.last_launch_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    pg.drain(stream)  # every tick's gathered result is complete inside the timed region
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    try:
        task_ms, sort_ms = eng.general_timing_ms()  # last step's own CUDA-event split (same stream)
    except Exception:  # noqa: BLE001
        task_ms = sort_ms = None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    tasks_total = world * T
    value = tasks_total / (ms_per_step * 1e-3)
    po, ao = eng.download()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, po, ao)
    new_hosts_checksum = int(ao.result["new_hosts"].astype(np.int64).sum())
    order_ok = bool((np.sort(po.order[: args.tasks_per_distro]) == np.arange(args.tasks_per_distro)).all())
    H, G = hosts.n_hosts, distros.n_groups
    del po, ao
    # the device copy of the headline workload is no longer needed
    del keep, cols
    torch.cuda.empty_cache()

    # ---- end to end through the public API: host buffers in and out, every step ----
    e2e_reps = max(1, min(args.e2e_distros, args.distros) // args.block)
    we = tile_host(blk, e2e_reps)

    def pinned_like(a):
        v = a.view(np.int32) if a.dtype == np.uint32 else a  # torch pins signed views; same bytes
        p = torch.from_numpy(v).pin_memory().numpy()
        return p.view(a.dtype)
    for name, _ in we.tasks.COLUMNS:
        setattr(we.tasks, name, pinned_like(getattr(we.tasks, name)))
    if we.tasks.n_edges:
        we.tasks.dep_off, we.tasks.dep_idx = pinned_like(we.tasks.dep_off), pinned_like(we.tasks.dep_idx)
    for name, _ in we.hosts.COLUMNS:
        setattr(we.hosts, name, pinned_like(getattr(we.hosts, name)))
    h2d = we.tasks.nbytes() + we.distros.nbytes() + we.hosts.nbytes()
    pe, ae = eng.plan_and_alloc_batch(we.tasks, we.distros, we.hosts, we.now)  # warm-up (buffers sized)
    d2h = pe.nbytes() + ae.nbytes()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        pe, ae = eng.plan_and_alloc_batch(we.tasks, we.distros, we.hosts, we.now)
        if world > 1:
            gather.gather()
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.e2e_steps
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * we.n_tasks / float(t.item())
    clocks = sampler.stop() if sampler else None  # sampled from before the timed loop to the end of the e2e loop
    # ---- the same table kept resident, a tick's worth of changes sent instead (evg_update_tasks + evg_download_queue):
    #      5% of the rows get new priority / durations / dependency bits each step, the persisted slice (first 10 000
    #      ranks of every distro, scheduler/task_queue_persister.go:14-55) comes back.  Reported NEXT TO the headline
    #      e2e, never as it: the headline uploads every column every step.
    delta = None
    if world == 1 and not args.no_delta:
        from evergreen_b200 import _lib as L
        from evergreen_b200.soa import TaskSoA
        rng = np.random.default_rng(11)
        n_upd = max(1, we.n_tasks // 20)
        upd = []
        for _ in range(args.e2e_steps + 1):
            rows = np.sort(rng.choice(we.n_tasks, size=n_upd, replace=False)).astype(np.int64)
            vals = TaskSoA(**{name: getattr(we.tasks, name)[rows].copy() for name, _ in we.tasks.COLUMNS})
            vals.priority = rng.integers(0, 101, n_upd).astype(np.int32)
            vals.expected_ns = (vals.expected_ns + rng.integers(0, 10 ** 9, n_upd)).astype(np.int64)
            vals.flags = (vals.flags | L.EVG_TF_DEPS_MET).astype(np.uint32)
            upd.append((pinned_like(rows), TaskSoA(**{name: pinned_like(getattr(vals, name)) for name, _ in vals.COLUMNS})))
        eng.upload(we.tasks, we.distros, we.hosts)
        eng.update_tasks(*upd[0]); eng.run(we.now); off, items = eng.download_queue(task_off=we.distros.task_off)  # warm-up
        d_bytes = int(items.nbytes + off.nbytes)
        t0 = time.perf_counter()
        for k in range(args.e2e_steps):
            eng.update_tasks(*upd[k + 1])
            eng.run(we.now)
            off, items = eng.download_queue(task_off=we.distros.task_off)
        dt_s = (time.perf_counter() - t0) / args.e2e_steps
        delta = {"value": we.n_tasks / dt_s, "unit": "tasks/s", "ms_per_step": dt_s * 1e3, "changed_rows_per_step": int(n_upd),
                 "h2d_bytes_per_step": int(48 * n_upd), "d2h_bytes_per_step": d_bytes,
                 "api": "Engine.update_tasks (evg_update_tasks: 5% of the rows, 48 B each) + evg_run_resident + Engine.download_queue "
                        "(evg_download_queue: 40 B x the first 10 000 ranks of every distro)"}
        del upd, off, items
    del we, pe, ae

    sharded = None
    if world > 1 and not args.no_shapes:  # every rank takes part
        sharded = measure_sharded_shapes(torch, dist, edist, eng, stream, dev, rank, world, args.shape_steps)
    line = None
    if rank == 0:
        peak, peak_src = load_peaks()
        step_s = ms_per_step * 1e-3
        ab = alg_bytes(T, E, H, G, D_local)  # per GPU per step
        roof = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src, "traffic": None,
                "whole_tick": {"achieved": ab / step_s / 1e9, "frac": ab / step_s / 1e9 / peak, "algorithmic_bytes_per_step": int(ab)}}
        if task_ms:
            kb = 48 * T + 4 * E  # the per-task pass reads every input column once; its outputs are scratch
            roof.update({"kernel": "k_gtask (general path: 128-bit column loads, 32-bit scoring, queue-info fold, work-list append), "
                                   "CUDA events on its stream around the launch in the last timed step",
                         "kernel_ms": task_ms, "algorithmic_bytes_per_launch": int(kb), "achieved": kb / (task_ms * 1e-3) / 1e9,
                         "frac": kb / (task_ms * 1e-3) / 1e9 / peak, "kernel_share_of_step": task_ms / ms_per_step,
                         "sort_ms": sort_ms, "sort_share_of_step": sort_ms / ms_per_step})
            tr = load_traffic(T)
            if tr and tr.get("kernel") == "k_gtask":
                roof["traffic"] = tr["bytes_per_launch"]
                roof["traffic_source"] = f"{tr['bytes_per_task']:.1f} B/task x {T} tasks; {tr['source']}"
        else:
            roof.update({"achieved": roof["whole_tick"]["achieved"], "frac": roof["whole_tick"]["frac"], "kernel": "whole tick"})
        line = {
            "metric": METRIC, "value": value, "unit": "tasks/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": f"{HEADLINE}: {D_local} distros x {args.tasks_per_distro} tasks each per GPU (of configs[2]'s 10000: "
                                   "what fits HBM next to the work buffers), Zipf priorities, 5% unmet + 2% met in-queue dependencies, "
                                   f"10% of tasks in task groups, {H} hosts; a {args.block}-distro block from synth (splitmix64) tiled "
                                   f"{reps}x on the device with a per-tile clock shift",
                       "distros_total": D_total, "tasks_total": tasks_total, "global_batch": tasks_total,
                       "parallelism": f"distro-sharded x{world} (LPT), 1 all-gather of 16 B/distro per step"
                                      + (", issued on a second stream under the next tick's planner (double-buffered)" if world > 1 else ""),
                       "l2": f"inputs ({(48 * T + 8 * T + 4 * E) / 1e9:.1f} GB of columns per GPU) exceed the 126 MB L2; no flush needed"},
            "decisions_per_s": D_total / step_s,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "tasks/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": float(t.item()) * 1e3,
                    "workload": f"the same shape on {e2e_reps * args.block} distros ({e2e_reps * args.block * args.tasks_per_distro} tasks) per GPU",
                    "api": "Engine.plan_and_alloc_batch (evg_plan_and_alloc_batch), pinned host columns",
                    "cpu_affinity": "GPU-local NUMA node" if prev_affinity else "unbound",
                    "resident_delta": delta},
            "gpu_launches": int(launches_per_step * args.steps),
            "roofline": roof,
            "checksum_new_hosts": new_hosts_checksum, "first_distro_is_a_permutation": order_ok,
        }
        if not args.no_shapes and world == 1:
            eng.bind_result_buffer(0, 0)  # the shapes have other distro counts: results go to the context's own buffer
            line["shapes"] = measure_shapes(torch, eng, stream, peak, args.shape_steps)
        if sharded is not None:
            line["shapes"] = sharded
        if world == 1 and not args.no_delta:
            # the string side of marshalling (group keys / versions / dependency ids -> dense ids), host C++ behind the
            # ABI (evg_intern_columns); columns of Evergreen-shaped strings, 1e6 tasks in 100 distros
            try:
                sys.path.insert(0, os.path.join(ROOT, "profiles"))
                import intern_bench
                ib = intern_bench.run(100, 10000, threads=(1, usable_cores()[0]))
                line["e2e"]["host_interning"] = {"tasks_per_s": ib["runs"][-1]["tasks_per_s"], "threads": ib["runs"][-1]["threads"],
                                                 "one_thread_tasks_per_s": ib["runs"][0]["tasks_per_s"], "string_bytes_per_task": ib["string_bytes"] / ib["tasks"],
                                                 "api": "evg_intern_columns (host C++): task-group keys, versions, dependency ids of 1e6 tasks"}
            except Exception as e:  # noqa: BLE001
                line["e2e"]["host_interning"] = {"error": str(e)}
        if not args.no_cpu_baseline and world == 1:
            if prev_affinity:
                os.sched_setaffinity(0, prev_affinity)  # the baseline gets every host core back
            cb, _ = cpu_baseline(blk, args.ref_sample, usable_cores()[0])
            line["cpu_baseline"] = cb
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())

"""Full tick (evg_run_resident) against the persisted-head tick (evg_run_resident_head, cap 10 000) in one process.

Workloads: bench.py's headline (configs[2] per-distro reading, 4000 distros x 100 000 tasks, the columns tiled on the
device exactly as bench.py tiles them), BASELINE configs[3] per-distro (8 x 1M tasks) and configs[4] (100k distros,
power-law sizes).  Per workload, after warm-up, full and head ticks alternate (CUDA events around each tick on the
engine's stream) and the rows every distro persists -- the first 10 000 ranks, evg_download_queue -- are checked equal
between the two kinds.  On the headline's host-tiled e2e slice (bench.py's resident_delta leg) it also times
update_tasks + tick + queue download for both kinds, the head kind with its breakdown rows (evg_download_queue_bd).

    python profiles/persisted_head.py --out persisted_head.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  headline_block / tile_device / tile_tables / tile_host: the same inputs as bench.py


def card(torch):
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return {"name": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": pl}


def alternate(torch, eng, stream, now, steps, warmup, task_off):
    """Alternating full / head ticks; per kind the mean ms per tick and the mean general-path sort stage."""
    def tick(head):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        if head:
            eng.run_head(now)
        else:
            eng.run(now)
        e1.record(stream)
        e1.synchronize()
        try:
            sort = eng.general_timing_ms()[1]
        except Exception:  # noqa: BLE001  a tick without general-path distros
            sort = None
        return e0.elapsed_time(e1), sort
    for _ in range(warmup):
        tick(False)
        tick(True)
    res = {False: [], True: []}
    for _ in range(steps):
        for head in (False, True):
            res[head].append(tick(head))
    out = {}
    for head, name in ((False, "full"), (True, "head")):
        ms = [a for a, _ in res[head]]
        sorts = [b for _, b in res[head] if b is not None]
        out[name] = {"ms_per_tick": float(np.mean(ms)), "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)),
                     "sort_stage_ms": float(np.mean(sorts)) if sorts else None}
    # the persisted rows of both kinds, every distro
    eng.run(now)
    off_f, items_f = (x.copy() for x in eng.download_queue(0, task_off))
    eng.run_head(now)
    off_h, items_h = eng.download_queue(0, task_off)
    out["rows_checked"] = int(items_f.shape[0])
    out["head_rows_equal_full"] = bool(np.array_equal(off_f, off_h) and items_f.tobytes() == items_h.tobytes())
    del items_f
    out["head_speedup"] = out["full"]["ms_per_tick"] / out["head"]["ms_per_tick"]
    return out


def resident_delta(eng, we, steps):
    """bench.py's resident_delta leg for both kinds: 5% of the rows edited, a tick, the persisted rows downloaded."""
    from evergreen_b200 import _lib as L
    from evergreen_b200.soa import TaskSoA
    rng = np.random.default_rng(11)
    n_upd = max(1, we.n_tasks // 20)
    upd = []
    for _ in range(2 * steps + 2):
        rows = np.sort(rng.choice(we.n_tasks, size=n_upd, replace=False)).astype(np.int64)
        vals = TaskSoA(**{name: getattr(we.tasks, name)[rows].copy() for name, _ in we.tasks.COLUMNS})
        vals.priority = rng.integers(0, 101, n_upd).astype(np.int32)
        vals.expected_ns = (vals.expected_ns + rng.integers(0, 10 ** 9, n_upd)).astype(np.int64)
        vals.flags = (vals.flags | L.EVG_TF_DEPS_MET).astype(np.uint32)
        upd.append((rows, vals))
    eng.upload(we.tasks, we.distros, we.hosts)

    def full(k):
        eng.update_tasks(*upd[k]); eng.run(we.now)
        return eng.download_queue(task_off=we.distros.task_off)

    def head(k):
        eng.update_tasks(*upd[k]); eng.run_head(we.now, 0, L.EVG_OPT_BREAKDOWN)
        return eng.download_queue(task_off=we.distros.task_off, breakdown=True)
    out = {}
    full(0); head(1)  # warm-up
    for name, fn, k0 in (("full", full, 2), ("head_with_breakdown", head, 2 + steps)):
        t0 = time.perf_counter()
        for k in range(steps):
            q = fn(k0 + k)
        dt = (time.perf_counter() - t0) / steps
        out[name] = {"ms_per_step": dt * 1e3, "tasks_per_s": we.n_tasks / dt, "d2h_rows": int(q[1].shape[0])}
    out["tasks"] = int(we.n_tasks)
    out["changed_rows_per_step"] = int(n_upd)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--distros", type=int, default=4000)
    ap.add_argument("--block", type=int, default=40)
    ap.add_argument("--tasks-per-distro", type=int, default=100_000)
    ap.add_argument("--e2e-distros", type=int, default=400)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    from evergreen_b200 import scheduler, synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 path only")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    eng = scheduler.Engine(0, stream.cuda_stream)
    result = {"card": card(torch), "steps": args.steps, "warmup": args.warmup, "cap": 10000, "workloads": {}}

    reps = max(1, args.distros // args.block)
    blk = bench.headline_block(0, args.block, args.tasks_per_distro)
    distros, hosts = bench.tile_tables(blk, reps)
    cols, keep, T, E = bench.tile_device(torch, dev, blk, reps)
    eng.upload_device(cols, T, distros, hosts, n_edges=E)
    name = f"headline: {distros.n_distros} distros x {args.tasks_per_distro} tasks (bench.py's inputs)"
    result["workloads"][name] = alternate(torch, eng, stream, blk.now, args.steps, args.warmup, distros.task_off)
    print(name, json.dumps(result["workloads"][name]), file=sys.stderr, flush=True)
    del keep, cols
    torch.cuda.empty_cache()
    we = bench.tile_host(blk, max(1, min(args.e2e_distros, args.distros) // args.block))
    result["resident_delta"] = resident_delta(eng, we, args.e2e_steps)
    print("resident_delta", json.dumps(result["resident_delta"]), file=sys.stderr, flush=True)
    del we

    for name, make in (("configs[3] per-distro reading: 8 distros x 1M tasks each, 40 hosts", lambda: synth.config(4, 0.0008, each=True)),
                       ("configs[4]: 100k distros, power-law queue sizes 1..1M, mixed providers", lambda: synth.config(5))):
        w = make()
        eng.upload(w.tasks, w.distros, w.hosts)
        result["workloads"][name] = alternate(torch, eng, stream, w.now, args.steps, args.warmup, w.distros.task_off)
        print(name, json.dumps(result["workloads"][name]), file=sys.stderr, flush=True)
    result["card_after"] = card(torch)
    eng.close()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

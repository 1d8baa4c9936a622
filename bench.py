#!/usr/bin/env python
"""bench.py - participant-steps/s of the batched env.step() hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the fused tick (physics -> pose -> collisions -> out-of-bound -> status) over one
batch of synthetic scenarios.  At N=1 the workload is BASELINE.json configs[1]: 4096 scenarios x 64
participants, SingleTrackKinematics + OBB collision, synthetic grid map.  For N>1 every rank steps its own
4096 x 64 shard (weak scaling; scenarios are independent) and the ranks exchange the done mask with one
all-gather per step.

Timing rules followed: W >= 3 warm-up steps; inputs larger than L2 - the timed steps rotate over R
independent world replicas whose state + actions + outputs exceed the 126 MB L2 (R x 14.2 MB), so every
step streams its state from HBM; device timing with CUDA events on the launching stream, barrier +
synchronize on both sides, max over ranks; SM clocks and throttle reasons sampled with nvidia-smi while
the timed region is repeated.  The K-step timed region is captured in a CUDA graph (the kernels are a few
microseconds each; a Python launch loop would measure the interpreter) and is repeated `reps` times, the
median repetition is reported.

`--impl reference` times the reference's own execution model for this path - one Python call per
participant with NumPy scalar float64 arithmetic and per-pose predicate loops (oracle/scalar_port.py, a
restatement: the reference's shapely/gymnasium dependencies are not installable here) - on all host cores.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "participant_steps_per_sec"
UNIT = "participant-steps/s"
N_SCN, M_PART = 4096, 64

# algorithmic bytes per participant-step of the fused kernel (DESIGN.md "Roofline"): reads x, y, heading,
# speed (16) + action (8) + type id (1); writes x, y, heading, speed, vx, vy (24) + event byte (1) +
# hit_index (2) + hit_segment (2); per scenario step_count r/w (8) + status (1) + done (1).
BYTES_PER_PARTICIPANT = 16 + 8 + 1 + 24 + 1 + 2 + 2
BYTES_PER_SCENARIO = 8 + 1 + 1


def usable_cores() -> int:
    """Host cores this process may really use: the scheduler affinity mask, capped by the cgroup CPU quota (a container that
    reports 128 CPUs may be allowed 8 of them - a worker pool sized by os.cpu_count() then only thrashes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota = None
        if os.path.exists("/sys/fs/cgroup/cpu.max"):
            q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
            if q != "max":
                quota = float(q) / float(per)
        elif os.path.exists("/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        if quota is not None:
            n = max(1, min(n, int(quota + 0.5)))
    except Exception:
        pass
    return max(1, n)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_scene(config: str, seed: int, n=None, m=None):
    from tactics2d_b200 import synthetic
    from tactics2d_b200.map import load_collidable_segments

    if config == "c2":
        return synthetic.config2(n or N_SCN, m or M_PART, seed=seed)
    if config == "c3":
        seg, bounds = load_collidable_segments("highD_1")
        return synthetic.config3(n or 4096, m or 64, seed=seed, segments=seg, bounds=bounds)
    if config == "c4":
        seg, bounds = load_collidable_segments("inD_1")
        return synthetic.config4(n or 16384, m or 32, seed=seed, segments=seg, bounds=bounds)
    if config == "c5":
        seg, bounds = load_collidable_segments("rounD_0")
        return synthetic.config5(n or 65536, m or 128, seed=seed, segments=seg, bounds=bounds)
    raise SystemExit(f"unknown config {config}")


def make_scene_name(config: str) -> str:
    return {"c2": f"C2 {N_SCN}x{M_PART} kinematics + OBB collision, synthetic grid map",
            "c3": "C3 4096x64 dynamics + map polylines", "c4": "C4 16384x32 mixed vehicle/cyclist/pedestrian",
            "c5": "C5 65536x128 kinematics + broadphase stress"}[config]


DUMP_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict) -> None:
    """Write `arrays` (each with the scenario axis first) to `path`/<name>.npy as float32, the integer outputs converted
    exactly, plus scenario_index.npy (float64): the scenario rows written.  When the whole batch would exceed DUMP_BYTES,
    a fixed seeded sample of scenario rows is written, the same rows for every array, so that two builds run with the
    same arguments can be compared array by array."""
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].size for a in arrays.values()) * 4 + 8
    keep = min(n, (DUMP_BYTES - (64 << 10)) // row_bytes)          # 64 KiB left for the .npy headers
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a[rows].astype(np.float32))
    np.save(os.path.join(path, "scenario_index.npy"), rows.astype(np.float64))
    print(f"[bench] wrote {len(arrays) + 1} arrays ({keep} of {n} scenarios) to {path}", file=sys.stderr)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ts, line in self.lines:
            if not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arms
_CPU_JOB = {}   # filled before the worker pool forks: the workers share the batch copy-on-write and receive only index ranges


def _cpu_worker(rng):
    from oracle import scalar_port as SP

    lo, hi = rng
    j = _CPU_JOB
    SP.tick_scenarios({k: v[lo:hi] for k, v in j["state"].items()}, j["tid"][lo:hi], j["act"][lo:hi], j["table"], j["seg"], j["bounds"])
    return hi - lo


def cpu_port_throughput(scene, n_scn: int, procs: int, steps: int = 1, warmup: int = 0, per_job: int = 32):
    """participant-steps/s of the reference-style per-agent Python loop over the first `n_scn` scenarios per step, fanned
    over `procs` worker processes in jobs of `per_job` scenarios (a job of one scenario would time the pool's dispatch,
    not the loop)."""
    import multiprocessing as mp

    from tactics2d_b200 import synthetic

    n_scn = min(n_scn, scene.shape[0])
    _CPU_JOB.update(state={k: v[:n_scn] for k, v in scene.state().items()}, tid=scene.type_id[:n_scn],
                    act=synthetic.random_actions(77, (n_scn, scene.shape[1])), table=scene.table.as_oracle_table(),
                    seg=scene.segments, bounds=scene.bounds)
    per_job = max(1, min(per_job, -(-n_scn // max(1, procs))))
    jobs = [(lo, min(lo + per_job, n_scn)) for lo in range(0, n_scn, per_job)]
    times = []
    if procs <= 1:
        for i in range(warmup + steps):
            t = time.perf_counter()
            for j in jobs:
                _cpu_worker(j)
            if i >= warmup:
                times.append(time.perf_counter() - t)
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            for i in range(warmup + steps):
                t = time.perf_counter()
                pool.map(_cpu_worker, jobs, chunksize=1)
                if i >= warmup:
                    times.append(time.perf_counter() - t)
    total = n_scn * scene.shape[1] * len(times)
    return total / sum(times), sum(times) / len(times)


def cpu_c_throughput(scene, reps=3):
    """The compiled float64 oracle (C + OpenMP, all cores) on the full batch - a stronger CPU figure."""
    from oracle import c_oracle as CO
    from tactics2d_b200 import synthetic

    table = scene.table.as_oracle_table()
    act = synthetic.random_actions(78, scene.shape)
    best = None
    for _ in range(reps):
        t = time.perf_counter()
        new = CO.physics(scene.state(), scene.type_id, act, table)
        CO.events(new["x"], new["y"], new["heading"], scene.type_id, table, scene.segments, scene.bounds)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    return scene.x.size / best


def run_reference(args):
    """The reference's execution model for this path on the host cores, on the SAME configuration as the GPU arm: every
    step is the whole batch (4096 x 64 at C2), 32 scenarios per job, one worker process per core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    scene = make_scene(args.config, seed=1, n=args.scenarios or None)
    n, m = scene.shape
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    # bounded: the whole run must end within a few minutes - ~2 k participant-steps/s per core measured for the port
    est = n * m / (1900.0 * max(1, cores)) * (steps + warmup)
    if est > 150.0:
        warmup = min(warmup, 1)
        steps = max(1, min(steps, int(150.0 / max(1e-9, n * m / (1900.0 * cores))) - warmup))
    value, t_step = cpu_port_throughput(scene, n, cores, steps=steps, warmup=warmup, per_job=32)
    sample = (f"the whole batch every step: {n} scenarios x {m} participants, {steps} timed steps after {warmup} warm-up, "
              f"{cores} worker processes x jobs of 32 scenarios (per-agent Python loop = the reference's execution model; "
              f"a restatement: shapely/GEOS and gymnasium are not installable here, oracle/scalar_port.py)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": scene.name, "scenarios_per_gpu": n, "participants": m,
                   "model": "SingleTrackKinematics" if args.config in ("c2", "c5") else args.config,
                   "interval_ms": 100, "delta_t_ms": 5, "map_segments": 0 if scene.segments is None else int(len(scene.segments)),
                   "timed_steps": steps},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry

    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        entry.build()
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world_size > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION/INFO
        os.environ["NCCL_DEBUG"] = os.environ.get("T2D_NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=device)
        dist.barrier()
    from tactics2d_b200 import BatchedWorld, _lib, synthetic

    lib = _lib.load()
    K, W = args.steps, max(args.warmup, 3)
    n_cfg = args.scenarios or None
    if args.sharded:   # the configuration's N is the whole job: every rank takes a contiguous 1 / world_size share of it
        from tactics2d_b200.distributed import shard_range
        total = args.scenarios or {"c2": N_SCN, "c3": 4096, "c4": 16384, "c5": 65536}[args.config]
        lo, hi = shard_range(total, rank, world_size)
        n_cfg = hi - lo
    scene0 = make_scene(args.config, seed=1 + 1000 * rank, n=n_cfg)
    n, m = scene0.shape
    bytes_per_launch = n * m * BYTES_PER_PARTICIPANT + n * BYTES_PER_SCENARIO
    l2_bytes = torch.cuda.get_device_properties(device).L2_cache_size
    R = args.replicas or max(4, int(np.ceil(2.5 * l2_bytes / bytes_per_launch)))
    R = min(R, max(2, int(60e9 // max(1, bytes_per_launch))))

    worlds, actions, pools = [], [], []
    for r in range(R):
        sc = scene0 if r == 0 else make_scene(args.config, seed=1 + 1000 * rank + r, n=n_cfg)
        w = BatchedWorld(n, m, sc.table, device=device, max_step=0)
        w.set_map(sc.segments, sc.bounds)
        w.set_state(sc.x, sc.y, sc.heading, sc.speed, vx=sc.vx, vy=sc.vy, type_id=sc.type_id)
        worlds.append(w)
        actions.append(torch.from_numpy(synthetic.random_actions(9000 + 1000 * rank + r, (n, m))).to(device))
        pools.append({k: getattr(w, k).clone() for k in ("x", "y", "heading", "speed", "vx", "vy")})
    ones = torch.ones(n, dtype=torch.uint8, device=device)
    # The one exchange of the path: every rank gets every rank's done mask of each step.  Default: our own all-gather
    # kernel over peer memory (t2d_exchange_allgather: put to every rank, signal, wait, copy - one CTA per rank and step);
    # --exchange nccl uses all_gather_into_tensor instead.  Either runs on a side stream under the next tick.
    peer = None
    if world_size > 1 and args.exchange == "peer":
        from tactics2d_b200.distributed import PeerDoneExchange

        try:
            peer = PeerDoneExchange(n, device, lag=args.lag)
        except RuntimeError as e:   # every rank raises together (the set-up is agreed on collectively): use NCCL instead
            peer = None
            args.exchange = "nccl"
            if rank == 0:
                print(f"[bench] {e}; falling back to --exchange nccl", file=sys.stderr)

    # rows of the gathered mask: the peer kernel pads every rank's row to a multiple of 16 bytes
    row = peer.pad if peer is not None else n
    done_all = torch.zeros(world_size * row, dtype=torch.uint8, device=device) if world_size > 1 else None

    def restore():
        for w, p in zip(worlds, pools):
            w.reset(ones, p)

    # The one exchange of the path: all-gather of this step's done mask.  It runs on a side stream behind an
    # event, so that the collective of step i overlaps the kernel of step i+1 (the next tick does not consume
    # it; a learner / reset scheduler does); the streams are joined before the timed region ends.
    comm_stream = torch.cuda.Stream(device) if world_size > 1 else None

    def one_step(i):
        r = i % R
        out = worlds[r].step(actions[r])
        if world_size > 1:
            main = torch.cuda.current_stream(device)
            ev = torch.cuda.Event()
            ev.record(main)
            comm_stream.wait_event(ev)
            with torch.cuda.stream(comm_stream):
                if peer is not None:
                    peer(out.done, done_all)
                else:
                    dist.all_gather_into_tensor(done_all, out.done)
        return out

    def join_comm():
        if world_size > 1:
            torch.cuda.current_stream(device).wait_stream(comm_stream)

    def barrier():
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # warm-up (also JIT-free: the library is prebuilt) --------------------------------------------
    for i in range(W):
        one_step(i)
    join_comm()
    barrier()

    # self-check of the exchange, every run: the masks our peer-memory kernel delivers (call k -> step k - lag) must
    # equal NCCL's all_gather of the same masks
    exchange_check = None
    if peer is not None:
        history, ok, checked = [], True, 0
        ref = torch.zeros(world_size * n, dtype=torch.uint8, device=device)
        for t in range(args.lag + 4):
            out = worlds[t % R].step(actions[t % R])
            got = peer(out.done, done_all).clone()
            dist.all_gather_into_tensor(ref, out.done)
            torch.cuda.synchronize()
            history.append(ref.clone())
            k = peer.calls - 1 - args.lag        # the step this call delivered (counted over all calls so far)
            h = len(history) - 1 - args.lag      # ... as an index into this loop's history
            if h >= 0:
                ok = ok and bool(torch.equal(got.view(world_size, peer.pad)[:, :n].reshape(-1), history[h]))
                checked += 1
        flag = torch.tensor([1 if ok else 0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        exchange_check = {"ok": bool(flag.item()), "steps_compared": checked, "against": "all_gather_into_tensor (NCCL)"}
        if not exchange_check["ok"]:
            if rank == 0:
                print("[bench] peer-memory done exchange disagrees with NCCL all_gather", file=sys.stderr)
            os._exit(4)
        restore()
        barrier()

    # capture the K-step timed region in a CUDA graph ----------------------------------------------
    def capture():
        """(graph, our launches recorded in it), or (None, K) when capture is off or fails: the eager loop is timed then."""
        if args.no_graph:
            return None, K
        try:
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                for i in range(min(3, K)):
                    one_step(i)
                join_comm()
            torch.cuda.current_stream(device).wait_stream(side)
            barrier()
            g = torch.cuda.CUDAGraph()
            l_cap = lib.t2d_launch_count()
            with torch.cuda.graph(g):
                for i in range(K):
                    one_step(i)
                join_comm()
            return g, int(lib.t2d_launch_count() - l_cap)   # our kernels recorded in the graph (tick, done exchange)
        except Exception as e:   # e.g. NCCL capture unsupported: fall back to the eager loop
            if rank == 0:
                print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); timing the eager loop", file=sys.stderr)
            torch.cuda.synchronize()
            return None, K

    graph, graph_launches = capture()

    def timed_region():
        restore()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.t2d_launch_count()
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            for i in range(K):
                one_step(i)
            join_comm()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world_size > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        launches = graph_launches if graph is not None else int(lib.t2d_launch_count() - l0)
        return float(ms.item()), launches

    timed_region()  # one untimed pass through the exact timed path

    # N > 1: the tick's early L2 prefetch of its inputs is a pure tuning knob (t2d_set_prefetch; results do not depend on it).
    # On one GPU it is a gain; next to the exchange kernel on 8 GPUs it measured slower, so the library's policy leaves it off
    # there.  Rather than trust either number, time both settings here - same graph, same collectives, the max over ranks of
    # a few repetitions each, identical on every rank - and keep the faster one for the timed region.
    prefetch_cal = None
    if world_size > 1 and peer is not None and graph is not None and not args.no_prefetch_cal:
        cal = {}
        for mode in (0, 1):
            for w in worlds:
                w.set_prefetch(mode)
            graph, graph_launches = capture()
            timed_region()
            cal[mode] = (float(np.median([timed_region()[0] for _ in range(args.prefetch_cal_reps)])) / K * 1e3, graph, graph_launches)
        pick = 0 if cal[0][0] <= cal[1][0] else 1
        for w in worlds:
            w.set_prefetch(pick)
        graph, graph_launches = cal[pick][1], cal[pick][2]
        prefetch_cal = {"us_per_step_off": cal[0][0], "us_per_step_on": cal[1][0], "picked": "on" if pick else "off",
                        "reps_each": args.prefetch_cal_reps}
        cal = None
        timed_region()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_wall0 = time.time()
    reps_ms, launches = [], K
    budget_s, t_begin = args.min_seconds, time.time()
    while True:
        ms, launches = timed_region()
        reps_ms.append(ms)
        more = len(reps_ms) < args.min_reps or (time.time() - t_begin < budget_s and len(reps_ms) < args.max_reps)
        if world_size > 1:
            # every repetition holds collectives (barrier, max over ranks), so all ranks must run the same number of them:
            # rank 0's wall clock decides for everybody (each rank reading its own clock can disagree on the last one
            # and leave a rank waiting in a barrier nobody else enters)
            flag = torch.tensor([1 if more else 0], dtype=torch.int32, device=device)
            dist.broadcast(flag, src=0)
            more = bool(flag.item())
        if not more:
            break
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:
        # every repetition restores the worlds first, so the last timed step's results do not depend on how many ran
        last = worlds[(K - 1) % R]
        outs = {k: getattr(last, k) for k in ("x", "y", "heading", "speed", "vx", "vy")}
        outs.update({k: getattr(last.result, k) for k in ("flags", "hit_index", "hit_segment", "status", "done")})
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in outs.items()})
    ms_total = float(np.median(reps_ms))
    ms_per_step = ms_total / K
    value = world_size * n * m * K / (ms_total * 1e-3)

    # e2e: public API with HOST buffers, host<->device copies and a stream sync inside every timed step ----------------
    e2e = None
    if not args.no_e2e:
        from tactics2d_b200.controller import IDMController

        def timed_loop(step_fn, reps):
            restore()
            for i in range(max(W, R)):   # every world replica once: first calls build per-world state (staging buffers, graphs)
                step_fn(i)
            ms = []
            for _ in range(reps):
                restore()
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(K):
                    step_fn(i)
                e1.record()
                barrier()
                t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
                if world_size > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms.append(float(t.item()))
            return float(np.median(ms)) / K

        reps_e2e = max(3, min(args.min_reps, 10))
        # (1) the headline: the reference env's contract - the caller's policy drives the EGO, one (steering, accel) per
        # scenario (envs/parking.py:219-239); the other 63 participants are driven by on-device IDM controllers
        # (t2d_control), so 8 N bytes go up and 2 N come back per step (t2d_step_host_ego)
        rs = np.random.default_rng(7)
        cid = np.zeros((n, m), np.uint8)
        cid[:, 0] = 255
        lead = np.tile(np.arange(m, dtype=np.int16) - 1, (n, 1))
        npc_act = []
        for w in worlds:
            w.set_controllers([IDMController()], cid, lead_index=lead)
            npc_act.append(torch.zeros((n, m, 2), dtype=torch.float32, device=device))
        host_ego = [torch.from_numpy(rs.uniform(-1, 1, (n, 2)).astype(np.float32)).pin_memory() for _ in range(8)]

        def ego_step(i):
            r = i % R
            done_np, _ = worlds[r].step_host_ego(host_ego[i % len(host_ego)], npc_act[r])
            if world_size > 1:
                # t2d_step_host_ego delivers status / done to the HOST; the exchange takes the device copy of this step's mask
                worlds[r].result.done.copy_(torch.from_numpy(done_np), non_blocking=True)
                if peer is not None:
                    peer(worlds[r].result.done, done_all)
                else:
                    dist.all_gather_into_tensor(done_all, worlds[r].result.done)
        t_ego = timed_loop(ego_step, reps_e2e)
        e2e = {"value": world_size * n * m / (t_ego * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * 2 * 4 + (n if world_size > 1 else 0),
               "d2h_bytes_per_step": 2 * n,
               "ms_per_step": t_ego,
               "api": ("BatchedWorld.step_host_ego(ego_action) = t2d_step_host_ego: pinned-host ego actions [N, 2] -> device, on-device "
                       "IDM controllers for the other participants (t2d_control), the fused tick, status + done -> host, stream sync "
                       "per step (the caller reads done before choosing the next action)" +
                       ("" if world_size == 1 else "; + the done exchange (" + args.exchange + ")"))}
        for w in worlds:
            w.set_controllers(None, None)
        if world_size == 1:
            # (2) every participant's action from the host (the round-1 figure): 8 N M bytes up per step
            host_act = [torch.from_numpy(synthetic.random_actions(500 + r, (n, m))).pin_memory() for r in range(min(R, 8))]
            t_all = timed_loop(lambda i: worlds[i % R].step_host(host_act[i % len(host_act)]), reps_e2e)
            e2e["all_actions_from_host"] = {"value": n * m / (t_all * 1e-3), "unit": UNIT, "ms_per_step": t_all, "h2d_bytes_per_step": n * m * 2 * 4,
                                            "d2h_bytes_per_step": 2 * n, "api": "BatchedWorld.step_host(action [N, M, 2]) = t2d_step_host"}
            # (3) the Gym surface: BatchedTrafficEnv.step(ego action) -> observation views, reward, terminated, truncated, info,
            # with auto-reset; the ego action is uploaded from pinned host memory and reward / terminated / truncated are read
            # back every step (tick + env epilogue + masked reset: three launches of ours)
            from tactics2d_b200.envs import BatchedTrafficEnv

            env = BatchedTrafficEnv(scene0, device=device, max_step=200, auto_reset=True)
            env.reset(seed=0)
            act_dev = torch.empty((n, 2), dtype=torch.float32, device=device)
            h_rew = torch.empty(n, dtype=torch.float32).pin_memory()
            h_term = torch.empty(n, dtype=torch.bool).pin_memory()
            h_trunc = torch.empty(n, dtype=torch.bool).pin_memory()
            stream = torch.cuda.current_stream(device)

            def env_step(i):
                act_dev.copy_(host_ego[i % len(host_ego)], non_blocking=True)
                _, rew, term, trunc, _ = env.step(act_dev)
                h_rew.copy_(rew, non_blocking=True); h_term.copy_(term, non_blocking=True); h_trunc.copy_(trunc, non_blocking=True)
                stream.synchronize()
            l0 = lib.t2d_launch_count()
            env_step(0)
            per_call = int(lib.t2d_launch_count() - l0)
            t_env = timed_loop(env_step, reps_e2e)
            e2e["env_step"] = {"value": n * m / (t_env * 1e-3), "unit": UNIT, "ms_per_step": t_env, "h2d_bytes_per_step": n * 2 * 4,
                               "d2h_bytes_per_step": 6 * n, "our_launches_per_step": per_call,
                               "api": "BatchedTrafficEnv.step(ego action) with auto-reset: ego action H2D, reward + terminated + truncated D2H, sync"}
            env.close()

    if rank == 0:
        peak, peak_src = _peaks()
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(args.config)
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.sharded else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": scene0.name, "scenarios_per_gpu": n, "participants": m, "model": "SingleTrackKinematics" if args.config in ("c2", "c5") else args.config,
                       "interval_ms": 100, "delta_t_ms": 5, "map_segments": 0 if scene0.segments is None else int(len(scene0.segments)),
                       "l2_policy": f"inputs larger than L2: {R} world replicas x {bytes_per_launch / 1e6:.1f} MB rotate through the timed steps ({R * bytes_per_launch / 1e6:.0f} MB > {l2_bytes / 1e6:.0f} MB L2)",
                       "timed_region": "CUDA graph of K steps" if graph is not None else "eager launch loop of K steps",
                       "reps": len(reps_ms), "rep_ms_min": min(reps_ms), "rep_ms_max": max(reps_ms),
                       "collective": ("none (1 GPU)" if world_size == 1 else
                                      f"all-gather(done) per step by our own peer-memory kernel (t2d_exchange_allgather_lagged: put + signal per peer, wait, copy; lag {args.lag}: call k delivers the masks of step k - {args.lag}), side stream, overlaps the next tick" if peer is not None else
                                      "all_gather(done) per step (NCCL, side stream, overlaps the next tick)"),
                       "exchange_selfcheck": exchange_check, "prefetch_calibration": prefetch_cal},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "t2d_step_kernel",
                         "bytes_per_launch": bytes_per_launch,
                         "duration_us": ms_per_step * 1e3,
                         "note": "achieved = algorithmic bytes per launch / mean launch duration inside the timed CUDA-graph region"},
        }
        if world_size == 1 and not args.no_cpu_baseline:
            cores = usable_cores()
            n_s = 16
            v1, _ = cpu_port_throughput(scene0, n_s, 1)
            line["cpu_baseline"] = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"first {n_s} of {n} scenarios x {m} participants, 1 step, 1 process (per-agent Python loop; restatement - shapely/GEOS unavailable)"}
            try:
                line["cpu_baseline_compiled"] = {"value": cpu_c_throughput(scene0), "unit": UNIT, "cores": cores, "kind": "port",
                                                 "sample": f"all {n} x {m}, 1 step, C + OpenMP float64 oracle (oracle/c/oracle_tick.c), best of 3"}
            except Exception as e:
                line["cpu_baseline_compiled"] = {"error": str(e)}
        print(json.dumps(line), flush=True)
    if peer is not None:
        torch.cuda.synchronize()
        steps_done, timed_out = peer.status()
        if timed_out:
            print(f"[bench] rank {rank}: the done exchange timed out ({steps_done} steps exchanged)", file=sys.stderr)
            os._exit(3)
    if world_size > 1:
        # leave without tearing NCCL down under a live CUDA graph that captured its collectives (that teardown
        # can dead-lock): drop the graph, drain the device, meet the other ranks, then exit hard.
        graph = None
        import gc

        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    for w in worlds:
        w.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--exchange", choices=("peer", "nccl"), default="peer", help="N > 1: how the done masks are exchanged")
    ap.add_argument("--lag", type=int, default=2, help="peer exchange: deliver the gathered masks this many steps late (0 = synchronous)")
    ap.add_argument("--steps", type=int, default=96)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--replicas", type=int, default=0)
    ap.add_argument("--scenarios", type=int, default=0, help="scenarios per GPU (with --sharded: of the whole job) instead of the configuration's")
    ap.add_argument("--sharded", action="store_true", help="strong scaling: the configuration's scenarios are split across the ranks")
    ap.add_argument("--no-prefetch-cal", action="store_true", help="N > 1: keep the library's prefetch policy instead of timing both settings")
    ap.add_argument("--prefetch-cal-reps", type=int, default=15)
    ap.add_argument("--min-reps", type=int, default=5)
    ap.add_argument("--max-reps", type=int, default=400)
    ap.add_argument("--min-seconds", type=float, default=2.0)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (rank 0's "
                    "state and step results) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

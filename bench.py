#!/usr/bin/env python
"""Throughput benchmark of the MAPF reset()/step() hot path (BASELINE.json metric: agent-steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE config 3, SURVEY 8d "C3"): 65 536 envs x 16 agents PER GPU on a 32x32 map with
30 % i.i.d. obstacles (map seed 2026), sensor_range 2, lifelong goal resampling, lock metrics on,
256 steps per episode with the reset inside the step launch (like run_benchmark's `if done:
reset()`, scripts/benchmark_multi_agent_env.py:89-95), actions uniform over the valid mask.
A "step" is one pass of the hot path over the whole batch: ONE launch of the step kernel, which
also draws the next step's masked-uniform actions (the benchmark sampler fused in).  Envs shard independently across GPUs (weak scaling, no data-path collective); the one
NCCL all-reduce (episode/lock metric sums) runs once after the timed region.

The timed region is exactly `--steps` launches after `--warmup` untimed ones.  `--dump-outputs DIR` then writes what
the last timed step returned (rank 0's shard, a fixed sample of its envs) as float32 / float64 .npy files; the inputs
depend on the arguments only, so two builds run with the same arguments can be compared output for output.

Prints ONE JSON line (rank 0).  `value` = agent-steps/s with inputs resident in HBM; `e2e` = the
same metric through the C ABI's host-buffer entry point (mapf_step_host: pinned host actions in,
all observation/reward/done channels out, copies inside the timed region); `roofline` = the step
kernel against the measured HBM copy bandwidth; `cpu_baseline` = the CPU oracle (a C port of the
reference's Python env) on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))
sys.dont_write_bytecode = True   # the tree may be read-only: no __pycache__ is written next to the sources

METRIC = "agent_steps_per_sec"
UNIT = "agent-steps/s"
# mapf_step_kernel_kind() -> kernel symbol (include/mapf_b200.h)
def kernel_name(kind: int, num_agents: int, sensor_range: int) -> str:
    if kind == 2:
        return f"mapf_step_env_kernel<{sensor_range},...> (env-per-thread)"
    if kind == 3:
        return f"mapf_step_pair_kernel<{sensor_range},...> (two lanes per env)"
    g = 4 if num_agents <= 4 else 8 if num_agents <= 8 else 16 if num_agents <= 16 else 32
    return f"mapf_step_kernel<{g},{sensor_range},...> (lane-per-agent)"


SHAPES = {
    # BASELINE.json configs[2] (the one `metric` is quoted on): the default
    "c3": {"envs": 65536, "agents": 16, "lifelong": True, "steps_per_episode": 256, "map": "32x32",
           "what": "32x32 map (30% obstacles, seed 2026), lifelong goal resampling"},
    # configs[1]: the parity-replay shape, reported for throughput too
    "c2": {"envs": 4096, "agents": 4, "lifelong": False, "steps_per_episode": 100, "map": "10x20",
           "what": "ReferenceModel-2-1 map (10x20), episodic (terminate when all agents are home)"},
    # configs[3]: deadlock-heavy corridors
    "c4": {"envs": 65536, "agents": 32, "lifelong": False, "steps_per_episode": 256, "map": "32x32 corridors",
           "what": "32x32 map of 1-wide corridors, episodic, deadlock-heavy"},
}


def apply_shape(args):
    sh = SHAPES[args.shape]
    if args.envs is None:
        args.envs = sh["envs"]
    if args.agents is None:
        args.agents = sh["agents"]


def workload(args) -> tuple[dict, np.ndarray]:
    from dl_reference_models_b200 import maps

    sh = SHAPES[args.shape]
    if args.shape == "c2":
        grid = maps.get_grid("ReferenceModel-2-1")
    elif args.shape == "c4":
        grid = maps.corridor_grid(32, 32)
    else:
        grid = maps.random_obstacle_grid(32, 32, 0.30, 2026, min_free=2 * args.agents)
    cfg = {
        "num_agents": args.agents, "sensor_range": args.sensor_range, "steps_per_episode": sh["steps_per_episode"],
        "lifelong_mapf": sh["lifelong"], "enable_lock_metrics": True, "deterministic": False, "seed": 999,
        "deadlock_window_steps": 8, "livelock_window_steps": 16,
    }
    return cfg, grid


def config_dict(args, n_gpus: int) -> dict:
    return {
        "workload": f"{args.shape.upper()}: {args.envs} envs x {args.agents} agents per GPU, {SHAPES[args.shape]['what']}, "
                    f"sensor_range {args.sensor_range}, lock metrics on, "
                    f"{SHAPES[args.shape]['steps_per_episode']} steps/episode, in-launch auto-reset, "
                    "masked-uniform actions sampled on device",
        "envs_per_gpu": args.envs, "num_agents": args.agents, "map": SHAPES[args.shape]["map"],
        "sensor_range": args.sensor_range,
        "sharding": f"envs x{n_gpus} (independent shards, no data-path collective)",
        "l2": f"{args.replicas} rotating replicas of the batch (working set > 126 MB L2 between launches)",
    }


def algorithmic_bytes_per_agent_step(N: int, V: int, lock: bool = True, map_bytes: int = 0) -> float:
    """SURVEY 8(d): 33 + V^2 + 28*[lock] + (60 + map_bytes)/N."""
    return 33 + V * V + (28 if lock else 0) + (60 + map_bytes) / N


def measured_peaks() -> tuple[float, str]:
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "10"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def wait_first_sample(self, timeout: float = 10.0):
        t = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.01)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ts, r in self.rows:
            # a sample describes the interval before it: keep those taken under load
            if len(r) < 6 or self.t0 is None or ts < self.t0 + 0.02 or ts > self.t1 + 0.03:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class CpuPort:
    """The CPU oracle (C port of the reference's Python env) on all host cores, timed on bounded
    samples of the bench workload.  bench.py is one of the few places allowed to execute oracle/."""

    def __init__(self, args, threads: int | None = None):
        from oracle import oracle as orc

        self.orc, self.args = orc, args
        self.cfg, self.grid = workload(args)
        self.threads = threads or len(os.sched_getaffinity(0))
        self.envs = orc.bench_envs(self.cfg, self.grid, self.threads * 32)
        n, _, dt, _ = self._run(20)  # calibration: env-steps/s
        self.rate = n / max(dt, 1e-9)

    def _run(self, steps: int):
        return self.orc.bench_run(self.cfg, self.grid, len(self.envs), steps, mode="masked", threads=self.threads,
                                  envs=self.envs)

    def sample(self, seconds: float) -> dict:
        steps = int(max(4, min(1_000_000, seconds * self.rate / len(self.envs))))
        n, episodes, dt, used = self._run(steps)
        self.rate = n / max(dt, 1e-9)
        return {
            "value": n * self.args.agents / dt, "unit": UNIT, "cores": used, "kind": "port",
            "sample": f"{len(self.envs)} envs x {steps} steps ({n} env-steps, {episodes} episodes, {dt:.2f} s) of the "
                      f"same workload on {used} host threads; C port of the reference's Python env "
                      "(oracle/mapf_oracle.c)",
        }


def cpu_port_run(args, seconds: float = 12.0) -> dict:
    return CpuPort(args).sample(seconds)


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The
    reference is pure Python and cannot travel to the GPU box (it is not vendored), so this arm
    times its C port, the oracle -- a generous stand-in (the Python original is ~100x slower)."""
    if rank != 0:
        return
    total = args.warmup + args.steps
    per = min(15.0, 100.0 / max(1, total))
    port = CpuPort(args)
    vals, last = [], None
    t0 = time.perf_counter()
    for i in range(total):
        last = port.sample(per)
        if i >= args.warmup:
            vals.append(last["value"])
    wall = time.perf_counter() - t0
    v = float(np.mean(vals))
    cb = {"value": v, "unit": UNIT, "cores": last["cores"], "kind": "port",
          "sample": f"mean of {len(vals)} samples ({wall:.0f} s in total), the last one: " + last["sample"]}
    line = {
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # one step = one pass over the batch of the b200 arm's step (envs x agents agent-steps), at the measured CPU rate
        "ms_per_step": args.envs * args.agents / v * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int16/u8", "data": "synthetic", "impl": "reference", "config": config_dict(args, args.gpus), "cpu_baseline": cb,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "cpu_baseline_python": python_reference_run(args, seconds=10.0),
    }
    print(json.dumps(line), flush=True)


def source_sha16() -> str:
    """Hash of the kernel sources: ncu-derived numbers (roofline.traffic) are only valid for the build they came from."""
    import hashlib

    h = hashlib.sha256()
    for f in sorted((REPO / "dl_reference_models_b200" / "csrc").glob("*")):
        if f.suffix in (".cu", ".cuh", ".cpp", ".h"):
            h.update(f.read_bytes())
    return h.hexdigest()[:16]


def committed_traffic(shape: str, kind: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
    (profiles/traffic.json), only if it was taken on THIS build of the kernels; else None and the reason."""
    f = REPO / "profiles" / "traffic.json"
    if not f.exists():
        return None, "no capture committed (profiles/traffic.json)"
    try:
        t = json.loads(f.read_text())
    except Exception as exc:
        return None, f"profiles/traffic.json unreadable: {exc}"
    key = f"{shape}_{ {1: 'lane', 2: 'env', 3: 'pair'}.get(kind) }"
    ent = t.get(key)
    if not ent:
        return None, f"no capture for {key} in profiles/traffic.json"
    if ent.get("sources_sha16") != source_sha16():
        return None, (f"capture {ent.get('file')} was taken on kernel sources {ent.get('sources_sha16')}, this build is "
                      f"{source_sha16()}: stale, not reported")
    return float(ent["dram_bytes_per_launch"]), ent.get("file")


class SteadyBatch:
    """`replicas` independent batches of one shape in benchmark state: episode phases staggered uniformly over the
    episode length and randomly over the env ids (so 1/steps_per_episode of the envs end -- and are reset inside the
    launch -- in EVERY step, like run_benchmark's `if done: reset()` in steady state), lock windows full, masked
    sampler fused into the launch."""

    def __init__(self, args, shape: str, dev, rank: int, replicas: int, burn: int = 64):
        import copy

        import torch

        from dl_reference_models_b200 import _native as nat
        from dl_reference_models_b200.batched_env import BatchedMapfEnv

        a = copy.copy(args)
        a.shape, a.envs, a.agents = shape, (args.envs if shape == args.shape else None), (args.agents if shape == args.shape else None)
        apply_shape(a)
        self.args, self.shape = a, shape
        cfg, grid = workload(a)
        cfg["grid"] = grid
        self.cfg = cfg
        self.B, self.N, self.V = a.envs, a.agents, 2 * a.sensor_range + 1
        T = int(cfg["steps_per_episode"])
        self.envs = [BatchedMapfEnv(cfg, self.B, dev, env_id_base=(rank * replicas + r) * self.B) for r in range(replicas)]
        for r, e in enumerate(self.envs):
            e.reset()
            # uniform over the episode, placed at random over the env ids -- what independent episodes of varying
            # length settle into; B / T envs (exactly, when T divides B) end in every step
            g = torch.Generator().manual_seed(2026 + 131 * rank + r)
            phase = torch.randperm(self.B, generator=g) % T
            e.state["env_words"][:, nat.W_STEP_COUNT] = phase.to(device=dev, dtype=torch.int32)
            e._next = e.sample_actions(masked=True)
            e.fuse_sampler("masked")
        self.i = 0
        self.burn_steps = burn
        for _ in range(burn * replicas):   # untimed: fills the lock windows, gets goal arrivals and resets flowing
            self.step()
        self.kind = int(nat.lib().mapf_step_kernel_kind(self.envs[0]._h))

    def step(self):
        e = self.envs[self.i % len(self.envs)]
        self.i += 1
        e.step(e._next, auto_reset=True)
        self.last = e

    def launches(self) -> int:
        return sum(e.launch_count for e in self.envs)

    def metrics_vector(self):
        v = self.envs[0].metrics_vector().clone()
        for e in self.envs[1:]:
            v += e.metrics_vector()
        return v

    def check(self):
        for e in self.envs:
            e.raise_on_device_errors()

    def close(self):
        for e in self.envs:
            e.close()


DUMP_BYTES = 48 << 20   # .npy payload --dump-outputs writes at most


def dump_outputs(env, out_dir: str) -> None:
    """What the env's last step handed its caller -- every output channel, the actions the fused sampler drew for the
    next step, the agents' positions and goals -- as DIR/<name>.npy (info as float64, the rest float32), for a seeded
    sample of the envs that fits DUMP_BYTES (all of them when they fit); env_ids.npy lists the sampled envs."""
    import torch

    from dl_reference_models_b200 import _native as nat

    chans = {k: env.out[k] for k in nat.OUTPUT_FIELDS}
    chans.update(next_actions=env._actions, positions=env.state["positions"], goals=env.state["goals"])
    wide = {"info"}   # int32 counters: float64 keeps them exact
    per_env = sum(t[0].numel() * (8 if k in wide else 4) for k, t in chans.items())
    n = min(env.B, DUMP_BYTES // per_env)
    ids = np.sort(np.random.default_rng(0).choice(env.B, n, replace=False))
    idx = torch.from_numpy(ids).to(env.device)
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "env_ids.npy", ids.astype(np.float64))
    for k, t in chans.items():
        np.save(d / f"{k}.npy", t.index_select(0, idx).cpu().numpy().astype(np.float64 if k in wide else np.float32))


def timed_steps(step, K: int, barrier, torch) -> float:
    """Time exactly K steps (CUDA events on the launching stream, no host sync in between); returns the region's ms."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def timed_blocks(step, K: int, min_seconds: float, barrier, torch, max_blocks: int = 20000):
    """Time blocks of EXACTLY K steps (CUDA events on the launching stream, no host sync between blocks) until the
    region lasts >= min_seconds; returns the per-block times in ms.  One calibration block sizes the region."""
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(K):
        step()
    c1.record()
    torch.cuda.synchronize()
    est = max(c0.elapsed_time(c1), 1e-3)
    nblocks = int(min(max_blocks, max(5, -(-min_seconds * 1e3 // est))))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(nblocks + 1)]
    barrier()
    t_host0 = time.perf_counter()
    ev[0].record()
    for b in range(nblocks):
        for _ in range(K):
            step()
        ev[b + 1].record()
    barrier()
    t_host1 = time.perf_counter()
    return [ev[b].elapsed_time(ev[b + 1]) for b in range(nblocks)], ev[0].elapsed_time(ev[nblocks]), (t_host0, t_host1)


def probe_host_ceilings(torch, dev, barrier, handle) -> dict:
    """What bounds the host-buffer step, measured in this job with every rank probing at once: (1) device-to-host
    DMA into pinned memory (PCIe and, on a multi-GPU node, the host memory system behind it), (2) host-to-device DMA,
    (3) the host cores' streaming copy into cached memory (what the expansion threads and any consumer of the
    delivered arrays have to do).  GB/s per rank."""
    n = 64 << 20
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    out = {}
    for name, (src, dst) in (("d2h_gbs", (d, h)), ("h2d_gbs", (h, d))):
        dst.copy_(src, non_blocking=True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(8):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        out[name] = 8 * n / (e0.elapsed_time(e1) * 1e-3) / 1e9
    # the host cores' streaming fill / copy rate, on the threads (count, pinning) mapf_step_host expands with
    import ctypes as C

    from dl_reference_models_b200 import _native as nat

    th, fill, cp = C.c_int32(0), C.c_double(0.0), C.c_double(0.0)
    barrier()
    nat.check(nat.lib().mapf_host_memory_probe(handle, C.c_int64(256 << 20), C.byref(th), C.byref(fill), C.byref(cp)))
    out["host_fill_gbs"], out["host_copy_gbs"] = fill.value, cp.value
    threads = th.value
    out["host_copy_threads"] = threads
    return out


def run_b200(args, rank: int, local_rank: int, world: int):
    import ctypes as C

    import torch
    import torch.distributed as dist

    from dl_reference_models_b200 import _native as nat
    from dl_reference_models_b200.metrics import AsyncMetrics, summarize

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this framework has no CPU fallback; use --impl reference "
                         "for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def reduce_max(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def reduced_metrics(sb) -> tuple[dict, dict]:
        """The ONE collective of the path, checked on the hardware it runs on: all-reduce(sum) of the per-shard metric
        vector against the sum of the per-rank vectors gathered separately."""
        local = sb.metrics_vector()
        am = AsyncMetrics(local, world, stream=torch.cuda.Stream(dev) if world > 1 else None)
        total = am.result()
        if world > 1:
            parts = [torch.zeros_like(local) for _ in range(world)]
            dist.all_gather(parts, local)
            ref = torch.stack(parts).sum(0)
        else:
            ref = local
        ref_s = summarize(ref)
        keys = ("episodes", "length_sum", "goals_reached_sum", "deadlock_steps_sum", "livelock_steps_sum")
        ok = all(total[k] == ref_s[k] for k in keys) and abs(total["throughput_sum"] - ref_s["throughput_sum"]) <= 1e-9 * max(
            1.0, abs(ref_s["throughput_sum"]))
        chk = {"ok": bool(ok), "ranks": world, "episodes_allreduced": total["episodes"], "episodes_sum_of_ranks": ref_s["episodes"],
               "length_sum_allreduced": total["length_sum"], "length_sum_sum_of_ranks": ref_s["length_sum"]}
        if not ok:
            raise SystemExit(f"bench.py: metric all-reduce disagrees with the sum of the per-rank vectors: {chk}")
        return total, chk

    # ------------------------------------------------------------------ headline shape: device-resident steps
    sb = SteadyBatch(args, args.shape, dev, rank, args.replicas)
    B, N, V = sb.B, sb.N, sb.V
    for _ in range(W):
        sb.step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample()
    launches0 = sb.launches()
    sampler.mark_begin()
    region_ms = timed_steps(sb.step, K, barrier, torch)
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    launches = sb.launches() - launches0
    # one step = ONE launch of the step kernel (checked below): the region's CUDA-event time / K is the kernel's average
    # launch duration, launch gaps included
    assert launches == K, (launches, K)
    sb.check()
    if args.dump_outputs and rank == 0:
        dump_outputs(sb.last, args.dump_outputs)
    region_ms_max = reduce_max(region_ms)                    # slowest rank
    kernel_ms = region_ms_max / K
    metrics, allreduce_check = reduced_metrics(sb)

    # ------------------------------------------------------------------ the same batches through mapf_step_many: K steps per launch
    # (fused-sampler rollouts: every warp takes its tile through the K steps, each step's outputs go to its own rows
    # of a [K, B, ...] rollout buffer -- K x 45 MB of outputs per launch and replica, nothing kept in L2 between launches)
    many = None
    if not args.no_extra_shapes and sb.kind == 2:
        Km = 16
        for e in sb.envs:
            e._roll = e.rollout_buffers(Km)
        mi = [0]

        def many_step():
            e = sb.envs[mi[0] % len(sb.envs)]
            mi[0] += 1
            e.step_many(Km, out=e._roll)

        for _ in range(len(sb.envs)):
            many_step()
        mblocks, _, _ = timed_blocks(many_step, 4, min(args.min_seconds, 0.2), barrier, torch)
        sb.check()
        many_ms = reduce_max(float(np.median(mblocks))) / (4 * Km)
        many = {"steps_per_launch": Km, "ms_per_step": many_ms, "value": world * B * N / (many_ms * 1e-3), "unit": UNIT,
                "api": "mapf_step_many (K env steps per kernel launch, fused masked sampler, [K, B, ...] rollout buffers)"}
        for e in sb.envs:
            del e._roll
        torch.cuda.empty_cache()

    # ------------------------------------------------------------------ e2e: the C ABI's host-buffer entry point
    e2e_env = sb.envs[0]
    e2e_env.fuse_sampler(None)
    host_out = {
        "local_obs": torch.empty((B, N, V, V), dtype=torch.uint8).pin_memory(),
        "action_mask": torch.empty((B, N, 5), dtype=torch.int8).pin_memory(),
        "goal_delta": torch.empty((B, N, 2), dtype=torch.float32).pin_memory(),
        "blocking_prev": torch.empty((B, N), dtype=torch.uint8).pin_memory(),
        "reward": torch.empty((B, N), dtype=torch.float32).pin_memory(),
        "terminated": torch.empty((B,), dtype=torch.uint8).pin_memory(),
        "truncated": torch.empty((B,), dtype=torch.uint8).pin_memory(),
    }
    cout = nat.MapfOutputs(**{k: v.data_ptr() for k, v in host_out.items()})
    gen = torch.Generator().manual_seed(999 + rank)
    host_actions = [torch.randint(0, 5, (B, N), dtype=torch.int8, generator=gen).pin_memory() for _ in range(4)]
    delivered = sum(v.numel() * v.element_size() for v in host_out.values())
    lib = nat.lib()
    Ke, We = max(3, min(K, 50)), 18   # the first sixteen calls are the library's packed / packed + NT / plain calibration
    torch.cuda.synchronize(dev)
    for i in range(We):
        barrier()   # the ranks of a node calibrate their delivery mode in step, like workers that step in step
        nat.check(lib.mapf_step_host(e2e_env._h, C.c_void_p(host_actions[i % 4].data_ptr()), None, None,
                                     C.byref(cout), 1))
    e2e_blocks = []
    for rep in range(3):
        barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            nat.check(lib.mapf_step_host(e2e_env._h, C.c_void_p(host_actions[i % 4].data_ptr()), None, None,
                                         C.byref(cout), 1))
        torch.cuda.synchronize(dev)
        e2e_blocks.append(reduce_max((time.perf_counter() - t0) * 1e3))
    e2e_ms = float(np.median(e2e_blocks))
    checksum = float(host_out["reward"].sum())  # the step's result is really on the host
    # bytes that crossed PCIe in one call (the big per-agent channels travel bit-packed and are expanded into the
    # host arrays by the library's host threads inside the call; `delivered` is the size of the arrays filled)
    c_h2d, c_d2h = C.c_int64(0), C.c_int64(0)
    nat.check(lib.mapf_host_transfer_bytes(e2e_env._h, C.byref(c_h2d), C.byref(c_d2h)))
    h2d, d2h = int(c_h2d.value), int(c_d2h.value)
    # ---- the compact delivery (mapf_step_host_records): the same step, the big channels arrive as bit-packed records
    rs = int(lib.mapf_packed_record_bytes(V * V))
    rec_host = torch.empty((B * N * rs,), dtype=torch.uint8).pin_memory()
    small = {k: torch.empty_like(e2e_env.out[k], device="cpu").pin_memory()
             for k in ("blocking_prev", "terminated", "truncated")}
    csmall = nat.MapfOutputs(**{k: (small[k].data_ptr() if k in small else None) for k in nat.OUTPUT_FIELDS})
    for i in range(3):
        nat.check(lib.mapf_step_host_records(e2e_env._h, C.c_void_p(host_actions[i % 4].data_ptr()), C.c_void_p(rec_host.data_ptr()),
                                             C.byref(csmall), 1))
    rec_blocks = []
    for rep in range(3):
        barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            nat.check(lib.mapf_step_host_records(e2e_env._h, C.c_void_p(host_actions[i % 4].data_ptr()),
                                                 C.c_void_p(rec_host.data_ptr()), C.byref(csmall), 1))
        torch.cuda.synchronize(dev)
        rec_blocks.append(reduce_max((time.perf_counter() - t0) * 1e3))
    rec_ms = float(np.median(rec_blocks))
    nat.check(lib.mapf_host_transfer_bytes(e2e_env._h, C.byref(c_h2d), C.byref(c_d2h)))
    rec_h2d, rec_d2h = int(c_h2d.value), int(c_d2h.value)
    rec_checksum = int(rec_host[: 1 << 16].to(torch.int64).sum())
    ncores = len(os.sched_getaffinity(0))
    ceil = probe_host_ceilings(torch, dev, barrier, e2e_env._h)
    ceil = {k: (reduce_sum(v) if k.endswith("_gbs") else v) for k, v in ceil.items()}   # aggregate over the ranks

    # ------------------------------------------------------------------ the other named shapes, same N (BASELINE configs 4, 5)
    extra = {}
    if not args.no_extra_shapes:
        extra = extra_shapes(args, dev, rank, world, barrier, reduce_max, torch, dist)

    if rank == 0:
        peak, peak_src = measured_peaks()
        bytes_per_as = algorithmic_bytes_per_agent_step(N, V, True, 0)
        alg_bytes = bytes_per_as * B * N
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        value = world * B * N * K / (region_ms_max * 1e-3)
        traffic, traffic_src = (args.traffic_bytes, "--traffic-bytes") if args.traffic_bytes is not None else \
            committed_traffic(args.shape, sb.kind)
        e2e_value = world * B * N * Ke / (e2e_ms * 1e-3)
        pcie_floor_ms = (d2h / 1e9) / max(ceil["d2h_gbs"] / world, 1e-9) * 1e3 + (h2d / 1e9) / max(ceil["h2d_gbs"] / world, 1e-9) * 1e3
        # the expansion's own floor is not a hard one (part of the 45 MB it writes stays in the last-level cache, which
        # a fill probe over fresh memory does not see): reported beside the PCIe floor, not folded into it
        host_fill_ms = (delivered / 1e9) / max(ceil["host_fill_gbs"] / world, 1e-9) * 1e3 if d2h < delivered else 0.0
        floor_ms = pcie_floor_ms
        e2e_mode = int(lib.mapf_host_transfer_mode(e2e_env._h))

        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": region_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16/u8", "data": "synthetic", "impl": "b200", "config": config_dict(args, world),
            "timing": {"timed_steps": K, "region_ms": region_ms_max, "region_ms_rank0": region_ms,
                       "burn_in_steps_per_replica": sb.burn_steps,
                       "note": "one region of exactly `steps` launches after `warmup` untimed ones (slowest rank); "
                               "steady state: episode phases staggered, 1/steps_per_episode of the envs reset inside "
                               "every launch"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": kernel_name(sb.kind, N, args.sensor_range), "kernel_ms": kernel_ms,
                         "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_agent_step": bytes_per_as,
                         "peak_source": peak_src, "sources_sha16": source_sha16()},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "delivered_bytes_per_step": delivered, "steps": Ke,
                    "ms_per_step": e2e_ms / Ke,
                    "api": "mapf_step_host (C ABI, pinned host buffers)",
                    "transfer": ("bit-packed agent records over PCIe, expanded into the host arrays inside the call"
                                 + (" (non-temporal stores)" if e2e_mode == 2 else "")
                                 if d2h < delivered else "plain copies"),
                    "actions": "uniform random from pinned host buffers", "checksum": checksum,
                    "roofline": {"bound": "host DMA (PCIe on one GPU; the node's host memory system when several ranks share it)",
                                 "floor_ms_per_step": floor_ms, "pcie_floor_ms": pcie_floor_ms,
                                 "host_fill_time_ms": host_fill_ms, "frac": floor_ms / (e2e_ms / Ke),
                                 "measured_ceilings_aggregate": ceil, "host_cores": ncores, "delivery_mode": e2e_mode,
                                 "note": "ceilings probed in this job with all ranks at once: pinned D2H / H2D DMA, and the "
                                         "streaming fill / copy rate of the host threads the call expands with; floor = the "
                                         "bytes this step moves over PCIe / the rank's share of the measured DMA rates "
                                         "(delivery_mode: 0 plain copies, 1 packed, 2 packed with the non-temporal expansion; "
                                         "for 1 and 2 on a node shared by many ranks the host memory system, not PCIe, is the "
                                         "bound: see host_fill_time_ms)"}},
            "e2e_compact": {"value": world * B * N * Ke / (rec_ms * 1e-3), "unit": UNIT, "ms_per_step": rec_ms / Ke,
                            "h2d_bytes_per_step": rec_h2d, "d2h_bytes_per_step": rec_d2h, "steps": Ke,
                            "api": "mapf_step_host_records (C ABI, pinned host buffers): the observation / mask / goal-delta / "
                                   "reward channels are delivered as bit-packed records (mapf_unpack_records expands them "
                                   "on the consumer's side, bit for bit), nothing is expanded inside the call",
                            "pcie_floor_ms": (rec_d2h / 1e9) / max(ceil["d2h_gbs"] / world, 1e-9) * 1e3 +
                                             (rec_h2d / 1e9) / max(ceil["h2d_gbs"] / world, 1e-9) * 1e3,
                            "checksum": rec_checksum},
            "step_many": (dict(many, roofline={"bound": "hbm", "achieved": alg_bytes / (many["ms_per_step"] * 1e-3) / 1e9,
                                                "peak": peak, "unit": "GB/s",
                                                "frac": alg_bytes / (many["ms_per_step"] * 1e-3) / 1e9 / peak,
                                                "kernel": kernel_name(sb.kind, N, args.sensor_range) + " (K steps per launch)"})
                          if many else None),
            "gpu_launches": int(reduce_sum(launches) if world > 1 else launches), "clocks": clocks,
            "step_kernel": {1: "lane", 2: "env", 3: "pair"}.get(sb.kind),
            "episode_metrics": {k: metrics[k] for k in ("episodes", "goals_reached_mean", "deadlock_steps_mean",
                                                        "livelock_steps_mean", "throughput_mean", "length_mean")},
            "allreduce_check": allreduce_check,
            "extra_shapes": extra,
        }
    else:
        reduce_sum(launches) if world > 1 else None
    sb.close()
    if rank == 0:
        if not args.no_cpu_baseline:   # rank 0 at every N: the other ranks wait at the barrier below
            line["cpu_baseline"] = cpu_port_run(args, seconds=args.cpu_seconds)
            line["cpu_baseline_python"] = python_reference_run(args, seconds=min(20.0, 2 * args.cpu_seconds))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def extra_shapes(args, dev, rank, world, barrier, reduce_max, torch, dist) -> dict:
    """BASELINE configs[3] and [4] at the same N, short: C4 = 32 agents on corridors with the metric all-reduce issued
    every 256 steps on a side stream WHILE the steps keep launching; C5 = the on-device rollout loop (policy forward +
    env step) beside the env-only rate.  Each with its own roofline entry."""
    from dl_reference_models_b200 import policy_kernels
    from dl_reference_models_b200.metrics import AsyncMetrics
    from dl_reference_models_b200.rollout import ActionMaskPolicy, FusedCollector, collect

    peak, _ = measured_peaks()
    out = {}
    # ---- C4
    sb = SteadyBatch(args, "c4", dev, rank, replicas=2, burn=48)
    steps, every = 768, 256
    side = torch.cuda.Stream(dev)
    pending = []
    for _ in range(8):
        sb.step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        sb.step()
        if (i + 1) % every == 0:   # the reporting interval: snapshot + all-reduce on the side stream, steps go on
            pending.append(AsyncMetrics(sb.metrics_vector(), world, stream=side if world > 1 else None))
    e1.record()
    barrier()
    ms = reduce_max(e0.elapsed_time(e1))
    sb.check()
    reports = [p.result() for p in pending]
    bpa = algorithmic_bytes_per_agent_step(sb.N, sb.V, True, 0)
    if rank == 0:
        ach = bpa * sb.B * sb.N / (ms / steps * 1e-3) / 1e9
        out["c4"] = {"workload": config_dict(sb.args, world)["workload"], "value": world * sb.B * sb.N * steps / (ms * 1e-3),
                     "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "step_kernel": {1: "lane", 2: "env", 3: "pair"}.get(sb.kind),
                     "metric_allreduces_during_stepping": len(reports), "allreduce_every_steps": every,
                     "episodes_reported": [r["episodes"] for r in reports],
                     "deadlock_steps_mean": reports[-1]["deadlock_steps_mean"], "livelock_steps_mean": reports[-1]["livelock_steps_mean"],
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                  "bytes_per_agent_step": bpa, "kernel": kernel_name(sb.kind, sb.N, args.sensor_range)}}
    sb.close()
    # ---- C2: the parity-replay shape is launch-rate bound; mapf_step_many runs K env steps inside one launch
    sb = SteadyBatch(args, "c2", dev, rank, replicas=1, burn=32)
    env = sb.envs[0]
    Kc = 16
    res = {}
    for name, fn, per in (("single", sb.step, 1), ("many", lambda: env.step_many(Kc), Kc)):
        for _ in range(3):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(1, 512 // per)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        barrier()
        res[name] = reduce_max(e0.elapsed_time(e1)) / (reps * per)
    sb.check()
    bpa = algorithmic_bytes_per_agent_step(sb.N, sb.V, True, 0)
    if rank == 0:
        ach = bpa * sb.B * sb.N / (res["many"] * 1e-3) / 1e9
        out["c2"] = {"workload": config_dict(sb.args, world)["workload"], "unit": UNIT,
                     "value": world * sb.B * sb.N / (res["many"] * 1e-3), "ms_per_step": res["many"],
                     "one_launch_per_step": world * sb.B * sb.N / (res["single"] * 1e-3), "ms_per_step_one_launch_per_step": res["single"],
                     "steps_per_launch": Kc, "api": "mapf_step_many (K env steps per kernel launch, fused masked sampler)",
                     "step_kernel": {1: "lane", 2: "env", 3: "pair"}.get(sb.kind),
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                  "bytes_per_agent_step": bpa, "kernel": kernel_name(sb.kind, sb.N, args.sensor_range),
                                  "note": "4 096 envs x 4 agents: 1.6 MB per step, launch-latency bound, not bandwidth bound"}}
    sb.close()
    # ---- C5: rollout loop on the C3 envs
    sb = SteadyBatch(args, "c3", dev, rank, replicas=1, burn=32)
    env = sb.envs[0]
    T = 32
    # env only (fused uniform sampler), same batch
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(T):
        sb.step()
    e1.record()
    barrier()
    env_ms = reduce_max(e0.elapsed_time(e1))
    env.fuse_sampler(None)
    torch.manual_seed(1234 + rank)
    policy = ActionMaskPolicy(env.flat_obs_dim(include_action_mask=False)).to(dev)
    # (a) PyTorch model forward + CUDA env step, as BASELINE words it
    collect(env, policy, 2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    collect(env, policy, 8)
    e1.record()
    barrier()
    torch_ms = reduce_max(e0.elapsed_time(e1))
    # (b) the fused policy kernel (bf16 tensor-core MLP + masked draw) + env step: two launches per step
    fused = policy_kernels.FusedPolicy(policy, env)
    col = FusedCollector(env, fused, T)
    col.collect()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    col.collect()
    e1.record()
    barrier()
    fused_ms = reduce_max(e0.elapsed_time(e1))
    del col
    # (c) the same loop with the compact rollout: the env step writes the observation channels into the rollout rows,
    # the policy kernel stores no float32 feature block (features are expanded per minibatch by the learner)
    col = FusedCollector(env, fused, T, compact=True)
    col.collect()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    col.collect()
    e1.record()
    barrier()
    compact_ms = reduce_max(e0.elapsed_time(e1))
    sb.check()
    if rank == 0:
        n = world * sb.B * sb.N
        F = env.flat_obs_dim(include_action_mask=False)
        # bytes the two launches of one fused step move per agent: env step + policy reads (window, delta, pressure,
        # mask) and its batch rows (f32 features, mask, int64 action, logp, value)
        bpa = algorithmic_bytes_per_agent_step(sb.N, sb.V, True, 0) + (sb.V * sb.V + 8 + 1 + 5) + (4 * F + 5 + 8 + 4 + 4)
        # compact rollout: no float32 feature block, no mask copy (the env step's own channels ARE the batch rows)
        bpa_c = algorithmic_bytes_per_agent_step(sb.N, sb.V, True, 0) + (sb.V * sb.V + 8 + 1 + 5) + (8 + 4 + 4)
        best_ms, best_bpa, best_name = ((compact_ms, bpa_c, "fused policy kernel, compact rollout (uint8 window + float32 delta rows)")
                                        if compact_ms < fused_ms else
                                        (fused_ms, bpa, "fused policy kernel, float32 feature rows"))
        ach = best_bpa * sb.B * sb.N / (best_ms / T * 1e-3) / 1e9
        out["c5"] = {"workload": f"C5: rollout loop on {sb.B} envs x {sb.N} agents per GPU (C3 envs), action-mask MLP "
                                 f"{F}-64-64-(5,1)", "unit": UNIT,
                     "env_only": n * T / (env_ms * 1e-3), "torch_policy_loop": n * 8 / (torch_ms * 1e-3),
                     "fused_policy_loop": n * T / (fused_ms * 1e-3),
                     "fused_policy_loop_compact_rollout": n * T / (compact_ms * 1e-3),
                     "ms_per_step_compact_rollout": compact_ms / T,
                     "value": n * T / (best_ms * 1e-3), "ms_per_step": best_ms / T, "value_is": best_name, "steps": T,
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                  "bytes_per_agent_step": best_bpa, "kernel": "mapf_policy_act_kernel + step kernel (two launches per step)"}}
    del col, fused
    sb.close()
    return out


def python_reference_run(args, seconds: float = 20.0) -> dict:
    """The reference's own Python env, driven the way scripts/benchmark_multi_agent_env.py:59-107 drives it (`masked`
    mode, SURVEY F8 workaround: include_action_mask_in_obs=True), on P processes -- when the reference is on this
    box (/root/reference in the build container; it is not vendored and does not travel to the GPU box)."""
    import multiprocessing as mp

    root = None
    for cand in (Path("/root/reference"), REPO / "baseline" / "_ref"):
        if (cand / "src" / "environments" / "reference_model_multi_agent.py").exists():
            root = cand
            break
    if root is None:
        return {"available": False, "why": "absent on this box: the Python reference is not vendored (looked for "
                                           "/root/reference and baseline/_ref); the C port above is the CPU baseline"}
    P = len(os.sched_getaffinity(0))
    cfg, grid = workload(args)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_python_reference_worker, args=(str(root), cfg, grid, seconds, 123 + i, q)) for i in range(P)]
    t0 = time.perf_counter()
    for p in procs:
        p.start()
    res = [q.get() for _ in procs]
    for p in procs:
        p.join()
    wall = time.perf_counter() - t0
    bad = [r for r in res if "error" in r]
    if bad:
        return {"available": False, "why": f"reference import failed: {bad[0]['error']}"}
    env_steps = sum(r["steps"] for r in res)
    rate = sum(r["steps"] / r["elapsed"] for r in res)
    cpu = ""
    try:
        cpu = next(l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name"))
    except Exception:
        pass
    return {"available": True, "value": rate * args.agents, "unit": UNIT, "kind": "reference", "cores": P, "cpu": cpu,
            "per_process_env_steps_per_s": rate / P,
            "sample": f"{P} processes x run_benchmark-style loop (masked actions, resets inside) of the unmodified "
                      f"reference env at {root}, {env_steps} env-steps in {wall:.1f} s wall, same workload"}


def _python_reference_worker(root, cfg, grid, seconds, seed, q):
    try:
        import logging

        logging.disable(logging.CRITICAL)
        sys.path.insert(0, str(REPO / "oracle" / "ref_stubs"))
        sys.path.insert(1, root)
        from src.environments import get_grid as ref_get_grid
        from src.environments.reference_model_multi_agent import ReferenceModel

        rcfg = {"env_name": "ReferenceModel-2-1", "num_agents": cfg["num_agents"], "sensor_range": cfg["sensor_range"],
                "steps_per_episode": cfg["steps_per_episode"], "lifelong_mapf": cfg["lifelong_mapf"],
                "enable_lock_metrics": True, "deterministic": False, "seed": seed, "render_env": False,
                "deadlock_window_steps": cfg["deadlock_window_steps"], "livelock_window_steps": cfg["livelock_window_steps"],
                "include_action_mask_in_obs": True, "training_execution_mode": "CTDE"}
        orig = ref_get_grid.get_grid
        ref_get_grid.get_grid = lambda name: np.array(grid, dtype=np.uint8)   # synthetic map (SURVEY F10)
        try:
            env = ReferenceModel(rcfg)
        finally:
            ref_get_grid.get_grid = orig
        rng = np.random.default_rng(999 + seed)
        sl = env._obs_slices["action_mask"]
        obs, _ = env.reset()

        def do_step(obs):
            acts = {}
            for a in env.agents:   # scripts/benchmark_multi_agent_env.py:42-57
                valid = np.flatnonzero(obs[a][sl] > 0.5)
                acts[a] = int(rng.choice(valid)) if valid.size else 0
            obs, _, term, trunc, _ = env.step(acts)
            if term["__all__"] or trunc["__all__"]:
                obs, _ = env.reset()
            return obs

        for _ in range(50):
            obs = do_step(obs)
        t0 = time.perf_counter()
        n = 0
        while time.perf_counter() - t0 < seconds:
            for _ in range(20):
                obs = do_step(obs)
            n += 20
        q.put({"steps": n, "elapsed": time.perf_counter() - t0})
    except Exception as exc:  # noqa: BLE001
        q.put({"error": f"{type(exc).__name__}: {exc}"})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed step launches")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
    ap.add_argument("--shape", choices=tuple(SHAPES), default="c3",
                    help="named shape of BASELINE.json (default c3: the one the metric is quoted on)")
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the shape's)")
    ap.add_argument("--agents", type=int, default=None)
    ap.add_argument("--sensor-range", type=int, default=2)
    ap.add_argument("--replicas", type=int, default=4, help="independent batches rotated between launches (L2 defeat)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-shapes", action="store_true", help="skip the C4 / C5 legs of the JSON line")
    ap.add_argument("--min-seconds", type=float, default=0.5,
                    help="the step_many leg repeats blocks of launches until it lasts this long, at most 0.2 s "
                         "(median block reported)")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per step-kernel launch from the committed ncu --set full capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (a seeded sample of rank 0's envs) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    apply_shape(args)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun, one rank per GPU
        import socket
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), str(Path(__file__).resolve())] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()

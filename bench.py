#!/usr/bin/env python3
"""Benchmark of the PGTG hot path (BASELINE.json: env-steps/sec, device-timed, vs CPU PGTGEnv; % HBM
roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

A step = one fused tick (traffic, agent move, reward/termination, same-step auto-reset with
on-device map regeneration, observation write) over every env of the rank's shard. Under torchrun
each rank owns `envs_per_gpu` envs (weak scaling, global env ids, no data-path collective); the only
collective is the episode-statistics all-reduce at the end of the timed region.

Prints ONE JSON line (rank 0):
  value         whole-job env-steps/s of the headline workload (default-2M) with inputs resident in HBM
  e2e           the same through `pgtg_step_host` with pinned HOST buffers (copies inside the timed region)
  e2e_packed    through `pgtg_step_host_packed` (observation planes as bits, 92 B/env instead of 729)
  roofline      algorithmic bytes (SURVEY.md 8d formula) / measured kernel time vs MEASURED_PEAKS.json
  workloads     the other BASELINE configurations and the reference's consumer configuration, each timed
                in this same invocation (N = 1 only): env-steps/s, kernel ms, roofline fraction
  cpu_baseline  the CPU oracle port (C) on the host cores; cpu_baseline_python = the UNMODIFIED reference
                PGTGEnv (oracle/_ref or /root/reference) in a forked runner, one worker per host core

K sets the number of timed steps of the headline loop and of each other workload's loop. --dump-outputs DIR
writes what the last timed step returned to its caller as DIR/<name>.npy (see dump_outputs); the inputs depend on
the arguments alone, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# pgtg/train.py:21-38 of the reference, verbatim, + its TimeLimit(100) (train.py:39)
TRAIN_PY = dict(random_map_width=4, random_map_height=4, random_map_obstacle_probability=0.2, random_map_percentage_of_connections=0.8,
                traffic_density=0.2, conservative_driver_percentage=0.15, normal_driver_percentage=0.50, aggressive_driver_percentage=0.20,
                elderly_driver_percentage=0.10, reckless_driver_percentage=0.05, sliding_observation_window_size=5, max_allowed_deviation=15,
                use_sliding_observation_window=True, use_next_subgoal_direction=True, final_goal_bonus=200, standing_still_penalty=1)

# name -> (PGTGEnv kwargs, envs per GPU, cpu sample envs, extras)
WORKLOADS = {
    # BASELINE config 5 per-GPU shard == the "default map settings" the north star quotes the target on
    "default-2M": (dict(), 2 * 1024 * 1024, 16384, {}),
    # BASELINE config 3
    "traffic-64k": (dict(traffic_density=0.05, random_map_obstacle_probability=0.2), 65536, 4096, {}),
    # BASELINE config 4
    "large-1M": (dict(random_map_width=8, random_map_height=8, random_map_percentage_of_connections=0.8, traffic_density=0.2,
                      random_map_obstacle_probability=0.5), 1024 * 1024, 256, {}),
    # the reference's real consumer: train.py's constructor arguments, TimeLimit(100), FlattenObservation each step
    "train-py": (TRAIN_PY, 262144, 1024, dict(max_episode_steps=100, flat=True)),
    # gymnasium's vector contract: terminal observations of auto-reset envs are written too
    "default-2M+final_observation": (dict(), 2 * 1024 * 1024, 16384, dict(final_observation=True)),
    # the observation of train.py without cars: 11x11 sliding window + next_subgoal_direction (the lean SLIDE tick)
    "sliding-nsd-1M": (dict(use_sliding_observation_window=True, sliding_observation_window_size=5, use_next_subgoal_direction=True), 1024 * 1024, 8192, {}),
    # small smoke-sized run
    "default-64k": (dict(), 65536, 8192, {}),
}
EXTRA = ["traffic-64k", "large-1M", "train-py", "default-2M+final_observation", "sliding-nsd-1M"]


def mean_cars(kw: dict) -> float:
    """Mean number of cars per env of a configuration, from a small probe handle."""
    if not kw.get("traffic_density"):
        return 0.0
    from pgtg_b200 import PGTGVectorEnv

    env = PGTGVectorEnv(2048, seed=1, **kw)
    env.reset()
    n = float(env.get_state()["num_cars"].mean())
    env.close()
    return n


def algorithmic_bytes(kw: dict, n_cars: float) -> float:
    """SURVEY.md 8(d): bytes one env-step must move (int8 planes, scalars, agent state r/w, tile
    descriptors + used bits, car records r/w)."""
    C = len(kw.get("features_to_include_in_observation", [0] * 9))
    P = 9 if not kw.get("use_sliding_observation_window") else 1 + 2 * kw.get("sliding_observation_window_size", 4)
    T = kw.get("random_map_width", 4) * kw.get("random_map_height", 4)
    return C * P * P + 16 + 8 + 2 + 1 + 2 * 16 + T * 2 + 2 * ((T + 7) // 8) + 2 * 8 * n_cars


class ClockSampler:
    """nvidia-smi clocks and throttle reasons DURING the timed region (profiling guide recipe):
    one streaming `nvidia-smi -lms 50` process, rows kept only if sampled inside [begin, end]."""

    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t_begin = self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def begin(self):
        self.t_begin = time.time()

    def end(self):
        self.t_end = time.time()

    def stop(self) -> dict:
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        time.sleep(0.12)
        self.proc.terminate()
        self.thread.join(timeout=3)
        rows = [r for t, r in self.rows if self.t_begin - 0.02 <= t <= self.t_end + 0.08 and len(r) >= 10]
        if not rows:
            rows = [r for _, r in self.rows[-2:] if len(r) >= 10]
        num = lambda v: float(v) if v.replace(".", "", 1).isdigit() else None  # noqa: E731
        sm = [num(r[2]) for r in rows if num(r[2]) is not None]
        mx = [num(r[3]) for r in rows if num(r[3]) is not None]
        pw = [num(r[4]) for r in rows if num(r[4]) is not None]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons),
                    power_w_max=max(pw) if pw else None, samples=len(rows))


# ---- CPU arms ------------------------------------------------------------------------------------
def cpu_port(kw: dict, n_envs: int, seconds: float, threads: int, extras: dict) -> dict:
    """The oracle (C port of the reference tick, oracle/pgtg_oracle.c) on the host cores."""
    from oracle.oracle import OracleVectorEnv

    env = OracleVectorEnv(num_envs=n_envs, threads=threads, seed=1, max_episode_steps=extras.get("max_episode_steps"), **kw)
    env.reset()
    rng = np.random.default_rng(0)
    acts = [rng.integers(0, 9, n_envs).astype(np.int32) for _ in range(4)]
    env.step(acts[0])
    t0, steps = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        env.step(acts[steps % 4])
        steps += 1
    dt = time.perf_counter() - t0
    env.close()
    return dict(value=n_envs * steps / dt, unit="env-steps/s", cores=threads, kind="port",
                sample=f"{n_envs} envs x {steps} ticks ({dt:.1f} s) of the same workload, C oracle port, {threads} threads, incl. auto-reset")


def cpu_python(kw: dict, seconds: float, extras: dict) -> dict | None:
    """The UNMODIFIED reference PGTGEnv (environment.py:581, 1092), forked runner with one worker per host core
    (oracle/ref_pool.py: how train.py:54 consumes it), same kwargs, uniform random actions, same-step auto-reset."""
    from oracle.ref_pool import ReferencePool, reference_root

    if reference_root() is None:
        return None
    cores = os.cpu_count() or 1
    ref_kw = {k: v for k, v in kw.items()}
    pool = ReferencePool(ref_kw, workers=cores, envs_per_worker=4, seed=0, max_episode_steps=extras.get("max_episode_steps"))
    try:
        r = pool.run(seconds)
    finally:
        pool.close()
    return dict(value=r["value"], unit="env-steps/s", cores=cores, kind="reference",
                sample=f"{pool.num_envs} reference PGTGEnv ({cores} forked workers x 4) x {r['env_steps'] // pool.num_envs} ticks ({r['seconds']:.1f} s), "
                       f"{r['resets']} auto-resets, source {os.path.relpath(pool.root, ROOT) if pool.root.startswith(ROOT) else pool.root}")


def run_reference(args, kw, n_cpu, extras):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, all of them:
    the unmodified Python PGTGEnv from oracle/_ref (kind "reference") when staged, else the C oracle port."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle.ref_pool import ReferencePool, reference_root

    cores = os.cpu_count() or 1
    rng = np.random.default_rng(0)
    if reference_root() is not None:
        pool = ReferencePool(dict(kw), workers=cores, envs_per_worker=4, seed=0, max_episode_steps=extras.get("max_episode_steps"))
        n = pool.num_envs
        t0 = time.perf_counter()
        pool.step(rng.integers(0, 9, n))
        tick_s = max(time.perf_counter() - t0, 1e-3)
        # one "step" of this arm = `inner` ticks of every env of the pool: ~0.5 s, the whole run within ~2.5 minutes
        inner = max(1, min(int(0.5 / tick_s), int(150.0 / (tick_s * max(args.steps + args.warmup, 1)))))
        step = lambda: [pool.step(rng.integers(0, 9, n)) for _ in range(inner)]  # noqa: E731
        kind, close = "reference", pool.close
        sample = (f"{n} unmodified reference PGTGEnv ({cores} forked workers x 4, {os.path.basename(pool.root)}) x {inner} ticks per step, "
                  "uniform random actions, same-step auto-reset")
    else:
        from oracle.oracle import OracleVectorEnv

        env = OracleVectorEnv(num_envs=n_cpu, threads=cores, seed=1, max_episode_steps=extras.get("max_episode_steps"), **kw)
        env.reset()
        n, inner = n_cpu, 8
        step = lambda: [env.step(rng.integers(0, 9, n).astype(np.int32)) for _ in range(inner)]  # noqa: E731
        kind, close = "port", env.close
        sample = f"{n} envs x {inner} ticks per step, C oracle port of the reference tick (oracle/_ref not staged), {cores} threads, incl. auto-reset"
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    close()
    value = n * inner * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32+f64", "data": "synthetic", "config": {"workload": args.workload, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---- GPU side ------------------------------------------------------------------------------------
def make_env(name, N, dev, rank, final_observation=False):
    from pgtg_b200 import PGTGVectorEnv

    kw, _, _, extras = WORKLOADS[name]
    return PGTGVectorEnv(N, device=dev, seed=2026, env_id_base=rank * N, final_observation=final_observation or extras.get("final_observation", False),
                         max_episode_steps=extras.get("max_episode_steps"), **kw)


def action_pool(N, dev, rank):
    import torch

    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    return [torch.randint(0, 9, (N,), device=dev, dtype=torch.int32, generator=g) for _ in range(8)]


def time_kernels_alone(env, pool, steps, flat):
    """The tick kernel timed ALONE (overlap off: kernels back to back on this stream), CUDA events around each launch."""
    env.raw.set_overlap(False)
    for i in range(3):
        env.step(pool[i % 8])
    env.raw.enable_timing(steps)
    for i in range(steps):
        env.step(pool[i % 8])
        if flat:
            env.flat_observation()
    alone = env.raw.timing()
    env.raw.enable_timing(0)
    env.raw.set_overlap(not os.environ.get("PGTG_NO_OVERLAP"))
    return alone


DUMP_BUDGET = 60 * 2**20  # bytes of arrays; the rest of the 64 MiB allowed is headroom for the .npy headers


def dump_outputs(path, step_out, flat_obs=None):
    """Write what one `env.step` returned to its caller (observation dict, reward, terminated, truncated, info
    dict) and, for flattened workloads, the `flat_observation` tensor, one DIR/<name>.npy per array (nested keys
    joined with '.'). float64 arrays stay float64; everything else is written as float32, which holds its
    small integers exactly. When all envs do not fit DUMP_BUDGET, a fixed-seed sample of envs is written, the
    same rows of every array; env_index.npy lists them."""
    from collections.abc import Mapping

    import torch

    arrays = {}

    def collect(name, v):
        if isinstance(v, Mapping):
            for k in v:
                collect(f"{name}.{k}", v[k])
        elif isinstance(v, torch.Tensor):
            arrays[re.sub(r"[^\w.-]", "_", name)] = v

    for name, v in zip(("obs", "reward", "terminated", "truncated", "info"), step_out):
        collect(name, v)
    if flat_obs is not None:
        collect("obs_flat", flat_obs)
    n = next(iter(arrays.values())).shape[0]
    row_bytes = 8 + sum(v[0].numel() * (8 if v.dtype == torch.float64 else 4) for v in arrays.values())
    keep = min(n, DUMP_BUDGET // row_bytes)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name, v in arrays.items():
        rows = v.index_select(0, torch.from_numpy(idx).to(v.device)).cpu().numpy()
        np.save(os.path.join(path, f"{name}.npy"), rows.astype(np.float64 if v.dtype == torch.float64 else np.float32))


def measure_workload(name, dev, peak, steps=None):
    """One of the other configurations, timed in this invocation: a short device-timed loop + the kernels alone."""
    import torch

    kw, N, _, extras = WORKLOADS[name]
    flat = bool(extras.get("flat"))
    env = make_env(name, N, dev, 0)
    env.reset()
    pool = action_pool(N, dev, 0)
    for i in range(4):
        env.step(pool[i % 8])
        if flat:
            env.flat_observation()
    torch.cuda.synchronize()
    # size the loop from a probe step: ~0.4 s of device time, 8..200 steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); env.step(pool[0]); e1.record(); torch.cuda.synchronize()
    k = steps or int(max(8, min(200, 400.0 / max(e0.elapsed_time(e1), 1e-3))))
    launches0 = env.launch_count()
    e0.record()
    for i in range(k):
        env.step(pool[i % 8])
        if flat:
            env.flat_observation()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    launches = env.launch_count() - launches0
    alone = time_kernels_alone(env, pool, min(k, 30), flat)
    info = env.raw.kernel_info()
    stats = env.episode_stats(reset=True, all_reduce=False)
    env.close()
    del env
    torch.cuda.empty_cache()
    b_alg = algorithmic_bytes(kw, mean_cars(kw))
    return dict(env_steps_per_s=N * 1e3 / ms, envs=N, steps=k, ms_per_step=ms, kernel_ms=alone["tick_ms"], mapgen_ms=alone["mapgen_ms"],
                gpu_launches=int(launches), kernels=info, flat_observation=flat, final_observation=bool(extras.get("final_observation")),
                max_episode_steps=extras.get("max_episode_steps"), mean_episode_length=stats["mean_length"],
                roofline={"bound": "hbm", "algorithmic_bytes_per_env_step": b_alg, "achieved": b_alg * N / (alone["tick_ms"] * 1e-3) / 1e9,
                          "peak": peak, "unit": "GB/s", "frac": b_alg * N / (alone["tick_ms"] * 1e-3) / 1e9 / peak,
                          "whole_step_frac": b_alg * N / (ms * 1e-3) / 1e9 / peak})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="default-2M", choices=list(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (overrides the workload's)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=6.0)
    ap.add_argument("--python-seconds", type=float, default=4.0, help="the unmodified Python reference beside the GPU path (0 = skip)")
    ap.add_argument("--no-extra", action="store_true", help="skip the other workloads")
    ap.add_argument("--final-observation", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0's envs) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    kw, n_gpu_envs, n_cpu, extras = WORKLOADS[args.workload]
    if args.envs:
        n_gpu_envs = args.envs
    if args.impl == "reference":
        run_reference(args, kw, n_cpu, extras)
        return

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    N = n_gpu_envs
    flat = bool(extras.get("flat"))
    # host threads and the pinned buffers allocated below on the GPU's own NUMA node (the e2e legs are host-copy bound)
    from pgtg_b200.distributed import bind_to_gpu_numa_node

    full_affinity = os.sched_getaffinity(0)
    numa = None if os.environ.get("PGTG_NO_NUMA_BIND") else bind_to_gpu_numa_node(local)
    env = make_env(args.workload, N, dev, rank, args.final_observation)
    env.reset()
    pool = action_pool(N, dev, rank)
    for i in range(max(args.warmup, 3)):
        env.step(pool[i % 8])
        if flat:
            env.flat_observation()
    env.episode_stats(reset=True)  # first call loads the reduction kernel; not part of the timed region
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed region: K fused launches, inputs resident in HBM -------------------------
    launches0 = env.launch_count()
    env.raw.enable_timing(args.steps)  # CUDA events around each kernel, on the launching stream
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    barrier()
    if sampler:
        sampler.begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev0.record()
    for i in range(args.steps):
        kev[i][0].record()
        last = env.step(pool[i % 8])
        last_flat = env.flat_observation() if flat else None
        kev[i][1].record()
    stats = env.episode_stats(all_reduce=True)  # the only collective: 8 doubles, once
    ev1.record()
    barrier()
    if args.dump_outputs and rank == 0:  # before any further step overwrites the buffers `last` views
        dump_outputs(args.dump_outputs, last, last_flat)
    ms = ev0.elapsed_time(ev1)
    step_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    ktime = env.raw.timing()
    env.raw.enable_timing(0)
    launches = env.launch_count() - launches0
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * N * args.steps / (ms * 1e-3)

    # ---- the dominant kernel timed ALONE ------------------------------------------------------------
    alone_steps = min(args.steps, 40)
    alone = time_kernels_alone(env, pool, alone_steps, flat)
    env.episode_stats(reset=True)

    # ---- end to end through the host-buffer entries -------------------------------------------------
    C, P = env.hc.pod.num_channels, env.hc.window
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()  # noqa: E731
    out = dict(obs_map=pin((N, C, P, P), torch.int8), obs_position=pin((N, 2), torch.int32), obs_velocity=pin((N, 2), torch.int32),
               reward=pin((N,), torch.float64), terminated=pin((N,), torch.uint8), truncated=pin((N,), torch.uint8))
    hact = [torch.randint(0, 9, (N,), dtype=torch.int32).pin_memory().numpy() for _ in range(2)]

    def timed_host_loop(fn, steps):
        fn(hact[0])
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(hact[i % 2])
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        tt = torch.tensor([s], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return world * N * steps / float(tt.item())

    e2e_value = e2e_packed = None
    packed_bytes = 0
    if args.e2e_steps > 0:
        e2e_value = timed_host_loop(lambda a: env.step_host(a, out), args.e2e_steps)
        if hasattr(env, "step_host_packed"):
            pout = env.packed_host_buffers(pinned=True)
            packed_bytes = sum(v.nbytes for v in pout.values())
            e2e_packed = timed_host_loop(lambda a: env.step_host_packed(a, pout), args.e2e_steps * 4)
    os.sched_setaffinity(0, full_affinity)  # the CPU baselines below use every core the process was given
    if sampler:
        sampler.end()
    clocks = sampler.stop() if sampler else None
    h2d = N * 4
    d2h = sum(v.nbytes for v in out.values())
    info = env.raw.kernel_info()
    env.close()
    del env
    torch.cuda.empty_cache()

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        b_alg = algorithmic_bytes(kw, mean_cars(kw))
        kernel_ms = alone["tick_ms"]
        achieved = b_alg * N / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = None, "not measured in this run (ncu is not run inside bench.py)"
        tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
        if os.path.exists(tpath):
            rec = json.load(open(tpath)).get(args.workload)
            if isinstance(rec, dict):
                traffic, traffic_src = rec.get("bytes_per_launch"), rec.get("source")
        workloads = {}
        if world == 1 and not args.no_extra and args.workload == "default-2M":
            for name in EXTRA:
                try:
                    workloads[name] = measure_workload(name, dev, peak, args.steps)
                except Exception as exc:  # keep the headline line even if an extra workload fails
                    workloads[name] = {"error": repr(exc)}
        cpu = cpu_port(kw, n_cpu, args.cpu_seconds, os.cpu_count() or 1, extras) if args.cpu_seconds > 0 else None
        cpu_py = None
        if args.python_seconds > 0:
            try:
                cpu_py = cpu_python(kw, args.python_seconds, extras)
            except Exception as exc:
                cpu_py = {"error": repr(exc)}
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32+f64", "data": "synthetic",
            "config": {"workload": args.workload, "envs_per_gpu": N, "kwargs": kw, "actions": "uniform random, 8 resident int32 tensors cycled",
                       "rng": "philox4x32-10 per env", "auto_reset": "same step, on-device map regeneration", "kernels": info,
                       "final_observation": bool(args.final_observation or extras.get("final_observation")), "flat_observation": flat,
                       "l2": f"working set {(b_alg * N) / 1e6:.0f} MB per step > 126 MB L2 (no flush needed)"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps, "path": "pgtg_step_host: pinned host actions in, int8 observation planes / reward / flags out"},
            "e2e_packed": {"value": e2e_packed, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": packed_bytes,
                           "path": "pgtg_step_host_packed: observation planes as bits (pgtg_unpack_obs restores the int8 planes on the host), double-buffered"},
            "gpu_launches": int(launches),
            "numa": numa,  # what bind_to_gpu_numa_node did for this rank (None: topology not exposed)
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_env_step": b_alg, "kernel_ms": kernel_ms,
                         "kernel": info,
                         "note": "kernel_ms/achieved/frac: the tick kernel timed alone (overlap off, CUDA events around the launch, "
                                 f"{alone_steps} launches); in the pipeline it shares the SMs with the map-generation kernel",
                         "tick_ms_in_pipeline": ktime["tick_ms"], "mapgen_ms_in_pipeline": ktime["mapgen_ms"],
                         "mapgen_ms_alone": alone["mapgen_ms"], "step_ms": step_ms,
                         "whole_step_frac": b_alg * N / (step_ms * 1e-3) / 1e9 / peak},
            "workloads": workloads,
            "cpu_baseline": cpu,
            "cpu_baseline_python": cpu_py,
            "episode_stats": stats,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

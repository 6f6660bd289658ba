"""Level sets on the GPU: env-steps/s with a pool of generated maps against fresh maps per episode, and the level-serving
kernel against the map generator it replaces.

For each workload the handles (num_levels = 0 and each level-set size) are built once and timed in alternating rounds with
CUDA events around `steps` steps (whole step: tick + map filling, overlapped as in normal use); then each handle runs with
overlap off, so that the tick and the map-filling kernel (generator or level server) are timed alone. The card's name and
power limit are read in the same run. Writes one JSON document to stdout and, with --out, to a file.

    python tools/bench_levels.py --steps 60 --rounds 3 --out bench_levels.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (label, bench.py workload, extra kwargs, level-set sizes)
CASES = [
    ("default-2M", "default-2M", {}, [0, 200, 100_000]),
    ("default-2M+final_observation", "default-2M", dict(final_observation=True), [0, 200, 100_000]),
    ("sliding-nsd-1M", "sliding-nsd-1M", {}, [0, 200]),
    ("traffic-64k", "traffic-64k", {}, [0, 200]),
]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_levels.py measures the CUDA kernels: no CUDA device")
    from bench import WORKLOADS
    from pgtg_b200 import PGTGVectorEnv

    dev = torch.device("cuda", 0)
    result = dict(card=card(), steps=args.steps, rounds=args.rounds, workloads={})
    for label, wl, extra, sizes in CASES:
        kw, N, _, _ = WORKLOADS[wl]
        envs = {}
        for M in sizes:
            envs[M] = PGTGVectorEnv(N, device=dev, seed=2026, num_levels=M, **kw, **extra)
            envs[M].reset()
        g = torch.Generator(device=dev)
        g.manual_seed(1234)
        pool = [torch.randint(0, 9, (N,), device=dev, dtype=torch.int32, generator=g) for _ in range(8)]
        for env in envs.values():
            for i in range(args.warmup):
                env.step(pool[i % 8])
        torch.cuda.synchronize()
        times = {M: [] for M in sizes}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):  # alternating: one timed loop of every handle per round
            for M, env in envs.items():
                e0.record()
                for i in range(args.steps):
                    env.step(pool[i % 8])
                e1.record()
                torch.cuda.synchronize()
                times[M].append(e0.elapsed_time(e1) / args.steps)
        rows = {}
        for M, env in envs.items():
            env.raw.set_overlap(False)
            for i in range(3):
                env.step(pool[i % 8])
            env.raw.enable_timing(args.steps)
            for i in range(args.steps):
                env.step(pool[i % 8])
            alone = env.raw.timing()
            env.raw.enable_timing(0)
            best = min(times[M])
            rows[str(M)] = dict(kernel_info=env.raw.kernel_info(), step_ms=times[M], env_steps_per_s=N / (best * 1e-3),
                                tick_alone_ms=alone["tick_ms"], map_fill_alone_ms=alone["mapgen_ms"])
            env.close()
        result["workloads"][label] = dict(num_envs=N, levels=rows)
        del envs
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

"""The bits observation format on the GPU: env-steps/s and the tick alone, int8 against bits; the unpack kernel; a rollout proxy.

For each workload an int8 handle and a bits handle are built once and timed in alternating rounds with CUDA events around
`steps` steps. Then, per handle: the tick and map generation alone (overlap off, pgtg_timing); a rollout proxy, each step
followed by a copy of the step's planes into a T-slot store (int8: obs_map, bits: obs_packed). For the bits handle: the unpack
kernel to int8 over all N rows of one slot, and (train-py) to float32 against pgtg_flatten of the int8 handle. The card's name
and power limit are read in the same run. Writes one JSON document to stdout and, with --out, to a file.

    python tools/bench_obs_bits.py --steps 40 --rounds 3 --out bench_obs_bits.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (label, bench.py workload, extra kwargs)
CASES = [
    ("default-2M", "default-2M", {}),
    ("default-2M+final_observation", "default-2M", dict(final_observation=True)),
    ("sliding-nsd-1M", "sliding-nsd-1M", {}),
    ("traffic-64k", "traffic-64k", {}),
    ("train-py", "train-py", dict(max_episode_steps=100)),
]
SLOTS = 8  # rollout store of the proxy


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default=None, help="comma-separated labels")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_obs_bits.py measures the CUDA kernels: no CUDA device")
    from bench import WORKLOADS
    from pgtg_b200 import PGTGVectorEnv

    dev = torch.device("cuda", 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n):
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    result = dict(card=card(), steps=args.steps, rounds=args.rounds, workloads={})
    for label, wl, extra in CASES:
        if args.only and label not in args.only.split(","):
            continue
        kw, N, _, _ = WORKLOADS[wl]
        envs = {fmt: PGTGVectorEnv(N, device=dev, seed=2026, observation_format=fmt, **kw, **extra) for fmt in ("int8", "bits")}
        g = torch.Generator(device=dev)
        g.manual_seed(1234)
        pool = [torch.randint(0, 9, (N,), device=dev, dtype=torch.int32, generator=g) for _ in range(8)]
        for env in envs.values():
            env.reset()
            for i in range(args.warmup):
                env.step(pool[i % 8])
        torch.cuda.synchronize()
        times = {fmt: [] for fmt in envs}
        for _ in range(args.rounds):  # alternating: one timed loop of every handle per round
            for fmt, env in envs.items():
                times[fmt].append(timed(lambda i, env=env: env.step(pool[i % 8]), args.steps))
        rows = {}
        for fmt, env in envs.items():
            buf = env.obs_packed() if fmt == "bits" else env._t["obs_map"].view(N, -1)
            store = torch.empty((SLOTS,) + tuple(buf.shape), dtype=buf.dtype, device=dev)

            def rollout(i, env=env, store=store, fmt=fmt):
                env.step(pool[i % 8])
                store[i % SLOTS].copy_(env.obs_packed() if fmt == "bits" else env._t["obs_map"].view(N, -1))

            rollout_ms = min(timed(rollout, args.steps) for _ in range(args.rounds))
            env.raw.set_overlap(False)
            for i in range(3):
                env.step(pool[i % 8])
            env.raw.enable_timing(args.steps)
            for i in range(args.steps):
                env.step(pool[i % 8])
            alone = env.raw.timing()
            env.raw.enable_timing(0)
            env.raw.set_overlap(True)
            best = min(times[fmt])
            rows[fmt] = dict(kernel_info=env.raw.kernel_info(), step_ms=times[fmt], env_steps_per_s=N / (best * 1e-3), tick_alone_ms=alone["tick_ms"],
                             mapgen_alone_ms=alone["mapgen_ms"], rollout_step_plus_copy_ms=rollout_ms, rollout_slot_bytes=buf.numel() * buf.element_size())
            if fmt == "bits":
                rows[fmt]["unpack_int8_all_rows_ms"] = min(timed(lambda i: env.unpack(store[i % SLOTS]), args.steps) for _ in range(args.rounds))
        if label == "train-py":
            b, a = envs["bits"], envs["int8"]
            pos = torch.empty((SLOTS, N, 2), dtype=torch.int32, device=dev)
            vel, nsd = torch.empty_like(pos), torch.zeros((SLOTS, N), dtype=torch.int32, device=dev)
            bits = b.obs_packed().clone().unsqueeze(0).expand(SLOTS, -1).contiguous()
            def flat_one_slot(i):
                s = i % SLOTS
                b.unpack(bits[s], format="flat", position=pos[s], velocity=vel[s], next_subgoal_direction=nsd[s] if b.use_next_subgoal_direction else None)

            rows["bits"]["unpack_flat_one_slot_ms"] = min(timed(flat_one_slot, args.steps) for _ in range(args.rounds))
            rows["int8"]["flatten_ms"] = min(timed(lambda i: a.flat_observation(), args.steps) for _ in range(args.rounds))
            rows["bits"]["flatten_ms"] = min(timed(lambda i: b.flat_observation(), args.steps) for _ in range(args.rounds))
        result["workloads"][label] = dict(num_envs=N, formats=rows)
        for env in envs.values():
            env.close()
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

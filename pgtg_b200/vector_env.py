"""`PGTGVectorEnv` -- the batched, GPU-resident drop-in for rollouts of the reference `PGTGEnv`.

Mirrors the reference's public surface (pgtg/environment.py):
  * constructor keyword arguments and defaults of `PGTGEnv.__init__` (:302-359);
  * `single_action_space = Discrete(9)` (:415) and the observation Dict (:417-441);
  * `reset(seed)` (:581) and `step(action)` (:1092) with the reward / terminated / truncated
    semantics of the reference; truncation comes from `max_episode_steps` (the reference uses a
    `TimeLimit` wrapper, train.py:39);
  * gymnasium 0.28.1 vector semantics (the version pinned by the reference's poetry.lock): env i is
    seeded with `seed + i`, and an env that finishes is reset inside the same `step` call -- the
    returned observation is the first observation of the new episode, the terminal one is under
    `info["final_observation"]` when `final_observation=True`.

All state lives in HBM; `step` is one fused CUDA launch enqueued on torch's current stream with no
host synchronisation. Observations, rewards and flags are torch views (DLPack) of buffers owned
by the native handle -- valid until the next `step`/`reset`; clone what must outlive it.
"""
from __future__ import annotations

from collections.abc import Mapping, MutableMapping
from typing import Any

import numpy as np
import torch

from . import spaces
from .config import AGENT_DIRECTIONS, PROFILE_NAMES, RNG_PHILOX, RNG_TAPE, HostConfig, make_config
from ._names import ROUTE_NAMES
from .raw import RawEnv


class LazyInfo(MutableMapping):
    """`info` of a step: entries that cost a kernel launch (bit tests on `step_flags`) are computed on
    first access, so a rollout loop that ignores them pays nothing. A Mapping rather than a dict
    subclass, so that `dict(info)`, `{**info}` and wrappers that copy infos go through `__getitem__`
    and see the materialised values."""

    def __init__(self, *a, **k):
        self._d = dict(*a, **k)
        self._lazy = {}

    def lazy(self, key, fn):
        self._lazy[key] = fn
        self._d[key] = None

    def __getitem__(self, key):
        if key in self._lazy:
            self._d[key] = self._lazy.pop(key)()
        return self._d[key]

    def __setitem__(self, key, value):
        self._lazy.pop(key, None)
        self._d[key] = value

    def __delitem__(self, key):
        self._lazy.pop(key, None)
        del self._d[key]

    def __iter__(self):
        return iter(self._d)

    def __len__(self):
        return len(self._d)

    def __repr__(self):
        return f"LazyInfo({dict(self)!r})"


class LazyPlanes(Mapping):
    """`obs["map"]` of the bits observation format: the planes are expanded from the stored bits into the int8 buffer by one
    kernel (`pgtg_expand_obs`) on first access, then the usual per-key views of that buffer are returned. A loop that never
    looks at the planes pays nothing. Like the int8 views, valid until the next `step`/`reset`."""

    def __init__(self, keys, expand):
        self._keys = list(keys)
        self._expand = expand
        self._views = None

    def _get(self):
        if self._views is None:
            self._views = self._expand()
        return self._views

    def __getitem__(self, key):
        return self._get()[key]

    def __iter__(self):
        return iter(self._keys)

    def __len__(self):
        return len(self._keys)

    def __repr__(self):
        return f"LazyPlanes({self._keys!r}, expanded={self._views is not None})"


def _device_index(device) -> int:
    d = torch.device(device)
    if d.type != "cuda":
        raise RuntimeError("PGTGVectorEnv runs on CUDA devices only (there is no CPU fallback)")
    return torch.cuda.current_device() if d.index is None else d.index


class PGTGVectorEnv:
    metadata = {"render_modes": []}

    def __init__(self, num_envs: int = 1, map_path: str | None = None, *, device="cuda", conformance_draws=None,
                 **kwargs: Any):
        if not torch.cuda.is_available():
            raise RuntimeError("PGTGVectorEnv needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device_index = _device_index(device)
        self.device = torch.device("cuda", self.device_index)
        if conformance_draws is not None:
            kwargs["rng_mode"] = RNG_TAPE
        self._ctor = (num_envs, map_path, dict(kwargs))
        self._shadow = None
        self.hc: HostConfig = make_config(map_path, num_envs=num_envs, **kwargs)
        self.num_envs = num_envs
        with torch.cuda.device(self.device):
            self.raw = RawEnv(self.hc, device=self.device_index)
            self._t = {}
            for name in ("obs_map", "obs_position", "obs_velocity", "obs_next_subgoal_direction", "reward", "cost",
                         "terminated", "truncated", "step_state", "step_flags", "stats"):
                self._t[name] = torch.from_dlpack(self.raw.dlpack_capsule(name))
            if self.hc.pod.write_final_obs:
                for name in ("final_obs_map", "final_obs_position", "final_obs_velocity", "final_obs_next_subgoal_direction"):
                    self._t[name] = torch.from_dlpack(self.raw.dlpack_capsule(name))
            self._actions = torch.zeros(num_envs, dtype=torch.int32, device=self.device)
        if conformance_draws is not None:
            self.raw.load_draws(*conformance_draws)
        self.observation_format = self.hc.observation_format
        self._terminated = self._t["terminated"].view(torch.bool)
        self._truncated = self._t["truncated"].view(torch.bool)

        P = self.hc.window
        kw = self.hc.kwargs
        self.use_next_subgoal_direction = bool(kw["use_next_subgoal_direction"])
        self.separate_reward_cost = bool(kw["separate_reward_cost"])
        self.single_action_space = spaces.Discrete(9)
        obs_space = {
            "position": spaces.MultiDiscrete([9, 9], dtype=np.int32),
            "velocity": spaces.Box(low=-99, high=99, shape=(2,), dtype=np.int32),
            "map": spaces.Dict({k: spaces.MultiBinary((P, P)) for k in self.hc.observation_keys}),
        }
        if self.use_next_subgoal_direction:
            obs_space["next_subgoal_direction"] = spaces.Discrete(9, start=-1)
        self.single_observation_space = spaces.Dict(obs_space)
        self.action_space = spaces.MultiDiscrete([9] * num_envs)
        self.observation_space = spaces.batch_space(self.single_observation_space, num_envs)
        self._was_reset = False

    # ---- Gymnasium vector API ----------------------------------------------------------------
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _observation(self, final: bool = False) -> dict:
        pre = "final_" if final else ""
        m = self._t[pre + "obs_map"]
        keys = self.hc.observation_keys
        if self.observation_format == "bits":
            def expand():
                with torch.cuda.device(self.device):
                    self.raw.expand_obs(final, self._stream())
                return {k: m[:, i] for i, k in enumerate(keys)}
            planes = LazyPlanes(keys, expand)
        else:
            planes = {k: m[:, i] for i, k in enumerate(keys)}
        obs = {
            "position": self._t[pre + "obs_position"],
            "velocity": self._t[pre + "obs_velocity"],
            "map": planes,
        }
        if self.use_next_subgoal_direction:
            obs["next_subgoal_direction"] = self._t[pre + "obs_next_subgoal_direction"]
        return obs

    def reset(self, *, seed: int | list | np.ndarray | None = None, options: dict | None = None):
        seeds = None
        if seed is not None:
            seeds = np.asarray(seed, dtype=np.int64)
            if seeds.ndim == 0:  # env i of the whole (possibly sharded) job is seeded seed + global index
                seeds = int(seeds) + int(self.hc.pod.env_id_base) + np.arange(self.num_envs, dtype=np.int64)
            if seeds.shape != (self.num_envs,):
                raise ValueError("seed must be an int or one seed per env")
        with torch.cuda.device(self.device):
            self.raw.reset(seeds, None, self._stream())
        self._was_reset = True
        return self._observation(), self._info(reset=True)

    def _info(self, reset: bool = False) -> dict:
        ss = self._t["step_state"]
        info = LazyInfo()
        if not reset:
            fl = self._t["step_flags"]
            info.update(x=ss[:, 0], y=ss[:, 1], x_velocity=ss[:, 2], y_velocity=ss[:, 3], step_flags=fl)
            info.lazy("flat_tire", lambda: (fl & 1).bool())
            info.lazy("braking_applied", lambda: (fl & 2).bool())
            if self.separate_reward_cost:
                info["cost"] = self._t["cost"]
                info["safety_cost"] = self._t["cost"]
                info["performance_reward"] = self._t["reward"]
            if self.hc.pod.write_final_obs:
                info["final_observation"] = self._observation(final=True)
                info.lazy("_final_observation", lambda: self._terminated | self._truncated)
            if self.hc.pod.num_levels:  # the level of the episode that ended (meaningful where _final_observation is set)
                info.lazy("final_level", lambda: self.level_ids(previous=True))
        if self.hc.pod.num_levels:
            info.lazy("level", self.level_ids)
        return info

    def level_ids(self, previous: bool = False) -> torch.Tensor:
        """Level sets (num_levels > 0): every env's level as int32 [N] on the device -- of the current episode, or with
        previous=True of the episode before it, which for an env that auto-reset in the last step is the one that just ended.
        Recomputed from the envs' keys and episode counters by one small kernel; no host synchronisation."""
        with torch.cuda.device(self.device):
            return self.raw.levels(previous, self._stream())

    def step(self, actions):
        if not self._was_reset:
            raise RuntimeError("step() called before reset()")
        with torch.cuda.device(self.device):
            if isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype in (torch.int32, torch.int64) \
                    and actions.is_contiguous() and actions.shape == (self.num_envs,):
                ptr, nbytes = actions.data_ptr(), actions.element_size()
            else:
                a = torch.as_tensor(np.asarray(actions.cpu() if isinstance(actions, torch.Tensor) else actions), dtype=torch.int32)
                if a.shape != (self.num_envs,):
                    raise ValueError(f"expected {self.num_envs} actions")
                self._actions.copy_(a, non_blocking=True)
                ptr, nbytes = self._actions.data_ptr(), 4
            self.raw.step_device(ptr, nbytes, self._stream())
        return self._observation(), self._t["reward"], self._terminated, self._truncated, self._info()

    # ---- full-state checkpoint / clone (PGTGEnv.light_step, environment.py:1283-1299) ---------------------
    def save_state(self) -> np.ndarray:
        """Everything a tick reads or writes (SoA state, map rings and request queues, car lists with patience /
        delay, RNG state, light counters, consumed subgoals, episode statistics, outputs) as one host blob.
        Unlike the reference's `set_to_state` (quirk A.3-10) nothing is left out."""
        with torch.cuda.device(self.device):
            return self.raw.save_state()

    def load_state(self, blob: np.ndarray) -> None:
        with torch.cuda.device(self.device):
            self.raw.load_state(blob)
        self._was_reset = True

    def clone(self) -> "PGTGVectorEnv":
        """A second env in exactly this env's state (device-to-device copy), `copy.deepcopy(env)` of the reference."""
        if self.hc.pod.rng_mode == RNG_TAPE:
            raise NotImplementedError("clone() of a conformance-tape env is not supported")
        num_envs, map_path, kwargs = self._ctor
        other = PGTGVectorEnv(num_envs, map_path, device=self.device, **kwargs)
        with torch.cuda.device(self.device):
            if len(self.hc.rules) != len(other.hc.rules) or any(a is not b and a != b for a, b in zip(self.hc.rules, other.hc.rules)):
                other.hc.rules = [dict(r) for r in self.hc.rules]
                other.raw.update_rules(other.hc.rules)
            other.raw.copy_state_from(self.raw)
        other._was_reset = self._was_reset
        return other

    def light_step(self, actions):
        """PGTGEnv.light_step (environment.py:1283-1299): copy the env and execute one step on the copy; this env
        stays unchanged. The copy is kept and re-synchronised on every call. Returns the copy's step outputs."""
        if not self._was_reset:
            raise RuntimeError("light_step() called before reset()")
        if self._shadow is None:
            self._shadow = self.clone()
        else:
            with torch.cuda.device(self.device):
                self._shadow.raw.copy_state_from(self.raw)
        return self._shadow.step(actions)

    # ---- evaluator (pgtg/evaluator.py:284-339) --------------------------------------------------------------
    def evaluate(self, policy, number: int, max_steps: int = 100, GAMMA: float = 0.99):
        """ModularEvaluator.evaluate over the batch: run `policy(observation) -> actions` until at least `number`
        episodes have finished, at most `max_steps` steps each, discounting rewards with GAMMA ** t on the device.
        Returns (mean discounted return, (terminated, truncated, over max_steps, negative return)) -- the reference
        returns the list of returns; here the mean is reduced on the device. PGTGEnv never sets `truncated` itself,
        so that counter stays 0 and the episode cap shows up as "over max_steps"."""
        with torch.cuda.device(self.device):
            self.raw.set_evaluation(GAMMA, max_steps)
        obs, _ = self.reset()
        self.episode_stats(reset=True, all_reduce=False)
        done = 0.0
        while done < number:
            for _ in range(max(1, min(max_steps, 8))):
                obs, _, _, _, _ = self.step(policy(obs))
            with torch.cuda.device(self.device):
                _check(self.raw, self.raw.lib.pgtg_reduce_stats(self.raw._h, self._stream()))
            done = float(self._t["stats"][0].item())
        st = self.episode_stats(all_reduce=False)
        with torch.cuda.device(self.device):
            self.raw.set_evaluation(0.0, 0)
        n = max(st["episodes"], 1.0)
        return st["discounted_return_sum"] / n, (int(st["goals"] + st["crashes"]), 0, int(st["truncations"]), int(st["negative_returns"]))

    # ---- host-buffer steps --------------------------------------------------------------------------------
    def packed_host_buffers(self, pinned: bool = True) -> dict:
        """Host buffers for `step_host_packed` (pinned by default: the copies are asynchronous)."""
        N = self.num_envs
        mk = (lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()) if pinned else (lambda shape, dt: torch.empty(shape, dtype=dt).numpy())
        return dict(obs_packed=mk((self.raw.packed_obs_bytes() // 4,), torch.int32).view(np.uint32), obs_position=mk((N, 2), torch.int32),
                    obs_velocity=mk((N, 2), torch.int32), reward=mk((N,), torch.float64), terminated=mk((N,), torch.uint8), truncated=mk((N,), torch.uint8))

    def step_host_packed(self, actions: np.ndarray, out: dict | None = None, wait: bool = False) -> dict:
        """The tick through HOST buffers with the observation planes as BITS (92 B per env instead of 729 at the
        defaults) and double-buffered copies: with wait=False the call returns once everything is enqueued and the
        buffers are complete after `host_sync()`; alternate two buffer sets to overlap tick k + 1 with the copies of
        tick k. `unpack_obs` turns the bits back into the int8 [N, C, P, P] planes on the host."""
        if out is None:
            out = self.packed_host_buffers(pinned=False)
            wait = True
        with torch.cuda.device(self.device):
            self.raw.step_host_packed(actions, stream=self._stream(), wait=wait, **out)
        return out

    def host_sync(self) -> None:
        self.raw.host_sync()

    def unpack_obs(self, obs_packed: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        return self.raw.unpack_obs(obs_packed, out)

    def step_host(self, actions: np.ndarray, out: dict | None = None) -> dict:
        """The same tick through HOST buffers (`pgtg_step_host`): copies in and out inside the call.
        This is the entry a non-CUDA consumer (the reference-facing plugin boundary) uses."""
        N, C, P = self.num_envs, self.hc.pod.num_channels, self.hc.window
        if out is None:
            out = dict(obs_map=np.empty((N, C, P, P), np.int8), obs_position=np.empty((N, 2), np.int32),
                       obs_velocity=np.empty((N, 2), np.int32), reward=np.empty(N, np.float64),
                       terminated=np.empty(N, np.uint8), truncated=np.empty(N, np.uint8))
        with torch.cuda.device(self.device):
            self.raw.step_host(actions, stream=self._stream(), **out)
        return out

    def flat_observation(self):
        """float32 [N, D] tensor equal to gymnasium 0.28.1 `FlattenObservation` applied to every env's
        observation (what SB3's MlpPolicy consumes at train.py:39-61): sorted map planes, optional
        next_subgoal_direction one-hot, position one-hots, velocity. One extra kernel per call."""
        with torch.cuda.device(self.device):
            self.raw.flatten(self._stream())
            if "obs_flat" not in self._t:
                self._t["obs_flat"] = torch.from_dlpack(self.raw.dlpack_capsule("obs_flat"))
        return self._t["obs_flat"]

    # ---- bits observation format ------------------------------------------------------------------------------------
    def obs_packed(self) -> torch.Tensor:
        """observation_format="bits": the step's observation planes as stored by the tick, uint32 [ceil(N * C*P*P / 32)] on the
        device, env i at bit i * C*P*P (a view, valid until the next step: copy it into a rollout store to keep it)."""
        return self._packed_view("obs_packed")

    def final_obs_packed(self) -> torch.Tensor:
        """observation_format="bits" with final_observation=True: the terminal observations, same layout as `obs_packed`; rows
        of envs that did not finish in the last step are not meaningful."""
        return self._packed_view("final_obs_packed")

    def _packed_view(self, name: str) -> torch.Tensor:
        if self.observation_format != "bits":
            raise RuntimeError(f"{name}() needs observation_format='bits'")
        if name not in self._t:
            with torch.cuda.device(self.device):
                self._t[name] = torch.from_dlpack(self.raw.dlpack_capsule(name))
        return self._t[name]

    def unpack(self, bits: torch.Tensor, index: torch.Tensor | None = None, format: str = "int8", position: torch.Tensor | None = None,
               velocity: torch.Tensor | None = None, next_subgoal_direction: torch.Tensor | None = None) -> torch.Tensor:
        """Stored bits -> a new device tensor, one kernel, no host synchronisation. `bits`: S step slots of `obs_packed` copies
        (a [S, words] or [words] uint32 / int32 tensor); row r = s * N + i is env i of slot s. `index`: int64 rows to gather
        (default: all S * N in order). format="int8": [count, C, P, P] like obs["map"]; format="flat": float32 [count, D] like
        `flat_observation()`, with `position` / `velocity` ([S, N, 2] int32) and, when next_subgoal_direction is on,
        `next_subgoal_direction` ([S, N] int32) gathered with the same rows. A row outside [0, S * N) comes back as zeros and
        sets an error flag that `episode_stats` reports."""
        if format not in ("int8", "flat"):
            raise ValueError("format must be 'int8' or 'flat'")
        words = self.raw.packed_obs_bytes() // 4

        def dev(t, dtypes, what):
            if not (isinstance(t, torch.Tensor) and t.device == self.device and t.dtype in dtypes and t.is_contiguous()):
                raise ValueError(f"{what} must be a contiguous {'/'.join(map(str, dtypes))} tensor on {self.device}")
            return t

        dev(bits, (torch.uint32, torch.int32), "bits")
        if bits.numel() == 0 or bits.numel() % words:
            raise ValueError(f"bits must hold S slots of {words} words")
        slots, N = bits.numel() // words, self.num_envs
        count = slots * N
        if index is not None:
            count = dev(index, (torch.int64,), "index").numel()
        ptrs = [None, None, None]
        if format == "flat":
            needed = [(position, "position", 2), (velocity, "velocity", 2)]
            if self.use_next_subgoal_direction:
                needed.append((next_subgoal_direction, "next_subgoal_direction", 1))
            for k, (t, what, per) in enumerate(needed):
                if t is None or dev(t, (torch.int32,), what).numel() != slots * N * per:
                    raise ValueError(f"format='flat' needs {what} as int32 [{slots}, {N}{', 2' if per == 2 else ''}]")
                ptrs[k] = t.data_ptr()
            C, P = self.hc.pod.num_channels, self.hc.window
            out = torch.empty((count, C * P * P + (9 if self.use_next_subgoal_direction else 0) + 20), dtype=torch.float32, device=self.device)
        else:
            out = torch.empty((count, self.hc.pod.num_channels, self.hc.window, self.hc.window), dtype=torch.int8, device=self.device)
        with torch.cuda.device(self.device):
            self.raw.unpack_bits(bits.data_ptr(), slots, None if index is None else index.data_ptr(), count, format, out.data_ptr(),
                                 *ptrs, stream=self._stream())
        return out

    def save_map(self, path: str, env_index: int = 0) -> None:
        """EpisodeMap.save_map (map.py:173-184): the current map plan of one env as reference JSON."""
        import json

        from ._names import CARDINALS, MASK_NAMES, OBSTACLE_NAMES

        st = self.raw.get_state()
        W, H = self.hc.pod.map_w, self.hc.pod.map_h
        pl = st["plan"][env_index]
        rows = []
        for y in range(H):
            row = []
            for x in range(W):
                td = int(st["tiles"][env_index, y * W + x])
                tile = {"exits": [td & 1, (td >> 1) & 1, (td >> 2) & 1, (td >> 3) & 1]}
                if (td >> 4) & 7:
                    tile["obstacle_type"] = OBSTACLE_NAMES[((td >> 4) & 7) - 1]
                    tile["obstacle_mask"] = MASK_NAMES[(td >> 7) & 15]
                row.append(tile)
            rows.append(row)
        plan = {"width": W, "height": H, "map": rows, "start": [int(pl[0]), int(pl[1]), CARDINALS[pl[2]]],
                "goal": [int(pl[3]), int(pl[4]), CARDINALS[pl[5]]]}
        if not path.endswith(".json"):
            path += ".json"
        with open(path, "w", encoding="utf-8") as f:
            json.dump(plan, f, ensure_ascii=False, indent=4)

    def close(self):
        if self._shadow is not None:
            self._shadow.close()
            self._shadow = None
        self.raw.close()

    # ---- reference extras ------------------------------------------------------------------------
    def add_traffic_rule(self, rule_dict: dict):
        """PGTGEnv.add_traffic_rule (environment.py:569-571)."""
        if any(r["name"] == rule_dict["name"] for r in self.hc.rules):
            raise ValueError(f"Rule with name {rule_dict['name']} already exists.")
        self.hc.rules.append(rule_dict)
        self.raw.update_rules(self.hc.rules)

    def remove_traffic_rule(self, rule_name: str) -> bool:
        """PGTGEnv.remove_traffic_rule (environment.py:573-575)."""
        for i, r in enumerate(self.hc.rules):
            if r["name"] == rule_name:
                del self.hc.rules[i]
                self.raw.update_rules(self.hc.rules)
                return True
        return False

    def get_state(self) -> dict:
        """Host snapshot of every env (the tensors behind PGTGEnv.get_info, environment.py:1538)."""
        return self.raw.get_state()

    def get_info_arrays(self) -> dict:
        """The computed parts of PGTGEnv.get_info (environment.py:1538-1578) for every env, as arrays:
        agent_direction (index into AGENT_DIRECTIONS, :185-206), current_tile_type (exits N|E<<1|S<<2|W<<3,
        :1541-1549), profile_counts [N, 5] (get_driver_profile_stats, :1017-1035). Synchronises."""
        with torch.cuda.device(self.device):
            return self.raw.get_info()

    def get_info_dicts(self) -> list[dict]:
        """Per-env dicts shaped like PGTGEnv.get_info() (environment.py:1538-1578; debugging aid, synchronises).
        `traffic_rules.triggered_rules` is not kept per rule: `braking_applied` says whether any rule fired."""
        st = self.raw.get_state()
        with torch.cuda.device(self.device):
            extra = self.raw.get_info()
        flags = self._t["step_flags"].cpu().numpy()
        configured = {n: float(p) * 100 for n, p in zip(PROFILE_NAMES, np.diff(np.concatenate([[0.0], list(self.hc.pod.profile_cdf)])))}
        out = []
        for i in range(self.num_envs):
            cars = [dict(id=int(c[0]), x=int(c[1]), y=int(c[2]), route=ROUTE_NAMES[c[3]], driver_profile=PROFILE_NAMES[c[4]],
                         patience_counter=int(c[5])) for c in st["cars"][i, : st["num_cars"][i]]]
            tt = int(extra["current_tile_type"][i])
            counts = {n: int(v) for n, v in zip(PROFILE_NAMES, extra["profile_counts"][i])}
            total = int(st["num_cars"][i])
            stats = dict(counts=counts, percentages={k: (v / total) * 100 if total else 0 for k, v in counts.items()}, total_cars=total,
                         configured_percentages=configured)
            out.append(dict(x=int(st["agent"][i, 0]), y=int(st["agent"][i, 1]), x_velocity=int(st["agent"][i, 2]),
                            y_velocity=int(st["agent"][i, 3]), flat_tire=bool(st["flat_tire"][i]),
                            current_tile_type="".join(str((tt >> k) & 1) for k in range(4)), cars=cars, driver_profile_stats=stats,
                            traffic_rules=dict(active_rules=[r["name"] for r in self.hc.rules], braking_applied=bool(flags[i] & 2),
                                               agent_direction=AGENT_DIRECTIONS[int(extra["agent_direction"][i])])))
        return out

    def set_to_state(self, agent=None, flat_tire=None, num_cars=None, cars=None):
        """PGTGEnv.set_to_state (environment.py:1301-1342) for all envs: position, velocity,
        flat_tire and cars only; returns the refreshed observation."""
        with torch.cuda.device(self.device):
            self.raw.set_state(agent=agent, flat_tire=flat_tire, num_cars=num_cars, cars=cars)
            self.raw.observe(self._stream())
        return self._observation(), self._info(reset=True)

    def episode_stats(self, reset: bool = False, all_reduce: bool = True) -> dict:
        """Episode statistics accumulated on the device since the last reset of the counters.
        With torch.distributed initialised the 8 doubles are summed over ranks with one NCCL
        all-reduce -- the only collective in the system."""
        with torch.cuda.device(self.device):
            _check(self.raw, self.raw.lib.pgtg_reduce_stats(self.raw._h, self._stream()))
            s = self._t["stats"].clone()
            if all_reduce and torch.distributed.is_available() and torch.distributed.is_initialized():
                torch.distributed.all_reduce(s)
            if reset:
                _check(self.raw, self.raw.lib.pgtg_reset_stats(self.raw._h, self._stream()))
            flags = self.raw.error_summary()
        if flags:
            names = {1: "conformance tape overrun", 2: "conformance tape tag mismatch", 4: "conformance index out of range", 8: "goal unreachable",
                     16: "no route at a spawn square", 32: "more cars than max_cars", 64: "no start square",
                     128: "an action outside 0..8 was replaced by the no-op 4 (the reference raises KeyError)",
                     256: "an unpack index outside the stored rows (its output row is zeros)"}
            raise RuntimeError("env error flags: " + "; ".join(v for k, v in names.items() if flags & k))
        v = s.cpu().tolist()
        n = max(v[0], 1.0)
        return dict(episodes=v[0], mean_return=v[1] / n, mean_length=v[2] / n, goals=v[3], crashes=v[4], truncations=v[5],
                    discounted_return_sum=v[6], negative_returns=v[7])

    def launch_count(self) -> int:
        return self.raw.launch_count()


def _check(raw, rc):
    from . import _lib

    _lib.check(raw.lib, rc)


def make_vec(num_envs: int, **kwargs) -> PGTGVectorEnv:
    """`gymnasium.make("pgtg-v4", **kwargs)` rollouts, batched (the reference registers pgtg-v4,
    pgtg/__init__.py:7)."""
    return PGTGVectorEnv(num_envs, **kwargs)

"""Level sets (num_levels / start_level / level_sampling): a finite pool of generated maps served to the episodes.

Level j is the map a handle without levels gives an env of key start_level + j at its first episode after a seeded reset.
Each case runs the emulation of the kernel phases (tests/emu, built with the level-set backend calls) on the CPU and the CUDA
kernels on the GPU, against the oracle with level sets (tests/level_oracle_c: the unmodified oracle plus a pool built with
its own generator and the level and start-square draws of include/pgtg_b200.h)."""
import ctypes as C
import os
import subprocess
import warnings

import numpy as np
import pytest

import philox_compare as pc
from level_oracle import LevelOracle
from pgtg_b200.config import PgtgConfig, make_config

BACKENDS = ["emu_levels", pytest.param("cuda", marks=pytest.mark.gpu)]
EMU_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")


def _native(backend, n, **kw):
    from native_env import NativeAdapter

    if backend == "emu_levels":  # the emulation with the level-set backend calls (tests/emu/levels.mk)
        subprocess.check_call(["make", "-s", "-C", EMU_DIR, "-f", "levels.mk"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return NativeAdapter(backend, num_envs=n, **kw)


def _oracle(n, **kw):
    return LevelOracle(num_envs=n, threads=8, **kw)


def _levels(env, previous=False):
    return env.raw.levels(previous).cpu().numpy()


def _pool(env):
    tiles, plan = env.raw.level_pool()
    return tiles.cpu().numpy(), plan.cpu().numpy()


def _pack(plan8):
    """pgtg_state.plan rows [sx, sy, sdir, gx, gy, gdir, num_subgoals, 0] -> plan words without the start-square bits."""
    p = plan8.astype(np.uint32)
    return p[:, 0] | p[:, 1] << 4 | p[:, 2] << 8 | p[:, 3] << 10 | p[:, 4] << 14 | p[:, 5] << 18 | p[:, 6] << 20


# ---- 1. configuration checks ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw,match", [
    (dict(num_levels=4, rng_mode="numpy"), "philox"),
    (dict(num_levels=4, rng_mode="tape"), "philox"),
    (dict(num_levels=4, map_plan=pc.CROSSING), "map_path"),
    (dict(num_levels=-1), "num_levels"),
    (dict(num_levels=(1 << 24) + 1), "num_levels"),
    (dict(num_levels=4, start_level=-1), "start_level"),
    (dict(num_levels=4, start_level=2 ** 31), "start_level"),
    (dict(num_levels=4, level_sampling="round_robin"), "level_sampling"),
])
def test_invalid_level_configurations_raise(kw, match):
    with pytest.raises(ValueError, match=match):
        make_config(**kw)


def test_library_rejects_invalid_level_pods():
    """pgtg_create checks the same ranges on the POD itself (emulation build of the same host code)."""
    from native_env import build_emu
    from pgtg_b200 import _lib

    _native("emu_levels", 1)  # builds libpgtg_emu_levels.so
    lib = _lib.load(build_emu().replace("libpgtg_emu.so", "libpgtg_emu_levels.so"))
    for field, value, text in (("num_levels", (1 << 24) + 1, b"num_levels"), ("rng_mode", 2, b"PHILOX"), ("start_level", -5, b"start_level"),
                               ("level_sampling", 2, b"level_sampling")):
        hc = make_config(num_envs=4, num_levels=3)
        setattr(hc.pod, field, value)
        h = C.c_void_p()
        assert lib.pgtg_create(C.byref(hc.pod), 0, C.byref(h)) == -1 and text in lib.pgtg_last_error()
    plain = _lib.load(build_emu())  # a backend without the level-set calls refuses level sets instead of generating maps
    hc = make_config(num_envs=4, num_levels=3)
    assert plain.pgtg_create(C.byref(hc.pod), 0, C.byref(h)) == -1 and b"no level sets" in plain.pgtg_last_error()


def test_levels_off_leaves_the_pod_as_before():
    """num_levels = 0 writes nothing: the three fields sit in what were padding words, sizeof(pgtg_config) is unchanged."""
    a, b = make_config(num_envs=8, seed=3), make_config(num_envs=8, seed=3, num_levels=0, start_level=0, level_sampling="uniform")
    assert bytes(a.pod) == bytes(b.pod)
    assert a.pod.num_levels == a.pod.start_level == a.pod.level_sampling == 0
    assert C.sizeof(PgtgConfig) == 1848
    assert (PgtgConfig.num_levels.offset, PgtgConfig.level_sampling.offset, PgtgConfig.start_level.offset) == (84, 612, 1844)


# ---- 2. the pool is the seeded-reset maps ---------------------------------------------------------------------------------
POOL_CONFIGS = {
    "4x4_registers": dict(),
    "3x3_staged": dict(random_map_width=3, random_map_height=3),
    "6x2_random_ends": dict(random_map_start_position="random", random_map_goal_position="random", random_map_width=6,
                            random_map_height=2, random_map_percentage_of_connections=0.3),
    "8x8_obstacles": dict(random_map_width=8, random_map_height=8, random_map_percentage_of_connections=0.8,
                          random_map_obstacle_probability=0.5),
}


@pytest.mark.parametrize("M", [1, 5, 300])
@pytest.mark.parametrize("name", list(POOL_CONFIGS))
@pytest.mark.parametrize("backend", BACKENDS)
def test_pool_equals_seeded_reset_maps(backend, name, M):
    kw, start = POOL_CONFIGS[name], 1000 + M
    env = _native(backend, 3, num_levels=M, start_level=start, seed=77, **kw)
    assert f"mapgen=levels(M={M})" in env.raw.kernel_info()
    tiles, plan = _pool(env)
    assert tiles.shape == (M, env.hc.pod.map_w * env.hc.pod.map_h) and plan.shape == (M,)
    assert not (plan >> 29).any()
    ref = _native(backend, M, seed=5, env_id_base=9, **kw)  # neither seed nor env_id_base enters the pool
    ref.reset(seeds=start + np.arange(M))
    st = ref.get_state()
    assert np.array_equal(tiles, st["tiles"]) and np.array_equal(plan, _pack(st["plan"]))
    ot, op = _oracle(3, num_levels=M, start_level=start, **kw).level_pool()
    assert np.array_equal(tiles, ot) and np.array_equal(plan, op)
    env.close()
    ref.close()


# ---- 3 + 4. lock-step with the oracle, level ids and the served maps at every tick ---------------------------------------
LOCKSTEP = {
    "default": (dict(max_episode_steps=6), "lean"),
    "default_final": (dict(max_episode_steps=6, final_observation=True), "lean+final"),
    "sliding_nsd": (dict(use_sliding_observation_window=True, sliding_observation_window_size=3, use_next_subgoal_direction=True,
                         max_episode_steps=6), "lean+slide"),
    "config3_traffic": (dict(traffic_density=0.05, random_map_obstacle_probability=0.2, max_episode_steps=8), "traffic"),
    "penalties_timelimit": (pc.CONFIGS["penalties_timelimit"][0], "general"),
    "train_py": (dict(pc.TRAFFIC_CONFIGS["train_py"][0], max_episode_steps=8), "traffic"),
}


def _check_served_maps(env, tiles, plan, t):
    lv, st = _levels(env), env.get_state()
    assert np.array_equal(st["tiles"], tiles[lv]), f"tick {t}: state tiles are not the levels' tiles"
    assert np.array_equal(_pack(st["plan"]), plan[lv]), f"tick {t}: state plans are not the levels' plans"


def _lockstep_levels(env, ora, ticks, final, action_seed=0):
    """pc.compare with the level ids (current and previous episode) and the served maps checked at every tick."""
    tiles, plan = _pool(env)
    rng = np.random.default_rng(action_seed)
    env.reset()
    ora.reset()
    assert np.array_equal(_levels(env), ora.levels())
    _check_served_maps(env, tiles, plan, -1)
    episodes = 0
    for t in range(ticks):
        a = rng.integers(0, 9, ora.N).astype(np.int32)
        env.step(a)
        ora.step(a)
        for name in pc.ARRAYS:
            pc._eq(name, getattr(env, name), getattr(ora, name), t)
        done = (ora.terminated | ora.truncated).astype(bool)
        episodes += int(done.sum())
        if final and done.any():
            pc._eq("final_obs_map", env.final_obs_map[done], ora.final_obs_map[done], t)
        pc._eq("level", _levels(env), ora.levels(), t)
        pc._eq("final_level", _levels(env, True)[done], ora.levels(previous=True)[done], t)
        _check_served_maps(env, tiles, plan, t)
        if (t + 1) % 5 == 0:
            pc.compare_state(env, ora, t)
    pc.compare_state(env, ora, ticks)
    return episodes


@pytest.mark.parametrize("sampling", ["uniform", "env_index"])
@pytest.mark.parametrize("name", list(LOCKSTEP))
@pytest.mark.parametrize("backend", BACKENDS)
def test_level_set_matches_oracle(backend, name, sampling):
    kw, tick = LOCKSTEP[name]
    kw = dict(kw, num_levels=11, start_level=40, level_sampling=sampling, seed=21)
    n, ticks = (150, 24) if backend == "emu_levels" else (1500, 40)
    env, ora = _native(backend, n, **kw), _oracle(n, **kw)
    assert f"tick={tick}(" in env.raw.kernel_info() and "mapgen=levels(M=11)" in env.raw.kernel_info()
    assert _lockstep_levels(env, ora, ticks, kw.get("final_observation", False)) > 0
    if sampling == "env_index":
        assert np.array_equal(_levels(env), np.arange(n) % 11)
    env.close()
    ora.close()


@pytest.mark.parametrize("backend", BACKENDS)
def test_one_level_is_one_map_for_every_episode(backend):
    env = _native(backend, 200, num_levels=1, start_level=7, max_episode_steps=3, random_map_obstacle_probability=0.4)
    tiles, plan = _pool(env)
    env.reset()
    rng = np.random.default_rng(1)
    for t in range(10):
        env.step(rng.integers(0, 9, 200))
        st = env.get_state()
        assert (st["tiles"] == tiles[0]).all() and (_pack(st["plan"]) == plan[0]).all()
        assert not _levels(env).any()
    env.close()


# ---- 5. the uniform draw --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_uniform_level_frequencies_chi_square():
    from scipy.stats import chisquare

    n, M = 16384, 7
    env = _native("cuda", n, num_levels=M, seed=2024, max_episode_steps=1)
    env.reset()
    counts = np.bincount(_levels(env), minlength=M)
    for _ in range(3):  # every env starts a new episode at every tick
        env.step(np.zeros(n, np.int32) + 4)
        counts += np.bincount(_levels(env), minlength=M)
    assert counts.sum() >= 50000
    assert chisquare(counts).pvalue > 1e-3, counts
    env.close()


# ---- 6. env_index sampling across shards ------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
def test_env_index_shards_reproduce_one_handle(backend):
    n, M = (130, 9) if backend == "emu_levels" else (1030, 9)
    kw = dict(num_levels=M, start_level=3, level_sampling="env_index", seed=12, max_episode_steps=5, random_map_obstacle_probability=0.3)
    whole = _native(backend, n, **kw)
    parts = [_native(backend, n // 2, **kw), _native(backend, n - n // 2, env_id_base=n // 2, **kw)]
    for e in [whole] + parts:
        e.reset()
    rng = np.random.default_rng(3)
    for t in range(15):
        a = rng.integers(0, 9, n).astype(np.int32)
        whole.step(a)
        parts[0].step(a[: n // 2])
        parts[1].step(a[n // 2:])
        for name in ("obs_map", "obs_position", "reward", "terminated", "truncated"):
            pc._eq(name, np.concatenate([getattr(p, name) for p in parts]), getattr(whole, name), t)
        assert np.array_equal(_levels(whole), np.arange(n) % M)
        assert np.array_equal(np.concatenate([_levels(p) for p in parts]), np.arange(n) % M)
    for e in [whole] + parts:
        e.close()


# ---- 7. bit identity across tick kernels and pipeline modes ---------------------------------------------------------------
def _trace(env, ticks, seed=5):
    rng = np.random.default_rng(seed)
    env.reset()
    out = []
    for _ in range(ticks):
        env.step(rng.integers(0, 9, env.N).astype(np.int32))
        out.append([env.obs_map, env.obs_position, env.reward, env.terminated, env.truncated, _levels(env), env.get_state()["tiles"]])
    return out


def _same(a, b):
    for t, (x, y) in enumerate(zip(a, b)):
        for k, (u, v) in enumerate(zip(x, y)):
            assert np.array_equal(u, v), f"tick {t}, field {k}"


@pytest.mark.parametrize("backend", BACKENDS)
def test_general_tick_and_no_overlap_equal_the_lean_tick(backend, monkeypatch):
    kw = dict(num_levels=13, start_level=5, max_episode_steps=4, random_map_obstacle_probability=0.3, seed=8)
    n = 260 if backend == "emu_levels" else 2600
    lean = _native(backend, n, **kw)
    assert "tick=lean(" in lean.raw.kernel_info()
    ref = _trace(lean, 12)
    serial = _native(backend, n, **kw)
    serial.raw.set_overlap(False)
    _same(_trace(serial, 12), ref)
    monkeypatch.setenv("PGTG_NO_LEAN", "1")
    general = _native(backend, n, **kw)
    assert "tick=general(" in general.raw.kernel_info()
    _same(_trace(general, 12), ref)
    for e in (lean, serial, general):
        e.close()


# ---- 8. checkpoints and clones ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
def test_save_load_and_clone_continue_identically(backend):
    kw = dict(num_levels=6, start_level=90, max_episode_steps=5, traffic_density=0.05, seed=4)
    n = 150 if backend == "emu_levels" else 1500
    env = _native(backend, n, **kw)
    _trace(env, 7)
    blob = env.raw.save_state()
    twin = _native(backend, n, **kw)
    twin.raw.copy_state_from(env.raw)
    cont = _trace_from_here(env, 8)
    env.raw.load_state(blob)
    _same(_trace_from_here(env, 8), cont)
    _same(_trace_from_here(twin, 8), cont)
    other = _native(backend, n, **dict(kw, start_level=91))
    with pytest.raises(ValueError, match="level set"):
        other.raw.load_state(blob)
    with pytest.raises(ValueError, match="level set"):
        other.raw.copy_state_from(env.raw)
    plain = _native(backend, n, **dict(kw, num_levels=0))
    with pytest.raises(ValueError, match="level set"):
        plain.raw.load_state(blob)
    for e in (env, twin, other, plain):
        e.close()


def _trace_from_here(env, ticks, seed=6):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(ticks):
        env.step(rng.integers(0, 9, env.N).astype(np.int32))
        out.append([env.obs_map, env.reward, env.terminated, env.truncated, _levels(env), _levels(env, True)])
    return out


# ---- 9. the vector env ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vector_env_level_info():
    import torch

    from pgtg_b200 import PGTGVectorEnv

    env = PGTGVectorEnv(512, device="cuda:0", num_levels=20, start_level=3, max_episode_steps=4, final_observation=True)
    obs, info = env.reset(seed=1)
    assert torch.equal(info["level"], env.level_ids())
    pool = [t.clone() for t in env.raw.level_pool()]
    first, finals = [], 0
    for t in range(12):
        _, _, term, trunc, info = env.step(torch.randint(0, 9, (512,), device="cuda:0"))
        done = info["_final_observation"]
        assert torch.equal(info["level"], env.level_ids())
        assert torch.equal(info["final_level"][done], env.level_ids(previous=True)[done])
        finals += int(done.sum())
        first.append(env.level_ids().cpu())
    assert finals > 0
    env.reset(seed=2)
    second = [env.level_ids().cpu()]
    for t in range(11):
        env.step(torch.randint(0, 9, (512,), device="cuda:0"))
        second.append(env.level_ids().cpu())
    assert all(torch.equal(a, b) for a, b in zip(pool, env.raw.level_pool()))
    assert not all(torch.equal(a, b) for a, b in zip(first, second))
    plain = PGTGVectorEnv(8, device="cuda:0")
    _, info = plain.reset(seed=1)
    _, _, _, _, info = plain.step(torch.zeros(8, dtype=torch.int32, device="cuda:0"))
    assert "level" not in info and "final_level" not in info
    env.close()
    plain.close()

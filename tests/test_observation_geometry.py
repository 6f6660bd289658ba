"""Observation geometry in lock-step with the oracle (Philox mode): sliding windows k = 0..15 (plane edge P = 2k+1 from 1 to
31), 0..16 planes with repeated kinds, terminal observations, CTA sizes of 32 / 64 / 128 envs and the packed host step.

An env's observation is obs_bits = C * P * P cells. The kernels lay the CTA's envs end to end in one bitstring and expand it
32 cells at a time, so when obs_bits < 32 (k = 0, k = 1 with C <= 3, k = 2 with C = 1) one 32-cell vector covers three or
more envs; a wide window with many planes makes the bitstring outgrow shared memory, and the tick drops to 64 or 32 envs per
CTA. Every case runs the emulation of the kernel phases (tests/emu) on the CPU and the CUDA kernels on the GPU, and
asserts which tick kernel and CTA size the handle picked, so that a change of dispatch is visible."""
import warnings

import numpy as np
import pytest

import philox_compare as pc
from oracle.oracle import OracleVectorEnv
from pgtg_b200.config import DEFAULT_FEATURES

BACKENDS = ["emu", pytest.param("cuda", marks=pytest.mark.gpu)]

# feature lists -> C planes. "walls" / "wall" are one kind twice (the generic channel loop instead of the one-plane-per-kind
# path); "goals" twice is one key of the observation dict; unknown names are all-zero planes.
FEATURES = {
    "default": None,                                      # 9 planes
    "none": [],                                           # 0
    "one": ["walls"],                                     # 1
    "three": ["goals", "walls", "sand"],                  # 3
    "repeat": ["walls", "wall", "goals", "goals", "ice", "start", "final goal", "bogus"],  # 7, kinds repeat
    "sixteen": DEFAULT_FEATURES + ["wall", "subgoal", "final goal", "start", "used subgoal", "bogus", "unknown"],
}
# with cars: the traffic plane and the car_spawner plane
TRAFFIC_FEATURES = {
    "two": ["traffic", "car_spawner"],
    "ten": DEFAULT_FEATURES + ["car_spawner"],
    "sixteen": DEFAULT_FEATURES + ["wall", "subgoal", "final goal", "start", "used subgoal", "car_spawner", "bogus"],
}
PLANES = {"default": 9, "none": 0, "one": 1, "three": 3, "repeat": 7, "sixteen": 16}

# short episodes and obstacles: many envs finish in every tick, so terminal observations of neighbouring envs meet in one vector
CARFREE_BASE = dict(random_map_obstacle_probability=0.3, max_episode_steps=5, seed=31)


def _native(backend, n, **kw):
    from native_env import NativeAdapter

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return NativeAdapter(backend, num_envs=n, **kw)


def _make(backend, n, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return _native(backend, n, **kw), OracleVectorEnv(num_envs=n, threads=8, **kw)


def _size(backend, n, ticks, k):
    """The emulation leg runs the case as listed; the CUDA leg runs more envs (the oracle's cost grows with C * P * P)."""
    if backend == "emu":
        return n, ticks
    return (4 * n + 1, 2 * ticks) if (k or 0) < 12 else (n, ticks)


def _lockstep(env, ora, ticks, final):
    episodes = pc.compare(env, ora, ticks, state_every=4, final_obs=final)
    assert episodes > 0
    env.close()
    ora.close()


# ---- car-free grid: the lean SLIDE tick --------------------------------------------------------------------------------
# (window k or None for the fixed 9x9 window, features, final_observation, use_next_subgoal_direction, num_envs)
# Every k, every plane count and both flags; the first block holds each shape with obs_bits < 32 and terminal observations.
CARFREE = [
    (0, "default", True, False, 97),
    (0, "one", True, True, 300),
    (0, "three", True, False, 97),
    (0, "repeat", True, True, 97),
    (0, "sixteen", True, False, 97),
    (1, "one", True, False, 300),
    (1, "three", True, True, 97),
    (2, "one", True, True, 97),
    (0, "none", True, True, 97),
    (1, "default", False, True, 97),
    (2, "sixteen", False, False, 300),
    (3, "three", True, False, 97),
    (3, "repeat", False, True, 300),
    (7, "default", True, True, 97),
    (7, "none", False, False, 97),
    (8, "repeat", True, False, 300),
    (8, "one", False, True, 97),
    (9, "sixteen", True, True, 97),
    (9, "three", False, False, 97),
    (12, "default", True, False, 97),
    (12, "repeat", False, True, 97),
    (15, "one", True, False, 300),
    (15, "three", False, True, 97),
    (None, "repeat", True, False, 300),  # fixed window, repeated kinds: the general tick's generic channel loop
]


def _carfree_id(case):
    k, feats, final, nsd, n = case
    return f"{'fixed' if k is None else f'k{k}'}-{feats}{'-final' if final else ''}{'-nsd' if nsd else ''}-n{n}"


def _carfree_kwargs(k, feats, final, nsd):
    kw = dict(CARFREE_BASE, features_to_include_in_observation=FEATURES[feats], final_observation=final, use_next_subgoal_direction=nsd)
    if k is not None:
        kw.update(use_sliding_observation_window=True, sliding_observation_window_size=k)
    return kw


@pytest.mark.parametrize("case", CARFREE, ids=_carfree_id)
@pytest.mark.parametrize("backend", BACKENDS)
def test_carfree_window_geometry_matches_oracle(backend, case):
    k, feats, final, nsd, n = case
    n, ticks = _size(backend, n, 16, k)
    env, ora = _make(backend, n, **_carfree_kwargs(k, feats, final, nsd))
    assert env.C == PLANES[feats] and env.P == (9 if k is None else 2 * k + 1)
    tick = "general" if k is None else "lean+slide+final" if final else "lean+slide"
    assert f"tick={tick}(B=128)" in env.raw.kernel_info()
    _lockstep(env, ora, ticks, final)


# ---- traffic grid: the traffic tick, or the general tick where its shared memory does not fit ---------------------------
# (k, features, final_observation, map edge in tiles, num_envs, tick). On 7x7 tiles with traffic 0.3 (470 cars per env at
# most) the traffic tick's CTA needs ~184 KB plus 4 bytes per observation cell: 16 planes at k = 12 and 10 planes at k = 15
# pass its 220 KB and run the general tick.
TRAFFIC = [
    (0, "two", True, 4, 97, "traffic"),
    (1, "ten", False, 4, 97, "traffic"),
    (2, "sixteen", True, 4, 97, "traffic"),
    (3, "two", False, 4, 300, "traffic"),
    (7, "ten", True, 4, 97, "traffic"),
    (8, "sixteen", False, 4, 97, "traffic"),
    (9, "two", True, 4, 97, "traffic"),
    (12, "ten", False, 4, 97, "traffic"),
    (15, "sixteen", True, 4, 97, "traffic"),
    (0, "two", True, 7, 33, "traffic"),
    (9, "sixteen", False, 7, 33, "traffic"),
    (12, "sixteen", True, 7, 33, "general"),
    (15, "ten", True, 7, 33, "general"),
]


@pytest.mark.parametrize("case", TRAFFIC, ids=lambda c: f"k{c[0]}-{c[1]}{'-final' if c[2] else ''}-{c[3]}x{c[3]}-n{c[4]}-{c[5]}")
@pytest.mark.parametrize("backend", BACKENDS)
def test_traffic_window_geometry_matches_oracle(backend, case):
    k, feats, final, w, n, tick = case
    n, ticks = _size(backend, n, 12, k)
    env, ora = _make(backend, n, traffic_density=0.3, use_sliding_observation_window=True, sliding_observation_window_size=k,
                     features_to_include_in_observation=TRAFFIC_FEATURES[feats], final_observation=final, random_map_width=w,
                     random_map_height=w, random_map_obstacle_probability=0.3, max_episode_steps=6, seed=32)
    assert f"tick={tick}(" in env.raw.kernel_info()
    _lockstep(env, ora, ticks, final)


# ---- CTA size -----------------------------------------------------------------------------------------------------------
CTA = {
    "lean": (dict(random_map_obstacle_probability=0.3, max_episode_steps=5), "lean"),
    "lean+slide+final": (_carfree_kwargs(1, "three", True, True), "lean+slide+final"),
    "general": (dict(random_map_obstacle_probability=0.3, max_episode_steps=5, final_observation=True, already_visited_position_penalty=2,
                     use_next_subgoal_direction=True), "general"),
}


@pytest.mark.parametrize("block", [32, 64])
@pytest.mark.parametrize("name", list(CTA))
@pytest.mark.parametrize("backend", BACKENDS)
def test_forced_cta_size_matches_oracle_and_default_cta(backend, name, block, monkeypatch):
    """PGTG_BLOCK: the same envs in CTAs of 32 or 64 instead of 128 give the same bits as the oracle and as the B = 128 run."""
    kw, tick = CTA[name]
    kw = dict(kw, seed=kw.get("seed", 33))
    final = kw.get("final_observation", False)
    n, ticks = _size(backend, 300, 16, 1)
    ref = _native(backend, n, **kw)
    assert f"tick={tick}(B=128)" in ref.raw.kernel_info()
    monkeypatch.setenv("PGTG_BLOCK", str(block))
    env, ora = _make(backend, n, **kw)
    assert f"tick={tick}(B={block})" in env.raw.kernel_info()
    _lockstep(env, ora, ticks, final)
    _lockstep(_native(backend, n, **kw), ref, ticks, final)


@pytest.mark.parametrize("name,kw,n,ticks", [
    ("16planes-k15", _carfree_kwargs(15, "sixteen", True, True), 97, 10),
    ("16x16-k15", dict(_carfree_kwargs(15, "default", True, False), random_map_width=16, random_map_height=16,
                       random_map_percentage_of_connections=0.6, max_episode_steps=4), 97, 10),
])
@pytest.mark.parametrize("backend", BACKENDS)
def test_window_too_large_for_128_envs_per_cta(backend, name, kw, n, ticks):
    """A 31x31 window with 16 planes (15 376 cells per env), or with 9 planes on a 16x16-tile map (whose tile rows take
    66 KB of the CTA), does not fit 128 envs per CTA: the tick picks 64 by itself."""
    env, ora = _make(backend, n, **kw)
    assert "tick=lean+slide+final(B=64)" in env.raw.kernel_info()
    _lockstep(env, ora, ticks, True)


# ---- packed host step ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,final", [(0, True), (15, False)])
@pytest.mark.parametrize("backend", BACKENDS)
def test_packed_host_step_on_the_sliding_window(backend, k, final):
    """step_host_packed + unpack_obs on the lean SLIDE tick: the bits unpack to the int8 planes and to the oracle's planes
    (k = 0: 9 cells per env, a CTA's slice ends inside a word; k = 15: 8 649 cells per env)."""
    n, ticks = _size(backend, 333, 10, k)
    env, ora = _make(backend, n, **_carfree_kwargs(k, "default", final, True))
    assert f"tick=lean+slide{'+final' if final else ''}(B=128)" in env.raw.kernel_info()
    env.reset()
    ora.reset()
    rng = np.random.default_rng(4)
    buf = dict(obs_packed=np.zeros(env.raw.packed_obs_bytes() // 4, np.uint32), obs_position=np.zeros((n, 2), np.int32),
               obs_velocity=np.zeros((n, 2), np.int32), reward=np.zeros(n), terminated=np.zeros(n, np.uint8), truncated=np.zeros(n, np.uint8))
    finished = 0
    for t in range(ticks):
        a = rng.integers(0, 9, n).astype(np.int32)
        env.raw.step_host_packed(a, **buf)
        env.raw.host_sync()
        ora.step(a)
        planes = env.raw.unpack_obs(buf["obs_packed"], threads=3)
        assert np.array_equal(planes, env.obs_map), f"tick {t}: unpacked bits differ from obs_map"
        assert np.array_equal(planes, ora.obs_map), f"tick {t}: unpacked bits differ from the oracle's planes"
        for name in ("obs_position", "obs_velocity", "reward", "terminated", "truncated"):
            assert np.array_equal(buf[name], getattr(ora, name)), f"tick {t}: {name}"
        finished += int((ora.terminated | ora.truncated).sum())
    assert finished > 0
    env.close()
    ora.close()

"""Episode statistics (the 8 doubles of pgtg_stats: episodes, return sum, length sum, goals, crashes, truncations,
discounted-return sum, negative discounted returns) and the evaluator, against a float64 restatement of the bookkeeping
on the host, every tick, in lock-step with the oracle.

The device keeps these numbers with warp ballots, shuffle reductions, float64 shared-memory atomics, one row per CTA and a
one-block reduction, in each tick kernel (lean, general, traffic); the emulation (tests/emu) keeps them with a scalar loop.
So the CPU leg checks the host code and the reference itself, and the CUDA leg checks the kernels' bookkeeping.

Reference: per env, ret += r; disc += r * g[t] (multiply and add rounded separately, as the kernel does; g = gamma ** t,
0 past max_steps); t += 1; a finished episode records (ret, t, disc) and zeroes them, a reset zeroes them and records
nothing. Counts must match exactly. The two sums must be within k * 2^-53 * fsum(|x|) of math.fsum(x), with
k = ticks + ceil(rows / 32) + 64: one rounding per tick in a CTA row, one per row in a lane of the reduction, and the
warp trees; a relative tolerance would not do, the sums can cancel to near zero."""
import math
import os
import subprocess
import warnings

import numpy as np
import pytest

import philox_compare as pc
from oracle.oracle import OracleVectorEnv

BACKENDS = ["emu", pytest.param("cuda", marks=pytest.mark.gpu)]
GAMMA = 0.97
STRAIGHT = dict(width=1, height=1, start=[0, 0, "west"], goal=[0, 0, "east"], map=[[{"exits": [0, 1, 0, 1]}]])


def _native(backend, n, **kw):
    from native_env import NativeAdapter

    if backend == "emu_levels":  # the emulation with the level-set backend calls (tests/emu/levels.mk)
        subprocess.check_call(["make", "-s", "-C", os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"), "-f", "levels.mk"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return NativeAdapter(backend, num_envs=n, **kw)


def _oracle(n, levels=False, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if levels:
            from level_oracle import LevelOracle

            return LevelOracle(num_envs=n, threads=8, **kw)
        return OracleVectorEnv(num_envs=n, threads=8, **kw)


class Ref:
    """The bookkeeping of the statistics restated in float64, one env at a time."""

    def __init__(self, n, gamma=0.0, max_steps=0):
        self.g = np.power(gamma, np.arange(max_steps)) if gamma > 0 else None
        self.ret, self.disc, self.t = np.zeros(n), np.zeros(n), np.zeros(n, np.int64)
        self.restart()

    def restart(self):
        self.rets, self.discs, self.length, self.term, self.over, self.ticks = [], [], 0, 0, 0, 0

    def zero(self, mask):
        self.ret[mask] = 0
        self.disc[mask] = 0
        self.t[mask] = 0

    def tick(self, r, te, tr):
        r, te, tr = np.asarray(r, np.float64), np.asarray(te).astype(bool), np.asarray(tr).astype(bool)
        self.ret = self.ret + r
        if self.g is not None:
            gt = np.zeros_like(r)
            inside = self.t < len(self.g)
            gt[inside] = self.g[self.t[inside]]
            prod = r * gt
            self.disc = self.disc + prod
        self.t += 1
        self.ticks += 1
        done = te | tr
        self.rets += self.ret[done].tolist()
        self.discs += self.disc[done].tolist()
        self.length += int(self.t[done].sum())
        self.term += int(te.sum())
        self.over += int((tr & ~te).sum())
        self.zero(done)
        return int(done.sum())

    def check(self, got, n, where=""):
        k = self.ticks + -(-((n + 31) // 32) // 32) + 64
        assert got[0] == len(self.rets), f"{where} episodes {got[0]} != {len(self.rets)}"
        assert got[2] == self.length, f"{where} length sum {got[2]} != {self.length}"
        assert got[3] + got[4] == self.term, f"{where} goals + crashes {got[3]} + {got[4]} != terminated {self.term}"
        assert got[5] == self.over, f"{where} truncations {got[5]} != {self.over}"
        _close(got[1], self.rets, k, where + " return sum")
        if self.g is None:
            assert got[6] == 0 and got[7] == 0, f"{where} evaluation off, but stats[6:8] = {got[6:8]}"
        else:
            assert got[7] == sum(1 for v in self.discs if v < 0), f"{where} negative returns {got[7]}"
            _close(got[6], self.discs, k, where + " discounted-return sum")


def _close(got, xs, k, what):
    want, scale = math.fsum(xs), math.fsum(abs(x) for x in xs)
    assert abs(got - want) <= k * 2.0 ** -53 * scale, f"{what}: {got!r} vs fsum {want!r} (bound {k} ulp of {scale!r})"


def _random(rng, env, n):
    return rng.integers(0, 9, n).astype(np.int32)


def _stay(rng, env, n):  # mostly "no acceleration": long episodes, so the cap truncates
    return np.where(rng.random(n) < 0.9, 4, rng.integers(0, 9, n)).astype(np.int32)


def _seek_east(rng, env, n):
    """Even envs drive east at speed 1 (toward the goal of STRAIGHT), the odd ones and one step in five act at random:
    goals and crashes in the same warp."""
    v = env.obs_velocity
    a = ((np.clip(1 - v[:, 0], -1, 1) + 1) * 3 + np.clip(-v[:, 1], -1, 1) + 1).astype(np.int32)
    rnd = (np.arange(n) % 2 == 1) | (rng.random(n) < 0.2)
    return np.where(rnd, rng.integers(0, 9, n), a).astype(np.int32)


def lockstep(env, ora, ticks, gamma, m, final=False, policy=_random, seed=0, splits=True):
    """Every output compared with the oracle at every tick, the statistics with the reference at three points:
    before a stats(reset_after=True), and twice at the end (a second reduction with no step between must not change
    them). A masked reset and a seeded full reset happen on the way. -> the final statistics."""
    n = ora.N
    ref = Ref(n, gamma, m)
    if gamma > 0:
        env.raw.set_evaluation(gamma, m)
    env.reset()
    ora.reset()
    env.stats(reset_after=True)
    if splits:
        ora.stats(reset_after=True)
    rng = np.random.default_rng(seed)
    for t in range(ticks):
        if t == ticks // 3:
            mask = (rng.random(n) < 0.4).astype(np.uint8)
            env.reset(mask=mask)
            ora.reset(mask=mask)
            ref.zero(mask.astype(bool))
            for name in pc.ARRAYS[:4]:
                pc._eq(name, getattr(env, name), getattr(ora, name), t)
        if t == ticks // 2:
            got = env.stats(reset_after=True)
            ref.check(got, n, f"tick {t}:")
            if splits:
                want = ora.stats(reset_after=True)
                assert np.array_equal(got[[0, 2, 3, 4, 5]], want[[0, 2, 3, 4, 5]]), (got, want)
            ref.restart()
        if t == (2 * ticks) // 3:
            seeds = 5000 + 7 * np.arange(n, dtype=np.int64)
            env.reset(seeds=seeds)
            ora.reset(seeds=seeds)
            ref.zero(np.ones(n, bool))
        a = policy(rng, env, n)
        env.step(a)
        ora.step(a)
        for name in pc.ARRAYS:
            pc._eq(name, getattr(env, name), getattr(ora, name), t)
        done = ref.tick(env.reward, env.terminated, env.truncated)
        if final and done:
            d = (ora.terminated | ora.truncated).astype(bool)
            pc._eq("final_obs_map", env.final_obs_map[d], ora.final_obs_map[d], t)
    got = env.stats()
    assert np.array_equal(env.stats(), got), "a second reduction with no step in between changed the statistics"
    ref.check(got, n, "end:")
    if splits:
        want = ora.stats()
        assert np.array_equal(got[[0, 2, 3, 4, 5]], want[[0, 2, 3, 4, 5]]), (got, want)
    return got


# ---- lock-step cases --------------------------------------------------------------------------------------------------------
C3 = pc.CONFIGS["config3_traffic_obstacles"][0]
C4 = pc.CONFIGS["config4_big"][0]
TRAIN = pc.TRAFFIC_CONFIGS["train_py"][0]
SLIDE = dict(use_sliding_observation_window=True, sliding_observation_window_size=5, use_next_subgoal_direction=True)
# name -> kwargs, forced environment, expected kernel_info on the device (on the emulation: its prefix up to "("),
#         policy, evaluation cap m, (envs, ticks) on the emulation, (envs, ticks) on the device; None: device only
RAGGED = 8 * 128 + 37
CASES = {
    "lean": (dict(), {}, "tick=lean(B=128)", _random, 5, (150, 24), (RAGGED, 40)),
    "lean_B32": (dict(), {"PGTG_BLOCK": "32"}, "tick=lean(B=32)", _random, 5, (150, 24), (RAGGED, 40)),
    "lean_B64": (dict(), {"PGTG_BLOCK": "64"}, "tick=lean(B=64)", _random, 5, (150, 24), (RAGGED, 40)),
    "lean_final": (dict(final_observation=True), {}, "tick=lean+final(B=128)", _random, 5, (150, 24), (RAGGED, 40)),
    "lean_slide_nsd": (SLIDE, {}, "tick=lean+slide(B=128)", _random, 5, (150, 24), (RAGGED, 40)),
    "lean_slide_final": (dict(SLIDE, final_observation=True), {}, "tick=lean+slide+final(B=128)", _random, 5, (150, 24), (RAGGED, 40)),
    "lean_n1": (dict(), {}, "tick=lean(B=128)", _random, 3, (1, 30), (1, 40)),
    "lean_n5": (dict(), {}, "tick=lean(B=128)", _random, 3, (5, 30), (5, 40)),
    "general_penalties": (pc.CONFIGS["penalties_timelimit"][0], {}, "tick=general(B=128)", _random, 4, (150, 24), (RAGGED, 40)),
    "traffic_c3": (C3, {}, "tick=traffic(G=32,NT=128)", _stay, 6, (100, 24), (RAGGED, 40)),
    "traffic_c3_n5": (C3, {}, "tick=traffic(G=32,NT=128)", _stay, 4, (5, 30), (5, 40)),
    "traffic_train_py": (TRAIN, {}, "tick=traffic(G=32,NT=256)", _stay, 12, (40, 30), (4 * 128 + 37, 40)),
    "traffic_c4": (C4, {}, "tick=traffic(G=32,NT=1024)", _stay, 6, (6, 16), (69, 24)),
    "no_traffic_kernel": (C3, {"PGTG_NO_TRAFFIC_KERNEL": "1"}, "tick=general(B=128)", _stay, 6, (100, 24), (RAGGED, 40)),
    "traffic_G64": (C3, {"PGTG_TRAFFIC_G": "64"}, "tick=traffic(G=64,", _stay, 6, None, (RAGGED, 40)),
    "traffic_G128": (C3, {"PGTG_TRAFFIC_G": "128"}, "tick=traffic(G=128,", _stay, 6, None, (RAGGED, 40)),
    "traffic_NT256": (C3, {"PGTG_TRAFFIC_NT": "256"}, "tick=traffic(G=32,NT=256)", _stay, 6, None, (RAGGED, 40)),
    "traffic_NT1024": (C3, {"PGTG_TRAFFIC_NT": "1024"}, "tick=traffic(G=32,NT=1024)", _stay, 6, None, (RAGGED, 40)),
    "inline_mapgen": (dict(), {"PGTG_INLINE_MAPGEN": "1"}, "tick=lean(B=128)", _random, 5, None, (RAGGED, 40)),
    # goals: a straight one-tile map with a policy that drives to the goal, and 1x1 random maps
    "goals_straight": (dict(map_plan=STRAIGHT), {}, "tick=general(B=128)", _seek_east, 9, (150, 30), (RAGGED, 40)),
    "goals_1x1": (dict(random_map_width=1, random_map_height=1), {}, "tick=lean(B=128)", _random, 5, (150, 30), (RAGGED, 40)),
    "goals_1x1_traffic": (pc.CONFIGS["tiny_1x1"][0], {}, "tick=traffic(G=32,NT=128)", _random, 5, (130, 30), (RAGGED, 40)),
}
GOAL_CASES = ("goals_straight", "goals_1x1", "goals_1x1_traffic")


def _case_params():
    out = []
    for name, case in CASES.items():
        emu_ok = case[5] is not None
        for ev in ("eval_off", "eval_on"):
            out.append(pytest.param("cuda", name, ev, marks=pytest.mark.gpu, id=f"cuda-{name}-{ev}"))
            if emu_ok:
                out.append(pytest.param("emu", name, ev, id=f"emu-{name}-{ev}"))
    return out


@pytest.mark.parametrize("backend,name,ev", _case_params())
def test_statistics_match_reference_in_lockstep(backend, name, ev, monkeypatch):
    kw, envvars, info, policy, m, emu_size, dev_size = CASES[name]
    for k, v in envvars.items():
        monkeypatch.setenv(k, v)
    n, ticks = emu_size if backend == "emu" else dev_size
    gamma = GAMMA if ev == "eval_on" else 0.0
    kw = dict(kw, seed=kw.get("seed", 41))
    env = _native(backend, n, **kw)
    got_info = env.raw.kernel_info()
    assert (info if backend == "cuda" else info.split("(")[0] + "(") in got_info, got_info
    # the oracle has no discounting and no evaluation cap: it gets max_episode_steps = m when evaluation is on
    ora = _oracle(n, **(dict(kw, max_episode_steps=m) if gamma > 0 else kw))
    st = lockstep(env, ora, ticks, gamma, m, final=kw.get("final_observation", False), policy=policy)
    if gamma > 0:
        assert st[5] > 0 or n < 32, f"the cap m = {m} truncated nothing"
    if name in GOAL_CASES and n > 32:
        assert st[3] > 0 and st[4] > 0, f"goals {st[3]}, crashes {st[4]}: the case must finish with both"
    env.close()
    ora.close()


@pytest.mark.parametrize("ev", ["eval_off", "eval_on"])
@pytest.mark.parametrize("backend", ["emu_levels", pytest.param("cuda", marks=pytest.mark.gpu)])
def test_statistics_with_level_sets(backend, ev):
    """Level sets (num_levels = 7) on the lean tick; the oracle with level sets keeps no statistics, so goals and crashes
    are checked together against the terminated count."""
    n, ticks = (150, 24) if backend == "emu_levels" else (RAGGED, 40)
    gamma = GAMMA if ev == "eval_on" else 0.0
    kw = dict(num_levels=7, seed=43)
    env = _native(backend, n, **kw)
    assert "tick=lean(" in env.raw.kernel_info() and "mapgen=levels(M=7)" in env.raw.kernel_info()
    ora = _oracle(n, levels=True, **(dict(kw, max_episode_steps=5) if gamma > 0 else kw))
    st = lockstep(env, ora, ticks, gamma, 5, splits=False)
    assert st[0] > 0
    env.close()
    ora.close()


# ---- full-size legs (device only, no oracle) ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,n,ticks,m", [
    ("default_1M", dict(), 1 << 20, 40, 12),
    ("config3_64k", C3, 1 << 16, 24, 10),
    ("config4_32k", dict(C4, max_episode_steps=None), 1 << 15, 6, 4),
])
def test_full_size_statistics(name, kw, n, ticks, m):
    """Millions of finished episodes over thousands of CTA rows. The reference stays on the device in float64 tensors;
    each tick only the finished envs' values come to the host for fsum."""
    import torch

    env = _native("cuda", n, seed=47, **kw)
    env.raw.set_evaluation(GAMMA, m)
    env.reset()
    env.stats(reset_after=True)
    t_ = lambda name: env._tmod.from_dlpack(env.raw.dlpack_capsule(name))  # noqa: E731
    rew, te_d, tr_d = t_("reward"), t_("terminated"), t_("truncated")
    g = torch.tensor(np.power(GAMMA, np.arange(m)), dtype=torch.float64, device="cuda")
    ret = torch.zeros(n, dtype=torch.float64, device="cuda")
    disc = torch.zeros_like(ret)
    tt = torch.zeros(n, dtype=torch.int64, device="cuda")
    rets, discs, length, term, over = [], [], 0, 0, 0
    gen = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(ticks):
        a = torch.randint(0, 9, (n,), device="cuda", dtype=torch.int32, generator=gen)
        a = torch.where(torch.rand(n, device="cuda", generator=gen) < 0.5, torch.full_like(a, 4), a)
        env.raw.step_device(a.data_ptr(), 4, torch.cuda.current_stream().cuda_stream)
        r, te, tr = rew.clone(), te_d.bool(), tr_d.bool()
        ret = ret + r
        gt = torch.where(tt < m, g[tt.clamp(max=m - 1)], torch.zeros_like(r))
        prod = r * gt
        disc = disc + prod
        tt += 1
        done = te | tr
        rets += ret[done].tolist()
        discs += disc[done].tolist()
        length += int(tt[done].sum())
        term += int(te.sum())
        over += int((tr & ~te).sum())
        ret = torch.where(done, torch.zeros_like(ret), ret)
        disc = torch.where(done, torch.zeros_like(disc), disc)
        tt = torch.where(done, torch.zeros_like(tt), tt)
    st = env.stats()
    assert np.array_equal(env.stats(), st)
    k = ticks + -(-((n + 31) // 32) // 32) + 64
    assert st[0] == len(rets) and st[2] == length and st[3] + st[4] == term and st[5] == over, (st, len(rets), length, term, over)
    assert st[7] == sum(1 for v in discs if v < 0)
    _close(st[1], rets, k, "return sum")
    _close(st[6], discs, k, "discounted-return sum")
    assert st[0] > n // 4 and st[5] > 0
    env.close()


# ---- evaluation and the state around it -------------------------------------------------------------------------------------
OUT = ("obs_map", "obs_position", "obs_velocity", "obs_nsd", "reward", "terminated", "truncated", "step_state", "step_flags")
EVAL_KW = dict(random_map_obstacle_probability=0.3, sum_subgoals_reward=300, crash_penalty=5, seed=11)


def _roll(env, acts):
    out = []
    for a in acts:
        env.step(a)
        out.append({k: getattr(env, k).copy() for k in OUT})
    return out


def _same(a, b, what):
    for t, (x, y) in enumerate(zip(a, b)):
        for k in OUT:
            assert np.array_equal(x[k], y[k]), f"{what}: tick {t}: {k} differs"


def _acts(n, k, seed=1):
    rng = np.random.default_rng(seed)
    return [np.where(rng.random(n) < 0.6, 4, rng.integers(0, 9, n)).astype(np.int32) for _ in range(k)]


@pytest.mark.parametrize("cap", [0, 5])
@pytest.mark.parametrize("backend", BACKENDS)
def test_evaluation_off_restores_the_configured_cap(backend, cap):
    """After an evaluation with max_steps = 3, training episodes are capped as configured again (no cap, or 5), exactly
    as on a handle that never evaluated; each switch-on may use another table length and gamma."""
    n = 64
    kw = dict(max_episode_steps=cap or None, seed=5)
    a, b = _native(backend, n, **kw), _native(backend, n, **kw)
    for gamma, m in ((0.9, 40), (0.5, 3)):  # a long table, then a shorter one in its place
        a.raw.set_evaluation(gamma, m)
    a.reset()
    ref = Ref(n, 0.5, 3)
    a.stats(reset_after=True)
    for _ in range(7):
        a.step(np.full(n, 4, np.int32))
        ref.tick(a.reward, a.terminated, a.truncated)
    assert ref.over == 2 * n  # truncated at ticks 3 and 6
    ref.check(a.stats(), n)
    a.raw.set_evaluation(0, 0)
    seeds = 300 + np.arange(n, dtype=np.int64)
    a.reset(seeds=seeds)
    b.reset(seeds=seeds)
    noop = [np.full(n, 4, np.int32)] * 12
    first, second = _roll(a, noop), _roll(b, noop)
    _same(first, second, "after evaluation vs never evaluated")
    trunc = np.array([x["truncated"] for x in first])
    if cap:
        assert trunc[cap - 1].all() and trunc[2 * cap - 1].all() and trunc.sum() == 2 * n
    else:
        assert not trunc.any(), f"truncations at ticks {np.nonzero(trunc.any(1))[0] + 1} with no cap configured"
    a.close()
    b.close()


@pytest.mark.parametrize("backend", BACKENDS)
def test_evaluation_run_matches_a_replay_on_a_capped_twin(backend):
    """The evaluator on the raw API (switch on, reset, clear the counters, step until enough episodes, switch off):
    its statistics equal the reference computed on the outputs of a twin built with max_episode_steps = max_steps that
    replays the same actions from the same reset; afterwards a seeded reset gives exactly the outputs of a handle that
    never evaluated, over more than max_steps ticks."""
    n, m, number = 200, 9, 300
    env = _native(backend, n, **EVAL_KW)
    env.raw.set_evaluation(GAMMA, m)
    env.reset()
    env.stats(reset_after=True)
    rng = np.random.default_rng(2)
    acts = []
    while env.stats()[0] < number:
        acts.append(np.where(rng.random(n) < 0.7, 4, rng.integers(0, 9, n)).astype(np.int32))
        env.step(acts[-1])
    st = env.stats()
    env.raw.set_evaluation(0, 0)
    twin = _native(backend, n, **dict(EVAL_KW, max_episode_steps=m))
    twin.reset()
    ref = Ref(n, GAMMA, m)
    for a in acts:
        twin.step(a)
        ref.tick(twin.reward, twin.terminated, twin.truncated)
    ref.check(st, n)
    assert ref.over > 0 and ref.term > 0
    # after evaluation: seeded reset -> the outputs of a handle that never evaluated
    fresh = _native(backend, n, **EVAL_KW)
    seeds = 77 + np.arange(n, dtype=np.int64)
    env.reset(seeds=seeds)
    fresh.reset(seeds=seeds)
    later = _acts(n, 3 * m)
    _same(_roll(env, later), _roll(fresh, later), "seeded reset after evaluation")
    for x in (env, twin, fresh):
        x.close()


@pytest.mark.parametrize("backend", BACKENDS)
def test_blobs_and_copies_across_evaluation(backend):
    """Evaluation leaves the state layout alone: a blob saved before an evaluation loads afterwards and continues
    identically, a blob saved after it loads into a handle that never evaluated, and copies work both ways."""
    n, K = 150, 10
    kw = dict(traffic_density=0.1, random_map_obstacle_probability=0.4, seed=9)
    a, b = _native(backend, n, **kw), _native(backend, n, **kw)
    acts = _acts(n, 4 + K + 6, seed=4)
    a.reset()
    _roll(a, acts[:4])
    before = a.raw.save_state()
    a.raw.set_evaluation(GAMMA, 5)
    _roll(a, acts[4:8])
    a.raw.set_evaluation(0, 0)
    # before -> after
    a.raw.load_state(before)
    first = _roll(a, acts[4:4 + K])
    b.raw.load_state(before)
    _same(first, _roll(b, acts[4:4 + K]), "blob saved before evaluation")
    # after -> a handle that never evaluated
    c = _native(backend, n, **kw)
    blob = a.raw.save_state()
    c.raw.load_state(blob)
    _same(_roll(a, acts[-6:]), _roll(c, acts[-6:]), "blob saved after evaluation")
    # copies both ways, while evaluation is on in the source, and after
    a.raw.set_evaluation(GAMMA, 6)
    d = _native(backend, n, **kw)
    d.raw.copy_state_from(a.raw)
    a.raw.set_evaluation(0, 0)
    _same(_roll(a, acts[:K]), _roll(d, acts[:K]), "copy of an evaluated handle")
    a.raw.copy_state_from(d.raw)
    _same(_roll(a, acts[K:]), _roll(d, acts[K:]), "copy into an evaluated handle")
    for x in (a, b, c, d):
        x.close()


@pytest.mark.gpu
def test_vector_env_evaluate_replay_clone_and_light_step():
    """PGTGVectorEnv.evaluate against a replay of the recorded actions on a twin capped at max_steps; then clone(),
    light_step() and checkpoints of the evaluated env work and match."""
    import torch

    from pgtg_b200.vector_env import PGTGVectorEnv

    n, m, number = RAGGED, 8, 2000
    kw = dict(random_map_obstacle_probability=0.3, sum_subgoals_reward=300, crash_penalty=5, seed=13)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        env = PGTGVectorEnv(n, **kw)
        twin = PGTGVectorEnv(n, max_episode_steps=m, **kw)
        later = PGTGVectorEnv(n, **kw)
    env.reset(seed=21)
    blob = env.save_state()
    rng = np.random.default_rng(6)
    acts = []

    def policy(obs):
        acts.append(np.where(rng.random(n) < 0.7, 4, rng.integers(0, 9, n)).astype(np.int32))
        return acts[-1]

    mean, (terminated, truncated, over, negative) = env.evaluate(policy, number, max_steps=m, GAMMA=GAMMA)
    twin.reset(seed=21)
    twin.reset()  # (evaluate's own reset)
    ref = Ref(n, GAMMA, m)
    for a in acts:
        _, r, te, tr, _ = twin.step(a)
        ref.tick(r.cpu().numpy(), te.cpu().numpy(), tr.cpu().numpy())
    assert len(ref.rets) >= number and terminated == ref.term and truncated == 0 and over == ref.over
    assert negative == sum(1 for v in ref.discs if v < 0)
    k = ref.ticks + -(-((n + 31) // 32) // 32) + 64
    want = math.fsum(ref.discs) / len(ref.discs)
    assert abs(mean - want) <= k * 2.0 ** -53 * math.fsum(abs(v) for v in ref.discs) / len(ref.discs) + 2.0 ** -52 * abs(want)
    # the evaluated env keeps training without the cap, clones and light steps, and loads the blob saved before
    env.reset(seed=3)
    a = torch.as_tensor(_acts(n, 1, 9)[0])
    c = env.clone()
    light = [x.clone() if isinstance(x, torch.Tensor) else x for x in env.light_step(a)[1:4]]
    stepped = env.step(a)[1:4]
    cloned = c.step(a)[1:4]
    for x, y, z in zip(light, stepped, cloned):
        assert torch.equal(x, y) and torch.equal(y, z)
    env.load_state(blob)
    later.load_state(blob)
    for a in _acts(n, 3 * m, 10):
        _, r1, te1, tr1, _ = env.step(a)
        _, r2, te2, tr2, _ = later.step(a)
        assert torch.equal(r1, r2) and torch.equal(te1, te2) and torch.equal(tr1, tr2)
        assert not tr1.any(), "the evaluation cap outlived evaluate()"

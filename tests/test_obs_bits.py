"""The bits observation format (pgtg_set_obs_format / observation_format="bits") and the unpack kernel (pgtg_unpack_bits).

Two handles of one configuration, seed and action stream run side by side, one storing int8 planes (already checked against the
oracle by the other suites) and one storing bits: every tick the bits must be the int8 planes packed on the host, terminal
observations included, with identical scalars and the same tick kernel. Each case runs on the emulation of the kernel phases
(tests/emu, bits.mk) and, marked gpu, on the CUDA kernels."""
import ctypes as C
import os
import subprocess
import warnings

import numpy as np
import pytest

BACKENDS = ["emu_bits", pytest.param("cuda", marks=pytest.mark.gpu)]
EMU_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")

BASE = dict(random_map_obstacle_probability=0.3, max_episode_steps=5, seed=17)
SCALARS = ("obs_position", "obs_velocity", "obs_next_subgoal_direction", "reward", "cost", "terminated", "truncated", "step_state",
           "step_flags")


def _native(backend, n, **kw):
    from native_env import NativeAdapter

    if backend == "emu_bits":
        subprocess.check_call(["make", "-s", "-C", EMU_DIR, "-f", "bits.mk"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return NativeAdapter(backend, num_envs=n, **kw)


def _pair(backend, n, **kw):
    return _native(backend, n, **kw), _native(backend, n, observation_format="bits", **kw)


def _tensor(env, name):
    import torch

    return torch.from_dlpack(env.raw.dlpack_capsule(name))


def _host(env, name):
    """a copy of a handle buffer exported through DLPack (host memory for the emulation, device memory for CUDA)"""
    import torch

    t = _tensor(env, name)
    if t.is_cuda:
        torch.cuda.synchronize()
    t = t.cpu()
    return t.view(torch.int32).numpy().view(np.uint32).copy() if t.dtype == torch.uint32 else t.numpy().copy()


def _pack(planes):
    """int8 planes -> the uint32 words of pgtg_packed_obs_bytes (env i at bit i * C*P*P)"""
    b = np.packbits(np.ascontiguousarray(planes, np.uint8).reshape(-1), bitorder="little")
    b = np.concatenate([b, np.zeros(-len(b) % 4, np.uint8)])
    return b.view(np.uint32)


def _rows(words, n, ob):
    """bits -> [n, ob] 0/1"""
    return np.unpackbits(words.view(np.uint8), bitorder="little")[: n * ob].reshape(n, ob)


def _actions(rng, n):
    return rng.integers(0, 9, n).astype(np.int32)


def _check_tick(a, b, final, t):
    n, ob = a.N, a.C * a.P * a.P
    words = a.raw.packed_obs_bytes() // 4
    assert np.array_equal(_host(b, "obs_packed")[:words], _pack(a.obs_map)), f"tick {t}: obs_packed"
    for name in SCALARS:
        if name == "cost" and not a.hc.pod.separate_reward_cost:
            continue
        assert np.array_equal(a.array(name), b.array(name)), f"tick {t}: {name}"
    if final:
        done = (a.terminated | a.truncated).astype(bool)
        got = _rows(_host(b, "final_obs_packed")[:words], n, ob)
        assert np.array_equal(got[done], a.final_obs_map.reshape(n, ob)[done]), f"tick {t}: final_obs_packed"
        for name in ("final_obs_position", "final_obs_velocity"):
            assert np.array_equal(a.array(name)[done], b.array(name)[done]), f"tick {t}: {name}"
        return int(done.sum())
    return int((a.terminated | a.truncated).sum())


def _lockstep(backend, n, ticks, monkeypatch=None, env=None, tick=None, **kw):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    a, b = _pair(backend, n, **kw)
    assert a.raw.kernel_info() == b.raw.kernel_info()
    if tick:
        assert a.raw.kernel_info().startswith(f"tick={tick}"), a.raw.kernel_info()
    rng = np.random.default_rng(5)
    a.reset(), b.reset()
    _check_tick(a, b, False, -1)
    finished = 0
    for t in range(ticks):
        act = _actions(rng, n)
        a.step(act), b.step(act)
        finished += _check_tick(a, b, bool(kw.get("final_observation")), t)
    assert finished > 0
    assert a.raw.error_summary() == b.raw.error_summary() == 0
    a.close(), b.close()


TRAFFIC = dict(traffic_density=0.05, random_map_obstacle_probability=0.3, max_episode_steps=6, seed=9)
SLIDE = lambda k, **x: dict(BASE, use_sliding_observation_window=True, sliding_observation_window_size=k, **x)  # noqa: E731
# name -> (kwargs, tick, environment, emulation envs)
CASES = {
    "lean": (dict(BASE), "lean(B=128)", {}, 200),
    "lean+final": (dict(BASE, final_observation=True), "lean+final(B=128)", {}, 200),
    "lean+final-B32": (dict(BASE, final_observation=True), "lean+final(B=32)", {"PGTG_BLOCK": "32"}, 100),
    "lean-B64": (dict(BASE), "lean(B=64)", {"PGTG_BLOCK": "64"}, 150),
    "slide-k0-final": (SLIDE(0, final_observation=True, features_to_include_in_observation=["walls"]), "lean+slide+final", {}, 301),
    "slide-k1-final-nsd": (SLIDE(1, final_observation=True, use_next_subgoal_direction=True), "lean+slide+final", {}, 150),
    "slide-k15-16planes": (SLIDE(15, features_to_include_in_observation=["walls", "goals", "subgoals", "ice", "broken road", "sand",
                                                                       "traffic light green", "traffic light yellow", "traffic light red",
                                                                       "wall", "subgoal", "final goal", "start", "used subgoal", "bogus",
                                                                       "unknown"]), "lean+slide", {}, 40),
    "general-visited-repeat": (dict(BASE, final_observation=True, already_visited_position_penalty=1,
                                    features_to_include_in_observation=["walls", "wall", "goals", "goals", "ice", "start"]), "general", {}, 150),
    "traffic": (dict(TRAFFIC), "traffic", {}, 100),
    "traffic+final": (dict(TRAFFIC, final_observation=True, use_sliding_observation_window=True, sliding_observation_window_size=1,
                           features_to_include_in_observation=["traffic", "car_spawner"]), "traffic", {}, 100),
    "general-7x7-fallback": (dict(traffic_density=0.3, use_sliding_observation_window=True, sliding_observation_window_size=12,
                                  features_to_include_in_observation=["walls", "goals", "subgoals", "ice", "broken road", "sand",
                                                                      "traffic light green", "traffic light yellow", "traffic light red",
                                                                      "wall", "subgoal", "final goal", "start", "used subgoal", "car_spawner",
                                                                      "bogus"],
                                  final_observation=True, random_map_width=7, random_map_height=7, random_map_obstacle_probability=0.3,
                                  max_episode_steps=6, seed=32), "general", {}, 33),
    "no-traffic-kernel": (dict(TRAFFIC, final_observation=True), "general", {"PGTG_NO_TRAFFIC_KERNEL": "1"}, 100),
    "numpy": (dict(BASE, rng_mode="numpy", final_observation=True), "lean+final", {}, 100),
    "levels": (dict(BASE, num_levels=7, start_level=3, final_observation=True), "lean+final", {}, 150),
}


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("backend", BACKENDS)
def test_bits_lockstep_with_int8(backend, name, monkeypatch):
    kw, tick, env, n = CASES[name]
    _lockstep(backend, n if backend == "emu_bits" else 8 * n + 3, 14, monkeypatch, env, tick, **kw)


# ---- 2. obs_map is written on demand only --------------------------------------------------------------------------------------
def _fill_obs_map(env, value, final=False):
    name = "final_obs_map" if final else "obs_map"
    if env.backend == "emu":
        ptr = getattr(env.raw.bufs, name)
        C.memset(ptr, value, env.N * env.C * env.P * env.P)
    else:
        _tensor(env, name).fill_(value)


@pytest.mark.parametrize("backend", BACKENDS)
def test_obs_map_untouched_until_expand(backend):
    n = 130 if backend == "emu_bits" else 1300
    a, b = _pair(backend, n, final_observation=True, **BASE)
    a.reset(), b.reset()
    _fill_obs_map(b, 7), _fill_obs_map(b, 7, final=True)
    rng = np.random.default_rng(2)
    for _ in range(6):
        act = _actions(rng, n)
        a.step(act), b.step(act)
        assert (b.obs_map == 7).all() and (b.final_obs_map == 7).all()
    b.raw.expand_obs(False)
    assert np.array_equal(b.obs_map, a.obs_map)
    assert (b.final_obs_map == 7).all()
    b.raw.expand_obs(True)
    done = (a.terminated | a.truncated).astype(bool)
    assert np.array_equal(b.final_obs_map[done], a.final_obs_map[done])
    a.close(), b.close()


# ---- 3. every other call gives the same results in both formats ------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
def test_other_calls_agree(backend):
    n = 100 if backend == "emu_bits" else 1000
    kw = dict(TRAFFIC, use_next_subgoal_direction=True)
    a, b = _pair(backend, n, **kw)
    rng = np.random.default_rng(3)
    a.reset(), b.reset()
    for _ in range(4):
        act = _actions(rng, n)
        a.step(act), b.step(act)
    # masked reset: words straddling a reset env and a running one keep the running env's bits
    mask = (rng.random(n) < 0.5).astype(np.uint8)
    a.reset(mask=mask), b.reset(mask=mask)
    _check_tick(a, b, False, "masked reset")
    # set_to_state + observe
    st = a.get_state()
    agent = st["agent"].copy()
    agent[:, 2:] = 0
    a.set_state(agent=agent), b.set_state(agent=agent)
    a.observe(), b.observe()
    _check_tick(a, b, False, "observe")
    # flattened observation (read straight from the bits in bits mode)
    flat = []
    for env in (a, b):
        env.raw.flatten()
        flat.append(_host(env, "obs_flat"))
    assert np.array_equal(flat[0], flat[1])
    # host-buffer steps
    act = _actions(rng, n)
    outs = []
    for env in (a, b):
        o = dict(obs_map=np.empty((n, env.C, env.P, env.P), np.int8), obs_position=np.empty((n, 2), np.int32),
                 obs_velocity=np.empty((n, 2), np.int32), reward=np.empty(n), terminated=np.empty(n, np.uint8), truncated=np.empty(n, np.uint8))
        env.raw.step_host(act, **o)
        outs.append(o)
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k
    act = _actions(rng, n)
    outs = []
    for env in (a, b):
        o = dict(obs_packed=np.empty(env.raw.packed_obs_bytes() // 4, np.uint32), obs_position=np.empty((n, 2), np.int32),
                 obs_velocity=np.empty((n, 2), np.int32), reward=np.empty(n), terminated=np.empty(n, np.uint8), truncated=np.empty(n, np.uint8))
        env.raw.step_host_packed(act, wait=True, **o)
        outs.append(o)
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k
    assert np.array_equal(outs[1]["obs_packed"], _host(b, "obs_packed")[: len(outs[1]["obs_packed"])])
    # checkpoints and clones continue identically; a blob of one format does not load into the other
    blob_a, blob_b = a.raw.save_state(), b.raw.save_state()
    with pytest.raises(ValueError):
        a.raw.load_state(blob_b)
    with pytest.raises(ValueError):
        b.raw.load_state(blob_a)
    twin = _native(backend, n, observation_format="bits", **kw)
    twin.raw.copy_state_from(b.raw)
    with pytest.raises(ValueError):
        a.raw.copy_state_from(b.raw)
    acts = [_actions(rng, n) for _ in range(3)]
    later = []
    for act in acts:
        a.step(act), b.step(act), twin.step(act)
        _check_tick(a, b, False, "after save")
        _check_tick(a, twin, False, "clone")
        later.append(_host(b, "obs_packed"))
    a.raw.load_state(blob_a), b.raw.load_state(blob_b)
    for act, want in zip(acts, later):
        a.step(act), b.step(act)
        _check_tick(a, b, False, "after load")
        assert np.array_equal(_host(b, "obs_packed"), want)
    a.close(), b.close(), twin.close()


# ---- 4. unpack -------------------------------------------------------------------------------------------------------------------
class _Mem:
    """device arrays of the backend: aligned host memory for the emulation, torch CUDA tensors for CUDA"""

    def __init__(self, backend):
        self.cuda = backend == "cuda"
        self.keep = []

    def put(self, arr):
        arr = np.ascontiguousarray(arr)
        if self.cuda:
            import torch

            t = torch.from_numpy(arr.view(np.int32) if arr.dtype == np.uint32 else arr).cuda()
            self.keep.append(t)
            return t.data_ptr()
        raw = np.zeros(arr.nbytes + 64, np.uint8)
        off = (-raw.ctypes.data) % 32
        view = raw[off: off + arr.nbytes].view(arr.dtype).reshape(arr.shape)
        view[...] = arr
        self.keep.append(view)
        return view.ctypes.data

    def empty(self, shape, dtype):
        ptr = self.put(np.zeros(shape, dtype))
        return ptr, len(self.keep) - 1

    def get(self, i):
        x = self.keep[i]
        if self.cuda:
            import torch

            torch.cuda.synchronize()
            return x.cpu().numpy()
        return x.copy()


@pytest.mark.parametrize("nsd", [False, True])
@pytest.mark.parametrize("backend", BACKENDS)
def test_unpack_rows(backend, nsd):
    n = 70 if backend == "emu_bits" else 700
    kw = dict(BASE, use_next_subgoal_direction=nsd)
    a, b = _pair(backend, n, **kw)
    rng = np.random.default_rng(4)
    a.reset(), b.reset()
    words = b.raw.packed_obs_bytes() // 4
    slots, planes, flats, pos, vel, nsds = [], [], [], [], [], []
    for _ in range(3):
        act = _actions(rng, n)
        a.step(act), b.step(act)
        slots.append(_host(b, "obs_packed")[:words])
        planes.append(a.obs_map)
        a.raw.flatten()
        flats.append(_host(a, "obs_flat"))
        pos.append(b.obs_position), vel.append(b.obs_velocity), nsds.append(b.obs_nsd)
    bits, planes, flats = np.stack(slots), np.concatenate(planes), np.concatenate(flats)
    m = _Mem(backend)
    src, p_pos, p_vel, p_nsd = m.put(bits), m.put(np.stack(pos)), m.put(np.stack(vel)), m.put(np.stack(nsds))
    total = 3 * n
    # host unpack of the same bits
    host = np.empty((n, b.C, b.P, b.P), np.int8)
    b.raw.unpack_obs(slots[1].copy(), host)
    assert np.array_equal(host, planes[n: 2 * n])
    for index in (None, rng.permutation(total), rng.integers(0, total, 2 * total + 5), np.zeros(0, np.int64), np.array([total - 1] * 3)):
        rows = np.arange(total) if index is None else index
        p_idx = None if index is None else m.put(index.astype(np.int64)) if len(index) else m.put(np.zeros(1, np.int64))
        p8, i8 = m.empty((len(rows),) + planes.shape[1:], np.int8)
        b.raw.unpack_bits(src, 3, p_idx, len(rows), "int8", p8)
        assert np.array_equal(m.get(i8), planes[rows])
        pf, jf = m.empty((len(rows), flats.shape[1]), np.float32)
        b.raw.unpack_bits(src, 3, p_idx, len(rows), "flat", pf, p_pos, p_vel, p_nsd if nsd else None)
        assert np.array_equal(m.get(jf).view(np.uint32), flats[rows].view(np.uint32))
    assert b.raw.error_summary() == 0
    # an index outside the stored rows: a zero row and error flag 256
    index = np.array([0, total, -1, 5], np.int64)
    p8, i8 = m.empty((4,) + planes.shape[1:], np.int8)
    b.raw.unpack_bits(src, 3, m.put(index), 4, "int8", p8)
    got = m.get(i8)
    assert np.array_equal(got[[0, 3]], planes[[0, 5]]) and not got[[1, 2]].any()
    assert b.raw.error_summary() == 256
    pf, jf = m.empty((4, flats.shape[1]), np.float32)
    b.raw.unpack_bits(src, 3, m.put(index), 4, "flat", pf, p_pos, p_vel, p_nsd if nsd else None)
    got = m.get(jf)
    assert np.array_equal(got[[0, 3]], flats[[0, 5]]) and not got[[1, 2]].any()
    a.close(), b.close()


# ---- 5. errors ------------------------------------------------------------------------------------------------------------------
def test_format_errors():
    env = _native("emu_bits", 8, **BASE)
    lib, h = env.raw.lib, env.raw._h
    assert lib.pgtg_set_obs_format(h, 7) == -1 and b"unknown observation format" in lib.pgtg_last_error()
    assert lib.pgtg_expand_obs(h, 0, None) == -3  # int8 handle
    env.raw.set_obs_format("bits")
    env.raw.set_obs_format("int8")
    env.raw.set_obs_format("bits")
    env.reset()
    assert lib.pgtg_set_obs_format(h, 0) == -3 and b"before the first pgtg_reset" in lib.pgtg_last_error()
    assert lib.pgtg_expand_obs(h, 1, None) == -3  # no terminal observations in this configuration
    with pytest.raises(ValueError):
        env.raw.set_obs_format("half")
    env.close()
    from native_env import NativeAdapter

    from pgtg_b200.config import make_config

    with pytest.raises(ValueError):
        make_config(num_envs=4, observation_format="uint8")
    plain = NativeAdapter("emu", num_envs=4)  # a backend without the bits format refuses it
    assert plain.raw.lib.pgtg_set_obs_format(plain.raw._h, 1) == -1 and b"no bits observation format" in plain.raw.lib.pgtg_last_error()
    plain.close()


# ---- the vector env -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vector_env_bits():
    import torch

    from pgtg_b200 import PGTGVectorEnv
    from pgtg_b200.vector_env import LazyPlanes

    n = 3000
    kw = dict(BASE, final_observation=True, use_next_subgoal_direction=True, use_sliding_observation_window=True,
              sliding_observation_window_size=3)
    with pytest.raises(ValueError):
        PGTGVectorEnv(4, observation_format="float")
    a, b = PGTGVectorEnv(n, **kw), PGTGVectorEnv(n, observation_format="bits", **kw)
    oa, _ = a.reset(seed=1)
    ob, _ = b.reset(seed=1)
    assert isinstance(ob["map"], LazyPlanes)
    g = torch.Generator(device="cuda").manual_seed(0)
    store = torch.empty((4, b.obs_packed().numel()), dtype=torch.uint32, device="cuda")
    pos = torch.empty((4, n, 2), dtype=torch.int32, device="cuda")
    vel, nsd = torch.empty_like(pos), torch.empty((4, n), dtype=torch.int32, device="cuda")
    ref = []
    for t in range(4):
        act = torch.randint(0, 9, (n,), device="cuda", generator=g, dtype=torch.int32)
        oa, ra, ta, tra, ia = a.step(act)
        ob, rb, tb, trb, ib = b.step(act)
        store[t].copy_(b.obs_packed()), pos[t].copy_(ob["position"]), vel[t].copy_(ob["velocity"]), nsd[t].copy_(ob["next_subgoal_direction"])
        ref.append((torch.stack([oa["map"][k] for k in a.hc.observation_keys], 1).clone(), a.flat_observation().clone()))
        assert torch.equal(b.flat_observation(), ref[-1][1])
        for k in a.hc.observation_keys:
            assert torch.equal(ob["map"][k], oa["map"][k])
        done = ta | tra
        for k in a.hc.observation_keys:
            assert torch.equal(ib["final_observation"]["map"][k][done], ia["final_observation"]["map"][k][done])
        assert torch.equal(rb, ra) and torch.equal(tb, ta)
    idx = torch.randint(0, 4 * n, (5000,), device="cuda", generator=g)
    planes = torch.cat([r[0] for r in ref])
    flats = torch.cat([r[1] for r in ref])
    assert torch.equal(b.unpack(store, idx), planes[idx])
    assert torch.equal(b.unpack(store), planes)
    got = b.unpack(store, idx, format="flat", position=pos, velocity=vel, next_subgoal_direction=nsd)
    assert torch.equal(got, flats[idx])
    b.episode_stats()
    a.close(), b.close()

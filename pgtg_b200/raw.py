"""Thin object over one native handle (one GPU): the array-level API the vector env and the parity
tests share. Everything here is a direct call through the C ABI."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._names import CARDINALS
from .config import HostConfig, PgtgRule, direction_lut, rule_to_pod


class RawEnv:
    def __init__(self, hc: HostConfig, device: int = 0, lib_path: str | None = None):
        self.hc = hc
        self.lib = _lib.load(lib_path)
        self.device = device
        h = C.c_void_p()
        _lib.check(self.lib, self.lib.pgtg_create(C.byref(hc.pod), int(device), C.byref(h)))
        self._h = h
        c = hc.pod
        self.N, self.C, self.P, self.T = c.num_envs, c.num_channels, hc.window, c.map_w * c.map_h
        bufs = _lib.PgtgBuffers()
        _lib.check(self.lib, self.lib.pgtg_get_buffers(self._h, C.byref(bufs)))
        self.bufs = bufs
        self.max_cars = bufs.max_cars
        if hc.map_plan is not None:
            mp = hc.map_plan
            _lib.check(self.lib, self.lib.pgtg_load_fixed_map(
                self._h, mp.packed_tiles(), mp.width, mp.height, int(mp.start[0]), int(mp.start[1]),
                CARDINALS.index(mp.start[2]), int(mp.goal[0]), int(mp.goal[1]), CARDINALS.index(mp.goal[2])))
        # direction table evaluated by this interpreter's math.atan2, exactly like the reference
        radius = max(c.map_w, c.map_h) * 9 + 2
        lut = np.ascontiguousarray(direction_lut(radius))
        _lib.check(self.lib, self.lib.pgtg_load_direction_lut(self._h, lut.ctypes.data, radius))
        if hc.observation_format != "int8":
            self.set_obs_format(hc.observation_format)
        self._keep = []

    # -- control ------------------------------------------------------------------------------
    def load_draws(self, values, tags, offsets):
        v = np.ascontiguousarray(values, np.float64)
        t = np.ascontiguousarray(tags, np.uint8)
        o = np.ascontiguousarray(offsets, np.int64)
        assert o.shape == (self.N + 1,)
        _lib.check(self.lib, self.lib.pgtg_load_draws(self._h, v.ctypes.data, t.ctypes.data, o.ctypes.data))

    def reset(self, seeds=None, mask=None, stream: int = 0):
        s = None if seeds is None else np.ascontiguousarray(seeds, np.int64)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        _lib.check(self.lib, self.lib.pgtg_reset(self._h, None if s is None else s.ctypes.data,
                                                 None if m is None else m.ctypes.data, stream))

    def step_device(self, actions_ptr: int, action_bytes: int = 4, stream: int = 0):
        _lib.check(self.lib, self.lib.pgtg_step(self._h, actions_ptr, action_bytes, stream))

    def step_host(self, actions, obs_map=None, obs_position=None, obs_velocity=None, reward=None, terminated=None,
                  truncated=None, stream: int = 0):
        a = np.ascontiguousarray(actions, np.int32)
        assert a.shape == (self.N,)
        ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
        _lib.check(self.lib, self.lib.pgtg_step_host(self._h, a.ctypes.data, ptr(obs_map), ptr(obs_position),
                                                     ptr(obs_velocity), ptr(reward), ptr(terminated), ptr(truncated), stream))

    def observe(self, stream: int = 0):
        _lib.check(self.lib, self.lib.pgtg_observe(self._h, stream))

    def update_rules(self, rules: list):
        arr = (PgtgRule * max(1, len(rules)))()
        for i, r in enumerate(rules):
            arr[i] = rule_to_pod(r)
        _lib.check(self.lib, self.lib.pgtg_update_rules(self._h, arr, len(rules)))

    # -- state --------------------------------------------------------------------------------
    def get_state(self) -> dict:
        N, T, MC = self.N, self.T, self.max_cars
        out = dict(
            agent=np.zeros((N, 4), np.int32), flat_tire=np.zeros(N, np.uint8), light_counter=np.zeros(N, np.int32),
            elapsed=np.zeros(N, np.int32), num_cars=np.zeros(N, np.int32), cars=np.zeros((N, MC, 7), np.int32),
            tiles=np.zeros((N, T), np.uint16), plan=np.zeros((N, 8), np.int32), used=np.zeros((N, T), np.uint8),
            draw_cursor=np.zeros(N, np.int64), error=np.zeros(N, np.int32))
        st = _lib.PgtgState(**{k: v.ctypes.data for k, v in out.items()})
        _lib.check(self.lib, self.lib.pgtg_get_state(self._h, C.byref(st)))
        return out

    def get_info(self) -> dict:
        """The computed parts of PGTGEnv.get_info (environment.py:1538-1578) for every env."""
        out = dict(agent_direction=np.zeros(self.N, np.int32), current_tile_type=np.zeros(self.N, np.int32),
                   profile_counts=np.zeros((self.N, 5), np.int32))
        _lib.check(self.lib, self.lib.pgtg_get_info(self._h, out["agent_direction"].ctypes.data, out["current_tile_type"].ctypes.data,
                                                    out["profile_counts"].ctypes.data))
        return out

    def set_state(self, agent=None, flat_tire=None, num_cars=None, cars=None):
        keep, kw = [], {}
        for name, arr, dt in (("agent", agent, np.int32), ("flat_tire", flat_tire, np.uint8),
                              ("num_cars", num_cars, np.int32), ("cars", cars, np.int32)):
            if arr is not None:
                a = np.ascontiguousarray(arr, dt)
                keep.append(a)
                kw[name] = a.ctypes.data
        st = _lib.PgtgState(**kw)
        _lib.check(self.lib, self.lib.pgtg_set_state(self._h, C.byref(st)))

    def stats(self, reset_after: bool = False) -> np.ndarray:
        out = np.zeros(8, np.float64)
        _lib.check(self.lib, self.lib.pgtg_stats(self._h, out.ctypes.data, int(reset_after)))
        return out

    def flatten(self, stream: int = 0):
        """Launch the FlattenObservation kernel; -> (device pointer, D). Key order: sorted map keys."""
        keys = self.hc.observation_keys
        order = np.array([keys.index(k) for k in sorted(keys)], np.int32)
        ptr, dim = C.c_void_p(), C.c_int()
        _lib.check(self.lib, self.lib.pgtg_flatten(self._h, order.ctypes.data, stream, C.byref(ptr), C.byref(dim)))
        return ptr.value, dim.value

    # -- checkpoint / clone / evaluation / host-buffer steps ----------------------------------------------
    def save_state(self) -> np.ndarray:
        """Everything a tick reads or writes, as one host blob (pgtg_save_state)."""
        n = int(self.lib.pgtg_state_bytes(self._h))
        blob = np.empty(n, np.uint8)
        _lib.check(self.lib, self.lib.pgtg_save_state(self._h, blob.ctypes.data, n))
        return blob

    def load_state(self, blob: np.ndarray):
        b = np.ascontiguousarray(blob, np.uint8)
        _lib.check(self.lib, self.lib.pgtg_load_state(self._h, b.ctypes.data, b.nbytes))

    def copy_state_from(self, other: "RawEnv"):
        _lib.check(self.lib, self.lib.pgtg_copy_state(self._h, other._h))

    def set_evaluation(self, gamma: float, max_steps: int):
        _lib.check(self.lib, self.lib.pgtg_set_evaluation(self._h, float(gamma), int(max_steps)))

    def error_summary(self) -> int:
        v = C.c_uint32()
        _lib.check(self.lib, self.lib.pgtg_error_summary(self._h, C.byref(v)))
        return int(v.value)

    def packed_obs_bytes(self) -> int:
        return int(self.lib.pgtg_packed_obs_bytes(self._h))

    def step_host_packed(self, actions, obs_packed=None, obs_position=None, obs_velocity=None, reward=None, terminated=None,
                         truncated=None, wait: bool = True, stream: int = 0):
        a = np.ascontiguousarray(actions, np.int32)
        assert a.shape == (self.N,)
        self._keep = [a]  # (the copy of the actions is asynchronous)
        ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
        _lib.check(self.lib, self.lib.pgtg_step_host_packed(self._h, a.ctypes.data, ptr(obs_packed), ptr(obs_position), ptr(obs_velocity),
                                                            ptr(reward), ptr(terminated), ptr(truncated), int(bool(wait)), stream))

    def host_sync(self):
        _lib.check(self.lib, self.lib.pgtg_host_sync(self._h))

    def unpack_obs(self, obs_packed: np.ndarray, out: np.ndarray | None = None, threads: int = 0) -> np.ndarray:
        """bits -> int8 [N, C, P, P] on the host (multithreaded)."""
        import os

        if out is None:
            out = np.empty((self.N, self.C, self.P, self.P), np.int8)
        _lib.check(self.lib, self.lib.pgtg_unpack_obs(obs_packed.ctypes.data, out.ctypes.data, out.size, threads or (os.cpu_count() or 1)))
        return out

    def set_overlap(self, on: bool):
        _lib.check(self.lib, self.lib.pgtg_set_overlap(self._h, int(bool(on))))

    def enable_timing(self, max_steps: int):
        _lib.check(self.lib, self.lib.pgtg_enable_timing(self._h, int(max_steps)))

    def timing(self) -> dict:
        """-> mean device time (ms) of the tick and map-generation kernels over the recorded ticks."""
        a, b, n = C.c_double(), C.c_double(), C.c_int()
        _lib.check(self.lib, self.lib.pgtg_timing(self._h, C.byref(a), C.byref(b), C.byref(n)))
        k = max(n.value, 1)
        return dict(tick_ms=a.value / k, mapgen_ms=b.value / k, steps=n.value)

    def launch_count(self) -> int:
        return int(self.lib.pgtg_launch_count(self._h))

    def kernel_info(self) -> str:
        buf = C.create_string_buffer(256)
        _lib.check(self.lib, self.lib.pgtg_kernel_info(self._h, buf, 256))
        return buf.value.decode()

    def levels(self, previous: bool = False, stream: int | None = None):
        """Level of every env's current episode (previous=True: of the episode before it -- for an env that auto-reset in
        the last step, the one that just ended) as a torch int32 [N] on the handle's device; no host synchronisation."""
        import torch

        if getattr(self, "_level_device", None) is None:
            self._level_device = torch.from_dlpack(self.dlpack_capsule("level_plan")).device
        dev = self._level_device
        out = torch.empty(self.N, dtype=torch.int32, device=dev)
        if stream is None:
            stream = torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else 0
        _lib.check(self.lib, self.lib.pgtg_levels(self._h, out.data_ptr(), int(bool(previous)), stream))
        return out

    def level_pool(self):
        """-> (level_tiles uint16 [M, T], level_plan uint32 [M]) as torch views of the handle's pool."""
        import torch

        return torch.from_dlpack(self.dlpack_capsule("level_tiles")), torch.from_dlpack(self.dlpack_capsule("level_plan"))

    # -- bits observation format ---------------------------------------------------------------------------------
    def set_obs_format(self, fmt: str):
        """"int8" (the default) or "bits": how the ticks store the observation planes; only before the first reset."""
        if fmt not in _lib.OBS_FORMATS:
            raise ValueError(f"observation format must be one of {tuple(_lib.OBS_FORMATS)}")
        _lib.check(self.lib, self.lib.pgtg_set_obs_format(self._h, _lib.OBS_FORMATS[fmt]))
        self.hc.observation_format = fmt

    def expand_obs(self, final: bool = False, stream: int = 0):
        """Bits format: fill obs_map (final_obs_map) from obs_packed (final_obs_packed) on `stream`."""
        _lib.check(self.lib, self.lib.pgtg_expand_obs(self._h, int(bool(final)), stream))

    def unpack_bits(self, bits_ptr: int, slots: int, index_ptr: int | None, count: int, fmt: str, out_ptr: int,
                    position_ptr: int | None = None, velocity_ptr: int | None = None, nsd_ptr: int | None = None, stream: int = 0):
        """pgtg_unpack_bits on raw device pointers; fmt "int8" or "flat" (planes in sorted-key order, as `flatten`)."""
        if fmt not in _lib.UNPACK_FORMATS:
            raise ValueError(f"unpack format must be one of {tuple(_lib.UNPACK_FORMATS)}")
        keys = self.hc.observation_keys
        order = np.array([keys.index(k) for k in sorted(keys)] or [0], np.int32)
        _lib.check(self.lib, self.lib.pgtg_unpack_bits(self._h, bits_ptr, int(slots), index_ptr, int(count), _lib.UNPACK_FORMATS[fmt], out_ptr,
                                                       order.ctypes.data, position_ptr, velocity_ptr, nsd_ptr, stream))

    def dlpack_capsule(self, name: str):
        """-> a PyCapsule named "dltensor" for `torch.from_dlpack` / any DLPack consumer."""
        mt = C.c_void_p()
        _lib.check(self.lib, self.lib.pgtg_dlpack(self._h, name.encode(), C.byref(mt)))
        new = C.pythonapi.PyCapsule_New
        new.restype, new.argtypes = C.py_object, [C.c_void_p, C.c_char_p, C.c_void_p]
        return new(mt, b"dltensor", None)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.pgtg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

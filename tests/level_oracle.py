"""ctypes front-end of tests/level_oracle_c: the CPU oracle with level sets (test infrastructure only).

`LevelOracle` has the array-level surface of `oracle.oracle.OracleVectorEnv` that the lock-step harness uses (reset, step,
output arrays, get_state), plus `levels(previous)` and `level_pool()` in the layouts of the product's `pgtg_levels` and
`"level_tiles"` / `"level_plan"`."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import warnings

import numpy as np

from oracle.oracle import PgtgState
from pgtg_b200.config import PgtgConfig, make_config

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "level_oracle_c")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        subprocess.check_call(["make", "-s", "-C", _DIR])
        _LIB = C.CDLL(os.path.join(_DIR, "libpgtg_level_oracle.so"))
        _LIB.lvl_create.restype = C.c_void_p
        _LIB.lvl_create.argtypes = [C.POINTER(PgtgConfig)]
        for name in ("lvl_destroy", "ora_set_threads"):
            getattr(_LIB, name).restype = None
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class LevelOracle:
    def __init__(self, threads: int = 1, **kwargs):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            self.hc = make_config(**kwargs)
        c = self.hc.pod
        self.N, self.C, self.P, self.T = c.num_envs, c.num_channels, self.hc.window, c.map_w * c.map_h
        self.max_cars = max(1, c.max_cars)
        h = lib().lvl_create(C.byref(c))
        assert h, "level oracle: needs num_levels > 0 in Philox mode on procedural maps"
        self._h = C.c_void_p(h)
        lib().ora_set_threads(self._h, int(threads))
        N, Cc, P = self.N, self.C, self.P
        self.obs_map = np.zeros((N, Cc, P, P), np.int8)
        self.obs_position = np.zeros((N, 2), np.int32)
        self.obs_velocity = np.zeros((N, 2), np.int32)
        self.obs_nsd = np.zeros(N, np.int32)
        self.reward = np.zeros(N, np.float64)
        self.cost = np.zeros(N, np.float64)
        self.terminated = np.zeros(N, np.uint8)
        self.truncated = np.zeros(N, np.uint8)
        self.step_state = np.zeros((N, 4), np.int32)
        self.step_flags = np.zeros(N, np.uint8)
        self.final_obs_map = np.zeros((N, Cc, P, P), np.int8)
        self.final_obs_position = np.zeros((N, 2), np.int32)
        self.final_obs_velocity = np.zeros((N, 2), np.int32)
        self.final_obs_nsd = np.zeros(N, np.int32)

    def reset(self, seeds=None, mask=None):
        s = None if seeds is None else np.ascontiguousarray(seeds, np.int64)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        assert lib().lvl_reset(self._h, _p(s), _p(m), _p(self.obs_map), _p(self.obs_position), _p(self.obs_velocity), _p(self.obs_nsd)) == 0

    def step(self, actions):
        a = np.ascontiguousarray(actions, np.int32)
        assert a.shape == (self.N,)
        assert lib().lvl_step(self._h, _p(a), _p(self.obs_map), _p(self.obs_position), _p(self.obs_velocity), _p(self.obs_nsd),
                              _p(self.reward), _p(self.cost), _p(self.terminated), _p(self.truncated), _p(self.step_state),
                              _p(self.step_flags), _p(self.final_obs_map), _p(self.final_obs_position), _p(self.final_obs_velocity),
                              _p(self.final_obs_nsd)) == 0

    def get_state(self) -> dict:
        N, T, MC = self.N, self.T, self.max_cars
        out = dict(
            agent=np.zeros((N, 4), np.int32), flat_tire=np.zeros(N, np.uint8), light_counter=np.zeros(N, np.int32),
            elapsed=np.zeros(N, np.int32), num_cars=np.zeros(N, np.int32), cars=np.zeros((N, MC, 7), np.int32),
            tiles=np.zeros((N, T), np.uint16), plan=np.zeros((N, 8), np.int32), used=np.zeros((N, T), np.uint8),
            draw_cursor=np.zeros(N, np.int64), error=np.zeros(N, np.int32))
        st = PgtgState(**{k: v.ctypes.data for k, v in out.items()})
        assert lib().ora_get_state(self._h, C.byref(st)) == 0
        return out

    def levels(self, previous=False):
        out = np.zeros(self.N, np.int32)
        assert lib().lvl_levels(self._h, _p(out), int(bool(previous))) == 0
        return out

    def level_pool(self):
        M = self.hc.pod.num_levels
        tiles, plan = np.zeros((M, self.T), np.uint16), np.zeros(M, np.uint32)
        assert lib().lvl_pool(self._h, _p(tiles), _p(plan)) == 0
        return tiles, plan

    def close(self):
        if self._h:
            lib().lvl_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

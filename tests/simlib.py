"""TEST INFRASTRUCTURE: ctypes front-end of tests/hostsim (host build of the device headers)."""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
ASSETS = os.path.join(ROOT, "procgen2_b200", "data", "assets.bin")

_lib = None


def lib():
    global _lib
    if _lib is None:
        from tests.hostsim import build as hb
        L = ctypes.CDLL(hb.build())
        L.hs_create.restype = ctypes.c_void_p
        L.hs_create.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p]
        L.hs_create_mode.restype = ctypes.c_void_p
        L.hs_create_mode.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
        L.hs_destroy.argtypes = [ctypes.c_void_p]
        L.hs_reset.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.hs_step.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.hs_render_human.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        for n, t in (("hs_obs", ctypes.c_uint8), ("hs_reward", ctypes.c_float), ("hs_terminated", ctypes.c_uint8), ("hs_truncated", ctypes.c_uint8)):
            getattr(L, n).restype = ctypes.POINTER(t)
            getattr(L, n).argtypes = [ctypes.c_void_p]
        L.hs_read_field.restype = ctypes.c_long
        L.hs_read_field.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_long, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
        L.hs_last_error.restype = ctypes.c_char_p
        _lib = L
    return _lib


class HostSim:
    def __init__(self, game, num_envs, seed, max_episode_steps=0, distribution_mode=-1):
        L = lib()
        self.n = num_envs
        self.h = L.hs_create_mode(game.encode(), num_envs, seed, max_episode_steps, ASSETS.encode(), distribution_mode)
        if not self.h:
            raise RuntimeError(L.hs_last_error().decode())

    def _out(self):
        L = lib()
        obs = np.ctypeslib.as_array(L.hs_obs(self.h), shape=(self.n, 64, 64, 3)).copy()
        rew = np.ctypeslib.as_array(L.hs_reward(self.h), shape=(self.n,)).copy()
        term = np.ctypeslib.as_array(L.hs_terminated(self.h), shape=(self.n,)).copy().astype(bool)
        return obs, rew, term

    def reset(self, seeds=None):
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, np.int32)
        lib().hs_reset(self.h, seeds.ctypes.data if seeds is not None else None)
        return self._out()[0]

    def step(self, actions):
        a = np.ascontiguousarray(actions, np.int32)
        lib().hs_step(self.h, a.ctypes.data)
        return self._out()

    def render_human(self, env, width, height):
        out = np.empty((height, width, 3), np.uint8)
        if lib().hs_render_human(self.h, env, width, height, out.ctypes.data):
            raise RuntimeError("render_human: the %dx%d window spans more tile rows than the frame tables hold" % (width, height))
        return out

    def field(self, name):
        L = lib()
        esz, pe = ctypes.c_int(), ctypes.c_int()
        nbytes = L.hs_read_field(self.h, name.encode(), None, 0, ctypes.byref(esz), ctypes.byref(pe))
        if nbytes < 0:
            raise KeyError(name)
        buf = np.empty(nbytes, np.uint8)
        L.hs_read_field(self.h, name.encode(), buf.ctypes.data, nbytes, None, None)
        return buf, esz.value, pe.value

    def close(self):
        if self.h:
            lib().hs_destroy(self.h)
            self.h = None

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
        L.hs_create.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p] + [ctypes.c_int] * 3
        L.hs_destroy.argtypes = [ctypes.c_void_p]
        L.hs_reset.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.hs_step.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.hs_render_human.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        for n, t in (("hs_obs", ctypes.c_uint8), ("hs_reward", ctypes.c_float), ("hs_terminated", ctypes.c_uint8), ("hs_truncated", ctypes.c_uint8),
                     ("hs_final_obs", ctypes.c_uint8)):
            getattr(L, n).restype = ctypes.POINTER(t)
            getattr(L, n).argtypes = [ctypes.c_void_p]
        L.hs_read_field.restype = ctypes.c_long
        L.hs_read_field.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_long, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
        L.hs_write_field.restype = ctypes.c_long
        L.hs_write_field.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_long]
        L.hs_field_count.argtypes = [ctypes.c_void_p]
        L.hs_field_info.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_char_p] + [ctypes.POINTER(ctypes.c_int)] * 3
        L.hs_invalidate_views.argtypes = [ctypes.c_void_p]
        L.hs_last_error.restype = ctypes.c_char_p
        _lib = L
    return _lib


class HostSim:
    """auto_reset / final_obs: the engine's step variants (pg2_config). auto_reset=False: a finished env is not reset;
    final_obs=True: final_obs() = the terminal frame of every env that finished, written in the step it finished in."""

    def __init__(self, game, num_envs, seed, max_episode_steps=0, distribution_mode=-1, auto_reset=True, final_obs=False):
        L = lib()
        self.n = num_envs
        self.h = L.hs_create(game.encode(), num_envs, seed, max_episode_steps, ASSETS.encode(), distribution_mode,
                             1 if auto_reset else 0, 1 if final_obs else 0)
        if not self.h:
            raise RuntimeError(L.hs_last_error().decode())

    def _out(self):
        L = lib()
        obs = np.ctypeslib.as_array(L.hs_obs(self.h), shape=(self.n, 64, 64, 3)).copy()
        rew = np.ctypeslib.as_array(L.hs_reward(self.h), shape=(self.n,)).copy()
        term = np.ctypeslib.as_array(L.hs_terminated(self.h), shape=(self.n,)).copy().astype(bool)
        return obs, rew, term

    def truncated(self):
        return np.ctypeslib.as_array(lib().hs_truncated(self.h), shape=(self.n,)).copy().astype(bool)

    def final_obs(self):
        return np.ctypeslib.as_array(lib().hs_final_obs(self.h), shape=(self.n, 64, 64, 3)).copy()

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

    def field_list(self):
        """[(name, element size, elements per env, env-major)] of every field of the game state and CommonState."""
        L = lib()
        out = []
        name = ctypes.create_string_buffer(64)
        esz, pe, em = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        for i in range(L.hs_field_count(self.h)):
            assert L.hs_field_info(self.h, i, name, ctypes.byref(esz), ctypes.byref(pe), ctypes.byref(em)) == 0
            out.append((name.value.decode(), esz.value, pe.value, bool(em.value)))
        return out

    def write_field(self, name, data):
        a = np.ascontiguousarray(data)
        n = lib().hs_write_field(self.h, name.encode(), a.ctypes.data, a.nbytes)
        if n == -1:
            raise KeyError(name)
        if n != a.nbytes:
            raise ValueError("hs_write_field %s: %d bytes given" % (name, a.nbytes))

    def invalidate_views(self):
        """Mark every env's cached view stale (its cache is this sim's own, not that of the state's source)."""
        lib().hs_invalidate_views(self.h)

    def close(self):
        if self.h:
            lib().hs_destroy(self.h)
            self.h = None


def transplant(src, sim):
    """Copy every state field of `src` (a BatchedEnv or a HostSim of the same game, mode, N and max_episode_steps)
    into the HostSim `sim`, byte for byte: both lay a field out alike at equal N. Checks that `src` knows every field
    the sim has, with the same element size and count per env. The sim's view caches are invalidated."""
    for name, esz, pe, _ in sim.field_list():
        if isinstance(src, HostSim):
            buf, e2, p2 = src.field(name)
        else:
            buf, e2, p2 = src.read_field(name)
        assert (e2, p2) == (esz, pe), "field %s: %d x %d bytes per env in the source, %d x %d in the host-sim" % (name, p2, e2, pe, esz)
        sim.write_field(name, buf)
    sim.invalidate_views()


def read_state(src, fields):
    """{name: raw bytes (uint8 array)} of the given fields (HostSim.field_list() entries) of a BatchedEnv or HostSim."""
    return {name: (src.field(name) if isinstance(src, HostSim) else src.read_field(name))[0] for name, _, _, _ in fields}


def _elem(buf, esz, i):
    raw = bytes(buf[i * esz:(i + 1) * esz])
    v = int.from_bytes(raw, "little")
    if esz == 4:
        return "%d / %r (0x%08x)" % (np.frombuffer(raw, np.int32)[0], float(np.frombuffer(raw, np.float32)[0]), v)
    return "%d (0x%0*x)" % (v, 2 * esz, v)


def state_diff(want, got, fields, n, skip=(), lane_group=None):
    """Human-readable report of every field in which `got` differs from `want` (read_state of the same field list at n
    envs), naming the first differing element of each: env, slot / element index and both values (4-byte elements as
    int32 and float32, and in hex, which tells -0.0 from 0.0 and NaN payloads apart). `skip`: field names not compared.
    lane_group(env) -> text added to the env. Empty string: equal."""
    lines = []
    for name, esz, pe, env_major in fields:
        if name in skip:
            continue
        a, b = want[name], got[name]
        if np.array_equal(a, b):
            continue
        elem = np.flatnonzero((a.reshape(-1, esz) != b.reshape(-1, esz)).any(axis=1))
        i = int(elem[0])
        env, k = (i // pe, i % pe) if env_major else (i % n, i // n)
        envs = np.unique((elem // pe) if env_major else (elem % n))
        lines.append("field %s: %d elements of %d envs differ; first env %d%s, element %d: want %s, got %s" % (
            name, elem.size, envs.size, env, lane_group(env) if lane_group else "", k, _elem(a, esz, i), _elem(b, esz, i)))
    return "\n".join(lines)

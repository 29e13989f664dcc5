"""ctypes binding of the engine C ABI (include/pg2_engine.h) — the batched front-end.

`BatchedEnv` is the vectorised counterpart of the reference's `CEnv` (cenv/cenv.py:152-380):
same reset()/step() vocabulary, but N environments per call, observations resident in HBM
(exposed as torch tensors that alias the engine's buffers, no copy) and actions accepted either
from host memory or as a CUDA tensor. There is no CPU path: constructing it without the CUDA
extension or without a GPU raises.
"""
import ctypes
import os

import numpy as np

from . import build as _build

OBS_SHAPE = (64, 64, 3)
OBS_BYTES = 64 * 64 * 3
GAMES = ("bossfight", "caveflyer", "chaser", "climber", "coinrun", "jumper", "maze")


class _Config(ctypes.Structure):
    _fields_ = [("game", ctypes.c_char_p), ("num_envs", ctypes.c_int32), ("seed", ctypes.c_int32),
                ("first_env", ctypes.c_int32), ("device", ctypes.c_int32), ("max_episode_steps", ctypes.c_int32),
                ("assets_path", ctypes.c_char_p), ("auto_reset", ctypes.c_int32), ("distribution_mode", ctypes.c_int32),
                ("final_obs", ctypes.c_int32)]


_lib = None


class _Raw:
    """A device buffer of the engine, described for torch.as_tensor (__cuda_array_interface__)."""
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def load_library():
    """Load procgen2_b200/lib/libprocgen2_b200.so (built in-tree by procgen2_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PG2_ENGINE_LIB", _build.ENGINE)   # override: A/B experiments with alternative builds
    if not os.path.exists(path):
        raise RuntimeError("CUDA extension %s is missing: run `python -m procgen2_b200.build` "
                           "(there is no CPU fallback)" % path)
    L = ctypes.CDLL(path)
    vp = ctypes.c_void_p
    L.pg2_create.argtypes = [ctypes.POINTER(_Config), ctypes.POINTER(vp)]
    L.pg2_create.restype = ctypes.c_int32
    L.pg2_destroy.argtypes = [vp]
    L.pg2_destroy.restype = None
    L.pg2_reset.argtypes = [vp, vp]
    L.pg2_step.argtypes = [vp, vp]
    L.pg2_step_device.argtypes = [vp, vp]
    L.pg2_fetch.argtypes = [vp, vp, vp, vp, vp]
    L.pg2_step_pipelined.argtypes = [vp, vp, vp, vp, vp, vp]
    L.pg2_pipeline_flush.argtypes = [vp]
    L.pg2_fetch_final.argtypes = [vp, vp]
    for name in ("pg2_obs_device", "pg2_reward_device", "pg2_terminated_device", "pg2_truncated_device", "pg2_final_obs_device", "pg2_stream"):
        getattr(L, name).argtypes = [vp]
        getattr(L, name).restype = vp
    L.pg2_sync.argtypes = [vp]
    L.pg2_num_envs.argtypes = [vp]
    L.pg2_step_epw.argtypes = [vp]
    L.pg2_kernel_launches.argtypes = [vp]
    L.pg2_kernel_launches.restype = ctypes.c_int64
    L.pg2_state_bytes_per_env.argtypes = [vp]
    L.pg2_state_bytes_per_env.restype = ctypes.c_int64
    L.pg2_read_field.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int64, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
    L.pg2_read_field.restype = ctypes.c_int64
    L.pg2_write_field.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int64]
    L.pg2_write_field.restype = ctypes.c_int64
    L.pg2_snapshot.argtypes = [vp, vp, ctypes.c_int64]
    L.pg2_snapshot.restype = ctypes.c_int64
    L.pg2_restore.argtypes = [vp, vp, ctypes.c_int64]
    L.pg2_restore.restype = ctypes.c_int64
    L.pg2_profile.argtypes = [vp, ctypes.c_int32]
    L.pg2_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int64)]
    L.pg2_last_error.restype = ctypes.c_char_p
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise RuntimeError("procgen2_b200 engine error: %s" % load_library().pg2_last_error().decode())


class BatchedEnv:
    """N environments of one game on one GPU.

    env i is seeded ``seed + first_env + i`` and reproduces a reference process created with
    that seed (cenv_make -> cenv_reset -> cenv_step..., reset on terminate).

    final_obs=True (needs auto_reset): the engine also keeps the terminal frame of every env that finishes, the frame the
    reference returns from cenv_step before its caller resets it; read it with final_obs_view() or fetch_final()."""

    def __init__(self, game, num_envs, seed=0, device=0, first_env=0, max_episode_steps=0, assets_path=None, auto_reset=True,
                 distribution_mode=-1, final_obs=False):
        L = load_library()
        self.game, self.num_envs, self.device = game, int(num_envs), int(device)
        self._assets = assets_path.encode() if assets_path else None
        cfg = _Config(game.encode(), self.num_envs, int(np.int32(np.uint32(seed & 0xffffffff))), int(first_env), self.device,
                      int(max_episode_steps), self._assets, 1 if auto_reset else 0, int(distribution_mode), 1 if final_obs else 0)
        h = ctypes.c_void_p()
        _check(L.pg2_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        self._L = L
        self.final_obs = bool(final_obs)
        self._torch_views = None
        self._final_view = None

    # ---- host-buffer API (numpy) -------------------------------------------------------------
    def reset(self, seeds=None):
        p = None
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, np.int32)
            assert seeds.shape == (self.num_envs,)
            p = seeds.ctypes.data
        _check(self._L.pg2_reset(self._h, p))

    def step(self, actions):
        """actions: int32 host array of shape (num_envs,). Asynchronous."""
        a = np.ascontiguousarray(actions, np.int32)
        assert a.shape == (self.num_envs,)
        _check(self._L.pg2_step(self._h, a.ctypes.data))

    def step_device_ptr(self, ptr):
        _check(self._L.pg2_step_device(self._h, ctypes.c_void_p(ptr)))

    def fetch(self, obs=True, reward=True, terminated=True, truncated=False):
        """Blocking copy of the last results to fresh host arrays."""
        n = self.num_envs
        o = np.empty((n,) + OBS_SHAPE, np.uint8) if obs else None
        r = np.empty(n, np.float32) if reward else None
        t = np.empty(n, np.uint8) if terminated else None
        tr = np.empty(n, np.uint8) if truncated else None
        _check(self._L.pg2_fetch(self._h, *(x.ctypes.data if x is not None else None for x in (o, r, t, tr))))
        return o, r, (t.astype(bool) if t is not None else None), (tr.astype(bool) if tr is not None else None)

    def fetch_final(self):
        """Blocking copy of the terminal-frame buffer (final_obs engines): uint8 [N, 64, 64, 3]. Row e is the terminal frame
        of env e's last finished episode, written in the step it finished in (zero before any)."""
        out = np.empty((self.num_envs,) + OBS_SHAPE, np.uint8)
        _check(self._L.pg2_fetch_final(self._h, out.ctypes.data))
        return out

    def fetch_into(self, obs=None, reward=None, terminated=None, truncated=None):
        _check(self._L.pg2_fetch(self._h, *(x.ctypes.data if x is not None else None for x in (obs, reward, terminated, truncated))))

    def step_pipelined(self, actions, obs, reward, terminated, truncated=None):
        """Depth-1 pipelined step (pg2_step_pipelined): enqueue this step with its results going to the given
        (pinned) host arrays; returns when the PREVIOUS call's arrays are complete. Alternate two sets."""
        a = np.ascontiguousarray(actions, np.int32)
        assert a.shape == (self.num_envs,)
        _check(self._L.pg2_step_pipelined(self._h, a.ctypes.data, *(x.ctypes.data if x is not None else None
                                                                     for x in (obs, reward, terminated, truncated))))

    def flush(self):
        _check(self._L.pg2_pipeline_flush(self._h))

    def sync(self):
        _check(self._L.pg2_sync(self._h))

    # ---- device-resident API (torch) ---------------------------------------------------------
    def torch_views(self):
        """(obs u8 [N,64,64,3], reward f32 [N], terminated u8 [N], truncated u8 [N]) CUDA tensors
        aliasing the engine's HBM buffers (zero copy, via __cuda_array_interface__)."""
        if self._torch_views is None:
            import torch
            n = self.num_envs
            dev = torch.device("cuda", self.device)
            mk = lambda fn, shape, ts: torch.as_tensor(_Raw(fn(self._h), shape, ts), device=dev)
            self._torch_views = (mk(self._L.pg2_obs_device, (n,) + OBS_SHAPE, "|u1"), mk(self._L.pg2_reward_device, (n,), "<f4"),
                                 mk(self._L.pg2_terminated_device, (n,), "|u1"), mk(self._L.pg2_truncated_device, (n,), "|u1"))
        return self._torch_views

    def final_obs_view(self):
        """The terminal-frame buffer of a final_obs engine (uint8 [N, 64, 64, 3], what fetch_final copies) as a CUDA tensor
        aliasing the engine's HBM buffer, like torch_views(); None without final_obs."""
        if not self.final_obs:
            return None
        if self._final_view is None:
            import torch
            raw = _Raw(self._L.pg2_final_obs_device(self._h), (self.num_envs,) + OBS_SHAPE, "|u1")
            self._final_view = torch.as_tensor(raw, device=torch.device("cuda", self.device))
        return self._final_view

    def step_torch(self, actions):
        """actions: int32 CUDA tensor (num_envs,) on this engine's device."""
        assert actions.is_cuda and actions.dtype.is_floating_point is False and actions.numel() == self.num_envs
        self.step_device_ptr(actions.data_ptr())

    def profile(self, enable=True):
        """Start (and clear) / stop per-kernel CUDA-event timing of step()."""
        _check(self._L.pg2_profile(self._h, 1 if enable else 0))

    def profile_read(self):
        """-> ({"step": ms, "reset": ms, "render": ms} accumulated, steps)"""
        ms = (ctypes.c_float * 3)()
        steps = ctypes.c_int64()
        _check(self._L.pg2_profile_read(self._h, ms, ctypes.byref(steps)))
        return {"step": ms[0], "reset": ms[1], "render": ms[2]}, steps.value

    @property
    def stream_ptr(self):
        return self._L.pg2_stream(self._h)

    @property
    def step_epw(self):
        """Environments per warp in the step kernel (1: a whole warp per environment)."""
        return int(self._L.pg2_step_epw(self._h))

    @property
    def kernel_launches(self):
        return int(self._L.pg2_kernel_launches(self._h))

    @property
    def state_bytes_per_env(self):
        return int(self._L.pg2_state_bytes_per_env(self._h))

    # ---- state access (tests / checkpointing) ------------------------------------------------
    def read_field(self, name, dtype=None):
        esz, pe = ctypes.c_int32(), ctypes.c_int32()
        nbytes = self._L.pg2_read_field(self._h, name.encode(), None, 0, ctypes.byref(esz), ctypes.byref(pe))
        if nbytes < 0:
            raise KeyError(name)
        buf = np.empty(nbytes, np.uint8)
        assert self._L.pg2_read_field(self._h, name.encode(), buf.ctypes.data, nbytes, None, None) == nbytes
        if dtype is not None:
            buf = buf.view(dtype)
        return buf, esz.value, pe.value

    def write_field(self, name, array):
        a = np.ascontiguousarray(array)
        n = self._L.pg2_write_field(self._h, name.encode(), a.ctypes.data, a.nbytes)
        if n < 0:
            raise RuntimeError(self._L.pg2_last_error().decode())

    def snapshot(self):
        """Complete simulation state of the shard as bytes (pg2_snapshot): checkpoint / fork point."""
        n = self._L.pg2_snapshot(self._h, None, 0)
        buf = np.empty(n, np.uint8)
        got = self._L.pg2_snapshot(self._h, buf.ctypes.data, n)
        if got != n:
            raise RuntimeError("pg2_snapshot: %s" % self._L.pg2_last_error().decode())
        return buf

    def restore(self, blob):
        """Restore a snapshot() of an engine of the same game and size; subsequent steps replay bit for bit."""
        blob = np.ascontiguousarray(blob, np.uint8)
        got = self._L.pg2_restore(self._h, blob.ctypes.data, blob.size)
        if got != blob.size:
            raise RuntimeError("pg2_restore: %s" % self._L.pg2_last_error().decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.pg2_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

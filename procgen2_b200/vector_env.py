"""Batched front-end in the shape of `gymnasium.vector.VectorEnv`, next to the reference's single-env wrapper
(cenv/cenv.py:152-380): N environments of one game per object, observations / rewards / flags returned as CUDA tensors
that ALIAS the engine's HBM buffers (zero copy: `__cuda_array_interface__` -> torch; DLPack via `torch.utils.dlpack` /
`tensor.__dlpack__()`), actions accepted as a CUDA tensor, a numpy array or a list. It replaces the per-step numpy copies
of the reference wrapper (cenv/cenv.py:289-309: every observation buffer is copied out element by element into a dict).

Conventions (Gymnasium 1.x vector API):
  * `reset(seed=None, options=None) -> (obs, info)`, `step(actions) -> (obs, reward, terminated, truncated, info)`;
  * autoreset mode SAME_STEP: an env that terminates or is truncated is reset on device inside the same step, the
    returned observation is the first frame of the new episode (the reference's caller does the same by hand:
    "if terminated: obs = reset()", game_test.py:38-40). With `final_obs=True` the step's info also holds the frame the
    episode ended in, as Gymnasium 1.x's same-step autoreset does: `info["final_obs"]` (uint8 [num_envs, 64, 64, 3]; row
    e is valid where `info["_final_obs"][e]`, i.e. where env e terminated or was truncated in this step);
  * `seed`: int -> env i restarts its RNG stream from seed + i (cenv_reset option "seed", coinrun.cpp:313-317), or a
    sequence of num_envs ints; None continues the streams;
  * the returned tensors are views of buffers the next step overwrites: `.clone()` what must outlive a step
    (`copy=True` does it for you). Everything is enqueued on `env.stream`; `step` makes the caller's current torch stream
    wait for the results, so ordinary torch code can consume them without further synchronisation.
There is no CPU path: constructing it without the CUDA extension or without a GPU raises.
"""
import numpy as np

from .engine import BatchedEnv, OBS_SHAPE

try:  # optional: real Gymnasium spaces / base class when the package is there (it is not in the build image)
    import gymnasium as gym
    from gymnasium.vector import VectorEnv as _VectorEnvBase
except Exception:  # pragma: no cover
    gym = None

    class _VectorEnvBase:
        pass


class _Box:
    def __init__(self, low, high, shape, dtype):
        self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), np.dtype(dtype)

    def __repr__(self):
        return "Box(%s, %s, %s, %s)" % (self.low, self.high, self.shape, self.dtype)


class _Discrete:
    def __init__(self, n):
        self.n = int(n)

    def __repr__(self):
        return "Discrete(%d)" % self.n


class _MultiDiscrete:
    def __init__(self, nvec):
        self.nvec = np.asarray(nvec, np.int64)

    def __repr__(self):
        return "MultiDiscrete(%s)" % self.nvec


NUM_ACTIONS = 15   # coinrun.cpp:27, identical for the seven games


class ProcgenVectorEnv(_VectorEnvBase):
    """`num_envs` environments of `game` on CUDA device `device`, Gymnasium-VectorEnv style, tensors in HBM."""
    metadata = {"render_modes": ["rgb_array"], "autoreset_mode": "SameStep"}

    DISTRIBUTION_MODES = {None: -1, "default": -1, "easy": 0, "hard": 1, "memory": 2, "extreme": 2}

    def __init__(self, game, num_envs, seed=0, device=0, max_episode_steps=0, first_env=0, copy=False, distribution_mode=None,
                 final_obs=False):
        """distribution_mode: None (the mode the reference compiles in), "easy" / "hard" / "memory" / "extreme" or the integer
        of the reference's `Distribution_Mode` enum (games/<g>/tilemap.h); a mode the game does not have raises.
        final_obs: return the terminal observations of finished envs in the step's info (see the module docstring)."""
        import torch
        self._torch = torch
        mode = self.DISTRIBUTION_MODES.get(distribution_mode, distribution_mode) if not isinstance(distribution_mode, int) else distribution_mode
        if not isinstance(mode, int):
            raise ValueError("distribution_mode %r: expected one of %s or an integer" % (distribution_mode, sorted(k for k in self.DISTRIBUTION_MODES if k)))
        self.env = BatchedEnv(game, num_envs, seed=seed, device=device, first_env=first_env, max_episode_steps=max_episode_steps,
                              distribution_mode=mode, final_obs=final_obs)
        self.game, self.num_envs, self.copy = game, int(num_envs), bool(copy)
        self.device = torch.device("cuda", device)
        self.stream = torch.cuda.ExternalStream(self.env.stream_ptr, device=self.device)
        if gym is not None:
            self.single_observation_space = gym.spaces.Box(0, 255, OBS_SHAPE, np.uint8)
            self.single_action_space = gym.spaces.Discrete(NUM_ACTIONS)
            self.observation_space = gym.spaces.Box(0, 255, (self.num_envs,) + OBS_SHAPE, np.uint8)
            self.action_space = gym.spaces.MultiDiscrete([NUM_ACTIONS] * self.num_envs)
        else:
            self.single_observation_space = _Box(0, 255, OBS_SHAPE, np.uint8)
            self.single_action_space = _Discrete(NUM_ACTIONS)
            self.observation_space = _Box(0, 255, (self.num_envs,) + OBS_SHAPE, np.uint8)
            self.action_space = _MultiDiscrete([NUM_ACTIONS] * self.num_envs)
        self._obs, self._reward, self._terminated, self._truncated = self.env.torch_views()
        self._final_obs = self.env.final_obs_view()
        self._actions = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        self._done_event = torch.cuda.Event()

    # ---- results -----------------------------------------------------------------------------------------------
    def _publish(self):
        """The caller's current stream waits for the engine's stream; returns the (aliased or cloned) result tensors."""
        torch = self._torch
        self._done_event.record(self.stream)
        torch.cuda.current_stream(self.device).wait_event(self._done_event)
        out = (self._obs, self._reward, self._terminated.bool(), self._truncated.bool())
        return tuple(t.clone() for t in out) if self.copy else out

    def reset(self, *, seed=None, options=None):
        seeds = None
        if seed is not None:
            seeds = np.asarray(seed, np.int64)
            seeds = (seeds + np.arange(self.num_envs)) if seeds.ndim == 0 else seeds
            seeds = (seeds & 0xffffffff).astype(np.uint32).view(np.int32)
        self.env.reset(seeds)
        obs, _, _, _ = self._publish()
        return obs, {}

    def step(self, actions):
        torch = self._torch
        if not (torch.is_tensor(actions) and actions.is_cuda and actions.dtype == torch.int32 and actions.is_contiguous()):
            actions = torch.as_tensor(np.asarray(actions, np.int32) if not torch.is_tensor(actions) else actions, device=self.device).to(torch.int32).contiguous()
        assert actions.numel() == self.num_envs
        # the engine's stream must see the caller's actions: order it after the caller's current stream, and keep the
        # action buffer alive / unmodified until the step has read it by copying into the env's own staging tensor
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self.stream.wait_event(ev)
        with torch.cuda.stream(self.stream):
            self._actions.copy_(actions.view(-1), non_blocking=True)
            self.env.step_torch(self._actions)
        obs, reward, terminated, truncated = self._publish()
        info = {}
        if self._final_obs is not None:
            info = {"final_obs": self._final_obs.clone() if self.copy else self._final_obs, "_final_obs": terminated | truncated}
        return obs, reward, terminated, truncated, info

    # ---- interchange -----------------------------------------------------------------------------------------------
    def dlpack(self):
        """(obs, reward, terminated, truncated) as DLPack capsules over the engine's buffers (zero copy)."""
        from torch.utils import dlpack
        return tuple(dlpack.to_dlpack(t) for t in (self._obs, self._reward, self._terminated, self._truncated))

    @property
    def __cuda_array_interface__(self):
        """The observation buffer (uint8 [num_envs, 64, 64, 3]) for CuPy / Numba consumers."""
        return self._obs.__cuda_array_interface__

    def render(self):
        """Frame of env 0 as a host array (rgb_array)."""
        self.env.sync()
        return self._obs[0].cpu().numpy()

    def close(self, **kwargs):
        self.env.close()

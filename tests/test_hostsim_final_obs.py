"""Terminal frames of auto-reset episodes (final_obs) in the host-sim, every game and distribution mode.

(a) The terminal frame is what an env that is not reset returns: before every step, host-sim A (auto-reset, final_obs)
is transplanted into host-sim B (auto_reset = 0); then both take the same step. Every row of A's final_obs of an env that
finished in the step equals B's observation row, and rewards and flags are equal for all envs.
(b) final_obs changes nothing else: A with final_obs and A without it have identical observations, rewards, flags and
state over 300 steps."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import simlib
from tests.conftest import IMPLEMENTED
from tests.simlib import HostSim, read_state, state_diff, transplant
from tests.test_hostsim_state import NONDEFAULT_MODES

CASES = [(g, -1) for g in IMPLEMENTED] + NONDEFAULT_MODES


@pytest.fixture(scope="module", autouse=True)
def final_sim_lib(tmp_path_factory):
    """tests/hostsim/final_obs_sim.cpp (the host-sim plus the auto_reset = 0 and final_obs step variants), compiled into a
    temporary directory with the host-sim's flags and loaded as simlib's library for this module: it exports every hs_*
    entry point of the host-sim, so HostSim and transplant work on its sims unchanged."""
    from tests.hostsim import build as hb
    out = str(tmp_path_factory.mktemp("final_obs_sim") / "libpg2_hostsim_final.so")
    csrc = os.path.join(simlib.ROOT, "procgen2_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-g", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++",
                           os.path.join(hb.HERE, "final_obs_sim.cpp"), os.path.join(csrc, "assets.cpp"), "-lz", "-ldl", "-o", out])
    saved_lib, saved_build = simlib._lib, hb.build
    simlib._lib, hb.build = None, lambda force=False: out
    try:
        L = simlib.lib()
    finally:
        hb.build = saved_build
    L.hs_create_final.restype = ctypes.c_void_p
    L.hs_create_final.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p] + [ctypes.c_int] * 3
    L.hs_final_obs.restype = ctypes.POINTER(ctypes.c_uint8)
    L.hs_final_obs.argtypes = [ctypes.c_void_p]
    yield L
    simlib._lib = saved_lib


class FinalSim(HostSim):
    """A HostSim with the engine's step variants: auto_reset=False (a finished env is not reset), final_obs=True
    (final_obs() = the terminal frame of every env that finished, written in the step it finished in)."""

    def __init__(self, game, num_envs, seed, max_episode_steps=0, distribution_mode=-1, auto_reset=True, final_obs=False):
        L = simlib.lib()
        self.n = num_envs
        self.h = L.hs_create_final(game.encode(), num_envs, seed, max_episode_steps, simlib.ASSETS.encode(), distribution_mode,
                                   1 if auto_reset else 0, 1 if final_obs else 0)
        if not self.h:
            raise RuntimeError(L.hs_last_error().decode())

    def final_obs(self):
        return np.ctypeslib.as_array(simlib.lib().hs_final_obs(self.h), shape=(self.n, 64, 64, 3)).copy()


def _actions(game, rs, n):
    if game == "bossfight":   # fire most of the time: boss fights end in both ways
        return np.where(rs.rand(n) < 0.8, 9, rs.randint(0, 9, n)).astype(np.int32)
    return rs.randint(0, 15, n).astype(np.int32)


@pytest.mark.parametrize("game,mode", CASES)
def test_final_obs_is_the_frame_of_an_env_that_is_not_reset(game, mode):
    n, T, max_ep = 8, 160, 40
    rs = np.random.RandomState(11)
    a = FinalSim(game, n, 31, max_episode_steps=max_ep, distribution_mode=mode, final_obs=True)
    b = FinalSim(game, n, 32, max_episode_steps=max_ep, distribution_mode=mode, auto_reset=False)
    a.reset()
    b.reset()
    finished = terminations = 0
    for t in range(T):
        transplant(a, b)   # b draws from scratch, a from its cached base images where it has them
        acts = _actions(game, rs, n)
        _, ra, da = a.step(acts)
        ob, rb, db = b.step(acts)
        tra, trb = a.truncated(), b.truncated()
        np.testing.assert_array_equal(ra.view(np.uint32), rb.view(np.uint32), err_msg="reward, step %d" % t)
        np.testing.assert_array_equal(da, db, err_msg="terminated, step %d" % t)
        np.testing.assert_array_equal(tra, trb, err_msg="truncated, step %d" % t)
        done = da | tra
        fa = a.final_obs()
        for e in np.flatnonzero(done):
            assert np.array_equal(fa[e], ob[e]), "%s mode %d, step %d, env %d: final_obs differs from the frame of the env that was not reset" % (game, mode, t, e)
        finished += int(done.sum())
        terminations += int(da.sum())
    assert finished >= n, "too few episodes ended (%d)" % finished
    assert finished > terminations, "no truncation among the finished episodes"
    a.close()
    b.close()


@pytest.mark.parametrize("game,mode", CASES)
def test_final_obs_changes_nothing_else(game, mode):
    n, T, max_ep = 8, 300, 50
    rs = np.random.RandomState(5)
    on = FinalSim(game, n, 77, max_episode_steps=max_ep, distribution_mode=mode, final_obs=True)
    off = FinalSim(game, n, 77, max_episode_steps=max_ep, distribution_mode=mode)
    fields = on.field_list()
    assert np.array_equal(on.reset(), off.reset())
    assert not on.final_obs().any(), "reset wrote final_obs"
    seen = np.zeros(n, bool)
    for t in range(T):
        acts = _actions(game, rs, n)
        before = on.final_obs()
        oa, ra, da = on.step(acts)
        ob, rb, db = off.step(acts)
        np.testing.assert_array_equal(oa, ob, err_msg="obs, step %d" % t)
        np.testing.assert_array_equal(ra.view(np.uint32), rb.view(np.uint32), err_msg="reward, step %d" % t)
        np.testing.assert_array_equal(da, db, err_msg="terminated, step %d" % t)
        done = da | on.truncated()
        np.testing.assert_array_equal(on.truncated(), off.truncated(), err_msg="truncated, step %d" % t)
        after = on.final_obs()
        assert np.array_equal(after[~done], before[~done]), "step %d: rows of envs that did not finish were written" % t
        seen |= done
    diff = state_diff(read_state(off, fields), read_state(on, fields), fields, n)
    assert not diff, "%s mode %d:\n%s" % (game, mode, diff)
    assert seen.all(), "not every env finished an episode"
    on.close()
    off.close()


def test_final_obs_needs_auto_reset():
    with pytest.raises(RuntimeError, match="auto_reset"):
        FinalSim("maze", 2, 1, final_obs=True, auto_reset=False)

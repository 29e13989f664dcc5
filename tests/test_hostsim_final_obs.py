"""Terminal frames of auto-reset episodes (final_obs) in the host-sim, every game and distribution mode.

(a) The terminal frame is what an env that is not reset returns: before every step, host-sim A (auto-reset, final_obs)
is transplanted into host-sim B (auto_reset = 0); then both take the same step. Every row of A's final_obs of an env that
finished in the step equals B's observation row, and rewards and flags are equal for all envs.
(b) final_obs changes nothing else: A with final_obs and A without it have identical observations, rewards, flags and
state over 300 steps."""
import numpy as np
import pytest

from tests.conftest import IMPLEMENTED
from tests.simlib import HostSim, read_state, state_diff, transplant
from tests.test_hostsim_state import NONDEFAULT_MODES

CASES = [(g, -1) for g in IMPLEMENTED] + NONDEFAULT_MODES


def _actions(game, rs, n):
    if game == "bossfight":   # fire most of the time: boss fights end in both ways
        return np.where(rs.rand(n) < 0.8, 9, rs.randint(0, 9, n)).astype(np.int32)
    return rs.randint(0, 15, n).astype(np.int32)


@pytest.mark.parametrize("game,mode", CASES)
def test_final_obs_is_the_frame_of_an_env_that_is_not_reset(game, mode):
    n, T, max_ep = 8, 160, 40
    rs = np.random.RandomState(11)
    a = HostSim(game, n, 31, max_episode_steps=max_ep, distribution_mode=mode, final_obs=True)
    b = HostSim(game, n, 32, max_episode_steps=max_ep, distribution_mode=mode, auto_reset=False)
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
    on = HostSim(game, n, 77, max_episode_steps=max_ep, distribution_mode=mode, final_obs=True)
    off = HostSim(game, n, 77, max_episode_steps=max_ep, distribution_mode=mode)
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
        HostSim("maze", 2, 1, final_obs=True, auto_reset=False)

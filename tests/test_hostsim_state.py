"""The host-sim's field list is the whole state: a host-sim whose every field was overwritten with another one's
(transplant) steps exactly like that one, field for field, frame for frame. The GPU state-parity test
(test_gpu_state_parity.py) transplants the engine's state into a host-sim the same way, so a field missing from the list
would show up there as an engine bug; this test rules that out on the CPU."""
import numpy as np
import pytest

from tests.conftest import IMPLEMENTED
from tests.simlib import HostSim, read_state, state_diff, transplant

# every distribution mode other than a game's default that is built
NONDEFAULT_MODES = [("maze", 0), ("maze", 2), ("chaser", 1), ("chaser", 2), ("jumper", 0), ("jumper", 2), ("caveflyer", 0),
                    ("caveflyer", 2), ("bossfight", 0), ("coinrun", 0), ("climber", 0)]


@pytest.mark.parametrize("game,mode", [(g, -1) for g in IMPLEMENTED] + NONDEFAULT_MODES)
def test_transplant_carries_the_whole_state(game, mode):
    n, warm, T, max_ep = 8, 120, 80, 150
    rs = np.random.RandomState(3)
    acts = rs.randint(0, 15, size=(warm + T, n)).astype(np.int32)
    a = HostSim(game, n, 101, max_episode_steps=max_ep, distribution_mode=mode)
    b = HostSim(game, n, 202, max_episode_steps=max_ep, distribution_mode=mode)
    a.reset()
    b.reset()
    # two unrelated mid-episode states (bullets, explosions, particles, timers, used view caches, episode lengths):
    # a field the transplant missed keeps b's value, which then differs from a's
    for t in range(warm):
        a.step(acts[t])
        if t % 2:
            b.step(acts[t][::-1].copy())
    fields = a.field_list()
    assert fields == b.field_list()
    names = [f[0] for f in fields]
    assert len(set(names)) == len(names)
    assert {"mt", "mti", "ep_steps", "view_valid", "cam_x", "fault"} <= set(names)
    a.invalidate_views()   # both draw their next frame from scratch; after that each keeps its own cache
    # every byte of b differs from a before the transplant and equals it after
    want = read_state(a, fields)
    for name in names:
        b.write_field(name, ~want[name])
    transplant(a, b)
    diff = state_diff(want, read_state(b, fields), fields, n)
    assert not diff, "the transplant left fields out:\n" + diff
    # b's history (seed, actions, steps) was a different one: state outside the field list would diverge now
    resets = 0
    for t in range(warm, warm + T):
        oa, ra, da = a.step(acts[t])
        ob, rb, db = b.step(acts[t])
        diff = state_diff(read_state(a, fields), read_state(b, fields), fields, n)
        assert not diff, "%s mode %d, step %d:\n%s" % (game, mode, t, diff)
        np.testing.assert_array_equal(oa, ob, err_msg="pixels, step %d" % t)
        np.testing.assert_array_equal(ra.view(np.uint32), rb.view(np.uint32), err_msg="reward, step %d" % t)
        np.testing.assert_array_equal(da, db, err_msg="terminated, step %d" % t)
        np.testing.assert_array_equal(a.truncated(), b.truncated(), err_msg="truncated, step %d" % t)
        resets += int(np.sum(da | a.truncated()))
    assert resets >= n // 2, "too few episodes ended to cover level generation after the transplant"
    a.close()
    b.close()


def test_write_field_rejects_bad_input():
    s = HostSim("maze", 4, 1)
    with pytest.raises(KeyError):
        s.write_field("no_such_field", np.zeros(4, np.int32))
    with pytest.raises(ValueError):
        s.write_field("mti", np.zeros(3, np.int32))
    s.write_field("mti", np.arange(4, dtype=np.int32))
    np.testing.assert_array_equal(s.field("mti")[0].view(np.int32), np.arange(4))
    s.close()

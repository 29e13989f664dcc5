"""Terminal frames of auto-reset episodes (pg2_config::final_obs) on the GPU, on every schedule of the step.

1. Oracle: engine A (final_obs) against engine B (auto_reset = 0, the pinned reference behaviour) of the same shape. Before
   each checked step A's whole state is copied into B; both take the same step. For every env A reports finished, A's
   final_obs row equals B's observation row; rewards and flags are equal for all envs.
2. Truncation identity at scale, without any state copy: A (max_episode_steps = T) against C (no truncation) from the same
   seeds and actions. Every env whose first episode was cut at step T has A's final_obs row = C's observation at step T.
3. Nothing else moves: final_obs on against off, obs / reward / flags at every step and every state field at the end;
   the kernel launches per step (+1 on the inline-reset and overlap schedules, +0 with level prefetch).
4. Snapshot / restore and pipelined stepping carry the final frames.
5. The front-ends: the cenv option "final_observation" and ProcgenVectorEnv(final_obs=True)."""
import ctypes
import os
import shutil

import numpy as np
import pytest

from tests.simlib import HostSim, read_state, state_diff
from tests.test_hostsim_state import NONDEFAULT_MODES

pytestmark = pytest.mark.gpu

def _engine(monkeypatch, game, n, seed, max_ep=0, mode=-1, prefetch=None, graph=None, **kw):
    from procgen2_b200.engine import BatchedEnv
    for var, val in (("PG2_PREFETCH", prefetch), ("PG2_GRAPH", graph)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))
    env = BatchedEnv(game, n, seed=seed, max_episode_steps=max_ep, distribution_mode=mode, **kw)
    monkeypatch.delenv("PG2_PREFETCH", raising=False)
    monkeypatch.delenv("PG2_GRAPH", raising=False)
    return env


def _fields(game, mode):
    s = HostSim(game, 1, 1, distribution_mode=mode)
    f = s.field_list()
    s.close()
    return f


def _actions(game, rs, n):
    if game == "bossfight":   # fire most of the time: the agent dies sooner
        return np.where(rs.rand(n) < 0.8, 9, rs.randint(0, 9, n)).astype(np.int32)
    return rs.randint(0, 15, n).astype(np.int32)


def _no_fault(env):
    fault = env.read_field("fault")[0]
    assert not fault.any(), "fault flags set in %d envs" % np.count_nonzero(fault)


# (game, N, mode, max_episode_steps, PG2_PREFETCH, PG2_GRAPH, warm-up steps, checked steps, terminations expected)
ORACLE = [
    ("bossfight", 16384, -1, 40, None, None, 30, 16, True),       # inline reset
    ("chaser", 4096, -1, 40, None, None, 30, 16, False),          # overlap (no termination within the window)
    ("coinrun", 4096, -1, 40, 1, None, 30, 16, True),             # level prefetch
    ("coinrun", 4096, -1, 32, None, None, 24, 16, False),         # inline (short episodes; no termination within the window)
    ("maze", 256, -1, 40, None, None, 30, 16, False),
    ("maze", 256, -1, 40, 0, None, 30, 16, False),
    ("maze", 32768, -1, 40, None, None, 34, 8, True),
    ("maze", 32768, -1, 40, 0, None, 34, 8, True),
    ("climber", 4096, -1, 40, None, None, 30, 16, True),
    ("climber", 4096, -1, 40, 0, None, 30, 16, True),
    ("caveflyer", 4096, -1, 40, None, None, 30, 16, True),
    ("caveflyer", 4096, -1, 40, 0, None, 30, 16, True),
    ("jumper", 4096, -1, 40, None, None, 30, 16, True),
    ("jumper", 4096, -1, 40, 0, None, 30, 16, True),
    ("coinrun", 512, -1, 1, None, None, 0, 4, False),             # every env finishes every step
    ("maze", 512, -1, 1, 1, None, 0, 4, False),                   # ... with level prefetch forced on
    ("bossfight", 512, -1, 1, None, None, 0, 4, False),
    ("chaser", 512, -1, 1, None, None, 0, 4, False),
    ("coinrun", 4096, -1, 32, None, 0, 24, 16, False),            # eager launches
    ("jumper", 4096, -1, 40, None, 0, 30, 16, True),
] + [(g, 64, m, 30, None, None, 22, 16, False) for g, m in NONDEFAULT_MODES]


@pytest.mark.parametrize("game,n,mode,max_ep,prefetch,graph,warm,T,terminations", ORACLE)
def test_final_obs_equals_the_frame_without_auto_reset(monkeypatch, game, n, mode, max_ep, prefetch, graph, warm, T, terminations):
    rs = np.random.RandomState(7)
    a = _engine(monkeypatch, game, n, 1000, max_ep, mode, prefetch, graph, final_obs=True)
    b = _engine(monkeypatch, game, n, 2000, max_ep, mode, prefetch, graph, auto_reset=False)
    fields = _fields(game, mode)
    a.reset()
    for _ in range(warm):
        a.step(_actions(game, rs, n))
    checked = np.zeros(2, np.int64)   # finished envs checked: terminated, truncated
    for t in range(T):
        for name, _, _, _ in fields:
            b.write_field(name, a.read_field(name)[0])
        acts = _actions(game, rs, n)
        a.step(acts)
        b.step(acts)
        _, ra, da, tra = a.fetch(obs=False, truncated=True)
        ob, rb, db, trb = b.fetch(truncated=True)
        fa = a.fetch_final()
        np.testing.assert_array_equal(ra.view(np.uint32), rb.view(np.uint32), err_msg="reward, step %d" % t)
        np.testing.assert_array_equal(da, db, err_msg="terminated, step %d" % t)
        np.testing.assert_array_equal(tra, trb, err_msg="truncated, step %d" % t)
        done = np.flatnonzero(da | tra)
        bad = [e for e in done if not np.array_equal(fa[e], ob[e])]
        assert not bad, "checked step %d: final_obs differs from the auto_reset = 0 frame in %d of %d finished envs, first env %d" % (
            t, len(bad), done.size, bad[0])
        checked += [int(da.sum()), int((tra & ~da).sum())]
    assert checked.sum() >= min(n, 64) * 3 // 4, "only %d finished envs checked" % checked.sum()
    assert checked[1] > 0, "no truncation among the checked envs"
    if terminations:
        assert checked[0] > 0, "no termination among the checked envs"
    _no_fault(a)
    _no_fault(b)
    a.close()
    b.close()


@pytest.mark.parametrize("game", ["bossfight", "caveflyer", "chaser", "climber", "coinrun", "jumper", "maze"])
def test_truncated_episode_frame_at_scale(monkeypatch, game):
    n, T = 4096, 60
    rs = np.random.RandomState(3)
    a = _engine(monkeypatch, game, n, 555, T, final_obs=True)
    c = _engine(monkeypatch, game, n, 555, 0)
    a.reset()
    c.reset()
    ended = np.zeros(n, bool)
    for t in range(T):
        acts = _actions(game, rs, n)
        a.step(acts)
        c.step(acts)
        _, _, da, tra = a.fetch(obs=False, reward=False, truncated=True)
        if t < T - 1:
            assert not tra.any()
            ended |= da
    cut = tra & ~ended
    assert cut.sum() >= n // 4, "only %d first episodes were cut at step %d" % (cut.sum(), T)
    fa = a.fetch_final()
    oc = c.fetch()[0]
    bad = np.flatnonzero([not np.array_equal(fa[e], oc[e]) for e in np.flatnonzero(cut)])
    assert bad.size == 0, "%d of %d truncated envs differ" % (bad.size, cut.sum())
    _no_fault(a)
    a.close()
    c.close()


# (game, N, max_episode_steps, PG2_PREFETCH, PG2_GRAPH, launches per step without final_obs, added with it)
SCHEDULES = [
    ("bossfight", 16384, 0, None, None, 3, 1),   # inline reset
    ("chaser", 4096, 0, None, None, 4, 1),       # overlap
    ("coinrun", 4096, 0, None, None, 3, 0),      # level prefetch: k_step, render, generator
    ("coinrun", 4096, 32, None, None, 3, 1),     # inline reset
    ("maze", 256, 0, None, None, 3, 0),
    ("maze", 256, 0, 0, None, 4, 1),             # overlap (maze and jumper generate slowly)
    ("jumper", 4096, 0, None, None, 3, 0),
    ("jumper", 4096, 0, 0, 0, 4, 1),             # overlap, eager
]


@pytest.mark.parametrize("game,n,max_ep,prefetch,graph,per_step,added", SCHEDULES)
def test_final_obs_changes_nothing_else(monkeypatch, game, n, max_ep, prefetch, graph, per_step, added):
    import torch
    T = 300
    rs = np.random.RandomState(9)
    on = _engine(monkeypatch, game, n, 42, max_ep, -1, prefetch, graph, final_obs=True)
    off = _engine(monkeypatch, game, n, 42, max_ep, -1, prefetch, graph)
    on.reset()
    off.reset()
    assert not on.fetch_final().any(), "reset wrote final_obs"
    von, voff = on.torch_views(), off.torch_views()
    fin = on.final_obs_view()
    l_on, l_off = on.kernel_launches, off.kernel_launches
    finished = 0
    for t in range(T):
        acts = _actions(game, rs, n)
        before = fin.clone() if t % 50 == 0 else None
        on.step(acts)
        off.step(acts)
        on.sync()
        off.sync()
        for x, y, what in zip(von, voff, ("obs", "reward", "terminated", "truncated")):
            assert torch.equal(x, y), "%s differs at step %d" % (what, t)
        done = (von[2] | von[3]).bool()
        finished += int(done.sum())
        if before is not None:   # rows of envs that did not finish were not written
            assert torch.equal(fin[~done], before[~done]), "step %d" % t
    assert finished > 0
    assert off.kernel_launches - l_off == per_step * T
    assert on.kernel_launches - l_on == (per_step + added) * T
    fields = _fields(game, -1)
    diff = state_diff(read_state(off, fields), read_state(on, fields), fields, n)
    assert not diff, diff
    _no_fault(on)
    on.close()
    off.close()


def test_snapshot_restore_and_pipelining(monkeypatch):
    game, n, max_ep, T = "maze", 256, 12, 20
    rs = np.random.RandomState(4)
    acts = [_actions(game, rs, n) for _ in range(T)]
    e = _engine(monkeypatch, game, n, 8, max_ep, final_obs=True)
    e.reset()
    for t in range(5):
        e.step(acts[t])
    blob = e.snapshot()

    def run():
        out = []
        for t in range(T):
            e.step(acts[t])
            out.append((e.fetch(obs=False, truncated=True), e.fetch_final()))
        return out

    first = run()
    e.restore(blob)
    second = run()
    for t, ((fa, xa), (fb, xb)) in enumerate(zip(first, second)):
        assert np.array_equal(xa, xb), "final frames after restore, step %d" % t
        for u, v in zip(fa[1:], fb[1:]):
            assert np.array_equal(u, v), "step %d" % t
    assert sum(int((f[2] | f[3]).sum()) for f, _ in first) > n
    off = _engine(monkeypatch, game, n, 8, max_ep)
    with pytest.raises(RuntimeError, match="does not belong"):
        off.restore(blob)
    with pytest.raises(RuntimeError, match="does not belong"):
        e.restore(off.snapshot())
    off.close()
    # depth-1 pipelined stepping: the final rows of each step equal those of pg2_step
    p = _engine(monkeypatch, game, n, 8, max_ep, final_obs=True)
    q = _engine(monkeypatch, game, n, 8, max_ep, final_obs=True)
    p.reset()
    q.reset()
    bufs = [(np.empty((n, 64, 64, 3), np.uint8), np.empty(n, np.float32), np.empty(n, np.uint8), np.empty(n, np.uint8)) for _ in range(2)]
    checked = 0
    for t in range(T):
        p.step_pipelined(acts[t], *bufs[t % 2])
        p.sync()
        _, _, dp, tp = p.fetch(obs=False, reward=False, truncated=True)
        fp = p.fetch_final()
        q.step(acts[t])
        _, _, dq, tq = q.fetch(obs=False, reward=False, truncated=True)
        fq = q.fetch_final()
        assert np.array_equal(dp, dq) and np.array_equal(tp, tq)
        done = dq | tq
        assert np.array_equal(fp[done], fq[done]), "pipelined step %d" % t
        checked += int(done.sum())
    p.flush()
    assert checked > n
    for x in (e, p, q):
        _no_fault(x)
        x.close()


def test_create_rejects_final_obs_without_auto_reset(monkeypatch):
    from procgen2_b200.engine import BatchedEnv
    with pytest.raises(RuntimeError, match="final_obs needs auto_reset"):
        BatchedEnv("maze", 4, auto_reset=False, final_obs=True)
    from procgen2_b200.vector_env import ProcgenVectorEnv
    v = ProcgenVectorEnv("maze", 4)
    assert v.env.final_obs_view() is None
    with pytest.raises(RuntimeError):
        v.env.fetch_final()
    v.close()


def _ptr(info, key, shard=0):
    lo, hi = (int(x) & 0xffffffff for x in info[key][2 * shard:2 * shard + 2])
    return lo | hi << 32


def _cenv(game, suffix, options):
    """One batch per loaded library (all cenv state is global): every CEnv gets a copy of the game's library."""
    from procgen2_b200.build import game_lib_path
    from procgen2_b200.cenv import CEnv
    path = os.path.join(os.path.dirname(game_lib_path(game)), "lib_final_obs_test_%s.so" % suffix)
    shutil.copyfile(game_lib_path(game), path)
    try:
        env = CEnv(path, options=options)
    finally:
        os.unlink(path)
    env.lib.cenv_device_buffer.restype = ctypes.c_void_p
    env.lib.cenv_device_buffer.argtypes = [ctypes.c_char_p, ctypes.c_int32]
    return env


def test_cenv_final_observation(monkeypatch):
    import torch
    from procgen2_b200.engine import _Raw
    game, n, seed, T, max_ep = "coinrun", 48, 91, 40, 15
    opts = {"seed": seed, "num_envs": n, "max_episode_steps": max_ep}
    host = _cenv(game, "host", dict(opts, final_observation=1))
    dev = _cenv(game, "dev", dict(opts, final_observation=1, host_copy=0))
    plain = _cenv(game, "plain", opts)
    ref = _engine(monkeypatch, game, n, seed, max_ep, final_obs=True)
    with pytest.raises(Exception):
        _cenv(game, "bad", dict(opts, final_observation=1, auto_reset=0))
    for e in (host, dev, plain):
        e.reset()
    ref.reset()
    rs = np.random.RandomState(1)
    checked = 0
    for t in range(T):
        acts = rs.randint(0, 15, n).astype(np.int32)
        _, _, _, _, ih = host.step(acts)
        _, _, _, _, idv = dev.step(acts)
        _, _, _, _, ip = plain.step(acts)
        ref.step(acts)
        _, _, d, tr = ref.fetch(obs=False, reward=False, truncated=True)
        fin = ref.fetch_final()
        done = d | tr
        assert set(ip) == {"reward", "terminated", "truncated", "screen_device", "reward_device", "terminated_device",
                           "truncated_device", "stream"}
        assert set(ih) == set(ip) | {"final_screen_device", "final_screen"}
        assert set(idv) == set(ip) | {"final_screen_device"}
        np.testing.assert_array_equal(ih["terminated"].astype(bool), d)
        np.testing.assert_array_equal(ih["truncated"].astype(bool), tr)
        got = ih["final_screen"].reshape(n, 64, 64, 3)
        assert np.array_equal(got[done], fin[done]), "host final_screen, step %d" % t
        for env, info in ((host, ih), (dev, idv)):
            p = _ptr(info, "final_screen_device")
            assert p == env.lib.cenv_device_buffer(b"final_screen", 0) != 0
            t_dev = torch.as_tensor(_Raw(p, (n, 64, 64, 3), "|u1"), device=torch.device("cuda", 0)).cpu().numpy()
            assert np.array_equal(t_dev[done], fin[done]), "device final_screen, step %d" % t
        checked += int(done.sum())
    assert checked >= n
    for e in (host, dev, plain):
        e.close()
    _no_fault(ref)
    ref.close()


@pytest.mark.parametrize("copy", [False, True])
def test_vector_env_final_obs(copy):
    import torch
    from procgen2_b200.vector_env import ProcgenVectorEnv
    n, T = 64, 40
    v = ProcgenVectorEnv("coinrun", n, seed=5, max_episode_steps=12, final_obs=True, copy=copy)
    w = ProcgenVectorEnv("coinrun", n, seed=5, max_episode_steps=12)
    ref = ProcgenVectorEnv("coinrun", n, seed=5, max_episode_steps=12, final_obs=True)
    v.reset()
    w.reset()
    ref.reset()
    rs = np.random.RandomState(2)
    seen = 0
    for t in range(T):
        acts = rs.randint(0, 15, n).astype(np.int32)
        obs, rew, term, trunc, info = v.step(acts)
        o2, r2, t2, tr2, info2 = w.step(acts)
        ref.step(acts)
        assert info2 == {}
        assert set(info) == {"final_obs", "_final_obs"}
        assert info["final_obs"].shape == (n, 64, 64, 3) and info["final_obs"].dtype == torch.uint8 and info["final_obs"].is_cuda
        assert info["_final_obs"].dtype == torch.bool and torch.equal(info["_final_obs"], term | trunc)
        assert (info["final_obs"].data_ptr() == v.env.final_obs_view().data_ptr()) != copy
        torch.cuda.synchronize()
        want = ref.env.fetch_final()
        mask = info["_final_obs"].cpu().numpy()
        assert np.array_equal(info["final_obs"].cpu().numpy()[mask], want[mask]), "step %d" % t
        assert torch.equal(obs, o2) and torch.equal(rew, r2) and torch.equal(term, t2) and torch.equal(trunc, tr2)
        seen += int(mask.sum())
    assert seen >= n
    for x in (v, w, ref):
        x.close()

"""GPU parity tests of the paths the first-round suite never drove against the oracle (pytest -m gpu on a B200, all
against the LIVE reference oracle/_ref, bit-exact):

  (a) the packed-warp k_step mapping (PG2_STEP_EPW = 2 / 4 / 32 environments per warp), which the engine selects by
      itself from 16 384 envs on for the thread-per-env games — incl. the real BASELINE configs[2] shape, bossfight at
      16 384 envs, checked on sampled envs;
  (b) max_episode_steps truncation (BASELINE configs[4]: short episodes), dozens of episodes per env: the oracle is
      driven as "step; every k steps: reset()" — hammers the persisted ECS bucket counts (Q25), the camera surviving
      reset (Q10) and level generation on a continuing MT19937 stream;
  (c) maze's 500-step timeout (maze.cpp:308-310), how BASELINE configs[0] episodes end;
  (d) GPU level generation over >= 512 seeds x 4 consecutive resets: full tile map + all 624 MT19937 words + position.
"""
import numpy as np
import pytest

from tests.conftest import IMPLEMENTED

pytestmark = pytest.mark.gpu

THREAD_PER_ENV_GAMES = ["maze", "bossfight", "caveflyer", "jumper"]   # G::LANE_AWARE == false: step_epw > 1 exists


def _mixed_actions(rs, T, n):
    return np.where(rs.rand(T, n) < 0.5, rs.randint(0, 15, size=(T, n)), rs.choice([6, 7, 8, 8, 5], size=(T, n))).astype(np.int32)


def _assert_no_fault(env):
    f = env.read_field("fault")[0].view(np.int32)
    assert not f.any(), "latent-UB / overflow flags set for envs %s" % np.nonzero(f)[0][:8]


def _check_state(env, refs, idx=None, tag=""):
    """Full MT19937 state + position + tile map of the engine's envs `idx` against the reference processes."""
    n = env.num_envs
    mt = env.read_field("mt")[0].view(np.uint32).reshape(n, 624)
    mti = env.read_field("mti")[0].view(np.int32)
    try:
        tb, _, pe = env.read_field("tiles")
        tiles = tb.reshape(n, pe)
    except KeyError:
        tiles = None
    for k, r in enumerate(refs):
        i = k if idx is None else int(idx[k])
        st, pos = r.rng_state()
        assert pos == mti[i], "%s MT19937 position, env %d" % (tag, i)
        np.testing.assert_array_equal(st, mt[i], err_msg="%s MT19937 words, env %d" % (tag, i))
        rt = r.tiles()
        if tiles is not None and rt.size:
            w, h = rt.shape
            np.testing.assert_array_equal((tiles[i, :w * h] & 15).reshape(w, h), rt, err_msg="%s tile map, env %d" % (tag, i))


# ---- (a) packed-warp step mapping ---------------------------------------------------------------------------------

@pytest.mark.parametrize("epw", [2, 4, 32])
@pytest.mark.parametrize("game", THREAD_PER_ENV_GAMES)
def test_step_epw_live_oracle(game, epw, reference, monkeypatch):
    from procgen2_b200.engine import BatchedEnv
    from tests.parity_util import check_against_oracle
    from tests.test_gpu_parity import EngineAdapter
    n, T, seed = 96, 400, 1300 + epw
    acts = _mixed_actions(np.random.RandomState(40 + epw), T, n)
    monkeypatch.setenv("PG2_STEP_EPW", str(epw))
    a = EngineAdapter(game, n, seed)
    monkeypatch.delenv("PG2_STEP_EPW")
    assert a.env.step_epw == epw
    refs = [reference.RefEnv(game, seed + i) for i in range(n)]
    episodes = check_against_oracle(a, refs, acts, tag="%s epw=%d" % (game, epw))
    _check_state(a.env, refs, tag=game)
    _assert_no_fault(a.env)
    assert episodes > 0 or game in ("maze", "jumper")
    for r in refs:
        r.close()
    a.env.close()


def test_bossfight_16384_sampled_oracle(reference):
    """BASELINE configs[2] as the engine runs it (16 384 envs, warp-per-env step with the bullet rings on the lanes):
    64 sampled envs, 50 steps, against reference processes with the same seeds."""
    from procgen2_b200.engine import BatchedEnv
    n, T, seed = 16384, 50, 7
    rs = np.random.RandomState(8)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    env = BatchedEnv("bossfight", n, seed=seed)
    assert env.step_epw == 1      # lane-aware since round 2: a whole warp per environment, bullets on the lanes
    idx = np.sort(rs.choice(n, 64, replace=False))
    idx[:4] = [0, 1, n - 2, n - 1]
    idx = np.unique(idx)
    refs = [reference.RefEnv("bossfight", seed + int(i)) for i in idx]
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0][idx], np.stack([r.reset() for r in refs]))
    for t in range(T):
        env.step(acts[t])
        o, r, d, _ = env.fetch()
        ro, rr, rd = [], [], []
        for k, e in enumerate(refs):
            oo, w, dd = e.step(acts[t, idx[k]])
            if dd:
                oo = e.reset()
            ro.append(oo); rr.append(w); rd.append(dd)
        np.testing.assert_array_equal(r[idx], np.array(rr, np.float32), err_msg="reward, step %d" % t)
        np.testing.assert_array_equal(d[idx], np.array(rd), err_msg="terminated, step %d" % t)
        np.testing.assert_array_equal(o[idx], np.stack(ro), err_msg="pixels, step %d" % t)
    _check_state(env, refs, idx, tag="bossfight@16384")
    _assert_no_fault(env)
    for r in refs:
        r.close()
    env.close()


# ---- (b) truncation = BASELINE configs[4] ------------------------------------------------------------------------------

@pytest.mark.parametrize("max_ep", [1, 3, 8, 32])
@pytest.mark.parametrize("game", IMPLEMENTED)
def test_truncation_live_oracle(game, max_ep, reference):
    from procgen2_b200.engine import BatchedEnv
    n, seed = 32, 2100 + max_ep
    T = max(24, 21 * max_ep)     # >= 21 episodes per env
    acts = _mixed_actions(np.random.RandomState(60 + max_ep), T, n)
    env = BatchedEnv(game, n, seed=seed, max_episode_steps=max_ep)
    refs = [reference.RefEnv(game, seed + i) for i in range(n)]
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0], np.stack([r.reset() for r in refs]), err_msg="reset frame")
    age = np.zeros(n, np.int64)
    episodes = 0
    for t in range(T):
        env.step(acts[t])
        o, rw, d, tr = env.fetch(truncated=True)
        ro, rr, rd, rt = [], [], [], []
        for i, e in enumerate(refs):
            oo, w, dd = e.step(acts[t, i])
            age[i] += 1
            trunc = (not dd) and age[i] >= max_ep
            if dd or trunc:
                oo = e.reset()
                age[i] = 0
                episodes += 1
            ro.append(oo); rr.append(w); rd.append(dd); rt.append(trunc)
        np.testing.assert_array_equal(rw, np.array(rr, np.float32), err_msg="reward, step %d" % t)
        np.testing.assert_array_equal(d, np.array(rd), err_msg="terminated, step %d" % t)
        np.testing.assert_array_equal(tr, np.array(rt), err_msg="truncated, step %d" % t)
        np.testing.assert_array_equal(o, np.stack(ro), err_msg="pixels, step %d" % t)
        if t % 16 == 15 or t == T - 1:
            _check_state(env, refs, tag="%s step %d" % (game, t))
    assert episodes >= 20 * n
    _assert_no_fault(env)
    for r in refs:
        r.close()
    env.close()


# ---- (c) maze timeout -----------------------------------------------------------------------------------------------------

def test_maze_timeout_live_oracle(reference):
    from tests.parity_util import check_against_oracle
    from tests.test_gpu_parity import EngineAdapter
    n, T, seed = 48, 520, 3100
    rs = np.random.RandomState(70)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    acts[:, : n // 2] = 4          # half of the envs never move: their episodes can only end by the 500-step timeout
    a = EngineAdapter("maze", n, seed)
    refs = [reference.RefEnv("maze", seed + i) for i in range(n)]
    episodes = check_against_oracle(a, refs, acts, tag="maze timeout")
    assert episodes >= n // 2
    _check_state(a.env, refs, tag="maze timeout")
    _assert_no_fault(a.env)
    for r in refs:
        r.close()
    a.env.close()


# ---- (d) level generation, many seeds ---------------------------------------------------------------------------------------

OTHER_MODES = [("maze", 0), ("maze", 2), ("chaser", 1), ("chaser", 2), ("jumper", 0), ("jumper", 2), ("caveflyer", 0), ("caveflyer", 2)]


@pytest.mark.parametrize("game,mode", [(g, None) for g in IMPLEMENTED] + OTHER_MODES)
def test_gpu_level_generation_many_seeds(game, mode, reference):
    """The warp-parallel generators (ordered BFS with atomicMin claims, unordered_set regrouping, bit-row automaton) exist
    only in the GPU build: 512 seeds x (make + 4 resets), tile map + complete RNG state + the reset frame every time
    (128 seeds for the distribution modes that have their own world size)."""
    from procgen2_b200.engine import BatchedEnv
    n, seed, chunk = (512 if mode is None else 128), 52000, 128
    env = BatchedEnv(game, n, seed=seed, distribution_mode=-1 if mode is None else mode)
    frames = []
    fields = []
    for rnd in range(5):
        mt = env.read_field("mt")[0].view(np.uint32).reshape(n, 624).copy()
        mti = env.read_field("mti")[0].view(np.int32).copy()
        try:
            tb, _, pe = env.read_field("tiles")
            tiles = tb.reshape(n, pe).copy()
        except KeyError:
            tiles = None
        fields.append((mt, mti, tiles))
        if rnd < 4:
            env.reset()
            frames.append(env.fetch()[0])
    _assert_no_fault(env)
    env.close()
    for c0 in range(0, n, chunk):
        refs = [reference.RefEnv(game, seed + i, mode=mode) for i in range(c0, min(n, c0 + chunk))]
        for rnd in range(5):
            mt, mti, tiles = fields[rnd]
            for k, r in enumerate(refs):
                i = c0 + k
                st, pos = r.rng_state()
                assert pos == mti[i], (game, rnd, i)
                np.testing.assert_array_equal(st, mt[i], err_msg="%s MT19937 words, level %d, seed %d" % (game, rnd, seed + i))
                rt = r.tiles()
                if tiles is not None and rt.size:
                    w, h = rt.shape
                    np.testing.assert_array_equal((tiles[i, :w * h] & 15).reshape(w, h), rt, err_msg="%s tile map, level %d, seed %d" % (game, rnd, seed + i))
            if rnd < 4:
                np.testing.assert_array_equal(frames[rnd][c0:c0 + len(refs)], np.stack([r.reset() for r in refs]),
                                              err_msg="%s reset frame %d" % (game, rnd))
        for r in refs:
            r.close()


# ---- (e) the captured step graph ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("game", ["coinrun", "bossfight", "maze", "jumper"])
def test_step_graph_equals_eager(game, monkeypatch):
    """One CUDA-graph launch per step (k_step node re-pointed at the caller's action buffer every step) against the eager
    three-launch sequence (PG2_GRAPH=0), with short episodes so that resets / level swaps happen inside the graph, and with
    the action tensor at a different device address every step."""
    import torch
    from procgen2_b200.engine import BatchedEnv
    n, T = 160, 90
    rs = np.random.RandomState(33)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    monkeypatch.setenv("PG2_GRAPH", "0")
    a = BatchedEnv(game, n, seed=71, max_episode_steps=12)
    monkeypatch.setenv("PG2_GRAPH", "1")
    b = BatchedEnv(game, n, seed=71, max_episode_steps=12)
    a.reset(); b.reset()
    dev_acts = torch.from_numpy(acts).cuda()
    for t in range(T):
        a.step(acts[t])
        b.step_torch(dev_acts[t])          # a view: a new device pointer each step
        oa, ra, da, ta = a.fetch(truncated=True)
        ob, rb, db, tb = b.fetch(truncated=True)
        np.testing.assert_array_equal(oa, ob, err_msg="pixels, step %d" % t)
        np.testing.assert_array_equal(ra, rb); np.testing.assert_array_equal(da, db); np.testing.assert_array_equal(ta, tb)
    b.sync()
    for name in ("mt", "mti", "fault"):
        np.testing.assert_array_equal(a.read_field(name)[0], b.read_field(name)[0])
    _assert_no_fault(b)
    a.close(); b.close()


# ---- (f) level prefetch under the worst case ----------------------------------------------------------------------------------

@pytest.mark.parametrize("game,n,max_ep", [("maze", 32768, 1), ("jumper", 8192, 1), ("climber", 16384, 2)])
def test_prefetch_when_every_env_finishes_every_step(game, n, max_ep, monkeypatch):
    """Large batch, one- / two-step episodes: every env finishes (again) before its next level can exist, so every stepping
    warp waits for the asynchronous generator while the GPU is full of them. No fault flag (= no bounded wait expired, no
    deadlock) and the same results as the inline-reset path."""
    from procgen2_b200.engine import BatchedEnv
    T = 16
    acts = np.random.RandomState(1).randint(0, 15, size=(T, n)).astype(np.int32)
    outs = []
    for pf in ("1", "0"):
        monkeypatch.setenv("PG2_PREFETCH", pf)
        env = BatchedEnv(game, n, seed=3, max_episode_steps=max_ep)
        env.reset()
        for t in range(T):
            env.step(acts[t])
        o, r, d, tr = env.fetch(truncated=True)
        _assert_no_fault(env)
        outs.append((o, r, d, tr, env.read_field("mti")[0].copy(), env.read_field("mt")[0].copy()))
        env.close()
    for a, b in zip(*outs):
        np.testing.assert_array_equal(a, b)


# ---- bossfight past its first seconds -----------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [None, 0])
def test_bossfight_whole_fight_live_oracle(mode, reference):
    """The lane-aware k_step<bossfight> (bullet rings as visited prefixes, ballots over 8-lane groups) through whole fights:
    a policy that dodges and fires (random actions die within ~50 steps) walks the boss through its shielded / unshielded
    phases, every attack pattern, the shield bounces, hp and its death — pixels, rewards, dones every step, RNG at the end."""
    from procgen2_b200.engine import BatchedEnv
    from tests.test_hostsim_parity import bossfight_policy
    n, seed, T = 16, 777, 1500
    rs = np.random.RandomState(seed)
    env = BatchedEnv("bossfight", n, seed=seed, distribution_mode=-1 if mode is None else mode)
    refs = [reference.RefEnv("bossfight", seed + i, mode=mode) for i in range(n)]
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0], np.stack([r.reset() for r in refs]))
    wins, longest, age = 0, 0, np.zeros(n, np.int64)
    for t in range(T):
        a = bossfight_policy(env.read_field, n, rs)
        env.step(a)
        o, rw, d, _ = env.fetch()
        for i, r in enumerate(refs):
            oo, w, dd = r.step(a[i])
            age[i] += 1
            if dd:
                oo = r.reset()
                wins += w > 0
                longest, age[i] = max(longest, age[i]), 0
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    _check_state(env, refs, tag="bossfight whole fight")
    _assert_no_fault(env)
    assert wins >= 1 and longest >= 400, (wins, longest)
    for r in refs:
        r.close()
    env.close()


# ---- chaser with orbs and eaten mobs --------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [None, 2])
def test_chaser_orbs_and_eaten_mobs_live_oracle(mode, reference):
    """The warp-per-env k_step<chaser> (point loop on the lanes, votes for "ate an orb") with a corridor-walking policy: the
    agent covers the maze, eats orbs (mobs flee and slow down) and now and then a mob (respawn on a free cell drawn from the
    RNG, SURVEY Q17) — paths uniform-random actions hardly reach. Easy 11x11 and extreme 19x19."""
    from procgen2_b200.engine import BatchedEnv
    n, seed, T = 16, 555, 1500
    rs = np.random.RandomState(seed)
    env = BatchedEnv("chaser", n, seed=seed, distribution_mode=-1 if mode is None else mode)
    refs = [reference.RefEnv("chaser", seed + i, mode=mode) for i in range(n)]
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0], np.stack([r.reset() for r in refs]))
    cur = rs.choice([1, 7, 3, 5], size=n)
    orbs, prev_eat = 0, np.zeros(n, np.float32)
    for t in range(T):
        cur = np.where(rs.rand(n) < 0.08, rs.choice([1, 7, 3, 5], size=n), cur)
        a = cur.astype(np.int32)
        env.step(a)
        o, rw, d, _ = env.fetch()
        eat = env.read_field("eat_timer")[0].view(np.float32).copy()
        orbs += int(((eat > prev_eat) & ~d.astype(bool)).sum())
        prev_eat = eat
        for i, r in enumerate(refs):
            oo, w, dd = r.step(a[i])
            if dd:
                oo = r.reset()
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    _check_state(env, refs, tag="chaser orbs")
    _assert_no_fault(env)
    assert orbs >= 5, orbs
    for r in refs:
        r.close()
    env.close()


# ---- purposeful action streams for the warp-per-env platformers ------------------------------------------------------------

@pytest.mark.parametrize("game,bias", [("coinrun", [8, 8, 7, 7, 5, 8, 6, 1, 4, 8]), ("climber", [2, 5, 8, 8, 2, 5, 1, 7, 5, 5])])
def test_biased_actions_live_oracle(game, bias, reference):
    """Run-right-and-jump (coinrun) / jump-a-lot (climber) action streams, held for 6 steps with 15 % noise: the agents get
    deep into their levels (crates, saws, lava, enemies, coins; 50x more rewarded steps than uniform-random actions), through
    the warp-per-env k_step with the entity loops on the lanes."""
    from procgen2_b200.engine import BatchedEnv
    n, seed, T = 32, 31415, 800
    rs = np.random.RandomState(seed)
    run = np.array(bias)[rs.randint(0, len(bias), size=(T // 6 + 1, n))]
    acts = np.repeat(run, 6, axis=0)[:T]
    acts = np.where(rs.rand(T, n) < 0.15, rs.randint(0, 15, size=(T, n)), acts).astype(np.int32)
    env = BatchedEnv(game, n, seed=seed)
    refs = [reference.RefEnv(game, seed + i) for i in range(n)]
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0], np.stack([r.reset() for r in refs]))
    rewarded = 0
    for t in range(T):
        env.step(acts[t])
        o, rw, d, _ = env.fetch()
        for i, r in enumerate(refs):
            oo, w, dd = r.step(acts[t, i])
            if dd:
                oo = r.reset()
            rewarded += w > 0
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    _check_state(env, refs, tag=game)
    _assert_no_fault(env)
    assert rewarded >= 3, rewarded
    for r in refs:
        r.close()
    env.close()


def test_bossfight_partial_last_warp_live_oracle(reference):
    """13 envs with 8 lanes each: the last warp of k_step<bossfight> holds ONE env and three idle lane groups."""
    from tests.parity_util import check_against_oracle
    from tests.test_gpu_parity import EngineAdapter
    n, T, seed = 13, 200, 8100
    acts = _mixed_actions(np.random.RandomState(3), T, n)
    a = EngineAdapter("bossfight", n, seed)
    refs = [reference.RefEnv("bossfight", seed + i) for i in range(n)]
    check_against_oracle(a, refs, acts, tag="bossfight 13 envs")
    _check_state(a.env, refs, tag="bossfight 13 envs")
    _assert_no_fault(a.env)
    for r in refs:
        r.close()
    a.env.close()

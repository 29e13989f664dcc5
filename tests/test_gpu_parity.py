"""GPU tests (pytest -m gpu on a B200): the CUDA engine, driven through its C ABI
(libprocgen2_b200.so via ctypes) and through the per-game cenv drop-in libraries, against
(1) the committed golden vectors generated from the compiled reference, (2) reference environments
(tests/reference.py: live when oracle/_ref is built, else the stand-in checked against recorded tapes), (3) size-independent properties at BASELINE sizes.
Everything is bit-exact: rewards, terminated, pixels, tile maps, MT19937 state."""
import numpy as np
import pytest

from tests.conftest import IMPLEMENTED, golden
from tests.parity_util import check_against_golden, check_against_oracle

pytestmark = pytest.mark.gpu


class EngineAdapter:
    def __init__(self, game, n, seed, **kw):
        from procgen2_b200.engine import BatchedEnv
        self.env = BatchedEnv(game, n, seed=seed, **kw)
        self.n = n

    def reset(self):
        self.env.reset()
        return self.env.fetch()[0]

    def step(self, actions):
        self.env.step(np.asarray(actions, np.int32))
        o, r, t, _ = self.env.fetch()
        return o, r, t

    def fields(self):
        out = {}
        for name, dt in (("mt", np.uint32), ("mti", np.int32), ("tiles", np.uint8)):
            try:
                b, esz, pe = self.env.read_field(name)
            except KeyError:
                continue
            out[name] = b.view(dt).reshape(self.n, pe) if pe > 1 else b.view(dt)
        return out


@pytest.mark.parametrize("game", IMPLEMENTED)
@pytest.mark.parametrize("stream", ["uniform", "biased"])
def test_golden(game, stream):
    a = check_against_golden(lambda n, seed: EngineAdapter(game, n, seed), golden(game), stream, read_fields=lambda a: a.fields())
    a.env.close()


@pytest.mark.parametrize("game", IMPLEMENTED)
def test_live_oracle(game, reference):
    n, T, seed = 48, 400, 900
    rs = np.random.RandomState(11)
    acts = np.where(rs.rand(T, n) < 0.5, rs.randint(0, 15, size=(T, n)), rs.choice([6, 7, 8, 8, 5], size=(T, n))).astype(np.int32)
    refs = [reference.RefEnv(game, seed + i) for i in range(n)]
    a = EngineAdapter(game, n, seed)
    episodes = check_against_oracle(a, refs, acts, tag=game)
    assert episodes > 0     # the auto-reset path was exercised
    a.env.close()


@pytest.mark.parametrize("game", IMPLEMENTED)
def test_cenv_dropin_single_env(game):
    """N=1 through lib<Game>.so + the CEnv wrapper = the reference's call pattern
    (make(seed) / reset / step / caller resets on terminate): golden env 0."""
    from procgen2_b200 import build
    from procgen2_b200.cenv import CEnv
    g = golden(game)
    env = CEnv(build.game_lib_path(game), options={"seed": int(g["seed"])})
    assert env.observation_space["screen"].low[0] == 0.0 and env.observation_space["screen"].high[0] == 255.0
    assert int(env.action_space["action"].nvec[0]) == 15
    obs, info = env.reset()
    np.testing.assert_array_equal(obs["screen"].reshape(64, 64, 3), g["uniform_frame0"][0])
    acts = g["uniform_actions"][:, 0]
    for t in range(len(acts)):
        obs, rew, term, trunc, info = env.step(int(acts[t]))
        assert rew == g["uniform_reward"][t, 0] and term == g["uniform_terminated"][t, 0] and not trunc
        if term:
            obs, _ = env.reset()
        key = "uniform_frame%d" % (t + 1)
        if key in g:
            np.testing.assert_array_equal(obs["screen"].reshape(64, 64, 3), g[key][0])
    env.close()


@pytest.mark.parametrize("game", IMPLEMENTED)
def test_cenv_dropin_batched(game):
    from procgen2_b200 import build
    from procgen2_b200.cenv import CEnv
    g = golden(game)
    acts = g["uniform_actions"]
    T, n = acts.shape
    env = CEnv(build.game_lib_path(game), options={"seed": int(g["seed"]), "num_envs": n})
    obs, _ = env.reset()
    np.testing.assert_array_equal(obs["screen"].reshape(n, 64, 64, 3), g["uniform_frame0"])
    for t in range(40):
        obs, rew, term, trunc, info = env.step(acts[t])
        np.testing.assert_array_equal(info["reward"], g["uniform_reward"][t])
        np.testing.assert_array_equal(info["terminated"].astype(bool), g["uniform_terminated"][t])
    np.testing.assert_array_equal(obs["screen"].reshape(n, 64, 64, 3), g["uniform_frame40"])
    env.close()


@pytest.mark.parametrize("game,n", [("coinrun", 4096), ("maze", 256)])
def test_sharding_invariance_at_baseline_size(game, n):
    """BASELINE configs 1/2 sizes: env i's trajectory does not depend on the batch it lives in
    (contiguous shards with first_env offsets == one big batch), checked by a checksum of
    per-env observation checksums, rewards and terminated flags over a short horizon."""
    import zlib
    if game not in IMPLEMENTED:
        pytest.skip("not implemented yet")
    T = 12
    rs = np.random.RandomState(3)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)

    def run(parts):
        outs = []
        for first, cnt in parts:
            a = EngineAdapter(game, cnt, 5, first_env=first)
            a.reset()
            res = []
            for t in range(T):
                o, r, d = a.step(acts[t, first:first + cnt])
                res.append((np.array([zlib.crc32(x.tobytes()) for x in o], np.uint32), r, d))
            outs.append(res)
            a.env.close()
        return [tuple(np.concatenate([outs[p][t][k] for p in range(len(parts))]) for k in range(3)) for t in range(T)]

    whole = run([(0, n)])
    split = run([(0, n // 2), (n // 2, n - n // 2)])
    for t in range(T):
        for k in range(3):
            np.testing.assert_array_equal(whole[t][k], split[t][k])


def test_manual_reset_equals_auto_reset():
    """auto_reset=0 (reference behaviour: the caller resets) gives the same stream as the
    on-device auto-reset when the caller resets every env that terminated — maze timeouts hit
    all envs at step 500 simultaneously."""
    from procgen2_b200.engine import BatchedEnv
    n = 8
    a = BatchedEnv("maze", n, seed=2, auto_reset=True)
    b = BatchedEnv("maze", n, seed=2, auto_reset=False)
    a.reset(); b.reset()
    acts = np.full(n, 4, np.int32)   # stay: no goal reached, every env times out at step 500
    for t in range(501):
        a.step(acts); b.step(acts)
        oa, ra, ta, _ = a.fetch()
        ob, rb, tb, _ = b.fetch()
        np.testing.assert_array_equal(ta, tb)
        if tb.all():
            b.reset()
            ob = b.fetch()[0]
        np.testing.assert_array_equal(oa, ob)
    a.close(); b.close()


def test_device_resident_views_and_reseed():
    import torch
    from procgen2_b200.engine import BatchedEnv
    env = BatchedEnv("maze", 16, seed=9)
    env.reset()
    obs, rew, term, trunc = env.torch_views()
    acts = torch.randint(0, 15, (16,), dtype=torch.int32, device="cuda")
    env.step_torch(acts)
    env.sync()
    host = env.fetch()[0]
    np.testing.assert_array_equal(obs.cpu().numpy(), host)
    # cenv_reset option "seed": reseeding reproduces the same level
    env.reset(seeds=np.arange(16, dtype=np.int32) + 100)
    f1 = env.fetch()[0]
    env.reset(seeds=np.arange(16, dtype=np.int32) + 100)
    f2 = env.fetch()[0]
    np.testing.assert_array_equal(f1, f2)
    env.close()


def test_pipelined_stepping_equals_sequential():
    """pg2_step_pipelined (double-buffered outputs, D2H on a second stream) returns, one call late, exactly what
    pg2_step + pg2_fetch return."""
    from procgen2_b200.engine import BatchedEnv
    n, T = 64, 60
    rs = np.random.RandomState(21)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    a = BatchedEnv("coinrun", n, seed=31)
    b = BatchedEnv("coinrun", n, seed=31)
    a.reset(); b.reset()
    seq = []
    for t in range(T):
        a.step(acts[t])
        o, r, d, _ = a.fetch()
        seq.append((o, r, d))
    bufs = [(np.empty((n, 64, 64, 3), np.uint8), np.empty(n, np.float32), np.empty(n, np.uint8)) for _ in range(2)]
    for t in range(T):
        b.step_pipelined(acts[t], *bufs[t & 1])
        if t > 0:   # the previous call's buffers are complete now
            o, r, d = bufs[(t - 1) & 1]
            np.testing.assert_array_equal(o, seq[t - 1][0]); np.testing.assert_array_equal(r, seq[t - 1][1])
            np.testing.assert_array_equal(d.astype(bool), seq[t - 1][2])
    b.flush()
    o, r, d = bufs[(T - 1) & 1]
    np.testing.assert_array_equal(o, seq[T - 1][0]); np.testing.assert_array_equal(r, seq[T - 1][1])
    a.close(); b.close()


@pytest.mark.parametrize("game", IMPLEMENTED)
def test_snapshot_restore_replays_bit_exact(game):
    """pg2_snapshot / pg2_restore (SURVEY §8f rank 4): stepping after a restore reproduces the steps that followed
    the snapshot bit for bit (observations, rewards, done flags, MT19937 streams) — also into a fresh engine, and
    across episode boundaries (auto-reset, level regeneration, bossfight's per-sub-step RNG)."""
    from procgen2_b200.engine import BatchedEnv
    n, T0, T1 = 96, 40, 120
    rs = np.random.RandomState(5)
    acts = rs.randint(0, 15, size=(T0 + T1, n)).astype(np.int32)
    a = BatchedEnv(game, n, seed=77, max_episode_steps=50)
    a.reset()
    for t in range(T0):
        a.step(acts[t])
    blob = a.snapshot()
    want = []
    for t in range(T0, T0 + T1):
        a.step(acts[t])
        o, r, d, tr = a.fetch(truncated=True)
        want.append((o, r, d, tr))
    mt_want = a.read_field("mt")[0].copy()
    # (1) same engine rewound, (2) a fresh engine that never saw the first T0 steps
    b = BatchedEnv(game, n, seed=12345, max_episode_steps=50)
    b.reset()
    for env in (a, b):
        env.restore(blob)
        np.testing.assert_array_equal(env.fetch()[0], np.frombuffer(blob, np.uint8)[-(n * 12288 + 6 * n):-6 * n].reshape(n, 64, 64, 3))
        for k, t in enumerate(range(T0, T0 + T1)):
            env.step(acts[t])
            o, r, d, tr = env.fetch(truncated=True)
            np.testing.assert_array_equal(o, want[k][0]); np.testing.assert_array_equal(r, want[k][1])
            np.testing.assert_array_equal(d, want[k][2]); np.testing.assert_array_equal(tr, want[k][3])
        np.testing.assert_array_equal(env.read_field("mt")[0], mt_want)
    with pytest.raises(RuntimeError):
        BatchedEnv(game, n + 1, seed=0).restore(blob)
    a.close(); b.close()


def test_cenv_dropin_num_devices_is_invisible():
    """cenv make-option "num_devices" (SURVEY §8e at the drop-in boundary): the batch sharded over two GPUs inside one
    library instance returns exactly what one GPU returns (seeds follow the global env index). Needs >= 2 GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from procgen2_b200.build import game_lib_path
    from procgen2_b200.cenv import CEnv
    n, T = 50, 60     # 25 + 25, and an uneven 3-way split is exercised by the shard arithmetic below when available
    rs = np.random.RandomState(4)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    ndev = 3 if torch.cuda.device_count() >= 3 else 2
    a = CEnv(game_lib_path("coinrun"), options={"seed": 11, "num_envs": n, "max_episode_steps": 25})
    ra = []
    obs, _ = a.reset()
    ra.append(obs["screen"].copy())
    for t in range(T):
        obs, _, _, _, info = a.step({"action": acts[t]})
        ra.append((obs["screen"].copy(), info["reward"].copy(), info["terminated"].copy(), info["truncated"].copy()))
    a.close()
    b = CEnv(game_lib_path("coinrun"), options={"seed": 11, "num_envs": n, "max_episode_steps": 25, "num_devices": ndev})
    obs, _ = b.reset()
    np.testing.assert_array_equal(obs["screen"], ra[0])
    for t in range(T):
        obs, _, _, _, info = b.step({"action": acts[t]})
        np.testing.assert_array_equal(obs["screen"], ra[t + 1][0])
        np.testing.assert_array_equal(info["reward"], ra[t + 1][1])
        np.testing.assert_array_equal(info["terminated"], ra[t + 1][2])
        np.testing.assert_array_equal(info["truncated"], ra[t + 1][3])
    b.close()


@pytest.mark.parametrize("game,max_ep", [("maze", 1), ("jumper", 2), ("caveflyer", 3), ("maze", 7)])
def test_level_prefetch_equals_inline_reset(game, max_ep, monkeypatch):
    """Level prefetch (next level generated one episode ahead into the shadow state, swapped in by k_swap) against the
    inline reset path (PG2_PREFETCH=0) on very short episodes: every env finishes every 1-3 steps, so envs finish again
    before their next level exists (k_swap_wait) and all four generator slots are in flight."""
    from procgen2_b200.engine import BatchedEnv
    n, T = 96, 40
    rs = np.random.RandomState(17)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    monkeypatch.setenv("PG2_PREFETCH", "0")
    a = BatchedEnv(game, n, seed=5, max_episode_steps=max_ep)
    monkeypatch.setenv("PG2_PREFETCH", "1")
    b = BatchedEnv(game, n, seed=5, max_episode_steps=max_ep)
    a.reset(); b.reset()
    np.testing.assert_array_equal(a.fetch()[0], b.fetch()[0])
    for t in range(T):
        a.step(acts[t]); b.step(acts[t])
        oa, ra, da, ta = a.fetch(truncated=True)
        ob, rb, db, tb = b.fetch(truncated=True)
        np.testing.assert_array_equal(oa, ob); np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(da, db); np.testing.assert_array_equal(ta, tb)
    b.sync()
    for name in ("mt", "mti", "tiles", "fault"):
        np.testing.assert_array_equal(a.read_field(name)[0], b.read_field(name)[0])
    a.close(); b.close()

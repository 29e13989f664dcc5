"""The whole state of the GPU step against the single-lane host-sim, one step at a time.

The other parity tests compare what reaches the outputs (pixels, rewards, done flags) plus the MT19937 state and the tile
map. Here every state field of the game and of CommonState is compared byte for byte after each checked step: positions,
velocities, timers, entity pools, both bossfight bullet rings with their indices and counts, ECS bucket counts,
ep_steps, camera, fault flags. Each checked step starts from the engine's own state, copied into a host-sim of the same
shape (tests/simlib.transplant); then both take the same step. The host-sim runs every env on one lane (StepCtx{0, 1})
with the level generated inline, so the comparison covers what only the device runs: the 8-lane bossfight groups and
their ballot-built ring prefixes, the 32-lane entity loops (coinrun and climber have 40 entity slots: a second pass),
the one-lane MT19937 twist of a lane group, the packed environments-per-warp mapping, and the level swap of the
prefetching games (swap_copy) with the shadow generator.

(a) plays the engine from its own seeds, (b) first writes edge states into the played engine (pg2_write_field, which
also regenerates the prefetched levels) and so into the host-sim. (c) are the assertions that the checked steps reached
what they exist for; (d) checks pg2_snapshot / pg2_restore on the whole state."""
import numpy as np
import pytest

from tests.simlib import HostSim, read_state, state_diff, transplant
from tests.test_hostsim_state import NONDEFAULT_MODES

pytestmark = pytest.mark.gpu

# Fields not compared, with the reason for each.
EXCLUDED = {}

# The one allowed difference. With level prefetch, an env that finished takes its next level from the shadow state, whose
# storage beyond what the level generator writes holds the shadow's own leftovers, while the inline reset (the host-sim)
# leaves the live leftovers there. The games never read that storage before writing it:
#   - entity slots k >= num_ents (coinrun, climber) / num_obj (caveflyer): every loop runs over k < the count;
#   - coinrun's particles of entity slot k (elements k * 10 .. k * 10 + 9) likewise;
#   - caveflyer's bullet ring: after a reset num_bullets = 0, so no slot is walked before the next shot writes it;
#   - jumper's tile map beyond the world's W * H cells (only memory mode has any: 2025 cells in 2048 bytes), which the
#     game never indexes; the generator leaves scratch bytes there.
# Allowed only in envs that took a prefetched level in the checked step, only in those elements, and only with prefetch
# on: the PG2_PREFETCH=0 configurations compare everything.
DEAD_AFTER_SWAP = {
    "coinrun": {f: ("num_ents", 1) for f in ("ent_type", "ent_x", "ent_y", "ent_vx", "ent_anim_t", "ent_frame", "ent_kind", "ent_flip",
                                             "part_timer")}
    | {f: ("num_ents", 10) for f in ("part_x", "part_y", "part_life")},
    "climber": {f: ("num_ents", 1) for f in ("ent_type", "ent_x", "ent_y", "ent_vx", "ent_spawn_x", "ent_anim_t", "ent_frame", "ent_flip")},
    "caveflyer": {f: ("num_obj", 1) for f in ("obj_type", "obj_x", "obj_y", "obj_vx", "obj_vy")}
    | {f: ("num_bullets", 1) for f in ("b_x", "b_y", "b_vx", "b_vy", "b_rot", "b_frame")},
    "jumper": {"tiles": "world"},
}
JUMPER_WORLD_CELLS = {-1: 40 * 40, 0: 20 * 20, 1: 40 * 40, 2: 45 * 45}   # Jumper::W * H of each distribution mode


def _mask_dead_after_swap(game, mode, fields, n, want, got, swapped):
    """Copy the host-sim's bytes over the engine's in the dead storage of the swapped envs (DEAD_AFTER_SWAP)."""
    rule = DEAD_AFTER_SWAP.get(game, {})
    got = dict(got)
    for name, esz, pe, env_major in fields:
        if name not in rule or not swapped.any():
            continue
        a = want[name].reshape(-1, esz)
        b = got[name].reshape(-1, esz).copy()
        if rule[name] == "world":   # env-major tile map: the cells of a swapped env beyond its world
            assert env_major
            k = np.arange(pe * n)
            dead = swapped[k // pe] & (k % pe >= JUMPER_WORLD_CELLS[mode])
        else:
            count_name, per = rule[name]
            count = want[count_name].view(np.int32)
            k = np.arange(pe)[:, None]
            dead = (swapped[None, :] & (k >= count[None, :] * per)).reshape(-1)
        b[dead] = a[dead]
        got[name] = b.reshape(-1)
    return got

BOSSFIGHT_LANES = 8   # BossFight::STEP_LANES: four envs per warp


def _engine(game, n, seed, max_ep, mode=-1, prefetch=None, epw=None, monkeypatch=None):
    from procgen2_b200.engine import BatchedEnv
    for var, val in (("PG2_PREFETCH", prefetch), ("PG2_STEP_EPW", epw)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))
    env = BatchedEnv(game, n, seed=seed, max_episode_steps=max_ep, distribution_mode=mode)
    monkeypatch.delenv("PG2_PREFETCH", raising=False)
    monkeypatch.delenv("PG2_STEP_EPW", raising=False)
    return env


PREFETCH_GAMES = ("maze", "coinrun", "climber", "caveflyer", "jumper")   # G::PREFETCH_LEVELS


def _prefetches(game, prefetch, max_ep):
    """Whether the engine generates levels ahead (Engine::init): PG2_PREFETCH decides if set, else coinrun only for
    episodes of at least 256 steps (CoinRun::PREFETCH_MIN_EPISODE)."""
    if game not in PREFETCH_GAMES:
        return False
    if prefetch is not None:
        return bool(prefetch)
    return not (game == "coinrun" and 0 < max_ep < 256)


def _lane_group(game, epw):
    if game == "bossfight":
        per_warp = 32 // BOSSFIGHT_LANES
        return lambda e: " (warp %d, lane group %d of %d)" % (e // per_warp, e % per_warp, per_warp)
    if epw > 1:
        return lambda e: " (warp %d, lane %d of %d envs per warp)" % (e // epw, e % epw, epw)
    return None


def _actions(game, rs, n):
    if game == "bossfight":   # fire most of the time: the agent's ring fills up
        return np.where(rs.rand(n) < 0.8, 9, rs.randint(0, 9, n)).astype(np.int32)
    return rs.randint(0, 15, n).astype(np.int32)


class Checker:
    """One-step differential: engine state -> host-sim, the same step on both, every field compared."""

    def __init__(self, env, game, mode, max_ep, tag, prefetch=False):
        self.env, self.game, self.mode, self.tag, self.prefetch = env, game, mode, tag, prefetch
        self.n = env.num_envs
        self.sim = HostSim(game, self.n, 1, max_episode_steps=max_ep, distribution_mode=mode)
        self.fields = self.sim.field_list()
        self.lane_group = _lane_group(game, env.step_epw)
        self.steps = 0
        self.done_count = np.zeros(self.n, np.int64)   # episodes that ended in the checked steps, per env
        self.before = self.after = None

    def step(self, actions):
        transplant(self.env, self.sim)
        self.before = read_state(self.sim, self.fields)
        self.env.step(actions)
        o, r, d, tr = self.env.fetch(truncated=True)
        so, sr, sd = self.sim.step(actions)
        st = self.sim.truncated()
        got = read_state(self.env, self.fields)
        want = read_state(self.sim, self.fields)
        where = "%s, checked step %d" % (self.tag, self.steps)
        if self.prefetch:
            got = _mask_dead_after_swap(self.game, self.mode, self.fields, self.n, want, got, d | tr)
        diff = state_diff(want, got, self.fields, self.n, skip=EXCLUDED, lane_group=self.lane_group)
        assert not diff, "%s: engine (got) vs host-sim (want)\n%s" % (where, diff)
        for name, a, b in (("reward", sr.view(np.uint32), r.view(np.uint32)), ("terminated", sd, d), ("truncated", st, tr)):
            bad = np.flatnonzero(a != b)
            assert bad.size == 0, "%s: %s of %d envs differ, first env %d: want %r, got %r" % (where, name, bad.size, bad[0], a[bad[0]], b[bad[0]])
        bad = np.flatnonzero((so != o).reshape(self.n, -1).any(axis=1))
        assert bad.size == 0, "%s: pixels of %d envs differ, first env %d" % (where, bad.size, bad[0])
        self.done_count += d | tr
        self.after = want
        self.steps += 1

    def field(self, state, name, dtype):
        _, esz, pe, em = next(f for f in self.fields if f[0] == name)
        a = state[name].view(dtype)
        return a.reshape(self.n, pe) if em else a.reshape(pe, self.n).T

    def close(self):
        self.sim.close()
        self.env.close()


# ---------------------------------------------------------------------------------------------------------------------
# (a) one-step differential from the engine's own state

# (game, N, mode, prefetch, epw, warm-up steps, max_episode_steps, checked steps)
CONFIGS = [
    ("bossfight", 13, -1, None, None, 260, 264, 10),      # 8-lane groups, partial last warp
    ("bossfight", 16384, -1, None, None, 400, 404, 8),    # the headline shape
    ("coinrun", 4096, -1, 0, None, 40, 24, 8),
    ("coinrun", 4096, -1, 1, None, 40, 4, 8),
    ("climber", 1000, -1, 0, None, 40, 24, 8),
    ("climber", 1000, -1, 1, None, 40, 4, 8),
    ("chaser", 4096, -1, None, None, 40, 24, 8),          # overlap-reset schedule
    ("maze", 256, -1, 0, None, 20, 6, 8),
    ("maze", 256, -1, 1, None, 20, 6, 8),
    ("maze", 32768, -1, 0, None, 20, 6, 8),               # the engine packs envs into warps by itself
    ("maze", 32768, -1, 1, None, 20, 6, 8),
] + [(g, 512, -1, pf, epw, 20, 6, 8) for g in ("caveflyer", "jumper") for epw in (2, 4, 32) for pf in (0, 1)] \
  + [(g, 256, m, None, None, 30, 12, 8) for g, m in NONDEFAULT_MODES]


@pytest.mark.parametrize("game,n,mode,prefetch,epw,warm,max_ep,T", CONFIGS,
                         ids=["%s-n%d-mode%d-pf%s-epw%s" % (c[0], c[1], c[2], c[3], c[4]) for c in CONFIGS])
def test_step_state_parity(game, n, mode, prefetch, epw, warm, max_ep, T, monkeypatch):
    env = _engine(game, n, 1000 + n, max_ep, mode, prefetch, epw, monkeypatch)
    if game == "maze" and n == 32768 and epw is None:
        assert env.step_epw > 1, "the packed mapping is what this shape exists for"
    if epw is not None:
        assert env.step_epw == epw
    tag = "%s mode %d, N=%d, envs per warp %d, PG2_PREFETCH=%s, max_episode_steps %d" % (game, mode, n, env.step_epw, prefetch, max_ep)
    rs = np.random.RandomState(n + warm)
    env.reset()
    for _ in range(warm):
        env.step(_actions(game, rs, n))
    ck = Checker(env, game, mode, max_ep, tag, _prefetches(game, prefetch, max_ep))
    m_max = a_max = 0
    for _ in range(T):
        ck.step(_actions(game, rs, n))
        if game == "bossfight":
            m_max = max(m_max, int(ck.field(ck.before, "m_num_bullets", np.int32).max()))
            a_max = max(a_max, int(ck.field(ck.before, "a_num_bullets", np.int32).max()))
    # (c) coverage
    assert ck.done_count.sum() > 0, "no env finished an episode in the checked steps: resets / level swaps not covered"
    if prefetch:   # an env that finishes twice takes a level its first finish queued for generation during these steps
        assert (ck.done_count >= 2).any(), "no env finished twice in the checked steps"
    # Rings longer than four passes of the 8-lane group. Random play does not fill the boss ring much further (a run at
    # this shape peaked at 36 bullets: they leave the screen about as fast as the boss fires them); full 64-bullet rings
    # and hits that stop the walk are written in test_bossfight_boss_ring_edges.
    if game == "bossfight" and n > 1000:
        assert m_max > 32 and a_max > 8, "boss ring peaked at %d bullets, agent ring at %d" % (m_max, a_max)
    ck.close()


# ---------------------------------------------------------------------------------------------------------------------
# (b) edge states written into both

def _write(env, name, fn, dtype):
    """Read field `name` of the engine, let fn edit it in place as [env, element] (slot-major fields are transposed for
    it), write it back."""
    buf, esz, pe = env.read_field(name)
    a = buf.view(dtype).reshape(pe, env.num_envs).T.copy()
    fn(a)
    env.write_field(name, np.ascontiguousarray(a.T))


def _set(env, name, values, dtype):
    _write(env, name, lambda a: a.__setitem__((slice(None), 0), values), dtype)


def _boss_ring_state(env, rs, variant_of_env):
    """Fill the boss's ring. variant_of_env(e) -> (m_next, num, p_hit, destroyed_before): live bullets (frame 0, moving at
    the game's bullet speed) scattered over the screen away from the agent; the bullet at walk position p_hit (0 = the
    newest, ring slot m_next - 1) sits on the agent; with destroyed_before, the bullets walked before it have just left the
    screen and are destroyed when visited. The game reaches this: the boss fires 8 bullets every 10 ticks, the ring holds
    64, bullets leave the screen in any order, and the agent can stand anywhere."""
    n = env.num_envs
    px = env.read_field("px")[0].view(np.float32)
    py = env.read_field("py")[0].view(np.float32)
    x = rs.uniform(-1.9, 1.9, (n, 64)).astype(np.float32)
    y = rs.uniform(-1.9, 1.9, (n, 64)).astype(np.float32)
    rot = rs.uniform(0, 2 * np.pi, (n, 64)).astype(np.float32)
    nxt, num = np.zeros(n, np.int32), np.zeros(n, np.int32)
    for e in range(n):
        m_next, cnt, p_hit, destroyed_before = variant_of_env(e)
        nxt[e], num[e] = m_next, cnt
        far = np.hypot(x[e] - px[e], y[e] - py[e]) < 0.5   # keep every other bullet clear of the agent
        y[e, far] = np.where(py[e] > 0, -1.8, 1.8)
        if p_hit is not None:
            slot = (64 + m_next - 1 - p_hit) % 64
            x[e, slot], y[e, slot] = px[e], py[e]
            if destroyed_before:
                for i in range(p_hit):
                    x[e, (64 + m_next - 1 - i) % 64] = 2.5   # off screen: destroyed when visited
    vx = (np.cos(rot) * np.float32(0.1)).astype(np.float32)
    vy = (-np.sin(rot) * np.float32(0.1)).astype(np.float32)
    for name, v in (("mb_x", x), ("mb_y", y), ("mb_vx", vx), ("mb_vy", vy), ("mb_rot", rot), ("mb_frame", np.zeros((n, 64), np.float32))):
        _write(env, name, lambda a, v=v: a.__setitem__(slice(None), v), np.float32)
    _set(env, "m_next_bullet", nxt, np.int32)
    _set(env, "m_num_bullets", num, np.int32)


def _agent_ring_state(env, rs, phase_of_env, hp_of_env, edge=False):
    """32 agent bullets (frame 0, not bouncing, as fired) all on the boss: on the shield in a shielded (even) phase, on
    the boss itself in an unshielded one. With edge, every bullet instead sits exactly on the screen border (its
    collision box touching it from inside or outside). The agent fires one bullet every 5 ticks while the ring has room."""
    n = env.num_envs
    bx = env.read_field("bx")[0].view(np.float32)
    by = env.read_field("by")[0].view(np.float32)
    x = np.repeat(bx[:, None], 32, 1) + rs.uniform(-0.3, 0.3, (n, 32)).astype(np.float32)
    y = np.repeat(by[:, None], 32, 1) + rs.uniform(-0.2, 0.2, (n, 32)).astype(np.float32)
    if edge:
        pos = np.array([-2.01, -1.99, 1.99, 2.01], np.float32)
        x = rs.choice(pos, (n, 32)).astype(np.float32)
        y = rs.uniform(-1.5, 1.5, (n, 32)).astype(np.float32)
        swap = rs.rand(n, 32) < 0.5
        x[swap], y[swap] = y[swap], x[swap]
    for name, v in (("ab_x", x), ("ab_y", y), ("ab_vx", np.zeros((n, 32), np.float32)), ("ab_vy", np.full((n, 32), -0.1, np.float32)),
                    ("ab_frame", np.zeros((n, 32), np.float32)), ("ab_bounce_timer", np.zeros((n, 32), np.float32))):
        _write(env, name, lambda a, v=v: a.__setitem__(slice(None), v), np.float32)
    _write(env, "ab_bouncing", lambda a: a.__setitem__(slice(None), 0), np.uint8)
    _set(env, "a_num_bullets", np.full(n, 32, np.int32), np.int32)
    _set(env, "a_next_bullet", (np.arange(n) * 7 % 32).astype(np.int32), np.int32)
    _set(env, "phase_index", np.array([phase_of_env(e) for e in range(n)], np.int32), np.int32)
    _set(env, "hp", np.array([hp_of_env(e) for e in range(n)], np.int32), np.int32)
    # the phase timer must not have expired this step (else the phase changes before the bullets arrive)
    _set(env, "phase_timer", np.full(n, 1.0, np.float32), np.float32)


def _bossfight(monkeypatch, n=64, max_ep=1000):
    env = _engine("bossfight", n, 77, max_ep, monkeypatch=monkeypatch)
    env.reset()
    rs = np.random.RandomState(9)
    for _ in range(40):
        env.step(_actions("bossfight", rs, n))
    return env, rs


BOSS_HIT_POS = (0, 7, 8, 31, 63)


def test_bossfight_boss_ring_edges(monkeypatch):
    env, rs = _bossfight(monkeypatch)
    variants = []
    for m_next in (0, 63):
        variants.append((m_next, 64, None, False))   # a full ring, nothing on the agent
        for p in BOSS_HIT_POS:
            for destroyed in (False, True):
                variants.append((m_next, 64, p, destroyed))
    assert len(variants) <= env.num_envs
    _boss_ring_state(env, rs, lambda e: variants[e % len(variants)])
    ck = Checker(env, "bossfight", -1, 1000, "bossfight boss ring edges, N=64")
    stay = np.full(env.num_envs, 4, np.int32)   # no movement, no fire: the agent stays on its bullet
    ck.step(stay)
    hit = ck.done_count > 0   # the agent died (and the env was reset)
    want_hit = np.array([variants[e % len(variants)][2] is not None for e in range(env.num_envs)])
    # a hit bullet is visited (and so stops the walk) unless destroyed bullets before it push it out of the prefix
    late = np.array([variants[e % len(variants)][2] == 63 and variants[e % len(variants)][3] for e in range(env.num_envs)])
    assert (hit[want_hit & ~late]).all() and not hit[~want_hit].any(), "the agent-hit scenarios did not play out as set up"
    for _ in range(3):
        ck.step(stay)
    ck.close()


@pytest.mark.parametrize("shielded", [True, False])
def test_bossfight_agent_ring_edges(shielded, monkeypatch):
    env, rs = _bossfight(monkeypatch)
    hp = lambda e: 1 + e % 3
    _agent_ring_state(env, rs, (lambda e: 2 * (e % 2)) if shielded else (lambda e: 1 + 2 * (e % 2)), hp)
    ck = Checker(env, "bossfight", -1, 1000, "bossfight agent ring on the %s boss, N=64" % ("shielded" if shielded else "unshielded"))
    stay = np.full(env.num_envs, 4, np.int32)
    ck.step(stay)
    live = ck.done_count == 0   # (an env whose agent died in the step was reset)
    if shielded:   # 32 bounce draws in ring order
        bouncing = ck.field(ck.after, "ab_bouncing", np.uint8)[live]
        assert bouncing.sum() >= 0.9 * 32 * bouncing.shape[0], "the bullets did not bounce off the shield"
    else:
        assert (ck.field(ck.after, "hp", np.int32)[live, 0] == 0).all(), "more hits than hp must leave hp at 0"
    for _ in range(3):
        ck.step(stay)
    ck.close()


def test_bossfight_bullets_on_the_screen_edge(monkeypatch):
    env, rs = _bossfight(monkeypatch)
    _agent_ring_state(env, rs, lambda e: 1, lambda e: 3, edge=True)
    ck = Checker(env, "bossfight", -1, 1000, "bossfight agent bullets on the screen edge, N=64")
    for _ in range(3):
        ck.step(np.full(env.num_envs, 4, np.int32))
    ck.close()


def test_bossfight_agent_at_screen_borders_and_corners(monkeypatch):
    """The ship clamped against each edge and corner of the screen (bossfight has no tile map: the screen is its
    world), moving into it. Holding a direction long enough puts the ship there."""
    env, rs = _bossfight(monkeypatch)
    n = env.num_envs
    # the ship's collision box is 0.3 x 0.2 around (px, py); the screen is [-2, 2] x [-2, 2]
    xs, ys = (-1.85, 0.0, 1.85), (-1.9, 0.0, 1.9)
    spots = [(x, y) for x in xs for y in ys if (x, y) != (0.0, 0.0)]
    # action pushing into the spot: x -1/0/+1 -> 0,1,2 / 3,4,5 / 6,7,8 (row), y -1/0/+1 within the row (y up = +1)
    push = np.array([3 * (1 + int(np.sign(spots[e % 8][0]))) + (1 - int(np.sign(spots[e % 8][1]))) for e in range(n)], np.int32)
    _set(env, "px", np.array([spots[e % 8][0] for e in range(n)], np.float32), np.float32)
    _set(env, "py", np.array([spots[e % 8][1] for e in range(n)], np.float32), np.float32)
    _set(env, "pvx", np.array([0.1 * np.sign(spots[e % 8][0]) for e in range(n)], np.float32), np.float32)
    _set(env, "pvy", np.array([0.1 * np.sign(spots[e % 8][1]) for e in range(n)], np.float32), np.float32)
    ck = Checker(env, "bossfight", -1, 1000, "bossfight ship at the screen borders, N=64")
    for _ in range(3):
        ck.step(push)
    ck.close()


# coinrun / climber: the per-entity loops run one entity per lane over 32 lanes, so slots 32-39 take a second pass.
# Generated levels have at most about 23 entities, so longer lists are written: the level's own entities repeated
# (same kind, position, velocity, animation and particles) up to the wanted count, each new slot appended to the sprite
# order. A level the generator filled with more saws, mobs or points would look the same.
ENT_SLOT_FIELDS = {
    "coinrun": {f: 1 for f in ("ent_type", "ent_x", "ent_y", "ent_vx", "ent_anim_t", "ent_frame", "ent_kind", "ent_flip", "part_timer")}
    | {f: 10 for f in ("part_x", "part_y", "part_life")},
    "climber": {f: 1 for f in ("ent_type", "ent_x", "ent_y", "ent_vx", "ent_spawn_x", "ent_anim_t", "ent_frame", "ent_flip")},
}
ENT_COUNTS = (31, 32, 33, 40)


@pytest.mark.parametrize("game", ["coinrun", "climber"])
def test_entity_lists_past_one_warp(game, monkeypatch):
    n = 128
    env = _engine(game, n, 31, 0, monkeypatch=monkeypatch)
    env.reset()
    rs = np.random.RandomState(12)
    for _ in range(10):
        env.step(_actions(game, rs, n))
    n0 = env.read_field("num_ents")[0].view(np.int32).copy()
    assert (n0 > 0).all() and (n0 < 31).all()
    target = np.array([ENT_COUNTS[e % len(ENT_COUNTS)] for e in range(n)], np.int32)
    for name, per in ENT_SLOT_FIELDS[game].items():
        buf, esz, pe = env.read_field(name)
        a = buf.reshape(pe, n, esz).copy()
        for e in range(n):
            for k in range(n0[e], target[e]):
                src = k % n0[e]
                a[k * per:(k + 1) * per, e] = a[src * per:(src + 1) * per, e]
        env.write_field(name, a.reshape(-1))
    order = env.read_field("sprite_order")[0].reshape(-1, n).copy()
    for e in range(n):
        order[n0[e]:target[e], e] = np.arange(n0[e], target[e])
    env.write_field("sprite_order", order.reshape(-1))
    _set(env, "num_ents", target, np.int32)
    ck = Checker(env, game, -1, 0, "%s with %s entities" % (game, "/".join(map(str, ENT_COUNTS))), _prefetches(game, None, 0))
    moved = np.zeros(n, bool)
    for _ in range(4):
        ck.step(_actions(game, rs, n))
        ents = ck.field(ck.before, "num_ents", np.int32)[:, 0]
        live = (ck.done_count == 0) & (ents > 32)
        x0, x1 = ck.field(ck.before, "ent_x", np.float32), ck.field(ck.after, "ent_x", np.float32)
        moved |= live & (x0[:, 32:] != x1[:, 32:]).any(axis=1)
    assert moved.any(), "no entity in slots 32-39 moved: the second pass did not run"
    ck.close()


MTI_POSITIONS = (0, 1, 311, 622, 623, 624)
ALL_GAMES = ["maze", "coinrun", "bossfight", "climber", "chaser", "caveflyer", "jumper"]


@pytest.mark.parametrize("game,prefetch", [(g, None) for g in ALL_GAMES] + [(g, 1) for g in ("maze", "coinrun", "climber", "caveflyer", "jumper")])
def test_rng_position_at_forced_reset(game, prefetch, monkeypatch):
    """mti at every twist boundary in the step that truncates: the level generator of k_reset (and with prefetch the
    shadow generator, regenerated by pg2_write_field) starts there. Any mti in [0, 624] is a position the stream passes."""
    n, max_ep = 96, 40
    env = _engine(game, n, 5, max_ep, prefetch=prefetch, monkeypatch=monkeypatch)
    env.reset()
    rs = np.random.RandomState(2)
    for _ in range(10):
        env.step(_actions(game, rs, n))
    mti = np.array([MTI_POSITIONS[e % len(MTI_POSITIONS)] for e in range(n)], np.int32)
    _set(env, "mti", mti, np.int32)
    _set(env, "ep_steps", np.full(n, max_ep - 1, np.int32), np.int32)
    ck = Checker(env, game, -1, max_ep, "%s RNG position at a forced reset, PG2_PREFETCH=%s" % (game, prefetch), _prefetches(game, prefetch, max_ep))
    ck.step(_actions(game, rs, n))
    assert ck.done_count.all(), "every env must have been truncated"
    after = ck.field(ck.after, "mti", np.int32)[:, 0]
    # a twist restarts the position at 0: the generation twisted where the position went down
    assert (after < mti)[mti >= 622].all(), "the level generation did not twist from the positions at the end of the state"
    for _ in range(3):
        ck.step(_actions(game, rs, n))
    ck.close()


@pytest.mark.parametrize("game", ["bossfight", "chaser"])
def test_rng_position_in_step(game, monkeypatch):
    """mti at every twist boundary before a step that draws: the one-lane collective twist of k_step."""
    n = 96 if game == "bossfight" else 64
    env = _engine(game, n, 6, 0, monkeypatch=monkeypatch)
    env.reset()
    rs = np.random.RandomState(3)
    for _ in range(150):   # chaser draws when a hatched mob reaches a junction
        env.step(_actions(game, rs, n))
    mti = np.array([MTI_POSITIONS[e % len(MTI_POSITIONS)] for e in range(n)], np.int32)
    _set(env, "mti", mti, np.int32)
    ck = Checker(env, game, -1, 0, "%s RNG position in k_step" % game)
    twisted = np.zeros(n, bool)
    for t in range(8):
        ck.step(_actions(game, rs, n))
        before, after = ck.field(ck.before, "mti", np.int32)[:, 0], ck.field(ck.after, "mti", np.int32)[:, 0]
        twisted |= (after < before) & (ck.done_count == 0)   # a twist restarts the position at 0 (not a reset)
        if t == 0 and game == "bossfight":   # draws every sub-step
            assert twisted[mti >= 622].all(), "the step did not twist from the positions at the end of the state"
    assert twisted.any(), "no env twisted in a step"
    ck.close()


def test_truncation_with_termination(monkeypatch):
    """maze: the agent on the goal (terminated) in the step that also reaches max_episode_steps: terminated wins,
    truncated stays 0. Walking onto the goal on the last allowed step reaches it."""
    n, max_ep = 64, 30
    env = _engine("maze", n, 8, max_ep, monkeypatch=monkeypatch)
    env.reset()
    rs = np.random.RandomState(4)
    for _ in range(5):
        env.step(_actions("maze", rs, n))
    on_goal = np.arange(n) % 2 == 0
    for a, g in (("agent_x", "goal_x"), ("agent_y", "goal_y")):
        ag = env.read_field(a)[0].view(np.float32).copy()
        gl = env.read_field(g)[0].view(np.float32)
        ag[on_goal] = gl[on_goal]
        env.write_field(a, ag)
    _set(env, "ep_steps", np.where(np.arange(n) % 4 < 2, max_ep - 1, 3).astype(np.int32), np.int32)
    ck = Checker(env, "maze", -1, max_ep, "maze truncation with termination")
    ck.step(np.full(n, 4, np.int32))
    o, r, d, tr = env.fetch(truncated=True)
    both = on_goal & (np.arange(n) % 4 < 2)
    assert d[both].all() and not tr[both].any()
    assert tr[~on_goal & (np.arange(n) % 4 < 2)].all()
    ck.close()


# ---------------------------------------------------------------------------------------------------------------------
# (d) snapshot / restore of the whole state

@pytest.mark.parametrize("game", ALL_GAMES)
def test_snapshot_restore_whole_state(game, monkeypatch):
    n, max_ep = 96, 30
    rs = np.random.RandomState(11)
    a = _engine(game, n, 21, max_ep, monkeypatch=monkeypatch)
    b = _engine(game, n, 99, max_ep, monkeypatch=monkeypatch)
    a.reset(); b.reset()
    for _ in range(45):
        a.step(_actions(game, rs, n))
    sim = HostSim(game, 1, 0)
    fields = sim.field_list()
    sim.close()
    want = read_state(a, fields)
    b.restore(a.snapshot())
    got = read_state(b, fields)
    assert not state_diff(want, got, fields, n, skip=("view_valid",)), state_diff(want, got, fields, n, skip=("view_valid",))
    assert not got["view_valid"].any(), "restore clears view_valid: the view caches are not part of the blob"
    # restore regenerates the prefetched levels from the restored state: their dead storage (DEAD_AFTER_SWAP) is the new
    # shadow's, not the one the source engine had built up
    swapped = np.zeros(n, bool)
    for t in range(20):
        acts = _actions(game, rs, n)
        a.step(acts); b.step(acts)
        oa, ra, da, ta = a.fetch(truncated=True)
        ob, rb, db, tb = b.fetch(truncated=True)
        want, got = read_state(a, fields), read_state(b, fields)
        if _prefetches(game, None, max_ep):
            swapped |= da | ta
            got = _mask_dead_after_swap(game, -1, fields, n, want, got, swapped)
        diff = state_diff(want, got, fields, n)
        assert not diff, "step %d after the restore:\n%s" % (t, diff)
        np.testing.assert_array_equal(oa, ob); np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(da, db); np.testing.assert_array_equal(ta, tb)
    a.close(); b.close()

"""CPU tests: the engine's device SOURCE (compiled for the host by tests/hostsim, single lane)
against the golden vectors generated from the compiled reference, and against reference environments
(tests/reference.py: live when oracle/_ref is built, else the stand-in checked against recorded tapes). The product path (CUDA) is covered by test_gpu_parity."""
import numpy as np
import pytest

from tests.conftest import IMPLEMENTED, golden
from tests.parity_util import check_against_golden, check_against_oracle
from tests.simlib import HostSim


class SimAdapter:
    def __init__(self, game, n, seed, **kw):
        self.sim = HostSim(game, n, seed, **kw)
        self.n = n

    def reset(self):
        return self.sim.reset()

    def step(self, actions):
        return self.sim.step(actions)

    def fields(self):
        out = {}
        for name, dt in (("mt", np.uint32), ("mti", np.int32), ("tiles", np.uint8)):
            try:
                b, esz, pe = self.sim.field(name)
            except KeyError:
                continue
            out[name] = b.view(dt).reshape(self.n, pe) if pe > 1 else b.view(dt)
        return out


@pytest.mark.parametrize("game", IMPLEMENTED)
@pytest.mark.parametrize("stream", ["uniform", "biased"])
def test_golden(game, stream):
    check_against_golden(lambda n, seed: SimAdapter(game, n, seed), golden(game), stream, read_fields=lambda a: a.fields())


@pytest.mark.parametrize("game", IMPLEMENTED)
def test_live_oracle(game, reference):
    n, T, seed = 8, 300, 77
    rs = np.random.RandomState(5)
    acts = np.where(rs.rand(T, n) < 0.5, rs.randint(0, 15, size=(T, n)), rs.choice([6, 7, 8, 8, 5], size=(T, n))).astype(np.int32)
    refs = [reference.RefEnv(game, seed + i) for i in range(n)]
    check_against_oracle(SimAdapter(game, n, seed), refs, acts, tag=game)


OTHER_MODES = [("maze", 0), ("maze", 2), ("chaser", 1), ("chaser", 2), ("jumper", 0), ("jumper", 2), ("caveflyer", 0), ("caveflyer", 2)]


@pytest.mark.parametrize("game,mode", [(g, None) for g in IMPLEMENTED] + OTHER_MODES)
def test_level_generation_many_seeds(game, mode, reference):
    """Level layouts + the complete MT19937 state for many seeds and consecutive resets — the compiled-in mode of every game
    and every distribution mode that has its own world size."""
    n, seed = 24, 31337
    sim = SimAdapter(game, n, seed, distribution_mode=-1 if mode is None else mode)
    refs = [reference.RefEnv(game, seed + i, mode=mode) for i in range(n)]
    for rnd in range(4):
        f = sim.fields()
        for i, r in enumerate(refs):
            st, pos = r.rng_state()
            assert pos == f["mti"][i], (rnd, i)
            np.testing.assert_array_equal(st, f["mt"][i])
            rt = r.tiles()
            if rt.size:
                w, h = rt.shape
                np.testing.assert_array_equal((f["tiles"][i, :w * h] & 15).reshape(w, h), rt)
        obs = sim.reset()
        np.testing.assert_array_equal(obs, np.stack([r.reset() for r in refs]))


def test_max_episode_steps_truncates():
    sim = HostSim("maze", 4, 1, max_episode_steps=5)
    sim.reset()
    for t in range(5):
        _, _, term = sim.step(np.full(4, 4, np.int32))   # action 4 = stay
    b, _, _ = sim.field("ep_steps")
    assert (b.view(np.int32) == 0).all()       # truncated at step 5 -> regenerated
    assert not term.any()                      # truncation is not termination


@pytest.mark.parametrize("game", IMPLEMENTED)
@pytest.mark.parametrize("max_ep", [1, 5])
def test_truncation_live_oracle(game, max_ep, reference):
    """max_episode_steps (BASELINE configs[4]) against the reference driven as "step; every k steps: reset()":
    pixels, rewards, terminated, truncated, and the RNG state + tile map at the end. (GPU twin with more envs,
    longer horizons and k up to 32: tests/test_gpu_parity_r2.py.)"""
    n, seed, T = 3, 600 + max_ep, 8 * max_ep + 3
    rs = np.random.RandomState(9)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    sim = SimAdapter(game, n, seed, max_episode_steps=max_ep)
    refs = [reference.RefEnv(game, seed + i) for i in range(n)]
    np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
    age = np.zeros(n, np.int64)
    for t in range(T):
        o, rw, d = sim.step(acts[t])
        tr = np.ctypeslib.as_array(__import__("tests.simlib", fromlist=["lib"]).lib().hs_truncated(sim.sim.h), shape=(n,)).astype(bool)
        for i, e in enumerate(refs):
            oo, w, dd = e.step(acts[t, i])
            age[i] += 1
            trunc = (not dd) and age[i] >= max_ep
            if dd or trunc:
                oo = e.reset()
                age[i] = 0
            assert w == rw[i] and dd == d[i] and trunc == tr[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="pixels, step %d env %d" % (t, i))
    f = sim.fields()
    for i, r in enumerate(refs):
        st, pos = r.rng_state()
        assert pos == f["mti"][i]
        np.testing.assert_array_equal(st, f["mt"][i])
        r.close()


def test_maze_timeout_live_oracle(reference):
    """maze.cpp:308-310: an env that never reaches the goal terminates at step 500."""
    n, seed, T = 2, 41, 503
    acts = np.full((T, n), 4, np.int32)
    acts[:, 1] = np.random.RandomState(1).randint(0, 15, size=T)
    refs = [reference.RefEnv("maze", seed + i) for i in range(n)]
    episodes = check_against_oracle(SimAdapter("maze", n, seed), refs, acts, tag="maze timeout")
    assert episodes >= 1
    for r in refs:
        r.close()


@pytest.mark.parametrize("game", IMPLEMENTED)
def test_human_render_live_oracle(game, reference):
    """cenv_render (render_game(false), coinrun.cpp:393-411): the scene drawn again with the window size as camera_size —
    square windows interleaved with stepping (the observations must not be disturbed), a non-square one at the end
    (there the reference's own step logic would afterwards see the window aspect, SURVEY Q11: not interleaved)."""
    n, seed = 2, 77
    for (W, H) in ((96, 96), (160, 100)):
        sim = SimAdapter(game, n, seed)
        refs = [reference.RefEnv(game, seed + i, width=W, height=H) for i in range(n)]
        np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
        rs = np.random.RandomState(3)
        for t in range(24):
            a = rs.randint(0, 15, size=n).astype(np.int32)
            o, _, _ = sim.step(a)
            for i, r in enumerate(refs):
                oo, w, d = r.step(a[i])
                np.testing.assert_array_equal(o[i], r.reset() if d else oo)
            if (W == H and t % 8 == 7) or t == 23:
                for i, r in enumerate(refs):
                    np.testing.assert_array_equal(sim.sim.render_human(i, W, H), r.render(), err_msg="%s %dx%d step %d env %d" % (game, W, H, t, i))
        for r in refs:
            r.close()


@pytest.mark.parametrize("game,mode", [("maze", 2), ("chaser", 2), ("jumper", 2), ("caveflyer", 0)])
def test_human_render_in_other_modes_live_oracle(game, mode, reference):
    """cenv_render of the instantiations with their own world size (zoom, sprite count and tile window differ)."""
    n, seed, W, H = 2, 91, 128, 128
    sim = SimAdapter(game, n, seed, distribution_mode=mode)
    refs = [reference.RefEnv(game, seed + i, width=W, height=H, mode=mode) for i in range(n)]
    np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
    rs = np.random.RandomState(4)
    for t in range(60):
        a = rs.randint(0, 15, size=n).astype(np.int32)
        o, _, _ = sim.step(a)
        for i, r in enumerate(refs):
            oo, w, d = r.step(a[i])
            np.testing.assert_array_equal(o[i], r.reset() if d else oo)
        if t % 20 == 19:
            for i, r in enumerate(refs):
                np.testing.assert_array_equal(sim.sim.render_human(i, W, H), r.render(), err_msg="%s mode %d step %d env %d" % (game, mode, t, i))
    for r in refs:
        r.close()


@pytest.mark.parametrize("game", ["climber", "coinrun", "bossfight"])
def test_easy_distribution_mode_live_oracle(game, reference):
    """Make-option distribution_mode = 0 (easy) against the reference with its compile-time Config::easy_mode flipped
    (climber: enemy probability .2 instead of .5, tilemap.cpp:118; coinrun: the flag only feeds a variable nothing reads,
    tilemap.cpp:148 — same levels as hard; bossfight: System_Mob_AI::Config::mode, boss bullets at half speed and shielded
    phases of 180 + 30 u instead of 180 + 80 u steps, common_systems.cpp:104, 202)."""
    n, seed, T, ep = (6, 9100, 120, 30) if game != "bossfight" else (4, 9100, 700, 350)
    rs = np.random.RandomState(12)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    sim = SimAdapter(game, n, seed, max_episode_steps=ep, distribution_mode=0)
    refs = [reference.RefEnv(game, seed + i, **(dict(mode=0) if game == "bossfight" else dict(easy_mode=True))) for i in range(n)]
    np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
    age = np.zeros(n, np.int64)
    for t in range(T):
        o, rw, d = sim.step(acts[t])
        for i, r in enumerate(refs):
            oo, w, dd = r.step(acts[t, i])
            age[i] += 1
            if dd or age[i] >= ep:
                oo = r.reset(); age[i] = 0
            assert w == rw[i] and dd == d[i]
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    f = sim.fields()
    for i, r in enumerate(refs):
        st, pos = r.rng_state()
        assert pos == f["mti"][i]
        np.testing.assert_array_equal(st, f["mt"][i])
        r.close()
    if game == "climber":   # the mode does change climber's levels (fewer enemies): easy and hard runs part ways
        easy, hard = SimAdapter(game, n, seed, distribution_mode=0), SimAdapter(game, n, seed, distribution_mode=1)
        assert any(not np.array_equal(easy.reset(), hard.reset()) for _ in range(6))
    if game == "bossfight":   # ... and bossfight's frames once the boss has fired
        easy, hard = SimAdapter(game, n, seed, distribution_mode=0), SimAdapter(game, n, seed, distribution_mode=1)
        easy.reset(); hard.reset()
        assert any(not np.array_equal(easy.step(acts[t])[0], hard.step(acts[t])[0]) for t in range(200))


@pytest.mark.parametrize("game,mode", [("maze", 0), ("maze", 2), ("chaser", 1), ("chaser", 2), ("jumper", 0), ("caveflyer", 0), ("jumper", 2), ("caveflyer", 2)])
def test_world_size_modes_live_oracle(game, mode, reference):
    """Distribution modes that change the world size (own instantiations, G = <Game>T<MODE>) against the reference with its
    compile-time Config::mode set through the probe: levels (tile map + RNG state), pixels, rewards, dones, truncation."""
    n, seed, T = 5, 8300 + mode, 150
    rs = np.random.RandomState(mode)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    sim = SimAdapter(game, n, seed, max_episode_steps=40, distribution_mode=mode)
    refs = [reference.RefEnv(game, seed + i, mode=mode) for i in range(n)]
    f = sim.fields()
    for i, r in enumerate(refs):   # level #1 (cenv_make)
        rt = r.tiles()
        w, h = rt.shape
        np.testing.assert_array_equal((f["tiles"][i, :w * h] & 15).reshape(w, h), rt, err_msg="tile map after make, env %d" % i)
    np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
    age = np.zeros(n, np.int64)
    for t in range(T):
        o, rw, d = sim.step(acts[t])
        for i, r in enumerate(refs):
            oo, w, dd = r.step(acts[t, i])
            age[i] += 1
            if dd or age[i] >= 40:
                oo = r.reset(); age[i] = 0
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    f = sim.fields()
    for i, r in enumerate(refs):
        st, pos = r.rng_state()
        assert pos == f["mti"][i]
        np.testing.assert_array_equal(st, f["mt"][i])
        r.close()


def bossfight_policy(read_field, n, rs):
    """Dodge the nearest boss bullet, otherwise line up under the boss and fire (action 9): random actions die within ~50
    steps, this survives long enough to walk the boss through all of its phases and to win. read_field(name) -> (bytes,
    element size, elements per env) of a state field (slot-major)."""
    def fld(name):
        buf, esz, pe = read_field(name)
        return buf.view(np.float32).reshape(pe, n) if pe > 1 else buf.view(np.float32)
    px, py, bx = fld("px"), fld("py"), fld("bx")
    mx, my, mf = fld("mb_x"), fld("mb_y"), fld("mb_frame")
    acts = np.zeros(n, np.int32)
    for i in range(n):
        live = mf[:, i] == 0.0
        dx, dy = mx[live, i] - px[i], my[live, i] - py[i]
        d2 = dx * dx + dy * dy
        if d2.size and d2.min() < 0.5:
            k = int(np.argmin(d2))
            mxv, myv = (-1 if dx[k] > 0 else 1), (1 if dy[k] > 0 else -1)
            if rs.rand() < 0.3:
                myv = 0
            acts[i] = (mxv + 1) * 3 + (myv + 1)
        elif abs(px[i] - bx[i]) > 0.25 and rs.rand() < 0.8:
            acts[i] = 7 if bx[i] > px[i] else 1
        else:
            acts[i] = 9 if rs.rand() < 0.8 else rs.randint(0, 15)
    return acts


@pytest.mark.parametrize("mode", [None, 0])
def test_bossfight_whole_fight_live_oracle(mode, reference):
    """bossfight beyond the first seconds (System_Mob_AI::update common_systems.cpp:199-390: shielded / unshielded phases,
    every attack pattern, hp, the boss's death and the win reward) with a policy that survives: pixels, rewards, dones every
    step, RNG state at the end, hard and easy mode."""
    n, seed, T = 8, 777, 1500
    rs = np.random.RandomState(seed)
    sim = SimAdapter("bossfight", n, seed, distribution_mode=-1 if mode is None else mode)
    refs = [reference.RefEnv("bossfight", seed + i, mode=mode) for i in range(n)]
    np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
    wins, longest, age = 0, 0, np.zeros(n, np.int64)
    for t in range(T):
        a = bossfight_policy(sim.sim.field, n, rs)
        o, rw, d = sim.step(a)
        for i, r in enumerate(refs):
            oo, w, dd = r.step(a[i])
            age[i] += 1
            if dd:
                oo = r.reset()
                wins += w > 0
                longest, age[i] = max(longest, age[i]), 0
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    f = sim.fields()
    for i, r in enumerate(refs):
        st, pos = r.rng_state()
        assert pos == f["mti"][i]
        np.testing.assert_array_equal(st, f["mt"][i])
        r.close()
    assert wins >= 1 and longest >= 400, (wins, longest)


@pytest.mark.parametrize("mode", [None, 2])
def test_chaser_orbs_and_eaten_mobs_live_oracle(mode, reference):
    """chaser with a corridor-walking policy (hold a direction, turn now and then): the agent covers the maze, eats orbs
    (System_Mob_AI::eat, mobs flee and slow down, common_systems.cpp:117-297) and, now and then, a mob (respawn as an egg on
    a free cell drawn from the RNG, y not flipped: SURVEY Q17) — paths uniform-random actions hardly reach."""
    n, seed, T = 16, 555, 1500
    rs = np.random.RandomState(seed)
    sim = SimAdapter("chaser", n, seed, distribution_mode=-1 if mode is None else mode)
    refs = [reference.RefEnv("chaser", seed + i, mode=mode) for i in range(n)]
    np.testing.assert_array_equal(sim.reset(), np.stack([r.reset() for r in refs]))
    cur = rs.choice([1, 7, 3, 5], size=n)
    orbs, prev_eat = 0, np.zeros(n, np.float32)
    for t in range(T):
        cur = np.where(rs.rand(n) < 0.08, rs.choice([1, 7, 3, 5], size=n), cur)
        a = cur.astype(np.int32)
        o, rw, d = sim.step(a)
        eat = sim.sim.field("eat_timer")[0].view(np.float32).copy()
        orbs += int(((eat > prev_eat) & ~d).sum())
        prev_eat = eat
        for i, r in enumerate(refs):
            oo, w, dd = r.step(a[i])
            if dd:
                oo = r.reset()
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    f = sim.fields()
    for i, r in enumerate(refs):
        st, pos = r.rng_state()
        assert pos == f["mti"][i]
        np.testing.assert_array_equal(st, f["mt"][i])
        r.close()
    assert orbs >= 5, orbs

"""GPU tests of the reference-facing and tensor-facing front-ends: the cenv drop-in's device-resident extension
(make-option "host_copy", device addresses as infos and through cenv_device_buffer, pinned host buffers) and the
Gymnasium-VectorEnv-shaped class — both against the live oracle / the host-copy path (pytest -m gpu)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _ptr(info, key, shard=0):
    lo, hi = (int(x) & 0xffffffff for x in info[key][2 * shard:2 * shard + 2])
    return lo | hi << 32


class _Raw:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def test_cenv_device_pointers_and_host_copy_off(reference):
    """A cenv.py-style caller gets the observations WITHOUT the device -> host copy: make-option host_copy = 0, the device
    addresses arrive as INT-pair infos of reset / step and through the exported cenv_device_buffer; the data behind them
    equals the host-copy path and the live oracle."""
    import torch
    from procgen2_b200.build import game_lib_path
    from procgen2_b200.cenv import CEnv
    n, T, seed = 24, 40, 610
    rs = np.random.RandomState(2)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    # one environment (batch) per loaded library, like the reference (all state is global): the second one gets a copy
    import os, shutil
    lib2 = os.path.join(os.path.dirname(game_lib_path("coinrun")), "libCoinRun_copy_for_test.so")
    shutil.copyfile(game_lib_path("coinrun"), lib2)
    a = CEnv(game_lib_path("coinrun"), options={"seed": seed, "num_envs": n})
    b = CEnv(lib2, options={"seed": seed, "num_envs": n, "host_copy": 0})
    os.unlink(lib2)
    b.lib.cenv_device_buffer.restype = ctypes.c_void_p
    b.lib.cenv_device_buffer.argtypes = [ctypes.c_char_p, ctypes.c_int32]
    oa, ia = a.reset()
    ob, ib = b.reset()
    assert {"screen_device", "reward_device", "terminated_device", "truncated_device", "stream"} <= set(ib)
    assert _ptr(ib, "screen_device") == b.lib.cenv_device_buffer(b"screen", 0) != 0
    assert b.lib.cenv_device_buffer(b"nonsense", 0) is None and b.lib.cenv_device_buffer(b"screen", 1) is None
    dev = torch.device("cuda", 0)
    screen = torch.as_tensor(_Raw(_ptr(ib, "screen_device"), (n, 64, 64, 3), "|u1"), device=dev)
    reward = torch.as_tensor(_Raw(_ptr(ib, "reward_device"), (n,), "<f4"), device=dev)
    np.testing.assert_array_equal(screen.cpu().numpy().reshape(-1), oa["screen"])
    assert not ob["screen"].any()      # host_copy = 0: the host "screen" buffer is never written
    refs = [reference.RefEnv("coinrun", seed + i) for i in range(n)]
    np.testing.assert_array_equal(screen.cpu().numpy(), np.stack([r.reset() for r in refs]))
    for t in range(T):
        oa, _, _, _, ia = a.step(acts[t])
        ob, _, _, _, ib = b.step(acts[t])
        assert _ptr(ib, "screen_device") == b.lib.cenv_device_buffer(b"screen", 0)
        np.testing.assert_array_equal(screen.cpu().numpy().reshape(-1), oa["screen"], err_msg="step %d" % t)
        np.testing.assert_array_equal(reward.cpu().numpy(), ia["reward"])
        np.testing.assert_array_equal(ib["reward"], ia["reward"])            # rewards / flags are still copied
        np.testing.assert_array_equal(ib["terminated"], ia["terminated"])
        ro = []
        for i, r in enumerate(refs):
            o, w, d = r.step(acts[t, i])
            ro.append(r.reset() if d else o)
        np.testing.assert_array_equal(screen.cpu().numpy(), np.stack(ro), err_msg="oracle, step %d" % t)
    a.close(); b.close()


def test_cenv_single_env_reports_no_infos():
    """num_envs = 1 without extension options keeps the reference's shape: no infos (coinrun.cpp:200-202)."""
    from procgen2_b200.build import game_lib_path
    from procgen2_b200.cenv import CEnv
    e = CEnv(game_lib_path("maze"), options={"seed": 3})
    _, info = e.reset()
    assert info == {}
    _, _, _, _, info = e.step(4)
    assert info == {}
    e.close()


@pytest.mark.parametrize("game,mode", [("coinrun", None), ("chaser", None), ("chaser", "extreme"), ("maze", "easy")])
def test_vector_env_matches_oracle(game, mode, reference):
    """ProcgenVectorEnv: zero-copy tensors, actions as CUDA tensor / numpy / list, same-step autoreset, seeds, and the
    `distribution_mode` keyword by name."""
    import torch
    from procgen2_b200.vector_env import ProcgenVectorEnv
    n, T, seed = 16, 60, 4400
    rs = np.random.RandomState(6)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    env = ProcgenVectorEnv(game, n, seed=seed, max_episode_steps=25, distribution_mode=mode)
    with pytest.raises(ValueError):
        ProcgenVectorEnv(game, n, distribution_mode="nightmare")
    assert env.single_observation_space.shape == (64, 64, 3) and env.observation_space.shape == (n, 64, 64, 3)
    assert env.single_action_space.n == 15
    obs, info = env.reset()
    assert obs.is_cuda and obs.dtype == torch.uint8 and tuple(obs.shape) == (n, 64, 64, 3) and info == {}
    assert obs.data_ptr() == env.env.torch_views()[0].data_ptr()     # a view of the engine's buffer, not a copy
    refs = [reference.RefEnv(game, seed + i, mode=ProcgenVectorEnv.DISTRIBUTION_MODES[mode] if mode else None) for i in range(n)]
    np.testing.assert_array_equal(obs.cpu().numpy(), np.stack([r.reset() for r in refs]))
    age = np.zeros(n, np.int64)
    for t in range(T):
        a = acts[t]
        arg = torch.from_numpy(a).cuda() if t % 3 == 0 else (a if t % 3 == 1 else a.tolist())
        obs, rew, term, trunc, info = env.step(arg)
        assert rew.dtype == torch.float32 and term.dtype == torch.bool and trunc.dtype == torch.bool
        ro, rr, rd, rt = [], [], [], []
        for i, r in enumerate(refs):
            o, w, d = r.step(a[i])
            age[i] += 1
            tr = (not d) and age[i] >= 25
            if d or tr:
                o = r.reset(); age[i] = 0
            ro.append(o); rr.append(w); rd.append(d); rt.append(tr)
        np.testing.assert_array_equal(obs.cpu().numpy(), np.stack(ro), err_msg="pixels, step %d" % t)
        np.testing.assert_array_equal(rew.cpu().numpy(), np.array(rr, np.float32))
        np.testing.assert_array_equal(term.cpu().numpy(), np.array(rd))
        np.testing.assert_array_equal(trunc.cpu().numpy(), np.array(rt))
    # interchange: DLPack capsules and __cuda_array_interface__ alias the same memory
    caps = env.dlpack()
    assert torch.utils.dlpack.from_dlpack(caps[0]).data_ptr() == obs.data_ptr()
    assert env.__cuda_array_interface__["data"][0] == obs.data_ptr()
    # reseeding reproduces the level (cenv_reset option "seed")
    f1 = env.reset(seed=99)[0].clone()
    f2 = env.reset(seed=np.arange(n) + 99)[0]
    assert torch.equal(f1, f2)
    assert env.render().shape == (64, 64, 3)
    env.close()


@pytest.mark.parametrize("game,mode", [("coinrun", None), ("bossfight", None), ("jumper", None), ("maze", None),
                                       ("chaser", 2), ("caveflyer", 2)])
def test_cenv_render_matches_oracle(game, mode, reference):
    """cenv_render of the drop-in library = the reference's human-mode frame (512x512 default window and a custom size),
    rendered on the device; with the make-option "distribution_mode" passed through the cenv options for two of the
    instantiations that have their own world size."""
    from procgen2_b200.build import game_lib_path
    from procgen2_b200.cenv import CEnv
    for opts in ({}, {"width": 200, "height": 200}):
        env = CEnv(game_lib_path(game), options=dict(seed=515, **opts, **({} if mode is None else {"distribution_mode": mode})))
        ref = reference.RefEnv(game, 515, mode=mode, **opts)
        obs, _ = env.reset()
        np.testing.assert_array_equal(obs["screen"].reshape(64, 64, 3), ref.reset())
        rs = np.random.RandomState(1)
        for t in range(20):
            a = int(rs.randint(0, 15))
            obs, _, term, _, _ = env.step(a)
            o, w, d = ref.step(a)
            if d:
                o = ref.reset(); obs, _ = env.reset()
            np.testing.assert_array_equal(obs["screen"].reshape(64, 64, 3), o)
            if t % 6 == 5:
                fr = env.render()
                assert fr.shape == ((512, 512, 3) if not opts else (200, 200, 3))
                np.testing.assert_array_equal(fr, ref.render(), err_msg="%s step %d" % (game, t))
        env.close(); ref.close()


@pytest.mark.parametrize("game", ["climber", "bossfight"])
def test_distribution_mode_option(game, reference):
    """cenv make-option "distribution_mode" = 0 (easy) on the GPU against the reference with its compile-time mode flipped
    through the probe (climber: Config::easy_mode; bossfight: System_Mob_AI::Config::mode); a (game, mode) pair that is
    not built is refused loudly."""
    from procgen2_b200.engine import BatchedEnv
    with pytest.raises(RuntimeError, match="distribution_mode"):
        BatchedEnv("climber", 4, distribution_mode=2)     # climber has no third mode
    n, seed, T, ep = (32, 9100, 90, 30) if game == "climber" else (12, 9100, 500, 250)
    rs = np.random.RandomState(12)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    env = BatchedEnv(game, n, seed=seed, max_episode_steps=ep, distribution_mode=0)
    refs = [reference.RefEnv(game, seed + i, **(dict(easy_mode=True) if game == "climber" else dict(mode=0))) for i in range(n)]
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0], np.stack([r.reset() for r in refs]))
    age = np.zeros(n, np.int64)
    for t in range(T):
        env.step(acts[t])
        o, rw, d, _ = env.fetch()
        for i, r in enumerate(refs):
            oo, w, dd = r.step(acts[t, i])
            age[i] += 1
            if dd or age[i] >= ep:
                oo = r.reset(); age[i] = 0
            assert w == rw[i] and dd == d[i]
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    for r in refs:
        r.close()
    env.close()


@pytest.mark.parametrize("game,mode,dim,max_ep,T", [("maze", 0, 15, 40, 150), ("maze", 2, 31, 40, 150),
                                                    ("chaser", 1, 13, 120, 300), ("chaser", 2, 19, 120, 300),
                                                    ("jumper", 0, 20, 100, 250), ("caveflyer", 0, 20, 100, 250),
                                                    ("jumper", 2, 45, 100, 250), ("caveflyer", 2, 45, 100, 250)])
def test_world_size_modes(game, mode, dim, max_ep, T, reference):
    """Distribution modes with their own world size = own instantiations (maze easy 15x15 / memory 31x31 with an agent-centred
    8x8 view: MazeT<MODE>; chaser hard 13x13 / extreme 19x19 with 5 enemies and 5 orbs: ChaserT<MODE>; jumper / caveflyer easy 20x20 and memory 45x45 with the unpruned cave), against the reference
    with its compile-time Config::mode set: tile maps + RNG after make, pixels / rewards / dones over truncated episodes."""
    from procgen2_b200.engine import BatchedEnv
    n, seed = 48, 8300 + mode
    rs = np.random.RandomState(mode)
    acts = rs.randint(0, 15, size=(T, n)).astype(np.int32)
    env = BatchedEnv(game, n, seed=seed, max_episode_steps=max_ep, distribution_mode=mode)
    refs = [reference.RefEnv(game, seed + i, mode=mode) for i in range(n)]
    tb, _, pe = env.read_field("tiles")
    tiles = tb.reshape(n, pe)
    for i, r in enumerate(refs):
        rt = r.tiles()
        w, h = rt.shape
        assert w == dim
        np.testing.assert_array_equal(tiles[i, :w * h].reshape(w, h), rt, err_msg="tile map after make, env %d" % i)
    env.reset()
    np.testing.assert_array_equal(env.fetch()[0], np.stack([r.reset() for r in refs]))
    age = np.zeros(n, np.int64)
    for t in range(T):
        env.step(acts[t])
        o, rw, d, _ = env.fetch()
        for i, r in enumerate(refs):
            oo, w, dd = r.step(acts[t, i])
            age[i] += 1
            if dd or age[i] >= max_ep:
                oo = r.reset(); age[i] = 0
            assert w == rw[i] and dd == d[i], (t, i)
            np.testing.assert_array_equal(o[i], oo, err_msg="step %d env %d" % (t, i))
    mt = env.read_field("mt")[0].view(np.uint32).reshape(n, 624)
    for i, r in enumerate(refs):
        np.testing.assert_array_equal(r.rng_state()[0], mt[i])
        r.close()
    assert not env.read_field("fault")[0].view(np.int32).any()
    env.close()

"""The rasteriser (pg2_render.cuh) against the written blit specification (oracle/raster.c) on synthetic scenes.

Every scene is drawn twice: by the production rasteriser for a synthetic game that copies one real game's render traits
(tests/raster/synth_game.cuh, drawn by tests/raster/harness.cu: the host-sim build here, the production kernels k_render /
k_render_human on the GPU), and by a plain reference that states render_game's painter's order with oracle/raster.c
(tests/raster/scene_ref.c). The frames must agree bit for bit. Each family of scenes drives one path of the rasteriser
and asserts from the per-frame report that it reached it.
"""
import ctypes
import os

import numpy as np
import pytest

from tests.raster import build as rbuild

# name: (harness index, MAX_POST, ROTATES, TILE_CLASSES, WIN_ROWS, HAS_TILES, STATIC_VIEW) -- the games' render traits
TRAITS = {
    "maze": (0, 4, False, 1, 28, True, True),
    "coinrun": (1, 192, False, 1, 16, True, False),
    "climber": (2, 48, False, 2, 23, True, False),
    "jumper": (3, 80, True, 2, 16, True, False),
    "bossfight": (4, 112, True, 1, 1, False, True),
    "caveflyer": (5, 112, True, 1, 11, True, False),
    "chaser2": (6, 208, False, 1, 22, True, True),
}
STATIC = [t for t, v in TRAITS.items() if v[6]]
TWO_CLASS = [t for t, v in TRAITS.items() if v[3] == 2]
TILED = [t for t, v in TRAITS.items() if v[5]]

MAX_CAND, MAP, NO_TILE, NUM_TEX = 320, 64, 255, 64
POST_DTYPE = np.dtype([("mode", "<i4"), ("tex", "<i4"), ("flip", "<i4"), ("pad", "<i4"), ("x", "<f4"), ("y", "<f4"),
                       ("w", "<f4"), ("h", "<f4"), ("scale", "<f4"), ("alpha", "<f4"), ("rotation", "<f4"), ("pad2", "<f4"),
                       ("angle", "<f8")])
SCENE_DTYPE = np.dtype([("cam_x", "<f4"), ("cam_y", "<f4"), ("cam_scale", "<f4"), ("bg_tex", "<i4"), ("bg_x", "<f4"),
                        ("bg_y", "<f4"), ("bg_scale", "<f4"), ("map_x0", "<i4"), ("map_y0", "<i4"), ("outside", "<i4"),
                        ("npost", "<i4"), ("pad", "<i4"), ("map", "u1", (MAP * MAP,)), ("post", POST_DTYPE, (MAX_CAND,))])
TEX_DTYPE = np.dtype([("offset", "<u4"), ("w", "<u2"), ("h", "<u2"), ("blend", "<u4")])
REPORT = ["wide", "npost", "reuse", "overflow", "fault", "slow", "quads", "quads_slow", "rb", "ambiguous", "rotated", "pre_blend",
          "bg_holes"]

# frames per trait set and family: the GPU draws GPU_SCALE times as many
CPU_FRAMES = {"game": 120, "two_classes": 80, "wide": 40, "background": 60, "post": 40}
GPU_SCALE = 10
HUMAN_WINDOWS = [(1, 1), (63, 65), (200, 200), (512, 512), (1000, 37), (64, 4096)]


# ---- libraries --------------------------------------------------------------------------------------------------------

_libs = {}


def _harness(kind):
    if kind not in _libs:
        path = rbuild.build_gpu() if kind == "gpu" else rbuild.build_host()
        L = ctypes.CDLL(path)
        assert L.rh_scene_bytes() == SCENE_DTYPE.itemsize and L.rh_report_words() == len(REPORT)
        L.rh_render.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                ctypes.c_long, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.rh_render_human.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_long,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        _libs[kind] = L
    return _libs[kind]


def _ref_lib():
    if "ref" not in _libs:
        L = ctypes.CDLL(rbuild.build_ref())
        L.scene_ref_render.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        _libs["ref"] = L
    return _libs["ref"]


class Textures:
    """64 synthetic textures in one atlas laid out as assets.cpp lays it out (atlas[0] = opaque black). Ids 0..15: tile
    shape class 0 (cls0 = (w, h)), 16..31: class 1, 32..39: backgrounds, 40..63: sprites. Opaque-copy textures store
    A = 255; alpha textures mix opaque, fully transparent and translucent texels."""

    def __init__(self, rng, cls0=(16, 16), cls1=(16, 16), tile_alpha=0.25, opaque_alpha_p=0.7):
        self.info = np.zeros(NUM_TEX, TEX_DTYPE)
        words = [np.array([0xff000000], np.uint32)]
        off = 1
        sprite_sizes = [(1, 1), (2, 3), (7, 5), (8, 8), (16, 16), (13, 21), (32, 24), (48, 40), (64, 64), (5, 64), (70, 9), (33, 33)]
        for t in range(NUM_TEX):
            if t < 32:
                w, h = cls0 if t < 16 else cls1
                blend = rng.random() < tile_alpha
            elif t < 40:
                w, h = [(96, 64), (64, 64), (200, 120), (40, 30), (128, 96), (301, 77), (64, 48), (17, 64)][t - 32]
                blend = t in (33, 35, 37)
            else:
                w, h = sprite_sizes[(t - 40) % len(sprite_sizes)]
                blend = t < 58
            rgb = rng.integers(0, 256, size=(h * w, 3), dtype=np.uint32)
            if blend:
                kind = rng.random(h * w)
                a = np.where(kind < opaque_alpha_p * 0.6, 255, np.where(kind < opaque_alpha_p, 0, rng.integers(1, 255, h * w)))
            else:
                a = np.full(h * w, 255)
            words.append((rgb[:, 0] | rgb[:, 1] << 8 | rgb[:, 2] << 16 | a.astype(np.uint32) << 24).astype(np.uint32))
            self.info[t] = (off, w, h, 1 if blend else 0)
            off += w * h
        self.atlas = np.concatenate(words)

    def wh(self, t):
        return int(self.info[t]["w"]), int(self.info[t]["h"])


# ---- drawing ----------------------------------------------------------------------------------------------------------

def render(kind, trait, scenes, tx, grid=0):
    """scenes: [npass, nenv] -> frames [npass, nenv, 64, 64, 3], reports [npass, nenv, len(REPORT)]"""
    scenes = np.ascontiguousarray(scenes, SCENE_DTYPE)
    npass, nenv = scenes.shape
    obs = np.zeros((npass, nenv, 64, 64, 3), np.uint8)
    rep = np.zeros((npass, nenv, len(REPORT)), np.int32)
    rc = _harness(kind).rh_render(TRAITS[trait][0], npass, nenv, scenes.ctypes.data, tx.info.ctypes.data, NUM_TEX, tx.atlas.ctypes.data,
                                  tx.atlas.size, grid, obs.ctypes.data, rep.ctypes.data)
    assert rc == 0, "harness failed (%s)" % kind
    return obs, rep


def render_human(kind, trait, scene, tx, width, height, grid=7):
    scene = np.ascontiguousarray(np.array(scene, SCENE_DTYPE).reshape(()))
    out = np.zeros((height, width, 3), np.uint8)
    rep = np.zeros(len(REPORT), np.int32)
    rc = _harness(kind).rh_render_human(TRAITS[trait][0], scene.ctypes.data, tx.info.ctypes.data, NUM_TEX, tx.atlas.ctypes.data,
                                        tx.atlas.size, width, height, grid, out.ctypes.data, rep.ctypes.data)
    assert rc == 0, "harness failed (%s)" % kind
    return out, rep


def reference(trait, scene, tx, width=64, height=64):
    scene = np.ascontiguousarray(np.array(scene, SCENE_DTYPE).reshape(()))
    out = np.zeros((height, width, 3), np.uint8)
    nclass = TRAITS[trait][3] if TRAITS[trait][5] else 0
    _ref_lib().scene_ref_render(scene.ctypes.data, tx.info.ctypes.data, tx.atlas.ctypes.data, nclass, width, height, out.ctypes.data)
    return out


def check_frame(got, want, family, trait, seed, frame, report, scene, tx, tmp_path):
    if np.array_equal(got, want):
        return
    ys, xs = np.nonzero(np.any(got != want, axis=2))
    y, x = int(ys[0]), int(xs[0])
    path = os.path.join(str(tmp_path), "scene_%s_%s_%d_%d.npz" % (family, trait, seed, frame))
    np.savez(path, scene=np.array(scene, SCENE_DTYPE), tex_info=tx.info, atlas=tx.atlas)
    flags = ", ".join("%s=%d" % (k, v) for k, v in zip(REPORT, report))
    pytest.fail("%s/%s seed %d frame %d: %d pixels differ, first (x=%d, y=%d) got %s want %s [%s]; scene saved to %s" % (
        family, trait, seed, frame, len(ys), x, y, tuple(got[y, x]), tuple(want[y, x]), flags, path))


def check_all(family, trait, seed, scenes, frames, reports, tx, tmp_path):
    npass, nenv = scenes.shape
    for p in range(npass):
        for e in range(nenv):
            assert reports[p, e, REPORT.index("overflow")] == 0, "%s/%s seed %d: tile window taller than WIN_ROWS" % (family, trait, seed)
            check_frame(frames[p, e], reference(trait, scenes[p, e], tx), family, trait, seed, p * nenv + e, reports[p, e], scenes[p, e], tx, tmp_path)


# ---- scene families ---------------------------------------------------------------------------------------------------

def min_cam_scale(trait):
    """Smallest camera scale whose tile window fits the trait's frame tables (WIN_ROWS rows, MAX_WIN = 32 columns)."""
    winr = TRAITS[trait][4]
    return max(4.0 / (winr - 2.5), 4.0 / 29.0) if TRAITS[trait][5] else 0.1


def new_scenes(n):
    s = np.zeros(n, SCENE_DTYPE)
    s["outside"] = NO_TILE
    s["map"] = NO_TILE
    return s


def base(rng, s, trait, tx, cs=None, density=0.35, classes=(0,), bg_tex=None, bg_cover=(0.6, 1.6)):
    """Camera, background and tile map of one scene."""
    cs = float(rng.uniform(min_cam_scale(trait), 1.6)) if cs is None else cs
    s["cam_scale"] = cs
    s["cam_x"] = rng.uniform(-200, 600)
    s["cam_y"] = rng.uniform(-200, 600)
    half = 32.0 / cs
    bt = int(rng.choice([32, 33, 34, 35, 36, 37, 38, 39])) if bg_tex is None else bg_tex
    bw, bh = tx.wh(bt)
    width = rng.uniform(*bg_cover) * 64.0          # on-screen width of the background in pixels
    s["bg_tex"] = bt
    s["bg_scale"] = width / (bw * cs)
    s["bg_x"] = s["cam_x"] - half - rng.uniform(-0.3, 0.5) * width / cs
    s["bg_y"] = s["cam_y"] - half - rng.uniform(-0.3, 0.5) * (bh * s["bg_scale"]) * cs / cs
    s["map_x0"] = int(np.floor(s["cam_x"] / 16.0)) - MAP // 2
    s["map_y0"] = int(np.floor(s["cam_y"] / 16.0)) - MAP // 2
    if TRAITS[trait][5]:
        ids = np.concatenate([np.arange(16) + 16 * c for c in classes if c < TRAITS[trait][3]])
        cells = rng.choice(ids, size=MAP * MAP).astype(np.uint8)
        s["map"] = np.where(rng.random(MAP * MAP) < density, cells, NO_TILE)
        s["outside"] = int(rng.choice([NO_TILE, ids[0]]))
    return cs


def sprite(rng, p, trait, s, tx, rotate_p=0.3, rect_p=0.15):
    """One post-blit request near the camera: a sprite with alpha-mod and flip, a rotated sprite or a screen rect."""
    cs = float(s["cam_scale"])
    t = int(rng.integers(40, 64))
    w, h = tx.wh(t)
    rot = TRAITS[trait][2]
    r = rng.random()
    if r < rect_p:
        p["mode"], p["tex"] = 3, t
        p["x"], p["y"] = rng.uniform(-20, 70), rng.uniform(-20, 70)
        p["w"], p["h"] = rng.uniform(0.5, 40), rng.uniform(0.5, 40)
        p["angle"] = float(rng.choice([0.0, 90.0, -90.0, 180.0, rng.uniform(-360, 360)])) if rot else 0.0
        return
    size = rng.uniform(1.0, 40.0)                 # on-screen pixels
    p["tex"] = t
    p["x"] = s["cam_x"] + rng.uniform(-44, 44) / cs
    p["y"] = s["cam_y"] + rng.uniform(-44, 44) / cs
    p["scale"] = size / (w * cs)
    p["alpha"] = 1.0 if rng.random() < 0.6 else rng.uniform(0.0, 1.0)
    if rot and r < rect_p + rotate_p:
        p["mode"] = 2
        p["rotation"] = float(rng.choice([0.0, np.pi / 2, -np.pi / 2, np.pi, rng.uniform(-7, 7)]))
    else:
        p["mode"], p["flip"] = 1, int(rng.random() < 0.4)


def posts(rng, s, trait, tx, n):
    s["npost"] = n
    for k in range(n):
        sprite(rng, s["post"][k], trait, s, tx)


def fam_game(trait, rng, n):
    tx = Textures(rng)
    sc = new_scenes(n)
    for i in range(n):
        base(rng, sc[i], trait, tx, classes=(0, 1))
        posts(rng, sc[i], trait, tx, int(rng.integers(0, min(TRAITS[trait][1], 40) + 1)))
    return tx, sc


def fam_two_classes(trait, rng, n):
    # 64x64 and 64x53 tile classes side by side, translucent and transparent tile texels
    tx = Textures(rng, cls0=(64, 64), cls1=(64, 53), tile_alpha=0.5)
    sc = new_scenes(n)
    for i in range(n):
        base(rng, sc[i], trait, tx, density=0.7, classes=(0, 1))
        posts(rng, sc[i], trait, tx, int(rng.integers(0, 4)))
    return tx, sc


def fam_wide(trait, rng, n):
    # tile textures whose samples overflow the candidate slots (sx > 255, sy * w > 65535), zoomed-out cameras
    tx = Textures(rng, cls0=(512, 160), cls1=(300, 240), tile_alpha=0.3)
    sc = new_scenes(n)
    for i in range(n):
        cs = min_cam_scale(trait) * (1.0 if i % 2 else rng.uniform(1.0, 3.0))
        base(rng, sc[i], trait, tx, cs=cs, density=0.8, classes=(0, 1))
        posts(rng, sc[i], trait, tx, int(rng.integers(0, min(TRAITS[trait][1], 6) + 1)))
    return tx, sc


def fam_background(trait, rng, n):
    # backgrounds with alpha, backgrounds that leave uncovered rows / columns or lie partly off screen, sparse tiles
    tx = Textures(rng, tile_alpha=0.5)
    sc = new_scenes(n)
    for i in range(n):
        base(rng, sc[i], trait, tx, density=0.1, bg_tex=int(rng.choice([33, 35, 37, 32, 34])), bg_cover=(0.2, 1.2))
        posts(rng, sc[i], trait, tx, int(rng.integers(0, 3)))
    return tx, sc


def fam_post(trait, rng, n):
    """Rotations at 0, +-90, 180 and arbitrary angles; 1-px, zero-size, negative-origin, fractional and huge rects; more
    than 128 candidates with invisible ones interleaved; exactly MAX_POST visible. Returns the visible count expected."""
    maxp, rot = TRAITS[trait][1], TRAITS[trait][2]
    tx = Textures(rng)
    sc = new_scenes(n)
    expect = np.full(n, -1)
    for i in range(n):
        s = sc[i]
        base(rng, s, trait, tx)
        kind = i % 4
        if kind == 0:   # exactly MAX_POST visible among > 128 candidates (mode 0 and zero-size rects interleaved)
            ncand = min(MAX_CAND, max(150, maxp + 100))
            vis = np.sort(rng.choice(ncand, size=maxp, replace=False))
            for k in range(ncand):
                p = s["post"][k]
                if k in vis:
                    p["mode"], p["tex"] = 3, int(rng.integers(40, 64))
                    p["x"], p["y"], p["w"], p["h"] = rng.uniform(0, 50), rng.uniform(0, 50), rng.uniform(1, 12), rng.uniform(1, 12)
                    p["angle"] = float(rng.choice([0.0, 90.0, 33.5])) if rot else 0.0
                elif k % 2:
                    p["mode"], p["tex"], p["x"], p["y"], p["w"], p["h"] = 3, 40, 10.0, 10.0, 0.0, 5.0
            s["npost"] = ncand
            expect[i] = maxp
        else:           # edge rects and rotations, and blits larger than the 16-bit destination range
            m = min(maxp, 24)
            s["npost"] = m
            for k in range(m):
                p = s["post"][k]
                t = int(rng.integers(40, 64))
                p["tex"] = t
                c = int(rng.integers(0, 8))
                if c == 0:
                    p["mode"], p["x"], p["y"], p["w"], p["h"] = 3, rng.integers(-2, 66), rng.integers(-2, 66), 1.0, 1.0
                elif c == 1:
                    p["mode"], p["x"], p["y"], p["w"], p["h"] = 3, rng.uniform(0, 64), rng.uniform(0, 64), float(rng.choice([0.0, 0.99])), 5.0
                elif c == 2:
                    p["mode"], p["x"], p["y"], p["w"], p["h"] = 3, -rng.uniform(0, 30), -rng.uniform(0, 30), rng.uniform(1, 60), rng.uniform(1, 60)
                elif c == 3:
                    p["mode"], p["x"], p["y"], p["w"], p["h"] = 3, rng.uniform(-3, 60) + 0.37, rng.uniform(-3, 60) + 0.71, rng.uniform(0.2, 9.5), rng.uniform(0.2, 9.5)
                elif c == 4:   # huge: starts far left / above, ends on screen (rotated about its centre where the traits rotate)
                    p["mode"], p["x"], p["w"] = 3, -float(rng.integers(33000, 70000)), 0.0
                    p["w"] = -p["x"] + rng.uniform(10, 100)
                    p["y"], p["h"] = rng.uniform(-10, 40), rng.uniform(3, 30)
                    if rng.random() < 0.5:
                        p["x"], p["y"], p["w"], p["h"] = p["y"], p["x"], p["h"], p["w"]
                    if rot and rng.random() < 0.6:
                        p["angle"] = float(rng.choice([90.0, -90.0, 180.0, 30.0, 0.01, rng.uniform(-360, 360)]))
                        if rng.random() < 0.5:   # centred on the screen, so that the rotated rect crosses it
                            p["x"], p["y"] = 32.0 - p["w"] / 2 + rng.uniform(-5, 5), 32.0 - p["h"] / 2 + rng.uniform(-5, 5)
                elif c == 5:   # huge sprite through render_texture
                    w, h = tx.wh(t)
                    p["mode"], p["scale"] = 1, float(rng.uniform(70000, 200000)) / (w * float(s["cam_scale"]))
                    p["x"] = s["cam_x"] - rng.uniform(0.2, 0.8) * w * p["scale"]
                    p["y"] = s["cam_y"] - rng.uniform(0.0, 0.05) * h * p["scale"]
                    p["flip"] = int(rng.random() < 0.5)
                    p["alpha"] = 1.0 if rng.random() < 0.5 else 0.6
                else:
                    sprite(rng, p, trait, s, tx, rotate_p=0.8, rect_p=0.1)
                    if p["mode"] == 3 and rot:
                        p["angle"] = float(rng.choice([0.0, 90.0, -90.0, 180.0, 270.0, rng.uniform(-720, 720)]))
    return tx, sc, expect


FAMILIES = {"game": fam_game, "two_classes": fam_two_classes, "wide": fam_wide, "background": fam_background, "post": fam_post}


def family_cases():
    out = []
    for fam in FAMILIES:
        for trait in TRAITS:
            if fam in ("two_classes",) and trait not in TWO_CLASS:
                continue
            if fam == "wide" and trait not in TILED:
                continue
            out.append((fam, trait))
    return out


def run_family(kind, fam, trait, seed, n, tmp_path, grid=0):
    rng = np.random.default_rng(seed)
    made = FAMILIES[fam](trait, rng, n)
    tx, sc = made[0], made[1]
    frames, rep = render(kind, trait, sc[None, :], tx, grid)
    check_all(fam, trait, seed, sc[None, :], frames, rep, tx, tmp_path)
    if fam == "post":
        sel = made[2] >= 0
        assert np.array_equal(rep[0, sel, REPORT.index("npost")], made[2][sel]), "post/%s seed %d: visible post blits miscounted" % (trait, seed)
        assert sc["npost"].max() > 128
    # coverage, from the host-sim build's report: the GPU build draws the same scenes from the same source, and only the
    # host build can look into the frame (RC_AMBIGUOUS cells, slow-path counters, rotated blits, background holes)
    cov = rep if kind == "host" else render("host", trait, sc[None, :], tx)[1]
    col = {k: cov[0, :, i] for i, k in enumerate(REPORT)}
    rot = TRAITS[trait][2]
    if fam == "game":
        assert col["quads"].sum() > 0 and col["npost"].max() > 0
        assert not rot or col["rotated"].sum() > 0, "no rotated post blit was drawn"
    elif fam == "two_classes":
        assert col["ambiguous"].sum() > 0, "no RC_AMBIGUOUS cell"
        assert col["rb"].sum() > 0, "no screen row with a second covering tile row"
        assert col["slow"].sum() > 0
    elif fam == "wide":
        assert col["wide"].mean() >= 0.5, "the wide path was reached by %d of %d frames" % (col["wide"].sum(), n)
        assert rep[0, :, REPORT.index("wide")].sum() > 0
    elif fam == "post":
        assert not rot or col["rotated"].sum() > 0, "no rotated post blit was drawn"
    elif fam == "background":
        assert col["slow"].sum() > 0
        assert col["pre_blend"].sum() > 0, "no background with alpha"
        assert col["bg_holes"].sum() > 0, "no screen row or column the background leaves uncovered"
    return rep


def cache_scenes(trait, rng, nenv, tx):
    """4 passes: the same base image with new posts (reuse), then half of the envs change their base (draw + store)."""
    sc = new_scenes(4 * nenv).reshape(4, nenv)
    for e in range(nenv):
        base(rng, sc[0, e], trait, tx, classes=(0, 1))
        for p in range(1, 4):
            sc[p, e] = sc[p - 1, e]
            if p == 2 and e % 2 == 0:
                base(rng, sc[p, e], trait, tx, classes=(0, 1))
        for p in range(4):
            posts(rng, sc[p, e], trait, tx, int(rng.integers(0, min(TRAITS[trait][1], 12) + 1)))
    return sc


def run_cache(kind, trait, seed, nenv, tmp_path, grid):
    rng = np.random.default_rng(seed)
    for wide in (False, True):
        if wide and not TRAITS[trait][5]:
            continue
        tx = Textures(rng, cls0=(512, 160), cls1=(300, 240)) if wide else Textures(rng)
        sc = cache_scenes(trait, rng, nenv, tx)
        frames, rep = render(kind, trait, sc, tx, grid)
        check_all("cache" + ("_wide" if wide else ""), trait, seed, sc, frames, rep, tx, tmp_path)
        reuse, w = rep[:, :, REPORT.index("reuse")], rep[:, :, REPORT.index("wide")]
        assert reuse[0].sum() == 0
        # a frame reuses the cached base image exactly when its base is unchanged and the previous frame was cacheable
        for p in range(1, 4):
            for e in range(nenv):
                same = p != 2 or e % 2 == 1
                assert reuse[p, e] == int(same and not w[p - 1, e] or (same and reuse[p - 1, e] == 1)), \
                    "cache/%s seed %d pass %d env %d: reuse %d (wide %s)" % (trait, seed, p, e, reuse[p, e], w[:, e])
        if not wide:
            assert reuse[1:].sum() > 0
        else:
            assert w[0].sum() > 0


def run_human(kind, trait, seed, tmp_path, windows=HUMAN_WINDOWS):
    rng = np.random.default_rng(seed)
    tx = Textures(rng)
    for j, (W, H) in enumerate(windows):
        sc = new_scenes(1)
        base(rng, sc[0], trait, tx, classes=(0, 1))
        posts(rng, sc[0], trait, tx, int(rng.integers(0, min(TRAITS[trait][1], 24) + 1)))
        out, rep = render_human(kind, trait, sc[0], tx, W, H)
        # the tile window of a tall frame can exceed the frame tables: then the frame must be reported incomplete
        if rep[REPORT.index("overflow")]:
            assert TRAITS[trait][5] and H > W, "human/%s %dx%d: unexpected overflow" % (trait, W, H)
            continue
        assert not (TRAITS[trait][5] and H >= 4 * W and H > 1000), "human/%s %dx%d: a window taller than the tables drew silently" % (trait, W, H)
        check_frame(out, reference(trait, sc[0], tx, W, H), "human_%dx%d" % (W, H), trait, seed, j, rep, sc[0], tx, tmp_path)


# ---- CPU tests (host-sim build of the same rasteriser) ----------------------------------------------------------------

@pytest.mark.parametrize("fam,trait", family_cases())
def test_family_host(fam, trait, tmp_path):
    run_family("host", fam, trait, 1000 + sorted(TRAITS).index(trait), CPU_FRAMES[fam], tmp_path)


@pytest.mark.parametrize("trait", STATIC)
def test_cache_host(trait, tmp_path):
    run_cache("host", trait, 2000 + sorted(TRAITS).index(trait), 12, tmp_path, 0)


@pytest.mark.parametrize("trait", sorted(TRAITS))
def test_human_host(trait, tmp_path):
    run_human("host", trait, 3000 + sorted(TRAITS).index(trait), tmp_path, [w for w in HUMAN_WINDOWS if w[0] * w[1] <= 64 * 4096])


def test_make_fast_huge_rect_host(tmp_path):
    """A 40 100-pixel rect starting at x = -40 000 covers the screen: the spec draws texels 40 000 .. 40 063 of it."""
    rng = np.random.default_rng(5)
    tx = Textures(rng)
    sc = new_scenes(1)
    base(rng, sc[0], "coinrun", tx)
    p = sc[0]["post"][0]
    p["mode"], p["tex"], p["x"], p["y"], p["w"], p["h"] = 3, 44, -40000.0, 8.0, 40100.0, 20.0
    sc[0]["npost"] = 1
    frames, rep = render("host", "coinrun", sc[None, :], tx)
    assert rep[0, 0, REPORT.index("npost")] == 1
    check_frame(frames[0, 0], reference("coinrun", sc[0], tx), "huge_rect", "coinrun", 5, 0, rep[0, 0], sc[0], tx, tmp_path)


# ---- GPU tests (the production kernels) -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("grid", [1, 0], ids=["one_cta", "occupancy"])
@pytest.mark.parametrize("fam,trait", family_cases())
def test_family_gpu(fam, trait, grid, tmp_path):
    run_family("gpu", fam, trait, 4000 + sorted(TRAITS).index(trait) + 100 * grid, CPU_FRAMES[fam] * (GPU_SCALE if grid == 0 else 2), tmp_path, grid)


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [1, 0], ids=["one_cta", "occupancy"])
@pytest.mark.parametrize("trait", STATIC)
def test_cache_gpu(trait, grid, tmp_path):
    run_cache("gpu", trait, 5000 + sorted(TRAITS).index(trait) + 100 * grid, 48 if grid else 400, tmp_path, grid)


@pytest.mark.gpu
@pytest.mark.parametrize("trait", sorted(TRAITS))
def test_human_gpu(trait, tmp_path):
    run_human("gpu", trait, 6000 + sorted(TRAITS).index(trait), tmp_path)


@pytest.mark.gpu
def test_render_human_rejects_what_it_cannot_draw():
    """pg2_render_human fails for a window whose tile rows exceed the frame tables, and for one wider than the 16-bit
    blit coordinates, instead of returning a silently wrong frame."""
    from procgen2_b200.engine import BatchedEnv, load_library
    L = load_library()
    L.pg2_render_human.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
    L.pg2_render_human.restype = ctypes.c_int32
    env = BatchedEnv("maze", 1, seed=3, device=0)
    try:
        env.reset()
        for (W, H), ok in (((64, 64), True), ((512, 512), True), ((64, 4096), False), ((66000, 4), False)):
            out = np.zeros((H, W, 3), np.uint8)
            rc = L.pg2_render_human(env._h, 0, W, H, out.ctypes.data_as(ctypes.c_void_p))
            assert (rc == 0) == ok, "%dx%d: rc %d" % (W, H, rc)
    finally:
        env.close()

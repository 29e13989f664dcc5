"""Every entry of the packed asset blob against the texels its source PNG decodes to, through (1) a plain Python reader
of the blob layout, (2) the PRODUCT's loader (assets.cpp via pg2_load_texture_host: the texels the engine uploads into
its device atlas), (3) the oracle's loader (oracle/assets_blob.cpp: the texels the reference games get from IMG_Load in
the stand-in). A packer or loader bug would otherwise be invisible: oracle and engine both read the same blob.

The PNGs themselves belong to the reference, not to this repository: tests/golden/assets_texels.json holds, per
texture, its size, whether it is alpha-blended, and the CRC32 of its RGBA texels (A = 255 for an opaque texture) by
the rule SDL_image + SDL_CreateTextureFromSurface follow: RGBA / LA / palette + tRNS = alpha-blended texture; RGB /
opaque palette = opaque copy. They were recorded from the blob after it had been checked bit for bit against every
PNG decoded independently with PIL."""
import ctypes
import json
import os
import struct
import subprocess
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOB = os.path.join(ROOT, "procgen2_b200", "data", "assets.bin")
TEXELS = os.path.join(ROOT, "tests", "golden", "assets_texels.json")


def blob_entries():
    with open(BLOB, "rb") as f:
        assert f.read(8) == b"PG2ASSET"
        ver, n = struct.unpack("<II", f.read(8))
        assert ver == 1
        out = []
        for _ in range(n):
            raw = f.read(152)
            name = raw[:120].split(b"\0", 1)[0].decode()
            w, h, ch, _, off, zs = struct.unpack("<IIIIQQ", raw[120:])
            out.append((name, w, h, ch, off, zs))
    return out


def recorded():
    """name -> (width, height, has_alpha, CRC32 of the RGBA texels)."""
    return {k: tuple(v) for k, v in json.load(open(TEXELS)).items()}


def rgba_crc(texels, has_alpha):
    a = np.array(texels, np.uint8)
    if not has_alpha:
        a[..., 3] = 255
    return zlib.crc32(a.tobytes()) & 0xffffffff


def test_blob_covers_every_texture_the_games_name():
    """Every texture name the engine asks for is in the blob (and the blob holds no duplicates)."""
    names = [e[0] for e in blob_entries()]
    assert len(names) == len(set(names)) and len(names) >= 200
    assert sorted(names) == sorted(recorded())


def test_blob_texels_equal_the_pngs():
    data = open(BLOB, "rb").read()
    want = recorded()
    for name, w, h, ch, off, zs in blob_entries():
        ww, wh, has_alpha, crc = want[name]
        assert (w, h) == (ww, wh), name
        assert ch == (4 if has_alpha else 3), name
        raw = np.frombuffer(zlib.decompress(data[off:off + zs]), np.uint8).reshape(h, w, ch)
        rgba = np.full((h, w, 4), 255, np.uint8)
        rgba[..., :ch] = raw
        assert rgba_crc(rgba, has_alpha) == crc, name


def test_product_loader_equals_the_pngs():
    from procgen2_b200 import build
    build.build()
    L = ctypes.CDLL(build.ENGINE)
    L.pg2_load_texture_host.restype = ctypes.c_int64
    L.pg2_load_texture_host.argtypes = [ctypes.c_char_p, ctypes.c_char_p] + [ctypes.POINTER(ctypes.c_int32)] * 3 + [ctypes.c_void_p, ctypes.c_int64]
    want = recorded()
    for name, w, h, ch, _, _ in blob_entries():
        _, _, has_alpha, crc = want[name]
        cw, chh, cb = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        out = np.empty(w * h, np.uint32)
        n = L.pg2_load_texture_host(BLOB.encode(), name.encode(), ctypes.byref(cw), ctypes.byref(chh), ctypes.byref(cb), out.ctypes.data, out.size)
        assert n == w * h and (cw.value, chh.value) == (w, h) and cb.value == has_alpha, name
        assert zlib.crc32(out.view(np.uint8).tobytes()) & 0xffffffff == crc, name
    assert L.pg2_load_texture_host(BLOB.encode(), b"assets/does/not/exist.png", None, None, None, None, 0) < 0


def test_oracle_loader_equals_the_pngs(tmp_path):
    lib = str(tmp_path / "libpg2o_assets.so")   # flags of oracle/build_ref.py
    subprocess.check_call(["g++", "-std=gnu++14", "-O2", "-fPIC", "-shared", os.path.join(ROOT, "oracle", "assets_blob.cpp"), "-lz", "-o", lib])
    L = ctypes.CDLL(lib)
    L.pg2o_blob_load.restype = ctypes.POINTER(ctypes.c_uint8)
    L.pg2o_blob_load.argtypes = [ctypes.c_char_p, ctypes.c_char_p] + [ctypes.POINTER(ctypes.c_int)] * 3
    want = recorded()
    for name, w, h, ch, _, _ in blob_entries():
        _, _, has_alpha, crc = want[name]
        cw, chh, ca = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        p = L.pg2o_blob_load(BLOB.encode(), name.encode(), ctypes.byref(cw), ctypes.byref(chh), ctypes.byref(ca))
        assert p and (cw.value, chh.value) == (w, h) and bool(ca.value) == bool(has_alpha), name
        # an opaque texture's alpha channel is not compared, as the games never read it
        assert rgba_crc(np.ctypeslib.as_array(p, shape=(h, w, 4)), has_alpha) == crc, name

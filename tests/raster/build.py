"""TEST INFRASTRUCTURE. Builds the rasteriser test harness (harness.cu) and the plain scene reference (scene_ref.c)
into tests/raster/_build/:
    libraster_host.so   g++ -DPG2_HOSTSIM build of the harness (runs without a GPU)
    libraster_gpu.so    nvcc build for sm_100a with the engine's flags (procgen2_b200.build.NVCC_FLAGS)
    libscene_ref.so     gcc -O2 -ffp-contract=off: scene_ref.c + the unchanged oracle/raster.c
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "_build")
CSRC = os.path.join(ROOT, "procgen2_b200", "csrc")


def _deps():
    out = [os.path.join(HERE, f) for f in ("harness.cu", "synth_game.cuh", "scene.h")]
    for d, _, files in os.walk(CSRC):
        out += [os.path.join(d, f) for f in files if f.endswith((".cuh", ".h"))]
    return out


def _build(target, deps, cmd):
    os.makedirs(OUT, exist_ok=True)
    if os.path.exists(target) and all(os.path.getmtime(d) <= os.path.getmtime(target) for d in deps):
        return target
    tmp = target + ".tmp%d" % os.getpid()
    subprocess.check_call(cmd + ["-o", tmp])
    os.replace(tmp, target)
    return target


def build_ref():
    src = [os.path.join(HERE, "scene_ref.c"), os.path.join(ROOT, "oracle", "raster.c")]
    return _build(os.path.join(OUT, "libscene_ref.so"), src + [os.path.join(HERE, "scene.h"), os.path.join(ROOT, "oracle", "raster.h")],
                  ["gcc", "-std=c99", "-O2", "-ffp-contract=off", "-fPIC", "-shared"] + src + ["-lm"])


def build_host():
    return _build(os.path.join(OUT, "libraster_host.so"), _deps(),
                  ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-DPG2_HOSTSIM", "-x", "c++",
                   os.path.join(HERE, "harness.cu")])


def build_gpu():
    sys.path.insert(0, ROOT)
    from procgen2_b200.build import NVCC_FLAGS
    return _build(os.path.join(OUT, "libraster_gpu.so"), _deps(),
                  ["nvcc"] + NVCC_FLAGS + ["-shared", os.path.join(HERE, "harness.cu")])


def build():
    return build_ref(), build_host(), build_gpu()


if __name__ == "__main__":
    print(build())

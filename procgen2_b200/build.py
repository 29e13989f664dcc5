"""In-tree build of the CUDA engine and the per-game cenv drop-in libraries (sm_100a only).

    python -m procgen2_b200.build [--force]

Outputs (git-ignored, travel to the GPU box with the working tree):
    procgen2_b200/lib/libprocgen2_b200.so     engine: kernels + pg2_* C ABI (include/pg2_engine.h)
    procgen2_b200/lib/lib<Game>.so            cenv ABI (include/cenv.h) for one game each, same file
                                              names as the reference's CMake targets

Float semantics: -fmad=false (no FMA contraction, like the reference's x86-64 baseline build,
SURVEY Q14), default IEEE division / sqrt, no fast-math, denormals kept.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib")
ENGINE = os.path.join(LIB, "libprocgen2_b200.so")

GAME_LIBS = {
    "maze": "Maze", "coinrun": "CoinRun", "bossfight": "BossFight", "chaser": "Chaser",
    "climber": "Climber", "caveflyer": "CaveFlyer", "jumper": "Jumper",
}

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off", "--expt-relaxed-constexpr",
]


def _sources():
    out = []
    for d, _, files in os.walk(CSRC):
        for f in files:
            if f.endswith((".cu", ".cuh", ".cpp", ".h")):
                out.append(os.path.join(d, f))
    out.append(os.path.join(ROOT, "include", "pg2_engine.h"))
    out.append(os.path.join(ROOT, "include", "cenv.h"))
    return out


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def game_lib_path(game):
    return os.path.join(LIB, "lib%s.so" % GAME_LIBS[game])


def build(force=False, verbose=False, ptxas_info=False):
    os.makedirs(LIB, exist_ok=True)
    deps = _sources()
    if force or _stale(ENGINE, deps):
        cmd = ["nvcc"] + NVCC_FLAGS + os.environ.get("PG2_NVCC_EXTRA", "").split() + (["-Xptxas", "-v"] if ptxas_info else []) + [
            "-shared", os.path.join(CSRC, "engine.cu"), os.path.join(CSRC, "engine_final.cu"), os.path.join(CSRC, "assets.cpp"),
            "-lz", "-ldl", "-o", ENGINE]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    abi = os.path.join(CSRC, "cenv_abi.cpp")
    if os.path.exists(abi):
        for game in GAME_LIBS:
            out = game_lib_path(game)
            if force or _stale(out, [abi, ENGINE, os.path.join(ROOT, "include", "cenv.h")]):
                cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-fvisibility=hidden",
                       '-DPG2_GAME="%s"' % game, "-I" + os.path.join(ROOT, "include"), abi,
                       "-L" + LIB, "-lprocgen2_b200", "-Wl,-rpath,$ORIGIN", "-o", out]
                if verbose:
                    print(" ".join(cmd))
                subprocess.check_call(cmd)
    return ENGINE


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True, ptxas_info="--ptxas" in sys.argv)
    print("ok")

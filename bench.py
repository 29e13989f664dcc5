#!/usr/bin/env python
"""Benchmark of the hot path: env-steps/s including the 64x64x3 render (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # reference C++ engine (oracle/_ref) on the host cores
    python bench.py --game coinrun --envs-per-gpu 32768 [--max-episode-steps 32]   # one explicit workload

Default (no --game): ONE JSON line that carries every single-GPU BASELINE.json config.
  headline  configs[2] bossfight, 16 384 envs per GPU — the largest single-GPU configuration (the metric is not quoted on
            one config): `value`, `ms_per_step`, `roofline`, `e2e`, `cpu_baseline` describe it;
  configs   [...] the same measurements for configs[0] (maze, 256 envs) and configs[1] (coinrun, 4 096 envs); under
            --gpus N > 1 additionally the per-GPU slices of configs[3] (each of the seven games, 32 768 / N envs per GPU)
            and configs[4] (coinrun, 32 768 envs per GPU, 32-step episodes).
A "step" is one cenv_step of every env of the batch (auto-reset with per-episode level regeneration on device). Weak
scaling for the headline: every rank owns `envs_per_gpu` envs (a contiguous slice of the global env index space, seeds
= base + global index), no collective on the step path.

Per workload:
  burn-in   BURN_IN untimed steps first, so that the episode phases of the envs are staggered and the timed window
            contains steady-state resets (`resets_per_step` is measured over the timed steps);
  value     device-resident throughput: actions already in HBM, observations stay in HBM; every step = ONE CUDA-graph
            launch, timed with CUDA events on the engine's stream, an L2 flush (256 MiB memset) between steps, outside the
            event pairs; `back_to_back` = the same steps without the flushes, one event pair around all of them (also
            covers asynchronous level generation that the flush gaps would otherwise hide);
  kernel_ms_per_step  a separate profiled pass (eager launches, CUDA events around each kernel) — not part of `value`;
  e2e       the same metric with HOST buffers through the C ABI: every step copies its actions H2D and its observations /
            rewards / flags D2H into pinned memory inside the timed region. `value` = pg2_step_pipelined (D2H of step
            t-1 overlaps the kernels of step t), `sequential` = pg2_step + pg2_fetch, `cenv` = the reference-facing
            plugin call itself, cenv_step of lib<Game>.so (ctypes, batched "action" in, "screen" out);
            `d2h_ceiling_gbs` = plain cudaMemcpyAsync of the observation bytes into pinned memory on this box, and
            `d2h_frac` = how much of that the pipelined path reaches;
  --steps   K timed steps in every timed loop of every workload (device-resident, back to back, profiled, e2e, cenv);
  --dump-outputs DIR   after the timed device-resident steps of each workload, what they handed the caller in the last
            step, as float32 .npy files `<game>_<envs>[_ep<k>]_<array>.npy`: `obs` of a fixed, seeded sample of DUMP_ENVS
            envs (`env_index` says which) and `reward` / `terminated` / `truncated` of every env (rank 0's shard). Inputs
            (env seeds, action stream) are the same from run to run, so two builds can be compared array for array.
  roofline  dominant kernel (k_render) against the measured HBM copy bandwidth in MEASURED_PEAKS.json, algorithmic bytes
            = 12 297 B per env-step (SURVEY.md §8d); traffic = dram bytes of one launch from the committed ncu capture
            (profiles/traffic.json) when one exists for the workload.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_ENV_STEP = 12288 + 4 + 4 + 1   # obs write + action read + reward write + done write
METRIC = "env-steps/sec incl. 64x64 RGB render"
UNIT = "env-steps/s"
BASE_SEED = 0
BURN_IN = 300
GAMES = ("bossfight", "caveflyer", "chaser", "climber", "coinrun", "jumper", "maze")

DUMP_ENVS = 64   # 64 x 12 288 B x 4 (float32) = 3.1 MB of observations per workload, 11 workloads at most

HEADLINE = dict(tag="configs[2]", game="bossfight", envs=16384, max_ep=0)
SINGLE_GPU_EXTRA = [dict(tag="configs[0]", game="maze", envs=256, max_ep=0), dict(tag="configs[1]", game="coinrun", envs=4096, max_ep=0)]


def describe(w):
    return "BASELINE.json %s: %s, %d envs per GPU, 64x64x3 uint8 obs, uniform-random actions, auto-reset with per-episode level " \
           "regeneration%s" % (w["tag"], w["game"], w["envs"], ", %d-step episodes" % w["max_ep"] if w["max_ep"] else "")


def measured_traffic(game, envs):
    """dram bytes per launch of the dominant kernel, from the committed ncu captures (profiles/traffic.json)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("%s@%d" % (game, envs))
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) if t else None
    except Exception:
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed regions."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own C++ engine (oracle/_ref) on the host cores

def _ref_proc(conn, game, seeds, action_seed):
    """Worker process: owns len(seeds) reference environments (one library copy each)."""
    sys.path.insert(0, ROOT)
    from oracle import ref_env
    envs = [ref_env.RefEnv(game, s) for s in seeds]
    for e in envs:
        e.reset()
    rs = np.random.RandomState(action_seed)
    conn.send("ready")
    while True:
        n = conn.recv()
        if n <= 0:
            break
        acts = rs.randint(0, 15, size=(n, len(envs)))
        t0 = time.perf_counter()
        for t in range(n):
            for i, e in enumerate(envs):
                if e.raw_step(acts[t, i]):
                    e.raw_reset()
        conn.send(time.perf_counter() - t0)


class ReferencePool:
    """The reference C++ engine (oracle/_ref) spread over the host cores: `procs` processes x
    `envs_per_proc` environments, env j seeded BASE_SEED + j, uniform-random actions, reset on
    terminate (game_test.py:38-40). run(n) advances every env n steps and returns env-steps/s."""

    def __init__(self, game, procs, envs_per_proc):
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.procs, self.envs_per_proc, self.workers = procs, envs_per_proc, []
        for p in range(procs):
            parent, child = ctx.Pipe()
            seeds = [BASE_SEED + p * envs_per_proc + i for i in range(envs_per_proc)]
            w = ctx.Process(target=_ref_proc, args=(child, game, seeds, 1234 + p), daemon=True)
            w.start()
            self.workers.append((w, parent))
        for _, c in self.workers:
            assert c.recv() == "ready"

    def run(self, n):
        t0 = time.perf_counter()
        for _, c in self.workers:
            c.send(n)
        for _, c in self.workers:
            c.recv()
        wall = time.perf_counter() - t0
        return self.procs * self.envs_per_proc * n / wall, wall

    def close(self):
        for w, c in self.workers:
            c.send(0)
        for w, _ in self.workers:
            w.join(timeout=5)


def reference_available():
    from oracle import ref_env
    return ref_env.available()


def run_reference(a, w):
    if not reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (reference sources absent)"}))
        return
    procs = os.cpu_count() or 1
    envs_per_proc = 8
    pool = ReferencePool(w["game"], procs, envs_per_proc)
    for _ in range(a.warmup):
        pool.run(a.ref_inner)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        pool.run(a.ref_inner)
    wall = time.perf_counter() - t0
    pool.close()
    v = procs * envs_per_proc * a.ref_inner * a.steps / wall
    sample = "%d procs x %d envs; one timed step = %d cenv_step per env (%s, seeds %d.., uniform actions, reset on terminate)" % (
        procs, envs_per_proc, a.ref_inner, w["game"], BASE_SEED)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * wall / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(w, a.gpus),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(w, world):
    return {"workload": describe(w), "game": w["game"], "envs_per_gpu": w["envs"], "global_envs": w["envs"] * world,
            "parallelism": "env-sharded x%d, no collective" % world,
            "l2": "flushed between timed steps (256 MiB memset outside the event pairs)", "base_seed": BASE_SEED,
            "max_episode_steps": w["max_ep"], "burn_in_steps": BURN_IN}


# ---------------------------------------------------------------------------------------------------

class Ctx:
    pass


def measure(c, w, steps, warmup, full):
    """One workload on this rank's GPU -> dict of the rank-local measurements (times are reduced by the caller).
    full: also the e2e legs and the profiled pass (headline / BASELINE single-GPU configs)."""
    import torch
    from procgen2_b200.engine import BatchedEnv
    N, game, dev = w["envs"], w["game"], c.dev
    env = BatchedEnv(game, N, seed=BASE_SEED, device=c.local_rank, first_env=c.rank * N, max_episode_steps=w["max_ep"])
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + c.rank)
    pool = 256   # synthetic uniform-random action stream, generated on device ahead of the timed region
    actions = torch.randint(0, 15, (pool, N), dtype=torch.int32, device=dev, generator=gen)
    stream = torch.cuda.ExternalStream(env.stream_ptr, device=dev)
    obs, rew, term, trunc = env.torch_views()
    out = {}
    bufs = None
    with torch.cuda.stream(stream):
        for t in range(BURN_IN):
            env.step_torch(actions[t % pool])
        for t in range(warmup):
            env.step_torch(actions[t % pool])
            c.flush.zero_()
    c.barrier()
    # ---- device-resident, one CUDA-graph launch per step, L2 flushed between steps
    launches0 = env.kernel_launches
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    done_count = torch.zeros((), dtype=torch.int64, device=dev)
    c.barrier()
    wall0 = time.perf_counter()
    with torch.cuda.stream(stream):
        for t in range(steps):
            starts[t].record(stream)
            env.step_torch(actions[(warmup + t) % pool])
            ends[t].record(stream)
            done_count += (term | trunc).sum()
            c.flush.zero_()
    c.barrier()
    out["wall_s"] = time.perf_counter() - wall0
    if c.dump:
        idx = np.sort(np.random.RandomState(0).choice(N, min(N, DUMP_ENVS), replace=False))
        out["outputs"] = {"env_index": idx.astype(np.float32),
                          "obs": obs[torch.from_numpy(idx).to(dev)].cpu().numpy().astype(np.float32),
                          "reward": rew.cpu().numpy().astype(np.float32),
                          "terminated": term.cpu().numpy().astype(np.float32),
                          "truncated": trunc.cpu().numpy().astype(np.float32)}
    out["launches"] = env.kernel_launches - launches0
    out["dev_ms"] = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    out["resets_per_step"] = float(done_count.item()) / steps
    # ---- back to back (no flush): one event pair around all steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for t in range(steps):
            env.step_torch(actions[t % pool])
        e1.record(stream)
    c.barrier()
    out["b2b_ms"] = e0.elapsed_time(e1)
    if full:
        # ---- profiled pass: per-kernel CUDA events (eager launches)
        env.profile(True)
        with torch.cuda.stream(stream):
            for t in range(steps):
                env.step_torch(actions[t % pool])
                c.flush.zero_()
        c.barrier()
        prof, prof_steps = env.profile_read()
        env.profile(False)
        out["kernel_ms"] = {k: v / max(prof_steps, 1) for k, v in prof.items()}
        # ---- end to end with host buffers
        host_actions = actions.cpu().numpy()
        bufs = []
        for _ in range(2):
            o = torch.empty((N, 64, 64, 3), dtype=torch.uint8).pin_memory()
            r = torch.empty(N, dtype=torch.float32).pin_memory()
            d = torch.empty(N, dtype=torch.uint8).pin_memory()
            bufs.append((o.numpy(), r.numpy(), d.numpy(), (o, r, d)))
        e2e_steps = steps
        out["e2e_steps"] = e2e_steps
        for t in range(3):
            env.step(host_actions[t % pool])
            env.fetch_into(*bufs[0][:3])
        c.barrier()
        t0 = time.perf_counter()
        for t in range(e2e_steps):
            env.step(host_actions[t % pool])
            env.fetch_into(*bufs[0][:3])
        c.barrier()
        out["seq_s"] = time.perf_counter() - t0
        # raw D2H ceiling of this box: the same observation bytes, plain async copies into pinned memory
        # (on torch's own stream: the pinned allocator remembers the streams a block was used on, and the engine's
        # stream does not outlive the engine)
        for _ in range(2):
            bufs[0][3][0].copy_(obs, non_blocking=True)
        c.barrier()
        t0 = time.perf_counter()
        for _ in range(10):
            bufs[0][3][0].copy_(obs, non_blocking=True)
        c.barrier()
        out["d2h_s_per_copy"] = (time.perf_counter() - t0) / 10
        for t in range(4):
            env.step_pipelined(host_actions[t % pool], *bufs[t & 1][:3])
        env.flush()
        c.barrier()
        t0 = time.perf_counter()
        for t in range(e2e_steps):
            env.step_pipelined(host_actions[t % pool], *bufs[t & 1][:3])
        env.flush()
        c.barrier()
        out["e2e_s"] = time.perf_counter() - t0
    fault = env.read_field("fault")[0].view(np.int32)
    assert not fault.any(), "fault flags set during the benchmark: %s" % np.unique(fault)
    del obs, rew, term, trunc, bufs
    c.barrier()
    env.close()
    if full:
        out["cenv_s"] = measure_cenv(c, w, host_actions, out["e2e_steps"])
    return out


def measure_cenv(c, w, host_actions, n_steps):
    """The reference-facing plugin call: cenv_make / cenv_step of lib<Game>.so through ctypes, batched actions in, the
    library's own (pinned) "screen" / reward / flag buffers out. Returns seconds for n_steps steps."""
    from procgen2_b200 import build
    from procgen2_b200 import cenv as pc
    lib = ctypes.CDLL(build.game_lib_path(w["game"]))
    lib.cenv_make.argtypes = [ctypes.c_char_p, ctypes.POINTER(pc.CEnv_Option), ctypes.c_int32]
    lib.cenv_reset.argtypes = [ctypes.POINTER(pc.CEnv_Option), ctypes.c_int32]
    lib.cenv_step.argtypes = [ctypes.POINTER(pc.CEnv_Key_Value), ctypes.c_int32]
    opts = {"seed": BASE_SEED + c.rank * w["envs"], "num_envs": w["envs"], "device": c.local_rank}
    if w["max_ep"]:
        opts["max_episode_steps"] = w["max_ep"]
    arr = (pc.CEnv_Option * len(opts))()
    keep = []
    for i, (k, v) in enumerate(opts.items()):
        keep.append(k.encode())
        arr[i].name, arr[i].value_type, arr[i].value = keep[-1], 0, pc.CEnv_Value(i=int(v))
    assert lib.cenv_make(b"", arr, len(opts)) == 0
    assert lib.cenv_reset(None, 0) == 0
    kv = pc.CEnv_Key_Value(b"action", 0, w["envs"], pc.CEnv_Value_Buffer())
    pool = host_actions.shape[0]

    def step(t):
        kv.value_buffer.i = host_actions[t % pool].ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
        assert lib.cenv_step(ctypes.byref(kv), 1) == 0

    for t in range(3):
        step(t)
    c.barrier()
    t0 = time.perf_counter()
    for t in range(n_steps):
        step(t)
    c.barrier()
    dt = time.perf_counter() - t0
    lib.cenv_close()
    return dt


def reduce_max(c, vals):
    import torch
    import torch.distributed as dist
    t = torch.tensor(vals, dtype=torch.float64, device=c.dev)
    if c.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def reduce_sum(c, vals):
    import torch
    import torch.distributed as dist
    t = torch.tensor(vals, dtype=torch.float64, device=c.dev)
    if c.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return [float(x) for x in t.tolist()]


def gather_ms(c, v):
    """per-rank value -> (min, max) over the ranks (the straggler is visible)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([v], dtype=torch.float64, device=c.dev)
    if c.world == 1:
        return v, v
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return float(lo.item()), float(hi.item())


def summarise(c, w, m, steps, warmup, full):
    """Rank-reduced result block of one workload (identical on every rank; rank 0 prints)."""
    N, world = w["envs"], c.world
    dev_ms, b2b_ms = reduce_max(c, [m["dev_ms"], m["b2b_ms"]])
    rank_lo, rank_hi = gather_ms(c, m["dev_ms"] / steps)
    resets, = reduce_sum(c, [m["resets_per_step"]])
    hbm_gbs, peak_src = peaks()
    blk = {"workload": describe(w), "game": w["game"], "envs_per_gpu": N, "global_envs": N * world, "max_episode_steps": w["max_ep"],
           "value": N * world * steps / (dev_ms * 1e-3), "unit": UNIT, "ms_per_step": dev_ms / steps,
           "ms_per_step_rank_min_max": [rank_lo, rank_hi],
           "back_to_back": {"value": N * world * steps / (b2b_ms * 1e-3), "ms_per_step": b2b_ms / steps},
           "resets_per_step": resets, "gpu_launches": int(m["launches"]), "wall_s_timed_region": m["wall_s"]}
    blk["roofline_whole_step"] = {"achieved": ALG_BYTES_PER_ENV_STEP * N / (dev_ms / steps * 1e-3) / 1e9, "peak": hbm_gbs, "unit": "GB/s",
                                  "frac": ALG_BYTES_PER_ENV_STEP * N / (dev_ms / steps * 1e-3) / 1e9 / hbm_gbs}
    if full:
        render_ms = m["kernel_ms"]["render"]
        achieved = ALG_BYTES_PER_ENV_STEP * N / (render_ms * 1e-3) / 1e9
        blk["kernel_ms_per_step"] = m["kernel_ms"]
        blk["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs,
                           "traffic": measured_traffic(w["game"], N), "kernel": "k_render<%s>" % w["game"], "kernel_ms": render_ms,
                           "peak_source": peak_src, "algorithmic_bytes_per_launch": ALG_BYTES_PER_ENV_STEP * N}
        e2e_s, seq_s, cenv_s, d2h_s = reduce_max(c, [m["e2e_s"], m["seq_s"], m["cenv_s"], m["d2h_s_per_copy"]])
        k = m["e2e_steps"]
        d2h_bytes = N * (12288 + 4 + 1)
        ceiling = N * 12288 / d2h_s / 1e9
        blk["e2e"] = {"value": N * world * k / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": d2h_bytes, "steps": k,
                      "api": "pg2_step_pipelined(host actions -> pinned host obs/reward/terminated), depth-1 pipeline",
                      "sequential": N * world * k / seq_s,
                      "cenv": {"value": N * world * k / cenv_s, "api": "cenv_step of lib<Game>.so (ctypes; batched \"action\" in, pinned \"screen\" + infos out)"},
                      "d2h_ceiling_gbs": ceiling, "d2h_gbs": d2h_bytes * k / e2e_s / 1e9, "d2h_frac": (d2h_bytes * k / e2e_s / 1e9) / ceiling}
    return blk


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--game", default=None, help="one explicit workload instead of the BASELINE set (with --envs-per-gpu, --max-episode-steps)")
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--max-episode-steps", type=int, default=0,
                    help="truncate episodes (engine extension; BASELINE configs[4] stresses level generation with short episodes)")
    ap.add_argument("--ref-inner", type=int, default=50, help="env steps per env per timed sample of the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="headline workload only (skip the other BASELINE configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step of each workload as DIR/<name>.npy")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    headline = dict(tag="custom", game=a.game, envs=a.envs_per_gpu, max_ep=a.max_episode_steps) if a.game else dict(HEADLINE)

    if a.impl == "reference":
        if rank == 0:
            run_reference(a, headline)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    c = Ctx()
    c.rank, c.world, c.local_rank = rank, world, local_rank
    c.dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "WARN"     # keep stdout to the one JSON line (no "NCCL version" banner)
        dist.init_process_group("nccl", device_id=c.dev)
    c.flush = torch.empty(256 << 20, dtype=torch.uint8, device=c.dev)
    c.dump = a.dump_outputs is not None and rank == 0

    def barrier():
        torch.cuda.synchronize(c.dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(c.dev)
    c.barrier = barrier

    sampler = ClockSampler(local_rank)
    sampler.start()
    m = measure(c, headline, a.steps, a.warmup, True)
    head = summarise(c, headline, m, a.steps, a.warmup, True)
    dumps = [(headline, m.get("outputs"))]
    extra = []
    if not a.game and not a.no_extra:
        todo = [(w, True) for w in SINGLE_GPU_EXTRA]
        if world > 1:
            todo += [(dict(tag="configs[3] slice", game=g, envs=32768 // world, max_ep=0), False) for g in GAMES]
            todo += [(dict(tag="configs[4] slice", game="coinrun", envs=32768, max_ep=32), False)]
        for w, full in todo:
            m = measure(c, w, a.steps, a.warmup, full)
            extra.append(summarise(c, w, m, a.steps, a.warmup, full))
            dumps.append((w, m.get("outputs")))
    sampler.stop_flag = True
    sampler.join(timeout=2)

    if c.dump:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for w, arrays in dumps:
            name = "%s_%d%s" % (w["game"], w["envs"], "_ep%d" % w["max_ep"] if w["max_ep"] else "")
            for k, v in arrays.items():
                np.save(os.path.join(a.dump_outputs, "%s_%s.npy" % (name, k)), v)
    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": workload_config(headline, world),
                "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"],
                "roofline_whole_step": head["roofline_whole_step"], "kernel_ms_per_step": head["kernel_ms_per_step"],
                "back_to_back": head["back_to_back"], "resets_per_step": head["resets_per_step"],
                "ms_per_step_rank_min_max": head["ms_per_step_rank_min_max"],
                "clocks": sampler.summary(), "wall_s_timed_region": head["wall_s_timed_region"], "configs": extra}
        if not a.no_cpu_baseline and world == 1:
            procs = os.cpu_count() or 1
            if reference_available():
                pool = ReferencePool(headline["game"], procs, 8)
                pool.run(a.ref_inner)
                n_cpu = max(a.ref_inner, 2000)   # ~1 s wall on every host core = 10-30 s of CPU work
                v, wall_cpu = pool.run(n_cpu)
                pool.close()
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": procs, "kind": "reference",
                                        "sample": "%d procs x 8 envs x %d steps in %.1f s (%s; reference C++ engine, unmodified, + canonical "
                                                  "CPU rasteriser = oracle/_ref)" % (procs, n_cpu, wall_cpu, headline["game"])}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

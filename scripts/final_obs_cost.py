"""Cost of returning terminal frames (BatchedEnv(final_obs=True)): device ms per step with the feature off and on.

    python scripts/final_obs_cost.py [--steps 200] [--rounds 2] [--out profiles/final_obs_cost.json]

For each workload, two engines (off, on) of the same game, size and seeds run the same device-resident action stream,
alternating in rounds of `steps` steps within this one process. Each step is timed with CUDA events on the engine's
stream, with a 256 MiB memset between steps (outside the event pair) that flushes the L2, as bench.py does. The two
engines' observations, rewards and flags are compared at every timed step and must be identical. The GPU's name and
power limit are recorded with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [("bossfight", 16384), ("chaser", 4096), ("coinrun", 4096), ("maze", 256), ("jumper", 4096)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        q = "nvidia-smi unavailable (%s)" % e
    return q


def main():
    import numpy as np
    import torch
    from procgen2_b200.engine import BatchedEnv

    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": gpu_info(), "steps": args.steps, "rounds": args.rounds,
              "l2": "flushed between timed steps (256 MiB memset outside the event pairs)", "workloads": []}
    for game, n in WORKLOADS:
        envs = {k: BatchedEnv(game, n, seed=12345, final_obs=(k == "on")) for k in ("off", "on")}
        gen = torch.Generator(device=dev)
        gen.manual_seed(99)
        pool = 256
        actions = torch.randint(0, 15, (pool, n), dtype=torch.int32, device=dev, generator=gen)
        streams = {k: torch.cuda.ExternalStream(e.stream_ptr, device=dev) for k, e in envs.items()}
        views = {k: e.torch_views() for k, e in envs.items()}
        ms = {"off": [], "on": []}
        launches = {"off": 0, "on": 0}
        resets = 0
        t_global = {"off": 0, "on": 0}
        for k, e in envs.items():
            e.reset()
            with torch.cuda.stream(streams[k]):
                for _ in range(args.warmup):
                    e.step_torch(actions[t_global[k] % pool])
                    t_global[k] += 1
        torch.cuda.synchronize()
        for r in range(args.rounds):
            for k in ("off", "on"):   # alternate: the same steps of both engines, one round after the other
                e, s = envs[k], streams[k]
                starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
                ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
                l0 = e.kernel_launches
                snaps = []
                with torch.cuda.stream(s):
                    for t in range(args.steps):
                        starts[t].record(s)
                        e.step_torch(actions[t_global[k] % pool])
                        ends[t].record(s)
                        t_global[k] += 1
                        o, rw, te, tr = views[k]
                        snaps.append((o.sum(dtype=torch.int64), rw.clone(), te.clone(), tr.clone()))
                        flush.zero_()
                torch.cuda.synchronize()
                launches[k] += e.kernel_launches - l0
                ms[k].append(sum(a.elapsed_time(b) for a, b in zip(starts, ends)) / args.steps)
                if k == "off":
                    ref = snaps
                else:
                    for t, (x, y) in enumerate(zip(ref, snaps)):
                        for u, v, what in zip(x, y, ("obs checksum", "reward", "terminated", "truncated")):
                            assert torch.equal(u, v), "%s %d: %s differs at timed step %d of round %d" % (game, n, what, t, r)
                    resets += sum(int((te | tr).sum()) for _, _, te, tr in snaps)
        # full frames compared once more at the end
        torch.cuda.synchronize()
        assert torch.equal(views["off"][0], views["on"][0]), "%s %d: final observations differ" % (game, n)
        off, on = float(np.mean(ms["off"])), float(np.mean(ms["on"]))
        row = {"game": game, "envs": n, "ms_per_step_off": ms["off"], "ms_per_step_on": ms["on"], "overhead_pct": 100.0 * (on - off) / off,
               "launches_per_step_off": launches["off"] / (args.steps * args.rounds),
               "launches_per_step_on": launches["on"] / (args.steps * args.rounds),
               "finished_per_step": resets / (args.steps * args.rounds), "outputs_identical": True}
        result["workloads"].append(row)
        print("%-10s %6d  off %.4f ms  on %.4f ms  %+.1f %%  launches %.0f -> %.0f  finished/step %.1f" % (
            game, n, off, on, row["overhead_pct"], row["launches_per_step_off"], row["launches_per_step_on"], row["finished_per_step"]), flush=True)
        for e in envs.values():
            e.close()
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

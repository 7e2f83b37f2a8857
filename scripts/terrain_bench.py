"""Walkers on arbitrary terrain (wb_terrain_env_*, terrain_step_kernel) against the specialised walker kernel (wb_env_*).

  python scripts/terrain_bench.py [--sizes 4096 65536] [--warmup 512] [--steps 50] [--ppo-envs 65536] [--horizon 64]
                                  [--out profiles/terrain_bench.json]

Every env-step time is a pair of CUDA events around one step_dev call.  Each configuration first runs `--warmup` untimed
env-steps of random actions (auto-reset on), then `--steps` timed ones with a 256 MB write between them, so that no timed step
finds the previous step's state in the 126 MB L2.  Measured:
  flat    the reference's flat floor: wb_env_step_dev (physics_lanes.cu) vs wb_terrain_env_step_dev with CreateFloor("Metal")
  rough   Environment.CreateRoughFloor (10 segments) with its own random heights per walker, wb_terrain_env_step_dev
  ppo     VectorPPO(terrain=per-walker rough floor): rollout env-steps/s, update samples/s, whole loop (one warm-up iteration)
The card's name and power limit are read in the same run and written next to the numbers."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import __graft_entry__ as ge

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
ap.add_argument("--warmup", type=int, default=512)
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--ppo-envs", type=int, default=65536)
ap.add_argument("--horizon", type=int, default=64)
ap.add_argument("--minibatch", type=int, default=65536)
ap.add_argument("--ppo-iters", type=int, default=2)
ap.add_argument("--out", default=os.path.join("profiles", "terrain_bench.json"))
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("terrain_bench: no CUDA device")
wb = ge.load_package()
wb.init(0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line}


def rough_floors(n, seed):
    rng = np.random.default_rng(seed)
    return [wb.CreateRoughFloor([int(h) for h in rng.integers(0, 100, 11)]) for _ in range(n)]


def time_env(env, n, stream):
    """median / mean ms of one env-step over args.steps timed steps (L2 flushed between them)"""
    rng = np.random.default_rng(0)
    acts = torch.from_numpy(rng.uniform(-1.0, 1.0, (8, n, 4)).astype(np.float32)).cuda()
    obs = torch.empty(n, 12, device="cuda")
    rew = torch.empty(n, device="cuda")
    done = torch.empty(n, device="cuda", dtype=torch.uint8)
    flush = torch.empty(64 * 1024 * 1024, device="cuda")  # 256 MB
    with torch.cuda.stream(stream):
        for t in range(args.warmup):
            env.step_dev(acts[t % 8], obs, rew, done)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for t, (a, b) in enumerate(ev):
            flush.zero_()
            a.record()
            env.step_dev(acts[t % 8], obs, rew, done)
            b.record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    return {"median_ms": float(np.median(ms)), "mean_ms": float(ms.mean()), "min_ms": float(ms.min()),
            "env_steps_per_s": n / (float(np.median(ms)) * 1e-3)}


result = {"card": card(), "warmup_steps": args.warmup, "timed_steps": args.steps, "l2_flush_bytes": 256 << 20, "flat": {}, "rough": {}}
stream = torch.cuda.Stream()
for n in args.sizes:
    walker = wb.EnvBatch(n, floor_materials="Metal", stream=stream.cuda_stream)
    terrain = wb.TerrainEnvBatch(n, wb.CreateFloor("Metal"), stream=stream.cuda_stream)
    result["flat"][str(n)] = {"wb_env_step_dev": time_env(walker, n, stream), "wb_terrain_env_step_dev": time_env(terrain, n, stream),
                              "physics_lanes": walker.get_variant()}
    walker.close()
    terrain.close()
    rough = wb.TerrainEnvBatch(n, rough_floors(n, n), stream=stream.cuda_stream)
    result["rough"][str(n)] = {"wb_terrain_env_step_dev": time_env(rough, n, stream)}
    rough.close()
    print(json.dumps({"n": n, "flat": result["flat"][str(n)], "rough": result["rough"][str(n)]}), flush=True)

vp = wb.VectorPPO(args.ppo_envs, horizon=args.horizon, minibatch_global=args.minibatch, seed=11, terrain=rough_floors(args.ppo_envs, 7))
vp.iterate()  # warm-up iteration
tot = {"rollout_ms": 0.0, "update_ms": 0.0, "samples_trained": 0}
for _ in range(args.ppo_iters):
    torch.cuda.synchronize()
    last = vp.iterate()
    for k in tot:
        tot[k] += last[k]
ro, up = tot["rollout_ms"] * 1e-3, tot["update_ms"] * 1e-3
steps = args.ppo_envs * args.horizon * args.ppo_iters
result["ppo"] = {"envs": args.ppo_envs, "horizon": args.horizon, "minibatch": args.minibatch, "iters": args.ppo_iters,
                 "rollout_env_steps_per_s": steps / ro, "update_samples_per_s": tot["samples_trained"] / up,
                 "loop_env_steps_per_s": steps / (ro + up), "rollout_s": ro, "update_s": up,
                 "episodes_finished_last": last["episodes_finished"], "mean_reward_last": last["mean_reward"]}
result["card_after"] = card()
print(json.dumps(result["ppo"]), flush=True)
os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
with open(args.out, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", args.out)

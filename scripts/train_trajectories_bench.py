"""PPOAgent.Train(Trajectory) per finished episode: the per-mini-batch path (PPOAgent.Train: wb_policy_forward +
wb_returns_advantages + one wb_ppo_train per mini-batch, each a synchronous host call) against one wb_ppo_train_trajectories call
for the whole list (PPOAgent.TrainTrajectories: one launch of ppo_episodes_kernel on the default networks).

  python scripts/train_trajectories_bench.py [--repeats 5] [--out profiles/train_trajectories_bench.json]

Hyper-parameters are the reference's (BatchSize 64, Epochs 5).  Every time is host wall clock around work that ends in a device
synchronise (both calls return synchronised), after an untimed warm-up call of the same shape; the table reports medians.
Measured:
  single   one 1 001-step episode (the max_timesteps cap): ms per episode, us per Adam step
  batch    E finished episodes, E in {16, 256, 4096}, lengths drawn from the episode lengths of a random-policy rollout of the
           library's walker environment (uniform actions in [-1, 1], auto-reset; E drawn at random from 2 x 4096 finished
           episodes); the sample contents are synthetic (they do not change the work: every sample takes the same code path)
  kernel   the one-launch kernel alone: CUDA events around wb_ppo_train_trajectories_dev on inputs already on the device
The card's name and power limit are read in the same run and written next to the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import __graft_entry__ as ge

ap = argparse.ArgumentParser()
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--episodes", type=int, nargs="+", default=[16, 256, 4096])
ap.add_argument("--rollout-envs", type=int, default=4096)
ap.add_argument("--out", default=os.path.join("profiles", "train_trajectories_bench.json"))
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("train_trajectories_bench: no CUDA device")
wb = ge.load_package()
wb.init(0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line}


def episode_lengths(n_envs, want, seed=0):
    """lengths of finished episodes of a uniform-random policy, in the order they finish (capped by max_timesteps)"""
    rng = np.random.default_rng(seed)
    env = wb.EnvBatch(n_envs)
    age = np.zeros(n_envs, np.int64)
    out = []
    while len(out) < want:
        _, _, done = env.step(rng.uniform(-1.0, 1.0, (n_envs, 4)).astype(np.float32))
        age += 1
        for i in np.flatnonzero(done):
            out.append(int(age[i]))
        age[done.astype(bool)] = 0
    return out[:want]


def trajectories(lengths, seed=1):
    rng = np.random.default_rng(seed)
    std = np.float32(np.exp(-1.0))
    out = []
    for T in lengths:
        t = wb.Trajectory()
        t.States = list(rng.normal(size=(T, 12)).astype(np.float32) * np.float32(0.3))
        a = rng.normal(size=(T, 4)).astype(np.float32) * std
        t.Actions = list(a)
        t.LogProbabilities = list((-np.log(std) - np.float32(0.9189385) - 0.5 * (a / std) ** 2).astype(np.float32))
        t.Rewards = list(rng.normal(size=T).astype(np.float32))
        out.append(t)
    return out


def timed(fn, repeats):
    fn()  # warm-up of the same shape
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts) * 1e3, ts


def device_ms(agent, trajs, repeats):
    """CUDA-event time of wb_ppo_train_trajectories_dev alone (inputs already on the device, mini-batches drawn once)"""
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    B = agent.hp.batch_size
    lengths = [len(t.States) for t in trajs]
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    blocks = [agent.rng.permutation(T)[j * B:(j + 1) * B] for T in lengths for _ in range(5) for j in range(T // B)]
    index = np.concatenate(blocks).astype(np.int32) if blocks else np.zeros(1, np.int32)
    cat = lambda attr, w: torch.from_numpy(np.concatenate([np.asarray(getattr(t, attr), np.float32).reshape(-1, w) for t in trajs])).cuda()
    dev = [cat("States", 12), cat("Actions", 4), cat("LogProbabilities", 4), cat("Rewards", 1), torch.from_numpy(index).cuda()]
    ts = []
    for r in range(repeats + 1):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib().wb_ppo_train_trajectories_dev(agent._h, len(trajs), ptr(offsets), 5, *[ptr(t) for t in dev], None, None, None, None, None))
        e1.record()
        torch.cuda.synchronize()
        if r:  # (the first call is the warm-up)
            ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def compare(lengths, repeats):
    trajs = trajectories(lengths)
    per_call = wb.PPOAgent(seed=2)  # default variant: the tensor-core kernel, one launch per mini-batch
    one_call = wb.PPOAgent(seed=2)
    steps = 5 * sum(T // 64 for T in lengths)
    ms_loop, raw_loop = timed(lambda: [per_call.Train(t) for t in trajs], repeats)
    ms_one, raw_one = timed(lambda: one_call.TrainTrajectories(trajs), repeats)
    ms_dev = device_ms(one_call, trajs, repeats)
    return {"episodes": len(lengths), "rows": int(sum(lengths)), "adam_steps": steps, "kernel_ms": ms_dev,
            "kernel_us_per_adam_step": ms_dev * 1e3 / max(steps, 1),
            "train_loop_ms": ms_loop, "train_trajectories_ms": ms_one, "speedup": ms_loop / ms_one,
            "train_loop_us_per_adam_step": ms_loop * 1e3 / max(steps, 1), "train_trajectories_us_per_adam_step": ms_one * 1e3 / max(steps, 1),
            "raw_s": {"train_loop": raw_loop, "train_trajectories": raw_one}}


result = {"card": card(), "batch_size": 64, "epochs": 5, "repeats": args.repeats}
result["single_1001"] = compare([1001], args.repeats)
lengths = episode_lengths(args.rollout_envs, 2 * max(args.episodes))
result["rollout_lengths"] = {"mean": float(np.mean(lengths)), "median": float(np.median(lengths)), "max": int(max(lengths)),
                             "below_batch": int(sum(T < 64 for T in lengths))}
pick = np.random.default_rng(3)  # E episodes drawn from the rollout's finished episodes (the first to finish are the shortest)
result["batch"] = [compare([lengths[i] for i in pick.choice(len(lengths), E, replace=False)], args.repeats if E < 4096 else max(1, min(args.repeats, 3)))
                   for E in args.episodes]
os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
with open(args.out, "w") as fh:
    json.dump(result, fh, indent=1)
print(json.dumps({k: v for k, v in result.items() if k != "batch"}, indent=1))
for row in result["batch"]:
    print({k: v for k, v in row.items() if k != "raw_s"})

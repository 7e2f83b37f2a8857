"""One PPO brain per walker (wb_population_*): IndependentPPO's env-step rate, the episode-training kernel's scaling in agents and the
population act kernel alone.

  python scripts/population_bench.py [--sizes 4096 65536] [--warmup 512] [--steps 1000] [--train-agents 1 148 296 1024]
                                     [--act-reps 200] [--out profiles/population_bench.json]

Every time is a median of CUDA-event intervals after warm-up, with a 256 MB write between timed steps / calls so that no timed
interval finds the previous one's data in the 126 MB L2.  Measured:
  loop    IndependentPPO(N) (default hyper-parameters, flat Metal floor): `--warmup` env-steps, then `--steps` timed ones, each split
          into act (wb_population_act_dev), env (wb_env_step_dev + the reward-sum update), synchronisation + host (the done bytes,
          the item table) and train (wb_population_train_dev on the steps where an episode ended).  Beside it, in the same run,
          VectorPPO(N)'s rollout rate (one shared brain, horizon 64), as context.
  train   wb_population_train_dev with K agents, one 1 001-step episode each (random states / actions, device-drawn indices).
  act     population_act_kernel alone (N agents) against wb_policy_act_dev with one shared brain; actor-weight bytes (N x 21 008)
          over the median time, as a share of 7.7 TB/s (the HBM3e bandwidth of the B200 data sheet).
The card's name, power limit and max SM clock are read in the same run and written next to the numbers."""
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
ap.add_argument("--steps", type=int, default=1000)
ap.add_argument("--train-agents", type=int, nargs="+", default=[1, 148, 296, 1024])
ap.add_argument("--act-reps", type=int, default=200)
ap.add_argument("--out", default=os.path.join("profiles", "population_bench.json"))
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("population_bench: no CUDA device")
wb = ge.load_package()
wb.init(0)
from ppo_bipedalwalker_b200._lib import check, lib, ptr  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
ACTOR_BYTES = 5252 * 4
flush = torch.empty(64 * 1024 * 1024, device="cuda")  # 256 MB


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line}


def med(ms):
    ms = np.asarray(ms, np.float64)
    return {"median_ms": float(np.median(ms)), "mean_ms": float(ms.mean()), "min_ms": float(ms.min())}


def bench_loop(n):
    loop = wb.IndependentPPO(n, seed=3)
    for _ in range(args.warmup):
        loop.step()
    loop.timing = []
    episodes0 = sum(len(e[1]) for e in loop._log)
    for _ in range(args.steps):
        flush.zero_()
        loop.step()
    torch.cuda.synchronize()
    ev = loop.timing
    loop.timing = None
    phase = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(4)] for e in ev])  # act, env, sync + host, train
    total = phase.sum(1)
    episodes = sum(len(e[1]) for e in loop._log) - episodes0
    log = loop.episode_log()
    timed = log[log["step"] >= args.warmup]
    adam_steps = int(sum(5 * (int(L) // 64) for L in timed["length"]))
    total_s = float(total.sum()) * 1e-3
    out = {"walkers": n, "timed_steps": args.steps, "env_steps_per_s": n * args.steps / total_s,
           "step_ms": med(total), "act_ms": med(phase[:, 0]), "env_ms": med(phase[:, 1]), "sync_host_ms": med(phase[:, 2]),
           "train_ms": med(phase[:, 3]), "share_of_time": dict(zip(["act", "env", "sync_host", "train"], (phase.sum(0) / total.sum()).tolist())),
           "episodes_trained": episodes, "episodes_per_s": episodes / total_s, "adam_steps": adam_steps, "adam_steps_per_s": adam_steps / total_s,
           "steps_with_training": int((phase[:, 3] > 0).sum()), "mean_episode_length": float(timed["length"].mean()) if len(timed) else 0.0}
    del loop
    torch.cuda.synchronize()
    vp = wb.VectorPPO(n, horizon=64, minibatch_global=min(65536, n * 64), seed=3)
    vp.iterate()
    rollout_ms = [vp.iterate()["rollout_ms"] for _ in range(2)]
    out["vector_ppo_rollout_env_steps_per_s"] = n * 64 / (float(np.median(rollout_ms)) * 1e-3)
    del vp
    return out


def bench_train(K, R=1001):
    pop = wb.PPOPopulation(K, seed=5)
    rng = np.random.default_rng(K)
    states = torch.from_numpy(rng.normal(size=(R, K, 12)).astype(np.float32)).cuda()
    actions = torch.from_numpy(rng.normal(0, 0.5, size=(R, K, 4)).astype(np.float32)).cuda()
    logp = torch.full((R, K, 4), -0.5, device="cuda")
    rewards = torch.from_numpy(rng.normal(size=(R, K)).astype(np.float32)).cuda()
    out = [torch.empty(R, K, device="cuda") for _ in range(3)]
    items = np.ascontiguousarray(np.stack([np.arange(K), np.arange(K), np.zeros(K, int), np.full(K, R)], 1), np.int32)
    pop.set_stream(torch.cuda.current_stream().cuda_stream)

    def call():
        check(lib().wb_population_train_dev(pop._h, K, ptr(items), R, K, 5, 1, ptr(states), ptr(actions), ptr(logp), ptr(rewards), None,
                                            *[ptr(o) for o in out], None, None))
    call()
    ms = []
    for _ in range(5):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    steps = 5 * (R // 64)
    r = med(ms)
    r.update({"agents": K, "episode_steps": R, "adam_steps_per_agent": steps, "us_per_adam_step": r["median_ms"] * 1e3 / steps})
    return r


def bench_act(n):
    stream = torch.cuda.current_stream().cuda_stream
    pop = wb.PPOPopulation(n, seed=9, stream=stream)
    shared = wb.PPOAgent(seed=9, stream=stream)
    states = torch.randn(n, 12, device="cuda")
    o = [torch.empty(n, 4, device="cuda") for _ in range(2)]

    def timed(fn):
        for t in range(10):
            fn(t)
        ms = []
        for t in range(args.act_reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(t)
            b.record()
            ms.append((a, b))
        torch.cuda.synchronize()
        return med([a.elapsed_time(b) for a, b in ms])

    res = {"walkers": n, "actor_bytes": n * ACTOR_BYTES}
    res["population_act"] = timed(lambda t: check(lib().wb_population_act_dev(pop._h, n, ptr(states), 1, t, ptr(o[0]), ptr(o[1]), None, None)))
    sec = res["population_act"]["median_ms"] * 1e-3
    res["population_act"]["actor_bytes_per_s"] = n * ACTOR_BYTES / sec
    res["population_act"]["share_of_7.7TBps"] = n * ACTOR_BYTES / sec / HBM_BYTES_PER_S
    for variant in (0, 1):
        shared.set_variant(variant)
        res[f"shared_brain_policy_act_variant{variant}"] = timed(
            lambda t: check(lib().wb_policy_act_dev(shared._h, n, ptr(states), 1, t, ptr(o[0]), ptr(o[1]), None, None)))
    return res


result = {"card": card(), "warmup_steps": args.warmup, "l2_flush_bytes": 256 << 20, "act": {}, "train": {}, "loop": {}}
for n in args.sizes:
    result["act"][str(n)] = bench_act(n)
    print(json.dumps(result["act"][str(n)]), flush=True)
for K in args.train_agents:
    result["train"][str(K)] = bench_train(K)
    print(json.dumps(result["train"][str(K)]), flush=True)
for n in args.sizes:
    result["loop"][str(n)] = bench_loop(n)
    print(json.dumps(result["loop"][str(n)]), flush=True)
result["card_after"] = card()
os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
with open(args.out, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", args.out)

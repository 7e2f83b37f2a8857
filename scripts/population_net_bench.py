"""One PPO brain per walker for networks other than the defaults: the any-topology population act kernel, the any-topology episode
training kernel and IndependentPPO with both non-default networks.

  python scripts/population_net_bench.py [--sizes 4096 65536] [--warmup 256] [--steps 500] [--train-agents 148 1024]
                                         [--act-reps 200] [--out profiles/population_net_bench.json]

Every time is a median of CUDA-event intervals after warm-up, with a 256 MB write between timed steps / calls so that no timed
interval finds the previous one's data in the 126 MB L2 (as scripts/population_bench.py).  Measured:
  act     wb_population_act_dev at N walkers for three actors: the default networks (population_act_kernel), the same bytes as a
          non-default network (Input |64| (ReLU) |64| (ReLU) |4| (TanH) Output, population_generic_act_kernel) and a 128-wide actor
          (Input |128| (LeakyReLU) |128| (LeakyReLU) |4| (TanH) Output).  Actor-weight bytes over the median time, as a share of
          7.7 TB/s (the HBM3e bandwidth of the B200 data sheet).
  train   one agent with one 1 001-step episode (5 epochs, B = 64) on wb_population_train_trajectories against
          wb_ppo_train_trajectories on a wb_policy with the same networks; then wb_population_train_dev with K agents.  Microseconds
          per Adam step.
  loop    IndependentPPO(N, actor=, critic=) with each non-default actor: env-steps/s and the act / env / sync + host / train split.
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
ap.add_argument("--warmup", type=int, default=256)
ap.add_argument("--steps", type=int, default=500)
ap.add_argument("--train-agents", type=int, nargs="+", default=[148, 1024])
ap.add_argument("--act-reps", type=int, default=200)
ap.add_argument("--out", default=os.path.join("profiles", "population_net_bench.json"))
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("population_net_bench: no CUDA device")
wb = ge.load_package()
wb.init(0)
from ppo_bipedalwalker_b200._lib import check, lib, ptr  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
CRITIC = "Input |64| (LeakyReLU) |1| Output"
ACTORS = {"default": wb.DEFAULT_ACTOR, "relu64": "Input |64| (ReLU) |64| (ReLU) |4| (TanH) Output",
          "leaky128": "Input |128| (LeakyReLU) |128| (LeakyReLU) |4| (TanH) Output"}
flush = torch.empty(64 * 1024 * 1024, device="cuda")  # 256 MB


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line}


def med(ms):
    ms = np.asarray(ms, np.float64)
    return {"median_ms": float(np.median(ms)), "mean_ms": float(ms.mean()), "min_ms": float(ms.min())}


def timed(fn, reps, warm=3):
    for t in range(warm):
        fn(t)
    ev = []
    for t in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(t)
        b.record()
        ev.append((a, b))
    torch.cuda.synchronize()
    return med([a.elapsed_time(b) for a, b in ev])


def bench_act(n):
    stream = torch.cuda.current_stream().cuda_stream
    states = torch.randn(n, 12, device="cuda")
    o = [torch.empty(n, 4, device="cuda") for _ in range(2)]
    res = {"walkers": n}
    for name, actor in ACTORS.items():
        pop = wb.PPOPopulation(n, seed=9, stream=stream, actor=actor, critic=CRITIC)
        r = timed(lambda t: check(lib().wb_population_act_dev(pop._h, n, ptr(states), 1, t, ptr(o[0]), ptr(o[1]), None, None)), args.act_reps)
        nbytes = n * pop.N_ACTOR * 4
        r.update({"actor": actor, "actor_bytes": nbytes, "bytes_per_us": nbytes / (r["median_ms"] * 1e3),
                  "share_of_7.7TBps": nbytes / (r["median_ms"] * 1e-3) / HBM_BYTES_PER_S})
        res[name] = r
        del pop
    return res


def episode(K, R, rng):
    return (torch.from_numpy(rng.normal(size=(R, K, 12)).astype(np.float32)).cuda(),
            torch.from_numpy(rng.normal(0, 0.5, size=(R, K, 4)).astype(np.float32)).cuda(), torch.full((R, K, 4), -0.5, device="cuda"),
            torch.from_numpy(rng.normal(size=(R, K)).astype(np.float32)).cuda())


def bench_train_one(actor, R=1001, reps=5):
    """One agent, one episode: the population entry against the per-mini-batch path of one wb_policy (the same host arrays)."""
    rng = np.random.default_rng(1)
    S, A, LP, Rw = [np.ascontiguousarray(x.cpu().numpy().reshape(R, -1)) for x in episode(1, R, rng)]
    index = np.concatenate([rng.permutation(R)[:R // 64 * 64] for _ in range(5)]).astype(np.int32)
    offsets = np.array([0, R], np.int32)
    pop = wb.PPOPopulation(1, seed=2, actor=actor, critic=CRITIC)
    agent = wb.PPOAgent(actor=actor, critic=CRITIC, seed=2)
    pop_ms = timed(lambda t: check(lib().wb_population_train_trajectories(pop._h, 1, ptr(np.zeros(1, np.int32)), ptr(offsets), 5, ptr(S), ptr(A),
                                                                          ptr(LP), ptr(Rw), ptr(index), None, None, None, None, None)), reps, 1)
    pol_ms = timed(lambda t: check(lib().wb_ppo_train_trajectories(agent._h, 1, ptr(offsets), 5, ptr(S), ptr(A), ptr(LP), ptr(Rw), ptr(index),
                                                                   None, None, None, None, None)), reps, 1)
    steps = 5 * (R // 64)
    return {"actor": actor, "adam_steps": steps, "population_us_per_adam_step": pop_ms["median_ms"] * 1e3 / steps,
            "policy_us_per_adam_step": pol_ms["median_ms"] * 1e3 / steps, "population": pop_ms, "policy": pol_ms,
            "note": "host entries: both times include the host-to-device copies of the episode and the final synchronisation"}


def bench_train(actor, K, R=1001):
    pop = wb.PPOPopulation(K, seed=5, actor=actor, critic=CRITIC, stream=torch.cuda.current_stream().cuda_stream)
    states, actions, logp, rewards = episode(K, R, np.random.default_rng(K))
    out = [torch.empty(R, K, device="cuda") for _ in range(3)]
    items = np.ascontiguousarray(np.stack([np.arange(K), np.arange(K), np.zeros(K, int), np.full(K, R)], 1), np.int32)
    r = timed(lambda t: check(lib().wb_population_train_dev(pop._h, K, ptr(items), R, K, 5, 1, ptr(states), ptr(actions), ptr(logp),
                                                            ptr(rewards), None, *[ptr(o) for o in out], None, None)), 3, 1)
    steps = 5 * (R // 64)
    r.update({"actor": actor, "agents": K, "episode_steps": R, "adam_steps_per_agent": steps, "us_per_adam_step": r["median_ms"] * 1e3 / steps})
    return r


def bench_loop(n, actor):
    loop = wb.IndependentPPO(n, seed=3, actor=actor, critic=CRITIC)
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
    total_s = float(total.sum()) * 1e-3
    out = {"walkers": n, "actor": actor, "timed_steps": args.steps, "env_steps_per_s": n * args.steps / total_s, "step_ms": med(total),
           "act_ms": med(phase[:, 0]), "env_ms": med(phase[:, 1]), "sync_host_ms": med(phase[:, 2]), "train_ms": med(phase[:, 3]),
           "share_of_time": dict(zip(["act", "env", "sync_host", "train"], (phase.sum(0) / total.sum()).tolist())),
           "episodes_trained": sum(len(e[1]) for e in loop._log) - episodes0}
    del loop
    torch.cuda.synchronize()
    return out


result = {"card": card(), "critic": CRITIC, "l2_flush_bytes": 256 << 20, "act": {}, "train_one": {}, "train": {}, "loop": {}}
for n in args.sizes:
    result["act"][str(n)] = bench_act(n)
    print(json.dumps(result["act"][str(n)]), flush=True)
for name in ("relu64", "leaky128"):
    result["train_one"][name] = bench_train_one(ACTORS[name])
    print(json.dumps(result["train_one"][name]), flush=True)
    for K in args.train_agents:
        result["train"][f"{name}/{K}"] = bench_train(ACTORS[name], K)
        print(json.dumps(result["train"][f"{name}/{K}"]), flush=True)
for name in ("relu64", "leaky128"):
    for n in args.sizes:
        result["loop"][f"{name}/{n}"] = bench_loop(n, ACTORS[name])
        print(json.dumps(result["loop"][f"{name}/{n}"]), flush=True)
result["card_after"] = card()
os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
with open(args.out, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", args.out)

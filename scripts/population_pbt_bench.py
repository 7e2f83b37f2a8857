"""Population-based training (PBT): the copy kernel alone and IndependentPPO with and without the schedule.

  python scripts/population_pbt_bench.py [--agents 32768] [--pairs 1 148 1024 16384] [--reps 50] [--sizes 4096 65536]
                                         [--warmup 512] [--steps 1000] [--out profiles/population_pbt_bench.json]

Every time is a median of CUDA-event intervals after warm-up, with a 256 MB write between timed calls / steps so that no timed
interval finds the previous one's data in the 126 MB L2.  Measured:
  copy    wb_population_copy_agents alone (the pinned table upload and the one launch) with k pairs of distinct agents in a population
          of `--agents`, for the default networks and a 128-wide actor; bytes moved = read + write of three rows (weights, Adam
          m, v) of `stride` floats per pair, over the median time, and that rate as a share of 7.7 TB/s (the HBM3e bandwidth of the
          B200 data sheet).
  loop    IndependentPPO(N) (default hyper-parameters, flat Metal floor) without PBT and with PBT(interval 50, fraction 0.2, window
          5, the default perturbation): `--warmup` env-steps, then `--steps` timed ones; env-steps/s, copies per timed step and the
          host time of the schedule (PBT.step, perf_counter) per step.
The card's name, power limit and max SM clock are read in the same run and written next to the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import __graft_entry__ as ge

ap = argparse.ArgumentParser()
ap.add_argument("--agents", type=int, default=32768)
ap.add_argument("--pairs", type=int, nargs="+", default=[1, 148, 1024, 16384])
ap.add_argument("--reps", type=int, default=50)
ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
ap.add_argument("--warmup", type=int, default=512)
ap.add_argument("--steps", type=int, default=1000)
ap.add_argument("--out", default=os.path.join("profiles", "population_pbt_bench.json"))
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("population_pbt_bench: no CUDA device")
wb = ge.load_package()
wb.init(0)
from ppo_bipedalwalker_b200._lib import check, lib, ptr  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
WIDE = ("Input |128| (LeakyReLU) |128| (LeakyReLU) |4| (TanH) Output", "Input |64| (LeakyReLU) |1| Output")
flush = torch.empty(64 * 1024 * 1024, device="cuda")  # 256 MB


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line}


def med(ms):
    ms = np.asarray(ms, np.float64)
    return {"median_ms": float(np.median(ms)), "mean_ms": float(ms.mean()), "min_ms": float(ms.min())}


def bench_copy(net):
    kw = {} if net == "default" else dict(actor=WIDE[0], critic=WIDE[1])
    pop = wb.PPOPopulation(args.agents, seed=1, stream=torch.cuda.current_stream().cuda_stream, **kw)
    stride = (pop.N_PARAMS + 6) // 4 * 4
    out = {"agents": args.agents, "n_params": pop.N_PARAMS, "stride_floats": stride, "pairs": {}}
    for k in args.pairs:
        perm = np.random.default_rng(k).permutation(args.agents)
        dst, src = np.ascontiguousarray(perm[:k], np.int32), np.ascontiguousarray(perm[k:2 * k], np.int32)

        def call():
            check(lib().wb_population_copy_agents(pop._h, k, ptr(dst), ptr(src), None))
        for _ in range(3):
            call()
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            call()
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        r = med(ms)
        moved = 2 * 3 * 4 * stride * k
        r.update({"bytes_moved": moved, "GB_per_s": moved / (r["median_ms"] * 1e-3) * 1e-9,
                  "share_of_7.7TBps": moved / (r["median_ms"] * 1e-3) / HBM_BYTES_PER_S})
        out["pairs"][str(k)] = r
        print(net, k, json.dumps(r), flush=True)
    del pop
    torch.cuda.synchronize()
    return out


def bench_loop(n, with_pbt):
    pbt = wb.PBT(50, fraction=0.2, window=5) if with_pbt else None
    host = []
    if pbt is not None:
        step = pbt.step

        def timed_step(*a):
            t0 = time.perf_counter()
            r = step(*a)
            host.append(time.perf_counter() - t0)
            return r
        pbt.step = timed_step
    loop = wb.IndependentPPO(n, seed=3, pbt=pbt)
    for _ in range(args.warmup):
        loop.step()
    loop.timing = []
    copies0, host0 = len(loop._exploit), len(host)
    for _ in range(args.steps):
        flush.zero_()
        loop.step()
    torch.cuda.synchronize()
    ev = loop.timing
    loop.timing = None
    total = np.array([e[0].elapsed_time(e[4]) for e in ev])
    total_s = float(total.sum()) * 1e-3
    out = {"walkers": n, "pbt": with_pbt, "timed_steps": args.steps, "env_steps_per_s": n * args.steps / total_s, "step_ms": med(total)}
    if pbt is not None:
        xlog = loop.exploit_log()
        timed = xlog[xlog["step"] >= args.warmup]
        out.update({"copies_timed": int(len(timed)), "copies_per_step": len(timed) / args.steps,
                    "steps_with_copies": int(len(set(timed["step"].tolist()))), "copies_total": int(len(xlog)),
                    "schedule_host_ms_per_step": med(np.array(host[host0:]) * 1e3)})
    del loop
    torch.cuda.synchronize()
    return out


result = {"card": card(), "l2_flush_bytes": 256 << 20, "copy": {}, "loop": {}}
for net in ("default", "wide128"):
    result["copy"][net] = bench_copy(net)
for n in args.sizes:
    for with_pbt in (False, True):
        key = f"{n}_{'pbt' if with_pbt else 'no_pbt'}"
        result["loop"][key] = bench_loop(n, with_pbt)
        print(key, json.dumps(result["loop"][key]), flush=True)
result["card_after"] = card()
os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
with open(args.out, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", args.out)

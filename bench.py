#!/usr/bin/env python
"""bench.py -- walker env-steps/s of the lockstep physics step (BASELINE.json configs[1]) + PPO samples/s (configs[2]),
with the other BASELINE configs beside them in the same JSON line.

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, one process per GPU; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path (oracle port; rank 0 only)
  python bench.py ... --dump-outputs DIR                   also write the headline's last timed step (obs, reward, done) as
                                                           DIR/<name>.npy in float32 (DIR/<name>_rank<r>.npy for N > 1), so
                                                           that two builds can be compared output for output on identical inputs

Headline workload (config.workload): 4096 lockstep walkers per GPU, Wood floor (Carpet walker), i.i.d. U(-1,1) actions per joint
per env-step (seeded, generated once), dt = 0x1.111134p-6, Iterations = 50, auto-reset on terminal.  One "step" = one fused
env-step kernel over all walkers of the rank.  Multi-GPU: environments are block-sharded, no data-path collective on the physics
path (weak scaling, 4096 walkers per GPU).

Both arms first run PREROLL (512) untimed env-steps so that the batch is in the state a long rollout is in: decorrelated (right
after construction all walkers are identical, which flatters a SIMT kernel: no divergence) and past every walker's first reset
(the reference's body list changes order exactly once, at the first Walker.Reset -- Walker.cs:212-223).

Timing: every timed step is bracketed by CUDA events on the launching stream; between timed steps an L2 flush (256 MiB memset)
runs OUTSIDE the event pairs; ms_per_step = sum of the K event intervals / K, max over ranks.  --steps K is the number of timed
steps of every leg that reports "steps" (headline, e2e, at_scale, contact_stress, secondary); ppo_loop and cfg1 time the fixed
samples they describe.
"e2e" = the same step through the public host-buffer call (EnvBatch.step -> wb_env_step) with pinned host actions in and host
obs/reward/done out every step, wall clock around the call.

Keys beside the base contract (every one of them measured in this run, on this box):
  roofline       HBM accounting of the headline kernel (824 B per env-step; and 752 B x 50 as if the record crossed HBM every substep)
  cpu_baseline   the oracle port of the same physics workload on the box's host threads, rank 0, at EVERY N (bounded sample)
  at_scale       the same step on 262 144 walkers per GPU (throughput regime) + iterations_1 (one substep per launch: the record
                 really crosses HBM every substep)
  secondary      BASELINE configs[2]: PPO samples/s on one 65 536-sample minibatch (ONE launch: gradient + reduction + Adam), with
                 its own e2e (pinned host minibatch through PPOAgent.TrainBatch -> wb_ppo_train), roofline (tensor) and cpu_baseline (the oracle's
                 per-sample PPOAgent.Train(Batch) restatement, one thread like the reference)
  cfg1           BASELINE configs[0]: ONE walker -- the oracle port on one host thread (env-steps/s with a policy forward + sample
                 per step, and the per-sample PPO update) beside the same single-walker loop through this library
  ppo_loop       BASELINE configs[3]: the full PPO loop (rollout + returns + minibatch updates) on 65 536 walkers sharded over the
                 N ranks; at N > 1 once with the gradient kernel's fused reduce + all-reduce + Adam tail over NVLink peer memory and once with the
                 NCCL all-reduce: env-steps/s, samples/s, microseconds per minibatch update, spread of the weight checksums
  contact_stress BASELINE configs[4]: 16 384 walkers over the 8 floor materials, spin start, device-resident env-steps/s
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402
import workloads  # noqa: E402

N_ENVS_PER_GPU = 4096
N_ENVS_AT_SCALE = 262144   # "at_scale": the same step with the GPU full (one lane per walker)
N_ENVS_LOOP = 65536        # configs[3]: global walker count of the full PPO loop
N_ENVS_STRESS = 16384      # configs[4]
PREROLL = 512              # untimed env-steps before the warm-up: see the module docstring
SEED = 1234
BYTES_PER_ENV_STEP = 2 * 376 + 16 + 56   # SURVEY 8d: read state + actions, write state + obs/reward/done = 824 B
BYTES_PER_SUBSTEP = 2 * 376              # if the state round-tripped HBM every substep (it does not: 50 substeps are fused)
FLOP_PER_SAMPLE = 32640                  # MLP fwd + bwd (SURVEY 8d)
PPO_SAMPLES = 65536
REF_PASSES_PER_STEP = 12                 # reference arm: env-step passes per "step" (a bounded sample, ~0.1 s of CPU work each)
METRIC = "walker env-steps/sec (SAT physics step)"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernel.  ncu cannot run inside the timed bench, so the
    figure is read from the committed summary of this round's `ncu --set full` capture of the same kernel and workload
    (profiles/ncu_summary.json, written by scripts/ncu_summary.py); the provenance string travels with it."""
    path = os.path.join(ROOT, "profiles", "ncu_summary.json")
    try:
        rec = json.load(open(path))[kernel_key]
        return rec["dram_bytes_per_launch"], f"profiles/ncu_summary.json[{kernel_key}] ({rec.get('source', 'ncu --set full capture')})"
    except Exception:
        return None, "no ncu capture of this kernel in profiles/ncu_summary.json"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    """All host threads this process may use.  Passed to the oracle EXPLICITLY: torchrun exports OMP_NUM_THREADS=1 to its workers,
    which would silently turn the "all host threads" CPU arm into a single-threaded one."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def workload_config(n_gpus):
    """Identical for both arms (the reference arm runs the same N x 4096 walkers on the host)."""
    return {"workload": f"{N_ENVS_PER_GPU} lockstep walkers per GPU, physics step only, Wood ground, random actions "
                        "(BASELINE.json configs[1])",
            "walkers_per_gpu": N_ENVS_PER_GPU, "iterations": 50, "dt": "0x1.111134p-6", "floor": "Wood", "walker": "Carpet",
            "actions": f"U(-1,1) numpy PCG64 seed [{SEED}, rank]", "auto_reset": True, "preroll_env_steps": PREROLL,
            "parallelism": f"env-shard x{n_gpus}, no data-path collective",
            "l2": "256 MiB memset between timed steps, outside the event pairs"}


# ------------------------------------------------------------------------------------------------ CPU legs (oracle = checker, timed here only)
def cpu_physics_baseline(O, budget_s=12.0, max_steps=4000, nthreads=0):
    """The oracle port on the host cores: the headline workload, a bounded sample (~budget_s of CPU work)."""
    nthreads = nthreads if nthreads > 0 else host_threads()
    n = N_ENVS_PER_GPU
    env = O.EnvBatch(n, floor="Wood")
    acts = workloads.walker_actions(SEED, 0, n, 8)
    for k in range(PREROLL):
        env.step(acts[k % 8], nthreads=nthreads)  # pre-roll + warm-up
    t0 = time.perf_counter()
    k = 0
    while k < max_steps and (time.perf_counter() - t0) < budget_s:
        env.step(acts[k % 8], nthreads=nthreads)
        k += 1
    dt = time.perf_counter() - t0
    return {"value": n * k / dt, "unit": "env-steps/s", "cores": nthreads, "kind": "port",
            "sample": f"{k} env-steps x {n} walkers (Wood floor, U(-1,1) actions, auto-reset) after {PREROLL} pre-roll steps, "
                      f"OpenMP over walkers, {dt:.1f} s"}


def ppo_bench_inputs(rng, mean_fn):
    return workloads.ppo_minibatch(rng, PPO_SAMPLES, mean_fn)


def cpu_ppo_baseline(O, actor_flat, critic_flat, batch, budget_s=10.0):
    """The oracle's per-sample PPOAgent.Train(Batch) + Adam (PPOAgent.cs:218-346, DenseLayer.cs:103-159) on the SAME minibatch
    the GPU leg trains on, one thread (the reference's update is sequential by construction: every sample accumulates into the
    same layer gradients).  Bounded: as many samples of the minibatch as fit the budget, at least 8192."""
    actor, critic = O.Net(12, O.ACTOR_LAYERS), O.Net(12, O.CRITIC_LAYERS)
    actor.set_params(actor_flat)
    critic.set_params(critic_flat)
    hp = O.hyper_defaults()
    hp.batch_size = PPO_SAMPLES
    done, t0, chunk = 0, time.perf_counter(), 8192
    while done == 0 or time.perf_counter() - t0 < budget_s:   # whole passes over the minibatch until the budget is used
        sl = slice(done % PPO_SAMPLES, done % PPO_SAMPLES + chunk)
        O.ppo_train_batch(actor, critic, hp, *[x[sl] for x in batch], optimise=True)
        done += chunk
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "samples/s", "cores": 1, "kind": "port",
            "sample": f"{done} samples = {done / PPO_SAMPLES:.1f} passes over the {PPO_SAMPLES}-sample minibatch in chunks of {chunk} (forward + "
                      f"clipped-surrogate gradient + backward per sample, Adam per chunk), one thread, {dt:.1f} s"}


def cfg1_cpu(O, env_steps=1500, train_samples=8192):
    """BASELINE configs[0]: ONE walker on one host thread -- Environment.Update per step (critic + actor forward, Box-Muller
    sample, clip, 50 substeps, reward; Environment.cs:64-92) and PPOAgent.Train on the collected samples (batch 64, per sample)."""
    rng = np.random.default_rng(SEED + 2)
    actor, critic = O.Net(12, O.ACTOR_LAYERS), O.Net(12, O.CRITIC_LAYERS)
    import ppo_bipedalwalker_b200 as wbpkg  # host-side Xavier initialiser only (numpy)
    critic.set_params(wbpkg.xavier_flat(12, wbpkg.ParseLayers(wbpkg.DEFAULT_CRITIC), rng))
    actor.set_params(wbpkg.xavier_flat(12, wbpkg.ParseLayers(wbpkg.DEFAULT_ACTOR), rng))
    hp = O.hyper_defaults()
    env = O.EnvBatch(1, floor="Wood")
    obs = env.get_obs()
    S, A, LP, R = [], [], [], []
    u = rng.random((env_steps, 8)).astype(np.float32)
    t0 = time.perf_counter()
    for k in range(env_steps):
        a, lp, _ = O.sample_actions(actor, hp, obs[0], u[k])
        critic.forward(obs[0])
        S.append(obs[0].copy())
        obs, rew, done = env.step(a[None, :], nthreads=1)
        A.append(a)
        LP.append(lp)
        R.append(rew[0])
    dt_roll = time.perf_counter() - t0
    S, A, LP = np.asarray(S, np.float32), np.asarray(A, np.float32), np.asarray(LP, np.float32)
    reps = (train_samples + env_steps - 1) // env_steps
    S, A, LP = np.tile(S, (reps, 1))[:train_samples], np.tile(A, (reps, 1))[:train_samples], np.tile(LP, (reps, 1))[:train_samples]
    adv = rng.normal(size=train_samples).astype(np.float32)
    ret = rng.normal(size=train_samples).astype(np.float32)
    t0 = time.perf_counter()
    for j in range(train_samples // 64):
        sl = slice(j * 64, (j + 1) * 64)
        O.ppo_train_batch(actor, critic, hp, S[sl], A[sl], LP[sl], adv[sl], ret[sl], optimise=True)
    dt_train = time.perf_counter() - t0
    return {"env_steps_per_s": env_steps / dt_roll, "ppo_update_samples_per_s": train_samples / dt_train, "cores": 1, "kind": "port",
            "sample": f"{env_steps} env-steps of one walker (policy forward + sample + 50 substeps each), then {train_samples // 64} "
                      "minibatches of 64 through the per-sample update + Adam"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (no C#/.NET toolchain in the image, so the
    strict-fp32 C port in oracle/ stands in for it -- 'kind': 'port'), all host threads, rank 0 only.  Same config as our arm:
    N x 4096 walkers; one "step" = REF_PASSES_PER_STEP env-step passes over all of them (a bounded sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    O = ge.load_oracle()
    n = N_ENVS_PER_GPU * max(1, args.gpus)
    env = O.EnvBatch(n, floor="Wood")
    acts = np.concatenate([workloads.walker_actions(SEED, r, N_ENVS_PER_GPU, 16) for r in range(max(1, args.gpus))], axis=1)
    cores = host_threads()
    R = REF_PASSES_PER_STEP
    for w in range(PREROLL + args.warmup * R):
        env.step(acts[w % 16], nthreads=cores)
    t0 = time.perf_counter()
    for k in range(args.steps * R):
        env.step(acts[k % 16], nthreads=cores)
    dt = time.perf_counter() - t0
    value = n * args.steps * R / dt
    sample = (f"{args.steps} steps x {R} env-step passes x {n} walkers after {PREROLL} pre-roll passes, OpenMP over walkers on {cores} host "
              f"threads, {dt:.1f} s")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "passes_per_step": R, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU legs
class Ctx:
    """What every leg needs: torch, the package, the stream, rank/world, an L2 flush and a barrier."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.local_rank, self.world = (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
                                                  int(os.environ.get("WORLD_SIZE", "1")))
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{self.local_rank}"))
        self.wb = ge.load_package()
        self.wb.init(self.local_rank)  # raises without a CUDA device: there is no CPU fallback
        torch.cuda.set_device(self.local_rank)
        self.stream = torch.cuda.current_stream().cuda_stream
        self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush(self):
        self.flush_buf.zero_()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed_steps(self, fn, k):
        """sum of k CUDA-event intervals around fn(i), an L2 flush before each one outside the interval (ms)."""
        torch = self.torch
        total = 0.0
        for i in range(k):
            self.flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(i)
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
        return total


def bench_headline(cx, K, W):
    torch, wb = cx.torch, cx.wb
    n = N_ENVS_PER_GPU
    env = wb.EnvBatch(n, floor_materials="Wood", stream=cx.stream)
    acts_all = workloads.walker_actions(SEED, cx.rank, n, PREROLL + W + K)
    acts_pre, acts_host = acts_all[:PREROLL], acts_all[PREROLL:]
    acts_pre_dev = torch.from_numpy(acts_pre).cuda()
    acts_dev = torch.from_numpy(acts_host).cuda()
    obs_d = torch.empty(n, 12, device="cuda")
    rew_d = torch.empty(n, device="cuda")
    done_d = torch.empty(n, dtype=torch.uint8, device="cuda")
    # ---- device-resident throughput ("value")
    for w in range(PREROLL):
        env.step_dev(acts_pre_dev[w], obs_d, rew_d, done_d)
    for w in range(W):
        env.step_dev(acts_dev[w], obs_d, rew_d, done_d)
    cx.barrier()
    sampler = ClockSampler(cx.local_rank) if cx.rank == 0 else None
    l0 = env.launch_count()
    ndone = [0]

    def one(k):
        env.step_dev(acts_dev[W + k], obs_d, rew_d, done_d)

    total_ms = cx.timed_steps(one, K)
    ndone = int(done_d.sum().item())
    # what a caller of step_dev receives from the last timed step (the buffers are reused by the e2e leg below)
    outputs = {"obs": obs_d.cpu().numpy(), "reward": rew_d.cpu().numpy(), "done": done_d.cpu().numpy().astype(np.float32)}
    cx.barrier()
    launches = env.launch_count() - l0
    dev_ms = cx.max_over_ranks(total_ms) / K
    kernel_ms_local = total_ms / K
    # ---- end to end through the public API: pinned host actions in, host obs/reward/done out, every step
    env2 = wb.EnvBatch(n, floor_materials="Wood", stream=cx.stream)
    for w in range(PREROLL):
        env2.step_dev(acts_pre_dev[w], obs_d, rew_d, done_d)
    acts_pin = torch.from_numpy(acts_host).pin_memory()
    obs_h = torch.empty(n, 12).pin_memory()
    rew_h = torch.empty(n).pin_memory()
    done_h = torch.empty(n, dtype=torch.uint8).pin_memory()
    out = (obs_h.numpy(), rew_h.numpy(), done_h.numpy())
    for w in range(W):
        env2.step(acts_pin[w], out=out)
    cx.barrier()
    e2e_ms = 0.0
    for k in range(K):
        cx.flush()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        env2.step(acts_pin[W + k], out=out)  # H2D + kernel + D2H + stream sync inside the call
        e2e_ms += (time.perf_counter() - t0) * 1e3
    cx.barrier()
    e2e_ms_step = cx.max_over_ranks(e2e_ms) / K
    clocks = sampler.stop() if sampler else None
    hbm, _, which = measured_peaks()
    achieved = n * BYTES_PER_ENV_STEP / (kernel_ms_local * 1e-3) / 1e9
    achieved_sub = n * 50 * BYTES_PER_SUBSTEP / (kernel_ms_local * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic("physics_lanes_kernel_4096")
    return {
        "value": cx.world * n / (dev_ms * 1e-3), "ms_per_step": dev_ms,
        "e2e": {"value": cx.world * n / (e2e_ms_step * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": n * 16,
                "d2h_bytes_per_step": n * (48 + 4 + 1), "ms_per_step": e2e_ms_step,
                "path": "EnvBatch.step -> wb_env_step with pinned host buffers: the kernel reads the actions and writes "
                        "obs/reward/done through the buffers' device aliases (zero-copy over PCIe), one stream sync per step"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": f"physics kernel variant {env.get_variant()} (lanes per walker; 1001 = compacting)",
                     "note": f"824 B/env-step x {n} walkers per launch / CUDA-event launch time; peak = {which} copy bandwidth. "
                             "The 50 substeps are fused on chip, so the kernel is issue/latency-bound, not HBM-bound",
                     "substep_granular": {"achieved": achieved_sub, "frac": achieved_sub / hbm,
                                          "note": "752 B/substep x 50 substeps, as if the state round-tripped HBM every substep"}},
        "clocks": clocks, "episodes_finished_in_last_timed_step": ndone, "outputs": outputs,
    }


def bench_at_scale(cx, K):
    torch, wb = cx.torch, cx.wb
    na = N_ENVS_AT_SCALE
    env3 = wb.EnvBatch(na, floor_materials="Wood", stream=cx.stream)
    rng = np.random.default_rng([SEED, cx.rank, 7])
    acts3 = torch.from_numpy(rng.uniform(-1.0, 1.0, (8, na, 4)).astype(np.float32)).cuda()
    obs3 = torch.empty(na, 12, device="cuda")
    rew3 = torch.empty(na, device="cuda")
    done3 = torch.empty(na, dtype=torch.uint8, device="cuda")
    for w in range(PREROLL + 3):
        env3.step_dev(acts3[w % 8], obs3, rew3, done3)
    cx.barrier()
    tot3 = cx.timed_steps(lambda k: env3.step_dev(acts3[k % 8], obs3, rew3, done3), K)
    cx.barrier()
    ms3 = cx.max_over_ranks(tot3) / K
    hbm_peak = measured_peaks()[0]
    traffic, traffic_src = ncu_traffic("physics_kernel_262144")
    at_scale = {"value": cx.world * na / (ms3 * 1e-3), "unit": "env-steps/s", "walkers_per_gpu": na, "ms_per_step": ms3, "steps": K,
                "kernel_variant": env3.get_variant(),
                "roofline": {"bound": "hbm", "achieved": na * BYTES_PER_ENV_STEP / (ms3 * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": na * BYTES_PER_ENV_STEP / (ms3 * 1e-3) / 1e9 / hbm_peak,
                             "substep_granular_frac": na * 50 * BYTES_PER_SUBSTEP / (ms3 * 1e-3) / 1e9 / hbm_peak,
                             "traffic": traffic, "traffic_source": traffic_src}}
    # ---- Iterations = 1 (SURVEY 8d asks for it): ONE substep per launch from the state of the same batch, so the 376-byte record really
    #      crosses HBM twice per substep -- the measured counterpart of the "substep-granular" accounting above
    hp1 = wb.default_hyperparams()
    hp1.iterations = 1
    env4 = wb.EnvBatch(na, floor_materials="Wood", hp=hp1, stream=cx.stream)
    env4.set_state(*env3.get_state())
    del env3
    for w in range(3):
        env4.step_dev(acts3[w % 8], obs3, rew3, done3)
    cx.barrier()
    tot4 = cx.timed_steps(lambda k: env4.step_dev(acts3[k % 8], obs3, rew3, done3), K)
    cx.barrier()
    ms4 = cx.max_over_ranks(tot4) / K
    at_scale["iterations_1"] = {
        "value": cx.world * na / (ms4 * 1e-3), "unit": "substeps/s (Hyperparameters.Iterations = 1: one substep per env-step and per launch)",
        "ms_per_step": ms4, "steps": K, "kernel_variant": env4.get_variant(),
        "roofline": {"bound": "hbm", "achieved": na * BYTES_PER_ENV_STEP / (ms4 * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": na * BYTES_PER_ENV_STEP / (ms4 * 1e-3) / 1e9 / hbm_peak,
                     "note": "824 B per walker per launch (state in + out, actions, obs/reward/done)"}}
    del env4
    return at_scale


def bench_contact_stress(cx, K):
    """configs[4]: 16 384 walkers, 2 048 per floor material, spin start, random actions; device-resident env-steps/s after 16 steps
    (parity of exactly this workload: tests/test_physics_gpu.py::test_contact_stress_sweep_at_baseline_size)."""
    torch, wb = cx.torch, cx.wb
    n = N_ENVS_STRESS
    rng = np.random.default_rng([SEED, cx.rank, 5])
    probe = wb.EnvBatch(n, stream=cx.stream)
    f, iv = probe.get_state()
    del probe
    floors = workloads.contact_stress_start(n, n // 8, f, rng)
    env = wb.EnvBatch(n, floor_materials=floors, stream=cx.stream)
    env.set_state(f, iv)
    acts = torch.from_numpy(rng.uniform(-1, 1, (8, n, 4)).astype(np.float32)).cuda()
    obs = torch.empty(n, 12, device="cuda")
    rew = torch.empty(n, device="cuda")
    done = torch.empty(n, dtype=torch.uint8, device="cuda")
    for i in range(16):
        env.step_dev(acts[i % 8], obs, rew, done)
    cx.barrier()
    tot = cx.timed_steps(lambda i: env.step_dev(acts[i % 8], obs, rew, done), K)
    cx.barrier()
    ms = cx.max_over_ranks(tot) / K
    return {"value": cx.world * n / (ms * 1e-3), "unit": "env-steps/s", "walkers_per_gpu": n, "ms_per_step": ms, "steps": K,
            "kernel_variant": env.get_variant(),
            "config": {"workload": "contact-stress sweep: 16384 walkers per GPU, 2048 per floor material (Ice..SuperRubber), initial spin "
                                   "U(-5,5) per body, random actions, timed from env-step 16 (BASELINE.json configs[4])"}}


def bench_ppo(cx, steps, warmup):
    """configs[2]: PPO MLP fwd/bwd + clipped-surrogate gradient + Adam on a 65536-sample minibatch (synthetic obs)."""
    torch, wb = cx.torch, cx.wb
    n = PPO_SAMPLES
    rng = np.random.default_rng(SEED + 1)
    hp = wb.default_hyperparams()
    hp.batch_size = n
    agent = wb.PPOAgent(hp=hp, seed=42, stream=cx.stream)
    actor0, critic0 = agent.actor.get_flat().copy(), agent.critic.get_flat().copy()
    batch = ppo_bench_inputs(rng, lambda s: agent.FeedForward(s)[0])
    dev = [torch.from_numpy(x).cuda() for x in batch]
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    L = lib()

    def one(_):
        check(L.wb_ppo_train_dev(agent._h, n, *[ptr(t) for t in dev]))  # ONE launch: gradient + grid barrier + reduction + Adam

    for _ in range(warmup):
        one(0)
    torch.cuda.synchronize()
    l0 = agent.launch_count()
    ms = cx.timed_steps(one, steps) / steps
    launches = agent.launch_count() - l0
    # end to end through the host-buffer API: pinned host minibatch in (the kernel reads it in place over PCIe), losses out
    pinned = [torch.from_numpy(x).pin_memory().numpy() for x in batch]
    for _ in range(2):
        agent.TrainBatch(*pinned)
    e2e_ms = 0.0
    for _ in range(steps):
        cx.flush()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        agent.TrainBatch(*pinned)   # wb_ppo_train: one launch reading the pinned minibatch in place, D2H of the losses, sync
        agent.sync()
        e2e_ms += (time.perf_counter() - t0) * 1e3
    e2e_ms /= steps
    _, tflops, which = measured_peaks()
    achieved = n * FLOP_PER_SAMPLE / (ms * 1e-3) / 1e12
    traffic, traffic_src = ncu_traffic("ppo_tc_kernel")
    out = {"metric": "PPO samples/sec (MLP fwd/bwd + clipped-surrogate grad + Adam)", "value": n / (ms * 1e-3), "unit": "samples/s",
           "ms_per_step": ms, "steps": steps, "dtype": "f32 (3xTF32 on tcgen05)",
           "config": {"workload": "65536-sample minibatch, synthetic obs (BASELINE.json configs[2])"},
           "gpu_launches": launches,
           "e2e": {"value": n / (e2e_ms * 1e-3), "unit": "samples/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": n * 22 * 4,
                   "d2h_bytes_per_step": 12, "path": "PPOAgent.TrainBatch -> wb_ppo_train: ONE launch (gradient + reduction + Adam) that reads the pinned host "
                                                      "minibatch in place over PCIe (zero-copy), then a 12-byte D2H of the losses + sync"},
           "roofline": {"bound": "tensor", "achieved": achieved, "peak": tflops, "unit": "TFLOP/s", "frac": achieved / tflops,
                        "traffic": traffic, "traffic_source": traffic_src,
                        "note": f"32640 flop/sample; peak = {which} dense bf16 (the kernel computes in fp32 accuracy: 3xTF32 on tcgen05)"}}
    return out, (actor0, critic0, batch)


def bench_cfg1_gpu(cx, env_steps=300):
    """configs[0] through this library: ONE walker, per step SampleActions (host state in, action out) + Environment.Update
    (host action in, observation out) -- the call pattern of the reference's game loop.  A single walker leaves the GPU idle:
    the number is reported for completeness (the path pays off from a few hundred lockstep walkers upwards)."""
    wb = cx.wb
    agent = wb.PPOAgent(seed=7, stream=cx.stream)
    env = wb.Environment(1, floor="Wood")
    obs = env.InitialState()
    rng = np.random.default_rng(3)
    u = rng.random((env_steps + 20, 1, 4, 2)).astype(np.float32)
    for k in range(20):
        a, lp, mu, sd = agent.SampleActions(obs, u[k])
        obs, r, d = env.Update(wb.DT_FRAME, a)
    cx.torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(env_steps):
        a, lp, mu, sd = agent.SampleActions(obs, u[20 + k])
        obs, r, d = env.Update(wb.DT_FRAME, a)
    dt = time.perf_counter() - t0
    return {"env_steps_per_s": env_steps / dt, "sample": f"{env_steps} env-steps of one walker, SampleActions + Environment.Update per step, "
                                                          "host buffers in and out every call"}


def bench_ppo_loop(cx, fused):
    """configs[3]: 65 536 walkers sharded over the ranks, horizon 64, global minibatch 65 536, one epoch: rollout (2 launches per
    env-step) + bootstrap value + returns + 64 minibatch updates, each ONE launch that reads its permuted rows of the pool,
    reduces, exchanges the gradient over NVLink peer memory and applies Adam (or: gather + gradient kernel + NCCL all-reduce + Adam)."""
    torch = cx.torch
    vp = cx.wb.VectorPPO(N_ENVS_LOOP, horizon=64, minibatch_global=65536, epochs=1, floor="Wood", seed=11, fused_allreduce=fused)
    vp.iterate()  # warm-up (also takes the walkers off the identical start state)
    cx.barrier()
    its = 2
    roll = upd = 0.0
    n_mb = 0
    for _ in range(its):
        s = vp.iterate()
        roll += s["rollout_ms"]
        upd += s["update_ms"]
        n_mb += s["minibatches"]
    cx.barrier()
    roll, upd = cx.max_over_ranks(roll), cx.max_over_ranks(upd)
    env_steps = its * N_ENVS_LOOP * 64
    cs = torch.tensor([vp.weights_checksum()], device="cuda", dtype=torch.float64)
    lo, hi = cs.clone(), cs.clone()
    if cx.world > 1:
        cx.dist.all_reduce(lo, op=cx.dist.ReduceOp.MIN)
        cx.dist.all_reduce(hi, op=cx.dist.ReduceOp.MAX)
    out = {"exchange": ("one launch per minibatch: gradient kernel with fused reduce + all-reduce (NVLink peer memory) + Adam tail"
                        if (vp.fused and cx.world > 1) else
                        "gather + gradient kernel + NCCL all-reduce + Adam kernel" if cx.world > 1 else
                        "single rank: one launch per minibatch (gradient + reduction + Adam), nothing exchanged"),
           "loop_env_steps_per_s": env_steps / ((roll + upd) * 1e-3), "rollout_env_steps_per_s": env_steps / (roll * 1e-3),
           "update_samples_per_s": n_mb * 65536 / (upd * 1e-3), "us_per_minibatch_update": upd / n_mb * 1e3,
           "minibatches": n_mb, "iterations": its, "weights_checksum_spread": float((hi - lo).item())}
    del vp
    return out


def dump_outputs(out_dir, arrays, suffix):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), np.ascontiguousarray(a, np.float32))


def run_ours(args):
    cx = Ctx()
    K, W = args.steps, args.warmup
    head = bench_headline(cx, K, W)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, head["outputs"], f"_rank{cx.rank}" if cx.world > 1 else "")
    at_scale = bench_at_scale(cx, K)
    stress = bench_contact_stress(cx, K)
    loops = []
    if not args.no_loop:
        loops.append(bench_ppo_loop(cx, fused=True))
        if cx.world > 1:
            loops.append(bench_ppo_loop(cx, fused=False))
    line = None
    if cx.rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "env-steps/s",
            "n_gpus": cx.world, "steps": K, "warmup": W, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(cx.world),
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "clocks": head["clocks"],
            "episodes_finished_in_last_timed_step": head["episodes_finished_in_last_timed_step"],
            "at_scale": at_scale, "contact_stress": stress,
        }
        if loops:
            line["ppo_loop"] = {"config": {"workload": f"full PPO loop, {N_ENVS_LOOP} walkers sharded over {cx.world} GPU(s), horizon 64, global "
                                                       "minibatch 65536, 1 epoch (BASELINE.json configs[3])"}, "runs": loops}
        if not args.no_ppo:
            line["secondary"], ppo_ctx = bench_ppo(cx, K, W)
            if cx.world == 1:
                line["cfg1"] = {"config": {"workload": "single BipedalWalker env, physics step + PPO rollout/update (BASELINE.json configs[0])"},
                                "gpu": bench_cfg1_gpu(cx)}
        # the CPU legs: rank 0 only, while the other ranks wait at the store barrier below without spinning on a core
        O = ge.load_oracle()
        line["cpu_baseline"] = cpu_physics_baseline(O)
        if not args.no_ppo:
            line["secondary"]["cpu_baseline"] = cpu_ppo_baseline(O, *ppo_ctx)
            if cx.world == 1:
                line["cfg1"]["cpu"] = cfg1_cpu(O)
    if cx.world > 1:
        store = cx.dist.distributed_c10d._get_default_store()
        if cx.rank == 0:
            store.set("wb_cpu_legs_done", "1")
        else:
            store.wait(["wb_cpu_legs_done"])
    if line is not None:
        print(json.dumps(line))
    if cx.world > 1:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-ppo", action="store_true")
    ap.add_argument("--no-loop", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline's last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

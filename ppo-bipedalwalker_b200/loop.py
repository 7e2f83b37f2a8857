"""Lockstep PPO loop over N walkers, everything resident on the GPU(s) (BASELINE.json configs[3]; SURVEY.md 8e / 8f rows 1-2).

What the reference does for ONE walker per episode -- Environment.Update (Environment.cs:64-92): record state, SampleActions,
TakeActions(Clip(a)), Step, record action / log-probability / reward, and at the end PPOAgent.Train (PPOAgent.cs:147-172):
values, returns, advantages, Epochs x shuffled mini-batches of Train(Batch) -- runs here for N walkers at once:

  rollout   `horizon` env-steps; per env-step TWO kernel launches: wb_policy_act_dev (actor + critic + Philox Box-Muller sampling +
            log-probabilities) and wb_env_step_dev (the fused physics step with auto-reset; wb_terrain_env_step_dev when the
            walkers train on a terrain other than the flat floor).  The trajectory (states, UNCLIPPED
            actions and their log-probabilities -- Environment.cs:87-88 --, rewards, dones, values) stays in HBM, time-major.
  update    wb_segment_returns_dev (MC return / the reference's GAE per episode fragment; a fragment that is still running at the
            end of the horizon is bootstrapped with the critic's value of the next observation -- the reference never meets this
            case because it trains on complete episodes only; `bootstrap=False` truncates instead), optionally
            PPOAgent.Normalize over the global pool (two 2 KB all-reduces), then `epochs` x (pool / minibatch)
            mini-batches: index permutation (sampling without replacement, remainder dropped, PPOAgent.cs:501-540) ->
            wb_ppo_train_indexed_dev: ONE launch per mini-batch (the tensor-core gradient kernel reads the permuted rows of the
            pool directly, reduces its per-CTA partials behind a grid barrier, all-reduces the 6 152-float buffer over NVLink
            peer memory and applies Adam in its tail).  `fused_allreduce=False`: wb_gather_minibatch_dev -> wb_ppo_grad_dev ->
            NCCL all-reduce -> wb_adam_step (the fallback and cross-check).

Multi-GPU (one process per GPU, torchrun): the walkers are block-sharded, rollouts never communicate; every rank draws its
share (minibatch / world) of each global mini-batch from its OWN pool, gradients are divided by the GLOBAL batch size inside
the kernel, so one all-reduce(sum) per mini-batch makes every rank apply the identical Adam step (weights stay bit-identical
across ranks).  PyTorch is used for device buffers, the permutation and process-group plumbing only.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np

from . import dist as _dist
from ._lib import ACT, OBS, Hyperparams, check, lib, ptr
from .env import DT_FRAME, EnvBatch, default_hyperparams
from .ppo import PPOAgent
from .scene import IObject, TerrainEnvBatch


class VectorPPO:
    def __init__(self, n_envs_global: int, horizon: int = 64, minibatch_global: int = 65536, epochs: int = 1,
                 floor="Metal", walker="Carpet", hp: Hyperparams | None = None, seed: int = 0, policy_variant: int | None = None,
                 fused_allreduce: bool = True, bootstrap: bool = True, terrain=None):
        """terrain: None (the reference's flat floor of material `floor`, wb_env_*), or an IObject list in its place (e.g.
        CreateRoughFloor(heights)) shared by every walker, or a list of n_envs_global such lists, indexed by the GLOBAL walker
        index (wb_terrain_env_*; `floor` is then unused: the terrain bodies carry their materials)."""
        import torch
        self.torch = torch
        self.rank, self.local_rank, self.world = _dist.world()
        # equal shards: every rank must issue the same number of gradient exchanges per update (an uneven split would leave
        # the fused exchange waiting for a peer that has no mini-batch left)
        assert n_envs_global % self.world == 0, "n_envs_global must be a multiple of the number of ranks"
        lo, hi = _dist.shard_range(n_envs_global, self.rank, self.world)
        self.n = hi - lo
        self.env_offset = lo
        self.n_global = n_envs_global
        self.T = horizon
        assert minibatch_global % self.world == 0, "the global mini-batch must split evenly over the ranks"
        self.mb_global = minibatch_global
        self.mb_local = minibatch_global // self.world
        self.pool_local = self.n * self.T
        assert self.pool_local >= self.mb_local, "local rollout pool smaller than the local mini-batch share"
        self.epochs = epochs
        self.bootstrap = bool(bootstrap)
        self.seed = seed
        self.hp = hp if hp is not None else default_hyperparams()
        self.hp.batch_size = minibatch_global  # the divisor B of every per-sample gradient (PPOAgent.cs:326,333)
        self.stream = torch.cuda.current_stream().cuda_stream
        if terrain is None:
            self.env = EnvBatch(self.n, floor_materials=floor, walker_materials=walker, hp=self.hp, stream=self.stream)
            self._env_step_dev = lib().wb_env_step_dev
        else:
            terrain = list(terrain)
            if terrain and not isinstance(terrain[0], IObject):  # one list per walker: this rank's block of the global index
                assert len(terrain) == n_envs_global, "a per-walker terrain needs one IObject list per walker"
                terrain = terrain[lo:hi]
            self.env = TerrainEnvBatch(self.n, terrain, walker_material=walker, hp=self.hp, stream=self.stream)
            self._env_step_dev = lib().wb_terrain_env_step_dev
        self.agent = PPOAgent(hp=self.hp, seed=seed, stream=self.stream)  # same seed -> identical Xavier weights on every rank
        if policy_variant is not None:
            self.agent.set_variant(policy_variant)
        dev = f"cuda:{torch.cuda.current_device()}"
        f32 = dict(device=dev, dtype=torch.float32)
        n, T = self.n, self.T
        self.states = torch.empty(T, n, OBS, **f32)
        self.actions = torch.empty(T, n, ACT, **f32)
        self.logp = torch.empty(T, n, ACT, **f32)
        self.rewards = torch.empty(T, n, **f32)
        self.values = torch.empty(T, n, **f32)
        self.dones = torch.empty(T, n, device=dev, dtype=torch.uint8)
        self.returns = torch.empty(T, n, **f32)
        self.adv = torch.empty(T, n, **f32)
        self.obs = torch.from_numpy(self.env.get_obs()).to(dev)  # Environment.InitialState
        self.mb = [torch.empty(self.mb_local, OBS, **f32), torch.empty(self.mb_local, ACT, **f32), torch.empty(self.mb_local, ACT, **f32),
                   torch.empty(self.mb_local, **f32), torch.empty(self.mb_local, **f32)]
        self.last_values = torch.empty(n, **f32)
        self.norm_stats = _dist.norm_stats_tensor(self.agent)
        self.grad_view = _dist.grad_tensor(self.agent)
        # multi-GPU: the gradient all-reduce is fused into the reduction kernel (NVLink peer memory, dist.connect_peers);
        # fused_allreduce=False keeps the NCCL all-reduce (same result, one more launch + the NCCL latency per mini-batch)
        self.fused = bool(fused_allreduce) and _dist.connect_peers(self.agent)
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(seed * 1000003 + self.rank)
        self.step_counter = 0
        self.iterations = 0

    # -- rollout: `horizon` lockstep env-steps, 2 launches each
    def rollout(self):
        L = lib()
        h_agent, h_env = self.agent._h, self.env._h
        for t in range(self.T):
            self.states[t].copy_(self.obs)
            # distinct Philox streams per rank: the counter is (local sample index, action dim, step)
            check(L.wb_policy_act_dev(h_agent, self.n, ptr(self.obs), self.seed * 7919 + self.rank, self.step_counter, ptr(self.actions[t]),
                                      ptr(self.logp[t]), None, ptr(self.values[t])))
            check(self._env_step_dev(h_env, ptr(self.actions[t]), C.c_float(DT_FRAME), 1, ptr(self.obs), ptr(self.rewards[t]),
                                     ptr(self.dones[t])))
            self.step_counter += 1

    # -- update: returns/advantages, epochs x mini-batches with one all-reduce each
    def update(self):
        torch = self.torch
        L = lib()
        h = self.agent._h
        last = None
        if self.bootstrap:  # V(s_T): one more critic forward on the observation the rollout ended on
            check(L.wb_policy_forward_dev(h, self.n, ptr(self.obs), None, ptr(self.last_values)))
            last = self.last_values
        normalize = bool(self.hp.normalize_advantages)
        if normalize and self.world > 1:
            self.hp.normalize_advantages = 0  # the stages run below with an all-reduce in between
            self.agent.set_hyperparams(self.hp)
        check(L.wb_segment_returns_dev(h, self.n, self.T, ptr(self.rewards), ptr(self.values), ptr(self.dones), ptr(last), ptr(self.returns),
                                       ptr(self.adv)))
        if normalize and self.world > 1:
            self.hp.normalize_advantages = 1
            self.agent.set_hyperparams(self.hp)
            pool_global = self.pool_local * self.world
            for stage in (0, 1, 2):  # PPOAgent.Normalize over the GLOBAL pool: sum -> all-reduce -> squared deviations -> all-reduce -> apply
                check(L.wb_normalize_advantages_dev(h, stage, self.pool_local, pool_global, ptr(self.adv)))
                if stage < 2:
                    _dist.allreduce_sum_(self.norm_stats)
        S, A, LP = self.states.view(-1, OBS), self.actions.view(-1, ACT), self.logp.view(-1, ACT)
        ADV, RET = self.adv.view(-1), self.returns.view(-1)
        n_mb = self.pool_local // self.mb_local
        losses = None
        for _ in range(self.epochs):
            perm = torch.randperm(self.pool_local, generator=self.gen, device=S.device, dtype=torch.int32)
            for j in range(n_mb):
                idx = perm[j * self.mb_local:(j + 1) * self.mb_local]
                if self.fused or self.world == 1:
                    # ONE launch per mini-batch: the gradient kernel reads rows idx[] of the pool (CreateBatches fused into its
                    # prefetch), reduces its partials, all-reduces them over NVLink peer memory and applies Adam in its tail
                    check(L.wb_ppo_train_indexed_dev(h, self.mb_local, ptr(idx), ptr(S), ptr(A), ptr(LP), ptr(ADV), ptr(RET)))
                else:
                    check(L.wb_gather_minibatch_dev(h, self.mb_local, ptr(idx), ptr(S), ptr(A), ptr(LP), ptr(ADV), ptr(RET), *[ptr(m) for m in self.mb]))
                    check(L.wb_ppo_grad_dev(h, self.mb_local, *[ptr(m) for m in self.mb]))
                    _dist.allreduce_sum_(self.grad_view)
                    check(L.wb_adam_step(h))
        if self.fused and self.world > 1:
            # a peer that never arrived leaves stale slices unapplied and the replicas out of step: fail loudly, once per update
            world, failed = C.c_int32(0), C.c_int32(0)
            check(L.wb_comm_status(h, C.byref(world), C.byref(failed)))
            if failed.value:
                raise RuntimeError("fused gradient exchange timed out: a rank never arrived; the replicas' weights may differ")
        losses = self.grad_view[-3:].clone()  # [sum g_V, sum mean_k g_mu, skipped] of the last mini-batch (PPOAgent.cs:331-332)
        return n_mb * self.epochs, losses

    def iterate(self):
        """One rollout + one update; returns a dict of device-timed statistics (this rank's share)."""
        torch = self.torch
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        self.rollout()
        e[1].record()
        n_mb, losses = self.update()
        e[2].record()
        e[2].synchronize()
        self.iterations += 1
        return {"rollout_ms": e[0].elapsed_time(e[1]), "update_ms": e[1].elapsed_time(e[2]), "minibatches": n_mb,
                "env_steps": self.n * self.T, "samples_trained": n_mb * self.mb_local,
                "mean_reward": float(self.rewards.mean().item()), "episodes_finished": int(self.dones.sum().item()),
                "losses": [float(x) for x in losses.tolist()]}

    def weights_checksum(self) -> float:
        """Sum of |w| over both networks -- identical on every rank when the data-parallel update is consistent."""
        return float(np.abs(self.agent.actor.get_flat()).sum() + np.abs(self.agent.critic.get_flat()).sum())


__all__ = ["VectorPPO"]

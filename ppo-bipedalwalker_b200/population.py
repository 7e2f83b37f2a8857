"""One PPO brain per walker: a population of independent agents (wb_population_*).

In the reference every walker owns its agent -- new Walker() builds its own PPOAgent(12, 4) (Walker.cs:25-34) -- and trains it on
each of its own episodes as soon as the episode ends (Environment.cs:91,157-164 -> PPOAgent.Train(Trajectory), PPOAgent.cs:147-172).
Running the reference N times gives N independent learners, which is how seed studies and hyper-parameter sweeps are run.

  PPOPopulation   P agents with the same two networks (the defaults, or any the DSL describes), each with its own weights, Adam
                  state, step counters and Hyperparams.  Agent a is exactly PPOAgent(actor=, critic=, seed=seeds[a], hp=hp[a]) (kernel
                  variant 1 for the default networks): same initial weights, same actions, same training.
  IndependentPPO  N walkers, N agents, the reference's episode semantics for every walker at once: no segments, no bootstrap; a
                  walker whose episode ended (Terminal, or steps > MaxTimesteps) trains its agent on the complete episode before it
                  acts again (Environment.Update -> TrainNetworks -> Reset).
  PBT             population-based training for IndependentPPO: lagging agents copy a leader's weights and Adam state and
                  perturb its hyper-parameters (an extension; the reference's agents are independent).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import ACT, OBS, Hyperparams, check, lib, ptr
from .env import DT_FRAME, EnvBatch, default_hyperparams
from .ppo import DEFAULT_ACTOR, DEFAULT_CRITIC, dense_shapes, resolve_networks, weights_lines, xavier_flat
from .scene import IObject, TerrainEnvBatch


def default_seeds(seed: int, n_agents: int) -> list[int]:
    """The agents' seeds when none are given: numpy's SeedSequence(seed).generate_state(n_agents, uint64)."""
    return [int(s) for s in np.random.SeedSequence(seed).generate_state(n_agents, np.uint64)]


class PPOPopulation:
    """n_agents independent PPOAgent(stateSize, actionSize) (PPOAgent.cs:23-37) on one device handle, all with the networks of the
    DSL strings actor / critic (PPOAgent.__init__'s fallbacks apply).

    hp: None (the defaults), one Hyperparams shared by every agent, or a list of n_agents of them (a sweep:
    [Settings(...).to_hyperparams(), ...]).  seeds[a] seeds agent a's numpy Generator exactly as PPOAgent(seed=seeds[a]) does: its
    Xavier initialisation, its Box-Muller uniforms and its mini-batch permutations; default: default_seeds(seed, n_agents)."""

    def __init__(self, n_agents: int, hp=None, seed: int = 0, seeds=None, stream: int | None = None, actor: str = DEFAULT_ACTOR,
                 critic: str = DEFAULT_CRITIC, stateSize: int = OBS, actionSize: int = ACT):
        if hp is None:
            hps = [default_hyperparams() for _ in range(n_agents)]
        elif isinstance(hp, Hyperparams):
            hps = [Hyperparams.from_buffer_copy(hp) for _ in range(n_agents)]
        else:
            hps = [Hyperparams.from_buffer_copy(h) for h in hp]
            if len(hps) != n_agents:
                raise ValueError(f"{len(hps)} Hyperparams for {n_agents} agents")
        self.n, self.hp = n_agents, hps
        self.stateSize, self.actionSize = stateSize, actionSize
        self.actor_structure, self.actor_layers, self.critic_structure, self.critic_layers = resolve_networks(actor, critic, actionSize)
        lists = []
        for layers in (self.actor_layers, self.critic_layers):
            lists += [np.array([k for k, _ in layers], np.int32), np.array([s for _, s in layers], np.int32)]
        h = C.c_void_p()
        check(lib().wb_population_create_net(n_agents, stateSize, actionSize, ptr(lists[0]), ptr(lists[1]), len(self.actor_layers),
                                             ptr(lists[2]), ptr(lists[3]), len(self.critic_layers), (Hyperparams * max(n_agents, 1))(*hps),
                                             C.byref(h)))
        self._h = h
        counts = []
        for which in (0, 1):
            n = C.c_int32(0)
            check(lib().wb_population_num_params(h, which, C.byref(n)))
            counts.append(n.value)
        self.N_ACTOR, self.N_PARAMS = counts[0], counts[0] + counts[1]
        self.n_dense = len(dense_shapes(stateSize, self.actor_layers)) + len(dense_shapes(stateSize, self.critic_layers))
        if stream is not None:
            self.set_stream(stream)
        self.seeds = default_seeds(seed, n_agents) if seeds is None else [int(s) for s in seeds]
        if len(self.seeds) != n_agents:
            raise ValueError(f"{len(self.seeds)} seeds for {n_agents} agents")
        self.rngs = []
        for a in range(n_agents):  # PPOAgent.__init__: critic first, then actor, from the agent's own generator
            rng = np.random.default_rng(self.seeds[a])
            critic_w = xavier_flat(stateSize, self.critic_layers, rng)
            actor_w = xavier_flat(stateSize, self.actor_layers, rng)
            self.set_weights(a, np.concatenate([actor_w, critic_w]))
            self.rngs.append(rng)

    def close(self):
        if getattr(self, "_h", None) and lib is not None:
            lib().wb_population_destroy(self._h)
            self._h = None

    __del__ = close

    def set_stream(self, cuda_stream: int):
        check(lib().wb_population_set_stream(self._h, C.c_void_p(cuda_stream)))

    def sync(self):
        check(lib().wb_population_sync(self._h))

    def launch_count(self) -> int:
        out = C.c_int64(0)
        check(lib().wb_population_launch_count(self._h, C.byref(out)))
        return out.value

    # -- per-agent state
    def get_weights(self, agent: int) -> np.ndarray:
        """[N_PARAMS] actor | critic of one agent (the flat layout of PPOAgent.actor / .critic get_flat, concatenated)."""
        out = np.empty(self.N_PARAMS, np.float32)
        check(lib().wb_population_get_weights(self._h, agent, ptr(out)))
        return out

    def set_weights(self, agent: int, flat):
        flat = np.ascontiguousarray(flat, np.float32)
        assert flat.size == self.N_PARAMS
        check(lib().wb_population_set_weights(self._h, agent, ptr(flat)))

    def get_grads(self, agent: int) -> np.ndarray:
        out = np.empty(self.N_PARAMS, np.float32)
        check(lib().wb_population_get_grads(self._h, agent, ptr(out)))
        return out

    def adam(self, agent: int):
        """(m [N_PARAMS], v [N_PARAMS], step counters [n_dense]: actor layers, then critic layers) of one agent."""
        m, v = np.empty(self.N_PARAMS, np.float32), np.empty(self.N_PARAMS, np.float32)
        steps = np.zeros(self.n_dense, np.int32)
        check(lib().wb_population_get_adam(self._h, agent, ptr(m), ptr(v), ptr(steps)))
        return m, v, steps

    def set_adam(self, agent: int, m, v, steps):
        """The mirror of adam(): m / v [N_PARAMS], step counters [n_dense]."""
        m, v = np.ascontiguousarray(m, np.float32), np.ascontiguousarray(v, np.float32)
        steps = np.ascontiguousarray(steps, np.int32)
        assert m.size == v.size == self.N_PARAMS and steps.size == self.n_dense
        check(lib().wb_population_set_adam(self._h, agent, ptr(m), ptr(v), ptr(steps)))

    def set_hyperparams(self, agent: int, hp: Hyperparams):
        check(lib().wb_population_set_hyperparams(self._h, agent, C.byref(hp)))
        self.hp[agent] = Hyperparams.from_buffer_copy(hp)

    def copy_agents(self, pairs, hp=None):
        """PBT's exploit step in one launch, enqueued on the population's stream: for each (dst, src) of pairs, dst's weights, Adam
        m / v and step counters become src's, bit for bit, and its hyper-parameters hp[i] (hp None: src's).  dst keeps its own
        generator rngs[dst], its count of trained episodes (which keys its device-drawn mini-batches) and its gradient buffer.  A
        dst listed twice, dst == src or an agent that is both a src and a dst is refused."""
        pairs = np.ascontiguousarray(np.asarray(pairs, np.int64).reshape(-1, 2), np.int32)
        dst, src = np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1])
        hps = None
        if hp is not None:
            if len(hp) != len(pairs):
                raise ValueError(f"{len(hp)} Hyperparams for {len(pairs)} pairs")
            hps = (Hyperparams * len(pairs))(*hp)
        check(lib().wb_population_copy_agents(self._h, len(pairs), ptr(dst), ptr(src), hps))
        new = [Hyperparams.from_buffer_copy(hps[i] if hps is not None else self.hp[s]) for i, s in enumerate(src)]
        for d, h in zip(dst, new):
            self.hp[d] = h

    def Save(self, agent: int):
        """PPOAgent.Save (PPOAgent.cs:192-213) of one agent -> (critic lines, actor lines) of the two .weights files."""
        flat = self.get_weights(agent)
        return (weights_lines(self.critic_structure, dense_shapes(self.stateSize, self.critic_layers), flat[self.N_ACTOR:]),
                weights_lines(self.actor_structure, dense_shapes(self.stateSize, self.actor_layers), flat[:self.N_ACTOR]))

    # -- acting
    def SampleActions(self, states, uniforms=None):
        """PPOAgent.SampleActions (PPOAgent.cs:381-398) of every agent on its walker's state: states [P][12] -> (actions, logp, mean,
        std), each [P][actionSize].  uniforms [P][actionSize][2] (injected), default: one draw of shape (1, actionSize, 2) from each
        agent's own generator."""
        ACT_ = self.actionSize
        s = np.ascontiguousarray(states, np.float32).reshape(self.n, self.stateSize)
        if uniforms is None:
            uniforms = np.concatenate([rng.random((1, ACT_, 2)) for rng in self.rngs])
        u = np.ascontiguousarray(uniforms, np.float32).reshape(self.n, ACT_, 2)
        actions, logp, mean = (np.empty((self.n, ACT_), np.float32) for _ in range(3))
        check(lib().wb_population_sample(self._h, self.n, ptr(s), ptr(u), ptr(actions), ptr(logp), ptr(mean)))
        std = np.array([[np.exp(np.float32(h.log_std))] * ACT_ for h in self.hp], np.float32)  # GetStandardDeviations, PPOAgent.cs:367-378
        return actions, logp, mean, std

    # -- training
    def TrainTrajectories(self, pairs, epochs: int = 5):
        """PPOAgent.Train(Trajectory) (PPOAgent.cs:147-172) for a list of (agent, Trajectory), in ONE call and one launch: every agent
        trains its own trajectories in list order, so it ends exactly where its PPOAgent.TrainTrajectories of its sub-list ends.  The
        permutations come from each agent's own generator in the order PPOAgent.TrainTrajectories draws them.  Fills Values /
        Returns / Advantages; returns [(criticLoss, actorLoss)] per pair."""
        pairs = list(pairs)
        if not pairs:
            return []
        agents = np.array([a for a, _ in pairs], np.int32)
        if agents.min() < 0 or agents.max() >= self.n:
            raise ValueError(f"agent outside 0..{self.n - 1}")
        trajectories = [t for _, t in pairs]
        lengths = [len(t.States) for t in trajectories]
        offsets = np.zeros(len(pairs) + 1, np.int32)
        offsets[1:] = np.cumsum(lengths)
        blocks = []
        for a, T in zip(agents, lengths):
            if T == 0:  # Train returns before drawing
                continue
            B, rng = self.hp[a].batch_size, self.rngs[a]
            for _ in range(epochs):
                perm = rng.permutation(T)
                blocks.extend(perm[j * B:(j + 1) * B] for j in range(T // B))
        index = np.ascontiguousarray(np.concatenate(blocks) if blocks else np.zeros(0), np.int32)
        rows = int(offsets[-1])

        def rows_of(attr, width):
            parts = [np.asarray(getattr(t, attr), np.float32).reshape(-1, width) for t in trajectories if len(t.States)]
            return np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros((0, width), np.float32))
        S, A, LP = rows_of("States", self.stateSize), rows_of("Actions", self.actionSize), rows_of("LogProbabilities", self.actionSize)
        R = rows_of("Rewards", 1).reshape(rows)
        V, G, Adv = (np.empty(rows, np.float32) for _ in range(3))
        losses = np.zeros((len(pairs), 2), np.float32)
        skipped = np.zeros(len(pairs), np.int32)
        check(lib().wb_population_train_trajectories(self._h, len(pairs), ptr(agents), ptr(offsets), epochs, ptr(S), ptr(A), ptr(LP), ptr(R),
                                                     ptr(index), ptr(V), ptr(G), ptr(Adv), ptr(losses), ptr(skipped)))
        for t, o, T in zip(trajectories, offsets, lengths):
            if T:
                t.Values, t.Returns, t.Advantages = list(V[o:o + T]), list(G[o:o + T]), list(Adv[o:o + T])
        return [(float(c), float(a)) for c, a in losses]


PERTURBABLE = ("alpha", "beta1", "beta2", "adam_epsilon", "gamma", "lambda_", "epsilon", "log_std")  # wb_hyperparams field order
DEFAULT_PERTURB = {"alpha": (1e-5, 1e-2), "epsilon": (0.05, 0.5), "log_std": (-3.0, 0.0)}


class PBT:
    """Population-based training schedule for IndependentPPO (host only: it decides the copies, IndependentPPO issues them).

    History and score.  Each agent keeps the reward sums of the episodes it finished since its last copy, or since the start.
    Its score is the float64 mean of the last `window` of them; an agent with fewer than `window` episodes is unranked.

    Snapshot.  After the training of every env-step t with (t + 1) % interval == 0, a snapshot of the ranked agents is taken:
    score descending, ties broken by the lower agent index first.  With m ranked agents, k = floor(fraction * m); the top set is
    the first k, the bottom set the last k (0 <= fraction <= 0.5, so the two are disjoint).  It replaces the previous snapshot.

    Copy.  An agent in the current snapshot's bottom set copies once per snapshot: at the end of the first env-step after the
    snapshot's step in which its own episode ends, after that step's training (its walker has just reset, so none of its old
    policy's actions are in flight).  A bottom agent whose episode has not ended when the next snapshot is taken does not copy.
    The copies of one step are taken in ascending dst order; dst's src is top[g.integers(k)], g = np.random.default_rng(seed),
    and dst then clears its history.

    Explore.  dst takes src's hyper-parameters; then, for each field of `perturb` (a dict field -> (lo, hi); Hyperparams field
    names, applied in wb_hyperparams field order), the value v becomes clip(float32(float64(v) * f), lo, hi) as a float32, with
    f = 0.8 if g.random() < 0.5 else 1.2.  Per dst the draws are: the src, then one per perturbed field.  Only the float fields
    alpha, beta1, beta2, adam_epsilon, gamma, lambda_, epsilon and log_std may be perturbed; default DEFAULT_PERTURB.

    Within env-step t: (1) the reward sums of the episodes that ended in t join their agents' histories, (2) the copies of t are
    decided, (3) if (t + 1) % interval == 0 the new snapshot is taken."""

    def __init__(self, interval: int, fraction: float = 0.2, window: int = 5, perturb=None, seed: int = 0):
        if int(interval) < 1:
            raise ValueError(f"interval must be at least 1, got {interval}")
        if not 0.0 <= float(fraction) <= 0.5:
            raise ValueError(f"fraction must be in [0, 0.5], got {fraction}")
        if int(window) < 1:
            raise ValueError(f"window must be at least 1, got {window}")
        perturb = DEFAULT_PERTURB if perturb is None else dict(perturb)
        for name, (lo, hi) in perturb.items():
            if name not in PERTURBABLE:
                raise ValueError(f"{name!r} cannot be perturbed (one of {', '.join(PERTURBABLE)})")
            if not lo <= hi:
                raise ValueError(f"{name}: lo {lo} > hi {hi}")
        self.interval, self.fraction, self.window = int(interval), float(fraction), int(window)
        self.perturb = {name: (float(perturb[name][0]), float(perturb[name][1])) for name in PERTURBABLE if name in perturb}
        self.rng = np.random.default_rng(seed)
        # per agent: its last `window` reward sums, oldest first (a shift register), and how many it has had since its last copy
        self.history, self.count = None, None
        self.top, self.bottom = [], None  # the current snapshot; bottom[a]: a has not copied yet

    def scores(self) -> dict:
        """{agent: score} of the ranked agents."""
        ranked = np.flatnonzero(self.count >= self.window) if self.count is not None else np.zeros(0, np.int64)
        return dict(zip(ranked.tolist(), self.history[ranked].mean(axis=1).tolist()))

    def step(self, t: int, agents, rewards, hp) -> list:
        """Env-step t ended the episodes of `agents` (each at most once) with the reward sums `rewards`; hp: every agent's current
        Hyperparams.  Returns the copies of this step: [(dst, src, dst's new Hyperparams)] in ascending dst order."""
        if self.history is None:
            self.history, self.count = np.zeros((len(hp), self.window)), np.zeros(len(hp), np.int64)
            self.bottom = np.zeros(len(hp), bool)
        ended = np.asarray(agents, np.int64).reshape(-1)
        self.history[ended, :-1] = self.history[ended, 1:]
        self.history[ended, -1] = np.asarray(rewards, np.float32).reshape(-1)
        self.count[ended] += 1
        copies = []
        for dst in np.sort(ended[self.bottom[ended]]).tolist():
            src = self.top[int(self.rng.integers(len(self.top)))]
            h = Hyperparams.from_buffer_copy(hp[src])
            for name, (lo, hi) in self.perturb.items():
                f = 0.8 if self.rng.random() < 0.5 else 1.2
                setattr(h, name, float(np.float32(min(max(np.float32(np.float64(getattr(h, name)) * f), lo), hi))))
            copies.append((dst, src, h))
            self.count[dst] = 0
            self.bottom[dst] = False
        if (t + 1) % self.interval == 0:
            ranked = np.flatnonzero(self.count >= self.window)
            order = ranked[np.lexsort((ranked, -self.history[ranked].mean(axis=1)))]
            k = int(np.floor(self.fraction * len(order)))
            self.top = order[:k].tolist()
            self.bottom[:] = False
            self.bottom[order[len(order) - k:] if k else []] = True
        return copies


class IndependentPPO:
    """N walkers, N independent agents (walker w acts with and trains agent w), resident on the GPU.

    Per env-step: the observations are copied into a time-major ring of R = max_timesteps + 1 rows (the longest episode), ONE
    wb_population_act_dev launch samples every walker's action with its own agent (Philox stream (act_seed, step)), ONE env-step
    launch (wb_env_step_dev, or wb_terrain_env_step_dev with `terrain`, accepted as VectorPPO accepts it) writes the rewards into the
    ring and resets finished walkers, and ONE synchronisation reads the N done bytes through a pinned buffer.  If any walker
    finished, ONE wb_population_train_dev launch trains each of those walkers' agents on its complete episode, with mini-batch
    indices drawn on the device (seed train_seed).  A ring column is only written by its own walker, and the walker has trained
    before it writes again.  episode_log() lists every finished episode: step, agent, length, reward sum and the two losses.

    pbt: a PBT schedule, or None.  With one, the synchronisation also reads the N running reward sums, and after the training
    launch the step issues the schedule's copies as ONE wb_population_copy_agents launch; exploit_log() lists them."""

    def __init__(self, n_envs: int, floor="Metal", walker="Carpet", hp=None, seed: int = 0, epochs: int = 5, terrain=None, seeds=None,
                 actor: str = DEFAULT_ACTOR, critic: str = DEFAULT_CRITIC, stateSize: int = OBS, actionSize: int = ACT,
                 pbt: PBT | None = None):
        if (stateSize, actionSize) != (OBS, ACT):
            raise ValueError(f"the walker observes {OBS} values and takes {ACT} actions; got stateSize={stateSize}, actionSize={actionSize}")
        import torch
        self.torch = torch
        self.n, self.epochs, self.seed = n_envs, epochs, seed
        self.act_seed, self.train_seed = 2 * seed, 2 * seed + 1
        self.stream = torch.cuda.current_stream().cuda_stream
        self.pop = PPOPopulation(n_envs, hp, seed=seed, seeds=seeds, stream=self.stream, actor=actor, critic=critic)
        env_hp = self.pop.hp[0]
        if any((h.iterations, h.max_timesteps) != (env_hp.iterations, env_hp.max_timesteps) for h in self.pop.hp):
            raise ValueError("the walkers step in lockstep: every agent's Hyperparams must share iterations and max_timesteps")
        if terrain is None:
            self.env = EnvBatch(n_envs, floor_materials=floor, walker_materials=walker, hp=env_hp, stream=self.stream)
            self._env_step_dev = lib().wb_env_step_dev
        else:
            terrain = list(terrain)
            if terrain and not isinstance(terrain[0], IObject):
                assert len(terrain) == n_envs, "a per-walker terrain needs one IObject list per walker"
            self.env = TerrainEnvBatch(n_envs, terrain, walker_material=walker, hp=env_hp, stream=self.stream)
            self._env_step_dev = lib().wb_terrain_env_step_dev
        self.R = env_hp.max_timesteps + 1
        dev = f"cuda:{torch.cuda.current_device()}"
        self.device = dev
        f32 = dict(device=dev, dtype=torch.float32)
        n, R = n_envs, self.R
        self.states = torch.empty(R, n, OBS, **f32)
        self.actions = torch.empty(R, n, ACT, **f32)
        self.logp = torch.empty(R, n, ACT, **f32)
        self.rewards = torch.empty(R, n, **f32)
        self.values = torch.empty(R, n, **f32)
        self.returns = torch.empty(R, n, **f32)
        self.adv = torch.empty(R, n, **f32)
        self.done = torch.zeros(n, device=dev, dtype=torch.uint8)
        self.done_host = torch.zeros(n, dtype=torch.uint8).pin_memory()
        self.idx_host = torch.zeros(n, dtype=torch.int64).pin_memory()
        self.ep_reward = torch.zeros(n, **f32)
        self.pbt = pbt
        if pbt is not None:
            self.reward_host = torch.zeros(n, dtype=torch.float32).pin_memory()
        self._exploit = []
        self.obs = torch.from_numpy(self.env.get_obs()).to(dev)  # Environment.InitialState
        self.start = np.zeros(n, np.int64)  # env-step at which each walker's running episode began
        self.t = 0
        self.timing = None  # a list: step() appends 5 recorded CUDA events (before act, env, sync + host, train, after)
        self._log = []

    def step(self) -> np.ndarray:
        """One env-step of every walker (Environment.Update, Environment.cs:64-92) and the training of every walker whose episode
        ended in it (TrainNetworks + Reset, :157-173).  Returns the N done flags."""
        torch, L = self.torch, lib()
        ev = None
        if self.timing is not None:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record()
        r = self.t % self.R
        self.states[r].copy_(self.obs)
        check(L.wb_population_act_dev(self.pop._h, self.n, ptr(self.obs), self.act_seed, self.t, ptr(self.actions[r]), ptr(self.logp[r]),
                                      None, None))
        if ev:
            ev[1].record()
        check(self._env_step_dev(self.env._h, ptr(self.actions[r]), C.c_float(DT_FRAME), 1, ptr(self.obs), ptr(self.rewards[r]),
                                 ptr(self.done)))
        self.ep_reward.add_(self.rewards[r])
        if ev:
            ev[2].record()
        self.done_host.copy_(self.done, non_blocking=True)
        if self.pbt is not None:
            self.reward_host.copy_(self.ep_reward, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        done = self.done_host.numpy().copy()
        if ev:
            ev[3].record()
        if done.any():
            w = np.flatnonzero(done)
            lengths = self.t - self.start[w] + 1
            items = np.ascontiguousarray(np.stack([w, w, self.start[w] % self.R, lengths], 1), np.int32)
            losses = torch.empty(len(w), 2, device=self.device, dtype=torch.float32)
            check(L.wb_population_train_dev(self.pop._h, len(w), ptr(items), self.R, self.n, self.epochs, self.train_seed, ptr(self.states),
                                            ptr(self.actions), ptr(self.logp), ptr(self.rewards), None, ptr(self.values),
                                            ptr(self.returns), ptr(self.adv), ptr(losses), None))
            # (through a pinned index buffer: no further synchronisation; the buffer is reused after the next step's sync)
            self.idx_host[:len(w)].copy_(torch.from_numpy(w))
            idx = self.idx_host[:len(w)].to(self.device, non_blocking=True)
            self._log.append((self.t, w, lengths, self.ep_reward.index_select(0, idx), losses))
            self.ep_reward.index_fill_(0, idx, 0.0)
            self.start[w] = self.t + 1
        if self.pbt is not None:
            w = np.flatnonzero(done)
            copies = self.pbt.step(self.t, w, self.reward_host.numpy()[w], self.pop.hp)
            if copies:
                self.pop.copy_agents([(d, s) for d, s, _ in copies], [h for _, _, h in copies])
                self._exploit += [(self.t, d, s, h) for d, s, h in copies]
        if ev:
            ev[4].record()
            self.timing.append(ev)
        self.t += 1
        return done

    def run(self, steps: int):
        for _ in range(steps):
            self.step()

    def episode_log(self) -> np.ndarray:
        """Every finished episode in order: step (the env-step it ended in), agent, length, reward (sum over the episode),
        critic_loss, actor_loss (the last mini-batch's, 0 for an episode shorter than the agent's BatchSize)."""
        dt = np.dtype([("step", np.int64), ("agent", np.int32), ("length", np.int32), ("reward", np.float32), ("critic_loss", np.float32),
                       ("actor_loss", np.float32)])
        out = np.zeros(sum(len(e[1]) for e in self._log), dt)
        i = 0
        for t, w, lengths, rew, losses in self._log:
            k = len(w)
            ls = losses.cpu().numpy()
            out["step"][i:i + k], out["agent"][i:i + k], out["length"][i:i + k] = t, w, lengths
            out["reward"][i:i + k], out["critic_loss"][i:i + k], out["actor_loss"][i:i + k] = rew.cpu().numpy(), ls[:, 0], ls[:, 1]
            i += k
        return out


    def exploit_log(self) -> np.ndarray:
        """Every copy of the PBT schedule in order: step (the env-step it ended), dst, src and dst's new hyper-parameters (the
        Hyperparams fields)."""
        fields = [(name, np.int32 if ctype is C.c_int32 else np.float32) for name, ctype in Hyperparams._fields_]
        out = np.zeros(len(self._exploit), [("step", np.int64), ("dst", np.int32), ("src", np.int32)] + fields)
        for i, (t, d, s, h) in enumerate(self._exploit):
            out[i] = (t, d, s) + tuple(getattr(h, name) for name, _ in fields)
        return out


__all__ = ["PPOPopulation", "IndependentPPO", "PBT", "default_seeds"]

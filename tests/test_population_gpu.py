"""One PPO brain per walker (wb_population_*, PPOPopulation, IndependentPPO): every agent of a population against a PPOAgent with
the same weights, hyper-parameters and draws -- initialisation, acting, training in both entries, the lockstep loop on the flat and
on a rough floor -- plus launches, streams and refused arguments."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LENGTHS = [37, 130, 0, 1001, 64, 200, 63]


def rollout(gpu, lengths, seed=0):
    """Real walker steps from the library's Environment under a seeded random policy (auto-reset), cut into trajectories."""
    env = gpu.Environment(1)
    roller = gpu.PPOAgent(seed=seed)
    state = env.InitialState()
    trajs = []
    for T in lengths:
        t = gpu.Trajectory()
        for _ in range(T):
            a, lp, _, _ = roller.SampleActions(state)
            t.States.append(state[0][:12].copy())
            state, reward, _ = env.Update(gpu.DT_FRAME, a, auto_reset=True)
            t.Actions.append(a[0].copy())
            t.LogProbabilities.append(lp[0].copy())
            t.Rewards.append(float(reward[0]))
        trajs.append(t)
    return trajs


def fresh(t):
    return type(t)(States=list(t.States), Actions=list(t.Actions), LogProbabilities=list(t.LogProbabilities), Rewards=list(t.Rewards))


def bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def hp_sweep(gpu, n, batch_sizes=(64, 100)):
    """Agents that differ in every hyper-parameter the population keeps per agent."""
    out = []
    for a in range(n):
        hp = gpu.default_hyperparams()
        hp.alpha, hp.beta1, hp.beta2 = 0.001 * (1 + 0.5 * (a % 3)), 0.9 - 0.02 * (a % 2), 0.999 - 0.001 * (a % 3)
        hp.adam_epsilon = 1e-8 * (1 + a % 2)
        hp.gamma, hp.lambda_, hp.epsilon = 0.9 + 0.02 * (a % 4), 0.95 - 0.05 * (a % 2), 0.2 + 0.05 * (a % 3)
        hp.log_std = -1.0 + 0.125 * (a % 5)
        hp.use_gae, hp.normalize_advantages = a % 2, (a // 2) % 2
        hp.batch_size = batch_sizes[a % len(batch_sizes)]
        out.append(hp)
    return out


def twin(gpu, pop, a, variant=1):
    """PPOAgent(seed=seeds[a], hp=hp[a]) on kernel variant 1: what agent a of the population must equal."""
    agent = gpu.PPOAgent(hp=pop.hp[a], seed=pop.seeds[a])
    agent.set_variant(variant)
    return agent


def agent_state(agent):
    m_a, v_a, it_a = agent.actor.get_adam()
    m_c, v_c, it_c = agent.critic.get_adam()
    return (np.concatenate([agent.actor.get_flat(), agent.critic.get_flat()]), np.concatenate([m_a, m_c]), np.concatenate([v_a, v_c]),
            np.concatenate([it_a, it_c]), np.concatenate([agent.actor.get_grads(), agent.critic.get_grads()]))


def pop_state(pop, a):
    m, v, steps = pop.adam(a)
    return pop.get_weights(a), m, v, steps, pop.get_grads(a)


def assert_same(x, y, what=""):
    for p, q, name in zip(x, y, ("weights", "adam m", "adam v", "step counters", "gradient buffer")):
        same = np.array_equal(bits(p), bits(q)) if p.dtype == np.float32 else np.array_equal(p, q)
        assert same, (what, name)


# ---- the documented device draw of the mini-batch indices, restated
def philox_x(c0, c1, c2, c3, seed):
    M = np.uint64(0xFFFFFFFF)
    c = [np.asarray(v, np.uint64) & M for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M, (k1 + np.uint64(0xBB67AE85)) & M
    return c[0]


def device_draw(L, B, epochs, episode, agent, seed):
    rows = np.arange(L)
    blocks = []
    for epoch in range(epochs):
        keys = philox_x(rows, epoch, episode, agent, seed)
        perm = np.lexsort((rows, keys))
        blocks.extend(perm[j * B:(j + 1) * B] for j in range(L // B))
    return np.concatenate(blocks).astype(np.int32) if blocks else np.zeros(0, np.int32)


def train_replay(gpu, agent, traj, index, epochs=5):
    """PPOAgent.TrainTrajectories of one trajectory with given mini-batch indices (wb_ppo_train_trajectories)."""
    T = len(traj.States)
    offsets = np.array([0, T], np.int32)
    S = np.ascontiguousarray(np.array(traj.States, np.float32).reshape(T, 12))
    A = np.ascontiguousarray(np.array(traj.Actions, np.float32).reshape(T, 4))
    LP = np.ascontiguousarray(np.array(traj.LogProbabilities, np.float32).reshape(T, 4))
    R = np.ascontiguousarray(np.array(traj.Rewards, np.float32))
    V, G, Adv = (np.empty(T, np.float32) for _ in range(3))
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    check(lib().wb_ppo_train_trajectories(agent._h, 1, ptr(offsets), epochs, ptr(S), ptr(A), ptr(LP), ptr(R), ptr(index), ptr(V), ptr(G),
                                          ptr(Adv), None, None))
    return V, G, Adv


def test_agent_a_starts_as_ppoagent_with_seed_a(gpu):
    seeds = [3, 17, 17, 2 ** 40 + 5, 0]
    pop = gpu.PPOPopulation(len(seeds), seeds=seeds)
    for a, s in enumerate(seeds):
        ref = gpu.PPOAgent(seed=s)
        assert np.array_equal(bits(pop.get_weights(a)), bits(np.concatenate([ref.actor.get_flat(), ref.critic.get_flat()])))
        assert pop.rngs[a].random() == ref.rng.random()
    critic_lines, actor_lines = pop.Save(3)
    assert (critic_lines, actor_lines) == gpu.PPOAgent(seed=seeds[3]).Save()
    default = gpu.PPOPopulation(4, seed=7)
    assert default.seeds == gpu.default_seeds(7, 4) and len(set(default.seeds)) == 4


def test_acting_equals_each_agents_policy(gpu, O):
    import torch
    P = 4096
    hps = []
    for a in range(P):
        hp = gpu.default_hyperparams()
        hp.log_std = -1.5 + a / P
        hps.append(hp)
    pop = gpu.PPOPopulation(P, hp=hps, seed=11)
    rng = np.random.default_rng(1)
    states = rng.normal(size=(P, 12)).astype(np.float32)
    d_states = torch.from_numpy(states).cuda()
    outs = [torch.empty(P, 4, device="cuda") for _ in range(3)] + [torch.empty(P, device="cuda")]
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    seed, step = 12345, 2 ** 33 + 7
    before = pop.launch_count()
    check(lib().wb_population_act_dev(pop._h, P, ptr(d_states), seed, step, *[ptr(o) for o in outs]))
    assert pop.launch_count() == before + 1
    act, logp, mean, value = [o.cpu().numpy() for o in outs]
    uni = rng.random((P, 4, 2)).astype(np.float32)
    s_act, s_logp, s_mean, s_std = pop.SampleActions(states, uni)
    for a in list(rng.choice(P, 14, replace=False)) + [0, P - 1]:
        ref = twin(gpu, pop, a)
        ref.actor.set_flat(pop.get_weights(a)[:5252])
        ref.critic.set_flat(pop.get_weights(a)[5252:])
        r = [torch.empty(P, 4, device="cuda") for _ in range(3)] + [torch.empty(P, device="cuda")]
        check(lib().wb_policy_act_dev(ref._h, P, ptr(d_states), seed, step, ptr(r[0]), ptr(r[1]), ptr(r[2]), ptr(r[3])))
        r = [x.cpu().numpy() for x in r]
        for got, want in zip((act, logp, mean, value), r):
            assert np.array_equal(bits(got[a]), bits(want[a])), a
        ra, rl, rm, rs = ref.SampleActions(states, uni)
        for got, want in zip((s_act, s_logp, s_mean, s_std), (ra, rl, rm, rs)):
            assert np.array_equal(bits(got[a]), bits(want[a])), a
        actor = O.Net(12, O.ACTOR_LAYERS)
        actor.set_params(pop.get_weights(a)[:5252])
        np.testing.assert_allclose(mean[a], actor.forward(states[a:a + 1])[0], rtol=0, atol=1e-5)


def test_host_training_equals_ppoagent_per_agent(gpu):
    trajs = rollout(gpu, LENGTHS, seed=1)
    t37, t130, t0, t1001, t64, t200, t63 = trajs
    hps = hp_sweep(gpu, 6)
    pop = gpu.PPOPopulation(6, hp=hps, seed=3)
    pairs = [(0, t37), (1, t130), (0, t0), (2, t1001), (1, t64), (3, t200), (0, t63), (0, t200), (2, t130), (5, t64)]
    untouched = {4: pop_state(pop, 4)}
    twins = {a: twin(gpu, pop, a) for a in range(6)}
    mine = [(a, fresh(t)) for a, t in pairs]
    losses = pop.TrainTrajectories(mine)
    for a, ref in twins.items():
        sub = [(i, fresh(t)) for i, (b, t) in enumerate(pairs) if b == a]
        if not sub:
            continue
        # B = 64: PPOAgent.Train per trajectory (the per-mini-batch kernels), independent of the episode kernel and bit-identical to
        # it at that size; B = 100 has no other form with the episode kernel's summation order
        ts = [t for _, t in sub]
        ref_losses = [ref.Train(t) for t in ts] if ref.hp.batch_size == 64 else ref.TrainTrajectories(ts)
        assert_same(pop_state(pop, a), agent_state(ref), a)
        assert np.array_equal(bits([losses[i] for i, _ in sub]), bits(ref_losses)), a
        for i, t in sub:
            for attr in ("Values", "Returns", "Advantages"):
                assert np.array_equal(bits(getattr(t, attr)), bits(getattr(mine[i][1], attr))), (a, attr)
        assert pop.rngs[a].random() == ref.rng.random()
    assert_same(pop_state(pop, 4), untouched[4], "unlisted agent")


def test_skipped_counts_per_item(gpu):
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    t = rollout(gpu, [130], seed=7)[0]
    t.LogProbabilities[5] = np.array([0.0, -200.0, 0.0, 0.0], np.float32)  # exp underflows: the sample is skipped
    pop = gpu.PPOPopulation(2, seed=5)
    S = np.ascontiguousarray(np.concatenate([np.array(t.States, np.float32)] * 2))
    A = np.ascontiguousarray(np.concatenate([np.array(t.Actions, np.float32)] * 2))
    L = np.ascontiguousarray(np.concatenate([np.array(t.LogProbabilities, np.float32)] * 2))
    R = np.ascontiguousarray(np.concatenate([np.array(t.Rewards, np.float32)] * 2))
    index = np.concatenate([np.random.default_rng(k).permutation(130)[:128] for k in range(10)]).astype(np.int32)
    skipped = np.zeros(2, np.int32)
    check(lib().wb_population_train_trajectories(pop._h, 2, ptr(np.array([1, 0], np.int32)), ptr(np.array([0, 130, 260], np.int32)), 5,
                                                 ptr(S), ptr(A), ptr(L), ptr(R), ptr(index), None, None, None, None, ptr(skipped)))
    expect = [sum(5 in index[k * 128 + j * 64:k * 128 + (j + 1) * 64] for k in range(e * 5, e * 5 + 5) for j in range(2)) for e in (0, 1)]
    assert list(skipped) == expect and min(expect) > 0


def ring_from(trajs, placements, R, Cols):
    """Time-major ring [R][C] holding trajectory k at (column, t0) (wrapping at R)."""
    S, A, LP = np.zeros((R, Cols, 12), np.float32), np.zeros((R, Cols, 4), np.float32), np.zeros((R, Cols, 4), np.float32)
    Rw = np.zeros((R, Cols), np.float32)
    for t, (c, t0) in zip(trajs, placements):
        rows = (t0 + np.arange(len(t.States))) % R
        S[rows, c], A[rows, c], LP[rows, c], Rw[rows, c] = t.States, t.Actions, t.LogProbabilities, t.Rewards
    return S, A, LP, Rw


def test_device_training_with_device_draws_across_the_ring_end(gpu):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    trajs = rollout(gpu, [130, 200, 150, 64, 37], seed=2)
    R, Cols, seed = 300, 3, 77
    hps = hp_sweep(gpu, 4)
    pop = gpu.PPOPopulation(4, hp=hps, seed=9)
    items = np.array([[0, 0, 250, 130], [1, 1, 10, 200], [0, 2, 200, 150], [2, 1, 220, 64], [0, 0, 120, 37]], np.int32)
    ring = ring_from(trajs, [(c, t0) for _, c, t0, _ in items], R, Cols)
    dev = [torch.from_numpy(x).cuda() for x in ring]
    out = [torch.zeros(R, Cols, device="cuda") for _ in range(3)]
    losses = torch.zeros(len(items), 2, device="cuda")
    skipped = torch.zeros(len(items), dtype=torch.int32, device="cuda")
    twins = {a: twin(gpu, pop, a) for a in range(4)}
    untouched = pop_state(pop, 3)
    before = pop.launch_count()
    check(lib().wb_population_train_dev(pop._h, len(items), ptr(items), R, Cols, 5, seed, *[ptr(x) for x in dev], None,
                                        *[ptr(x) for x in out], ptr(losses), ptr(skipped)))
    pop.sync()
    assert pop.launch_count() == before + 1
    V, G, Adv = [x.cpu().numpy() for x in out]
    episodes = {}
    for k, (a, c, t0, L) in enumerate(items):
        e = episodes.get(a, 0)
        episodes[a] = e + 1
        index = device_draw(L, hps[a].batch_size, 5, e, a, seed)
        rv, rg, ra = train_replay(gpu, twins[a], trajs[k], index)
        rows = (t0 + np.arange(L)) % R
        for got, want in zip((V, G, Adv), (rv, rg, ra)):
            assert np.array_equal(bits(got[rows, c]), bits(want)), k
    for a in range(3):
        assert_same(pop_state(pop, a), agent_state(twins[a]), a)
    assert_same(pop_state(pop, 3), untouched, "unlisted agent")


def record_loop(gpu, loop, steps):
    rec = {k: [] for k in ("states", "actions", "logp", "rewards", "dones")}
    for _ in range(steps):
        r = loop.t % loop.R
        done = loop.step()
        rec["states"].append(loop.states[r].cpu().numpy())
        rec["actions"].append(loop.actions[r].cpu().numpy())
        rec["logp"].append(loop.logp[r].cpu().numpy())
        rec["rewards"].append(loop.rewards[r].cpu().numpy())
        rec["dones"].append(done)
    return {k: np.array(v) for k, v in rec.items()}


def replay_agent(gpu, loop, rec, a, O=None):
    """Agent a alone, step by step: its actions are wb_policy_act_dev of its current weights; at each of its episode ends it trains
    with the restated device draw.  Returns the replaying PPOAgent (and the oracle pair when O is given)."""
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    ref = twin(gpu, loop.pop, a)
    steps, n = rec["dones"].shape
    out_a, out_l = torch.empty(steps, n, 4, device="cuda"), torch.empty(steps, n, 4, device="cuda")
    states = torch.from_numpy(rec["states"]).cuda()
    oracle = None
    if O is not None:
        actor, critic = O.Net(12, O.ACTOR_LAYERS), O.Net(12, O.CRITIC_LAYERS)
        actor.set_params(ref.actor.get_flat())
        critic.set_params(ref.critic.get_flat())
        ohp = O.hyper_defaults()
        ohp.batch_size = ref.hp.batch_size
        oracle = (actor, critic, ohp)
    start, episode = 0, 0
    for t in range(steps):
        check(lib().wb_policy_act_dev(ref._h, n, ptr(states[t]), loop.act_seed, t, ptr(out_a[t]), ptr(out_l[t]), None, None))
        if rec["dones"][t, a]:
            tr = gpu.Trajectory(States=list(rec["states"][start:t + 1, a]), Actions=list(rec["actions"][start:t + 1, a]),
                                LogProbabilities=list(rec["logp"][start:t + 1, a]), Rewards=list(rec["rewards"][start:t + 1, a]))
            L = t + 1 - start
            index = device_draw(L, ref.hp.batch_size, loop.epochs, episode, a, loop.train_seed)
            if oracle is not None:
                actor, critic, ohp = oracle
                S = np.array(tr.States, np.float32)
                values = critic.forward(S)[:, 0].copy()
                G, Adv = O.mc_returns(np.array(tr.Rewards, np.float32), values, ref.hp.gamma)
                acts, lp = np.array(tr.Actions, np.float32), np.array(tr.LogProbabilities, np.float32)
                B = ref.hp.batch_size
                for j in range(len(index) // B):
                    idx = index[j * B:(j + 1) * B]
                    O.ppo_train_batch(actor, critic, ohp, S[idx], acts[idx], lp[idx], Adv[idx], G[idx], optimise=True)
            train_replay(gpu, ref, tr, index, loop.epochs)
            start, episode = t + 1, episode + 1
    torch.cuda.synchronize()
    assert np.array_equal(bits(out_a[:, a].cpu().numpy()), bits(rec["actions"][:, a])), a
    assert np.array_equal(bits(out_l[:, a].cpu().numpy()), bits(rec["logp"][:, a])), a
    return ref, oracle


# (on the flat floor the first falls come after ~50 steps: a longer cap there, so that both episode endings occur)
@pytest.mark.parametrize("rough,max_timesteps,steps", [(False, 150, 400), (True, 40, 260)])
def test_independent_ppo_replays_agent_by_agent(gpu, O, rough, max_timesteps, steps):
    n = 64
    hp = gpu.default_hyperparams()
    hp.max_timesteps, hp.batch_size = max_timesteps, 16
    terrain = None
    if rough:
        rng = np.random.default_rng(4)
        terrain = [gpu.CreateRoughFloor(rng.integers(0, 100, 11)) for _ in range(n)]
    loop = gpu.IndependentPPO(n, hp=hp, seed=21, epochs=3, terrain=terrain)
    before = loop.pop.launch_count()
    rec = record_loop(gpu, loop, steps)
    dones = rec["dones"].astype(bool)
    assert loop.pop.launch_count() - before == steps + int(dones.any(1).sum())
    log = loop.episode_log()
    assert len(log) == int(dones.sum()) and (log["length"] <= hp.max_timesteps + 1).all()
    assert (log["length"] == hp.max_timesteps + 1).any() and (log["length"] < hp.max_timesteps + 1).any()  # both endings
    for a in range(n):
        ref, oracle = replay_agent(gpu, loop, rec, a, O if a == 0 else None)
        assert_same(pop_state(loop.pop, a), agent_state(ref), a)
        if oracle is not None:
            np.testing.assert_allclose(loop.pop.get_weights(a)[:5252], oracle[0].get_params(), rtol=0, atol=2e-5)
            np.testing.assert_allclose(loop.pop.get_weights(a)[5252:], oracle[1].get_params(), rtol=0, atol=2e-5)
    first = log[log["agent"] == 0][0]
    assert np.isclose(first["reward"], rec["rewards"][:first["length"], 0].astype(np.float64).sum(), rtol=1e-5, atol=1e-4)


def test_two_populations_on_two_streams(gpu):
    import torch
    trajs = rollout(gpu, [130, 200, 70], seed=5)

    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    paired = [gpu.PPOPopulation(2, seed=1, stream=s1.cuda_stream), gpu.PPOPopulation(2, seed=2, stream=s2.cuda_stream)]
    # device entries enqueued on both streams before either finishes
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    R = 400
    ring = ring_from(trajs, [(0, 0), (0, 130), (1, 0)], R, 2)
    items = np.array([[0, 0, 0, 130], [1, 0, 130, 200], [0, 1, 0, 70]], np.int32)
    bufs = []
    for p in paired:
        dev = [torch.from_numpy(x).cuda() for x in ring]
        out = [torch.zeros(R, 2, device="cuda") for _ in range(3)]
        bufs.append((dev, out))
    ref = [gpu.PPOPopulation(2, seed=s) for s in (1, 2)]
    torch.cuda.synchronize()
    for p, (dev, out) in zip(paired, bufs):
        check(lib().wb_population_train_dev(p._h, 3, ptr(items), R, 2, 5, 99, *[ptr(x) for x in dev], None, *[ptr(x) for x in out], None, None))
    torch.cuda.synchronize()
    for p, (dev, out) in zip(ref, bufs):
        rdev = [torch.from_numpy(x).cuda() for x in ring]
        rout = [torch.zeros(R, 2, device="cuda") for _ in range(3)]
        check(lib().wb_population_train_dev(p._h, 3, ptr(items), R, 2, 5, 99, *[ptr(x) for x in rdev], None, *[ptr(x) for x in rout], None, None))
        p.sync()
        for x, y in zip(out, rout):
            assert torch.equal(x, y)
    for a, b in zip(paired, ref):
        for k in range(2):
            assert_same(pop_state(a, k), pop_state(b, k), k)


def test_bad_arguments_are_refused_and_change_nothing(gpu):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    hp = gpu.default_hyperparams()
    bad_hp = gpu.default_hyperparams()
    bad_hp.batch_size = 0
    h = C.c_void_p()
    for n, hps in [(0, None), (2, (gpu.Hyperparams * 2)(hp, bad_hp))]:
        with pytest.raises(gpu.WalkerB200Error) as ei:
            check(lib().wb_population_create(n, hps, C.byref(h)))
        assert ei.value.code == 1
    pop = gpu.PPOPopulation(3, seed=1)
    before = [pop_state(pop, a) for a in range(3)]
    t = rollout(gpu, [130, 70], seed=8)
    S = np.ascontiguousarray(np.concatenate([np.array(x.States, np.float32) for x in t]))
    A = np.ascontiguousarray(np.concatenate([np.array(x.Actions, np.float32) for x in t]))
    L = np.ascontiguousarray(np.concatenate([np.array(x.LogProbabilities, np.float32) for x in t]))
    Rw = np.ascontiguousarray(np.concatenate([np.array(x.Rewards, np.float32) for x in t]))
    offsets = np.array([0, 130, 200], np.int32)
    index = np.concatenate([np.arange(128)] * 5 + [np.arange(64)] * 5).astype(np.int32)
    bad_index = index.copy()
    bad_index[-1] = 70
    host_cases = [(2, [0, 1], offsets, 5, bad_index), (2, [0, 1], np.array([0, 130, 100], np.int32), 5, index), (2, [0, 1], offsets, -1, index),
                  (0, [0, 1], offsets, 5, index), (2, [0, 3], offsets, 5, index), (2, [-1, 0], offsets, 5, index)]
    for n, agents, off, epochs, idx in host_cases:
        with pytest.raises(gpu.WalkerB200Error) as ei:
            check(lib().wb_population_train_trajectories(pop._h, n, ptr(np.array(agents, np.int32)), ptr(off), epochs, ptr(S), ptr(A), ptr(L),
                                                         ptr(Rw), ptr(idx), None, None, None, None, None))
        assert ei.value.code == 1
    R, Cols = 300, 2
    dev = [torch.from_numpy(x).cuda() for x in ring_from(t, [(0, 0), (1, 250)], R, Cols)]
    out = [torch.zeros(R, Cols, device="cuda") for _ in range(3)]
    dev_cases = [[[3, 0, 0, 130]], [[0, 2, 0, 130]], [[0, 0, 0, -1]], [[0, 0, 0, 301]], [[0, 0, 300, 10]], [[0, 0, -1, 10]]]
    for items in dev_cases:
        with pytest.raises(gpu.WalkerB200Error) as ei:
            check(lib().wb_population_train_dev(pop._h, len(items), ptr(np.array(items, np.int32)), R, Cols, 5, 1, *[ptr(x) for x in dev], None,
                                                *[ptr(x) for x in out], None, None))
        assert ei.value.code == 1
    for n_items, epochs in [(0, 5), (1, -1)]:
        with pytest.raises(gpu.WalkerB200Error):
            check(lib().wb_population_train_dev(pop._h, n_items, ptr(np.array([[0, 0, 0, 130]], np.int32)), R, Cols, epochs, 1,
                                                *[ptr(x) for x in dev], None, *[ptr(x) for x in out], None, None))
    d_states = torch.zeros(4, 12, device="cuda")
    o = [torch.empty(4, 4, device="cuda") for _ in range(2)]
    with pytest.raises(gpu.WalkerB200Error):
        check(lib().wb_population_act_dev(pop._h, 4, ptr(d_states), 1, 0, ptr(o[0]), ptr(o[1]), None, None))
    with pytest.raises(gpu.WalkerB200Error):
        check(lib().wb_population_sample(pop._h, 2, ptr(np.zeros((2, 12), np.float32)), ptr(np.zeros((2, 4, 2), np.float32)),
                                         ptr(np.zeros((2, 4), np.float32)), ptr(np.zeros((2, 4), np.float32)), None))
    assert pop.launch_count() == 0
    for a in range(3):
        assert_same(pop_state(pop, a), before[a], a)

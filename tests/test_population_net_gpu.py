"""One PPO brain per walker for networks other than the defaults (wb_population_create_net, the any-topology population kernels):
every agent against PPOAgent(actor=, critic=, seed=seeds[a], hp=hp[a]), which runs the any-topology kernel for these networks --
initialisation, acting, training in both entries, the lockstep loop, the default lists, refused arguments and streams."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LENGTHS = [37, 130, 0, 1001, 64, 200, 63]
NETS = [  # (state, action, actor, critic): the non-default topologies of test_ppo_gpu.py and a 128-wide actor
    (12, 4, "Input |32| (ReLU) |4| (TanH) Output", "Input |16| (ReLU) |16| (TanH) |1| Output"),
    (12, 4, "Input |128| (LeakyReLU) |48| (ReLU) |80| (TanH) |4| Output", "Input |96| (ReLU) |1| Output"),
    (7, 3, "Input |20| (TanH) |3| Output", "Input |5| (LeakyReLU) |9| (LeakyReLU) |1| (ReLU) Output"),
    (12, 4, "Input |4| Output", "Input |1| Output"),
    (12, 4, "Input |128| (LeakyReLU) |128| (LeakyReLU) |4| (TanH) Output", "Input |64| (LeakyReLU) |1| Output"),
]
IDS = ["small", "mixed", "state7", "linear", "wide128"]


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


def population(gpu, net, n, **kw):
    S, A, actor, critic = net
    return gpu.PPOPopulation(n, actor=actor, critic=critic, stateSize=S, actionSize=A, **kw)


def twin(gpu, pop, a):
    return gpu.PPOAgent(pop.stateSize, pop.actionSize, hp=pop.hp[a], actor=pop.actor_structure, critic=pop.critic_structure, seed=pop.seeds[a])


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


def trajectories(gpu, S, A, lengths, seed=0):
    """Seeded synthetic episodes (states, actions, log-probabilities around what a Gaussian policy gives, rewards)."""
    rng = np.random.default_rng(seed)
    out = []
    for T in lengths:
        t = gpu.Trajectory()
        for _ in range(T):
            t.States.append(rng.normal(size=S).astype(np.float32))
            t.Actions.append(rng.uniform(-1, 1, size=A).astype(np.float32))
            t.LogProbabilities.append(rng.uniform(-2.5, 0.5, size=A).astype(np.float32))
            t.Rewards.append(float(np.float32(rng.normal())))
        out.append(t)
    return out


def fresh(t):
    return type(t)(States=list(t.States), Actions=list(t.Actions), LogProbabilities=list(t.LogProbabilities), Rewards=list(t.Rewards))


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


def train_replay(agent, traj, index, epochs=5):
    """PPOAgent.TrainTrajectories of one trajectory with given mini-batch indices (wb_ppo_train_trajectories)."""
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    T, S, A = len(traj.States), agent.stateSize, agent.actionSize
    arr = [np.ascontiguousarray(np.array(x, np.float32).reshape(T, w)) for x, w in
           ((traj.States, S), (traj.Actions, A), (traj.LogProbabilities, A), (traj.Rewards, 1))]
    V, G, Adv = (np.empty(T, np.float32) for _ in range(3))
    check(lib().wb_ppo_train_trajectories(agent._h, 1, ptr(np.array([0, T], np.int32)), epochs, *[ptr(x) for x in arr], ptr(index), ptr(V),
                                          ptr(G), ptr(Adv), None, None))
    return V, G, Adv


def ring_from(trajs, placements, R, Cols, S, A):
    St, Ac, LP = np.zeros((R, Cols, S), np.float32), np.zeros((R, Cols, A), np.float32), np.zeros((R, Cols, A), np.float32)
    Rw = np.zeros((R, Cols), np.float32)
    for t, (c, t0) in zip(trajs, placements):
        rows = (t0 + np.arange(len(t.States))) % R
        St[rows, c], Ac[rows, c], LP[rows, c], Rw[rows, c] = t.States, t.Actions, t.LogProbabilities, t.Rewards
    return St, Ac, LP, Rw


@pytest.mark.parametrize("net", NETS, ids=IDS)
def test_agents_start_as_their_ppoagent(gpu, net):
    pop = population(gpu, net, 3, seeds=[3, 17, 2 ** 40 + 5])
    for a in range(3):
        ref = twin(gpu, pop, a)
        assert np.array_equal(bits(pop.get_weights(a)), bits(np.concatenate([ref.actor.get_flat(), ref.critic.get_flat()])))
        assert pop.Save(a) == ref.Save()
        assert (pop.N_ACTOR, pop.N_PARAMS - pop.N_ACTOR) == (ref.actor.num_params, ref.critic.num_params)
        assert pop.rngs[a].random() == ref.rng.random()


@pytest.mark.parametrize("net", NETS, ids=IDS)
def test_acting_equals_each_agents_policy(gpu, net):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    S, A = net[0], net[1]
    P = 256
    hps = []
    for a in range(P):
        hp = gpu.default_hyperparams()
        hp.log_std = -1.5 + a / P
        hps.append(hp)
    pop = population(gpu, net, P, hp=hps, seed=11)
    rng = np.random.default_rng(1)
    states = rng.normal(size=(P, S)).astype(np.float32)
    d_states = torch.from_numpy(states).cuda()
    outs = [torch.empty(P, A, device="cuda") for _ in range(3)] + [torch.empty(P, device="cuda")]
    seed, step = 12345, 2 ** 33 + 7
    before = pop.launch_count()
    check(lib().wb_population_act_dev(pop._h, P, ptr(d_states), seed, step, *[ptr(o) for o in outs]))
    assert pop.launch_count() == before + 1
    act, logp, mean, value = [o.cpu().numpy() for o in outs]
    uni = rng.random((P, A, 2)).astype(np.float32)
    s_act, s_logp, s_mean, _ = pop.SampleActions(states, uni)
    for a in list(rng.choice(P, 6, replace=False)) + [0, P - 1]:
        ref = twin(gpu, pop, a)
        ref.actor.set_flat(pop.get_weights(a)[:pop.N_ACTOR])
        ref.critic.set_flat(pop.get_weights(a)[pop.N_ACTOR:])
        r = [torch.empty(P, A, device="cuda") for _ in range(3)] + [torch.empty(P, device="cuda")]
        check(lib().wb_policy_act_dev(ref._h, P, ptr(d_states), seed, step, *[ptr(x) for x in r]))
        r = [x.cpu().numpy() for x in r]
        for got, want in zip((act, logp, mean, value), r):
            assert np.array_equal(bits(got[a]), bits(want[a])), a
        ra, rl, rm, _ = ref.SampleActions(states, uni)
        for got, want in zip((s_act, s_logp, s_mean), (ra, rl, rm)):
            assert np.array_equal(bits(got[a]), bits(want[a])), a


@pytest.mark.parametrize("net", NETS, ids=IDS)
def test_host_training_equals_ppoagent_per_agent(gpu, net):
    S, A = net[0], net[1]
    t37, t130, t0, t1001, t64, t200, t63 = trajectories(gpu, S, A, LENGTHS, seed=1)
    hps = hp_sweep(gpu, 5)
    pop = population(gpu, net, 5, hp=hps, seed=3)
    pairs = [(0, t37), (1, t130), (0, t0), (2, t1001), (1, t64), (3, t200), (0, t63), (0, t200), (2, t130)]
    untouched = pop_state(pop, 4)
    twins = {a: twin(gpu, pop, a) for a in range(4)}
    mine = [(a, fresh(t)) for a, t in pairs]
    losses = pop.TrainTrajectories(mine)
    for a, ref in twins.items():
        sub = [(i, fresh(t)) for i, (b, t) in enumerate(pairs) if b == a]
        ref_losses = ref.TrainTrajectories([t for _, t in sub])
        assert_same(pop_state(pop, a), agent_state(ref), a)
        assert np.array_equal(bits([losses[i] for i, _ in sub]), bits(ref_losses)), a
        for (i, _), (_, t) in zip(sub, sub):
            for attr in ("Values", "Returns", "Advantages"):
                assert np.array_equal(bits(getattr(t, attr)), bits(getattr(mine[i][1], attr))), (a, attr)
    assert_same(pop_state(pop, 4), untouched, "unlisted agent")


@pytest.mark.parametrize("net", NETS, ids=IDS)
def test_skipped_and_gradient_tail_equal_the_twin(gpu, net):
    """The loss sums and skipped counts of the gradient buffer's tail (read back through losses / skipped) equal the twin's, and
    the skipped count equals the number of mini-batch slots that hold a poisoned row (the wide networks put the thread that
    zeroes the tail and the thread that reads it in different warps)."""
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    S, A = net[0], net[1]
    t = trajectories(gpu, S, A, [130], seed=7)[0]
    poisoned = (5, 77)
    for r in poisoned:  # exp(-200) underflows: the sample is skipped
        t.LogProbabilities[r] = np.array([0.0, -200.0] + [0.0] * (A - 2), np.float32)
    pop = population(gpu, net, 1, seed=5)
    ref = twin(gpu, pop, 0)
    index = np.concatenate([np.random.default_rng(k).permutation(130)[:128] for k in range(5)]).astype(np.int32)
    arr = [np.ascontiguousarray(np.array(x, np.float32)) for x in (t.States, t.Actions, t.LogProbabilities, t.Rewards)]
    offsets = np.array([0, 130], np.int32)
    out = []
    for h, head in ((pop._h, (1, ptr(np.zeros(1, np.int32)), ptr(offsets), 5)), (ref._h, (1, ptr(offsets), 5))):
        call = lib().wb_population_train_trajectories if h is pop._h else lib().wb_ppo_train_trajectories
        losses, skipped = np.zeros(2, np.float32), np.zeros(1, np.int32)
        check(call(h, *head, *[ptr(x) for x in arr], ptr(index), None, None, None, ptr(losses), ptr(skipped)))
        out.append((losses, skipped))
    expect = sum(int(np.isin(poisoned, index[j * 64:(j + 1) * 64]).sum()) for j in range(len(index) // 64))
    assert expect > 0
    assert np.array_equal(bits(out[0][0]), bits(out[1][0]))
    assert out[0][1][0] == out[1][1][0] == expect
    assert_same(pop_state(pop, 0), agent_state(ref))


@pytest.mark.parametrize("net", [NETS[1], NETS[2]], ids=["mixed", "state7"])
def test_device_training_with_device_draws_across_the_ring_end(gpu, net):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    S, A = net[0], net[1]
    trajs = trajectories(gpu, S, A, [130, 200, 150, 64, 37], seed=2)
    R, Cols, seed = 300, 3, 77
    hps = hp_sweep(gpu, 4)
    pop = population(gpu, net, 4, hp=hps, seed=9)
    items = np.array([[0, 0, 250, 130], [1, 1, 10, 200], [0, 2, 200, 150], [2, 1, 220, 64], [0, 0, 120, 37]], np.int32)
    ring = ring_from(trajs, [(c, t0) for _, c, t0, _ in items], R, Cols, S, A)
    dev = [torch.from_numpy(x).cuda() for x in ring]
    out = [torch.zeros(R, Cols, device="cuda") for _ in range(3)]
    losses = torch.zeros(len(items), 2, device="cuda")
    twins = {a: twin(gpu, pop, a) for a in range(4)}
    untouched = pop_state(pop, 3)
    before = pop.launch_count()
    check(lib().wb_population_train_dev(pop._h, len(items), ptr(items), R, Cols, 5, seed, *[ptr(x) for x in dev], None,
                                        *[ptr(x) for x in out], ptr(losses), None))
    pop.sync()
    assert pop.launch_count() == before + 1
    V, G, Adv = [x.cpu().numpy() for x in out]
    episodes = {}
    for k, (a, c, t0, L) in enumerate(items):
        e = episodes.get(a, 0)
        episodes[a] = e + 1
        rv, rg, ra = train_replay(twins[a], trajs[k], device_draw(L, hps[a].batch_size, 5, e, a, seed))
        rows = (t0 + np.arange(L)) % R
        for got, want in zip((V, G, Adv), (rv, rg, ra)):
            assert np.array_equal(bits(got[rows, c]), bits(want)), k
    for a in range(3):
        assert_same(pop_state(pop, a), agent_state(twins[a]), a)
    assert_same(pop_state(pop, 3), untouched, "unlisted agent")


@pytest.mark.parametrize("rough,max_timesteps,steps", [(False, 150, 260), (True, 40, 200)])
def test_independent_ppo_with_custom_networks_replays_agent_by_agent(gpu, rough, max_timesteps, steps):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    n = 64
    hp = gpu.default_hyperparams()
    hp.max_timesteps, hp.batch_size = max_timesteps, 16
    terrain = None
    if rough:
        rng = np.random.default_rng(4)
        terrain = [gpu.CreateRoughFloor(rng.integers(0, 100, 11)) for _ in range(n)]
    actor, critic = NETS[4][2], NETS[1][3]
    loop = gpu.IndependentPPO(n, hp=hp, seed=21, epochs=3, terrain=terrain, actor=actor, critic=critic)
    assert loop.pop.N_PARAMS != 6149
    rec = {k: [] for k in ("states", "actions", "logp", "rewards", "dones")}
    for _ in range(steps):
        r = loop.t % loop.R
        done = loop.step()
        for k, src in (("states", loop.states), ("actions", loop.actions), ("logp", loop.logp), ("rewards", loop.rewards)):
            rec[k].append(src[r].cpu().numpy())
        rec["dones"].append(done)
    rec = {k: np.array(v) for k, v in rec.items()}
    assert rec["dones"].any()
    states = torch.from_numpy(rec["states"]).cuda()
    out_a, out_l = torch.empty(steps, n, 4, device="cuda"), torch.empty(steps, n, 4, device="cuda")
    for a in range(n):
        ref = twin(gpu, loop.pop, a)
        start, episode = 0, 0
        for t in range(steps):
            check(lib().wb_policy_act_dev(ref._h, n, ptr(states[t]), loop.act_seed, t, ptr(out_a[t]), ptr(out_l[t]), None, None))
            if rec["dones"][t, a]:
                tr = gpu.Trajectory(States=list(rec["states"][start:t + 1, a]), Actions=list(rec["actions"][start:t + 1, a]),
                                    LogProbabilities=list(rec["logp"][start:t + 1, a]), Rewards=list(rec["rewards"][start:t + 1, a]))
                train_replay(ref, tr, device_draw(t + 1 - start, 16, loop.epochs, episode, a, loop.train_seed), loop.epochs)
                start, episode = t + 1, episode + 1
        torch.cuda.synchronize()
        assert np.array_equal(bits(out_a[:, a].cpu().numpy()), bits(rec["actions"][:, a])), a
        assert np.array_equal(bits(out_l[:, a].cpu().numpy()), bits(rec["logp"][:, a])), a
        assert_same(pop_state(loop.pop, a), agent_state(ref), a)
    with pytest.raises(ValueError):
        gpu.IndependentPPO(4, actor=NETS[2][2], critic=NETS[2][3], stateSize=7, actionSize=3)


def test_default_lists_select_the_default_kernels(gpu):
    """wb_population_create_net with the default layer lists gives the bits of the default kernels (a PPOAgent on variant 1), which
    differ from those of the any-topology kernel (variant 2) on the same weights."""
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    hps = hp_sweep(gpu, 2)
    lists = [np.array(x, np.int32) for x in ([0, 2, 0, 2, 0, 3], [64, 0, 64, 0, 4, 0], [0, 2, 0], [64, 0, 1])]
    h = C.c_void_p()
    check(lib().wb_population_create_net(2, 12, 4, ptr(lists[0]), ptr(lists[1]), 6, ptr(lists[2]), ptr(lists[3]), 3,
                                         (gpu.Hyperparams * 2)(*hps), C.byref(h)))
    pop = gpu.PPOPopulation(2, hp=hps, seed=4)
    weights = [pop.get_weights(k) for k in range(2)]
    pop.close()
    pop._h = h
    for k in range(2):
        pop.set_weights(k, weights[k])
    assert (pop.N_ACTOR, pop.N_PARAMS) == (5252, 6149)
    states = torch.randn(2, 12, device="cuda")
    got = [torch.empty(2, 4, device="cuda") for _ in range(3)] + [torch.empty(2, device="cuda")]
    check(lib().wb_population_act_dev(h, 2, ptr(states), 3, 9, *[ptr(o) for o in got]))
    got = [o.cpu().numpy() for o in got]
    t = trajectories(gpu, 12, 4, [130, 64], seed=3)
    mine = pop.TrainTrajectories([(0, fresh(t[0])), (1, fresh(t[1]))])
    differs = False
    for k in range(2):
        ref, other = (gpu.PPOAgent(hp=hps[k], seed=pop.seeds[k]) for _ in range(2))
        ref.set_variant(1)
        other.set_variant(2)
        for agent in (ref, other):
            want = [torch.empty(2, 4, device="cuda") for _ in range(3)] + [torch.empty(2, device="cuda")]
            check(lib().wb_policy_act_dev(agent._h, 2, ptr(states), 3, 9, *[ptr(o) for o in want]))
            want = [o.cpu().numpy() for o in want]
            same = all(np.array_equal(bits(g[k]), bits(w[k])) for g, w in zip(got, want))
            if agent is ref:
                assert same, k
            else:
                differs |= not same
        assert np.array_equal(bits(mine[k]), bits(ref.TrainTrajectories([fresh(t[k])])[0])), k
        assert_same(pop_state(pop, k), agent_state(ref), k)
    assert differs  # (the two kernel families round differently: the comparison above tells them apart)


def test_bad_arguments_are_refused_and_change_nothing(gpu):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    bad = [  # (state, action, actor kinds/sizes, critic kinds/sizes)
        (12, 4, [(0, 256), (3, 0), (0, 4)], [(0, 1)]),
        (0, 4, [(0, 4)], [(0, 1)]),
        (12, 4, [(0, 8), (3, 0), (0, 5)], [(0, 1)]),
        (12, 4, [(0, 4)], [(0, 2)]),
        (12, 4, [(7, 4)], [(0, 1)]),
        (12, 4, [(1, 0)], [(0, 1)]),
        (12, 4, [(0, 4)] * 17, [(0, 1)]),
    ]
    for S, A, al, cl in bad:
        lists = [np.array([x[i] for x in layers], np.int32) for layers in (al, cl) for i in (0, 1)]
        h = C.c_void_p()
        codes = []
        for create in ("pop", "policy"):
            args = (S, A, ptr(lists[0]), ptr(lists[1]), len(al), ptr(lists[2]), ptr(lists[3]), len(cl))
            rc = (lib().wb_population_create_net(2, *args, None, C.byref(h)) if create == "pop"
                  else lib().wb_policy_create(*args, None, C.byref(h)))
            codes.append(rc)
        assert codes[0] == codes[1] != 0, (S, A, al, cl)
    net = NETS[0]
    pop = population(gpu, net, 3, seed=1)
    before = [pop_state(pop, a) for a in range(3)]
    d_states = torch.zeros(4, 12, device="cuda")
    o = [torch.empty(4, 4, device="cuda") for _ in range(2)]
    with pytest.raises(gpu.WalkerB200Error):
        check(lib().wb_population_act_dev(pop._h, 4, ptr(d_states), 1, 0, ptr(o[0]), ptr(o[1]), None, None))
    with pytest.raises(gpu.WalkerB200Error):
        check(lib().wb_population_sample(pop._h, 2, ptr(np.zeros((2, 12), np.float32)), ptr(np.zeros((2, 4, 2), np.float32)),
                                         ptr(np.zeros((2, 4), np.float32)), ptr(np.zeros((2, 4), np.float32)), None))
    t = trajectories(gpu, 12, 4, [1025], seed=8)[0]
    arr = [np.ascontiguousarray(np.array(x, np.float32)) for x in (t.States, t.Actions, t.LogProbabilities, t.Rewards)]
    index = np.zeros(5 * 1024, np.int32)
    with pytest.raises(gpu.WalkerB200Error) as ei:
        check(lib().wb_population_train_trajectories(pop._h, 1, ptr(np.zeros(1, np.int32)), ptr(np.array([0, 1025], np.int32)), 5,
                                                     *[ptr(x) for x in arr], ptr(index), None, None, None, None, None))
    assert ei.value.code == 4  # WB_ERR_UNSUPPORTED
    n_out = C.c_int32(0)
    with pytest.raises(gpu.WalkerB200Error):
        check(lib().wb_population_num_params(pop._h, 2, C.byref(n_out)))
    assert pop.launch_count() == 0
    for a in range(3):
        assert_same(pop_state(pop, a), before[a], a)


def test_two_populations_on_two_streams(gpu):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    net = NETS[1]
    trajs = trajectories(gpu, 12, 4, [130, 200, 70], seed=5)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    paired = [population(gpu, net, 2, seed=1, stream=s1.cuda_stream), population(gpu, net, 2, seed=2, stream=s2.cuda_stream)]
    R = 400
    ring = ring_from(trajs, [(0, 0), (0, 130), (1, 0)], R, 2, 12, 4)
    items = np.array([[0, 0, 0, 130], [1, 0, 130, 200], [0, 1, 0, 70]], np.int32)
    bufs = []
    for p in paired:
        bufs.append(([torch.from_numpy(x).cuda() for x in ring], [torch.zeros(R, 2, device="cuda") for _ in range(3)]))
    ref = [population(gpu, net, 2, seed=s) for s in (1, 2)]
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

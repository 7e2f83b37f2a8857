"""Population-based training on the device (wb_population_copy_agents / set_adam / set_hyperparams, IndependentPPO(pbt=)): every
agent against a PPOAgent twin given the same weights, Adam state, hyper-parameters and draws -- the setters, the copy kernel, refused
arguments, the PBT loop replayed in lockstep with the copies applied to the twins, and streams."""
import ctypes as C

import numpy as np
import pytest

from test_population_gpu import agent_state, assert_same, bits, device_draw, fresh, hp_sweep, pop_state, record_loop, ring_from, train_replay
from test_population_net_gpu import trajectories
from test_population_pbt_cpu import FLOATS, hp_dict, restate

pytestmark = pytest.mark.gpu

WIDE = ("Input |128| (LeakyReLU) |128| (LeakyReLU) |4| (TanH) Output", "Input |64| (LeakyReLU) |1| Output")
NETS = {"default": None, "wide128": WIDE}


def population(gpu, net, n, **kw):
    if NETS[net] is None:
        return gpu.PPOPopulation(n, **kw)
    return gpu.PPOPopulation(n, actor=NETS[net][0], critic=NETS[net][1], **kw)


def make_twin(gpu, pop, a, hp=None):
    """PPOAgent(seed=seeds[a]) with agent a's networks (variant 1 for the defaults, the any-topology kernel otherwise)."""
    hp = gpu.Hyperparams.from_buffer_copy(pop.hp[a] if hp is None else hp)
    agent = gpu.PPOAgent(hp=hp, actor=pop.actor_structure, critic=pop.critic_structure, seed=pop.seeds[a])
    if pop.actor_structure == gpu.DEFAULT_ACTOR and pop.critic_structure == gpu.DEFAULT_CRITIC:
        agent.set_variant(1)
    return agent


def give(twin, state, hp, n_actor):
    """set_flat / set_adam / set_hyperparams: the twin takes a population agent's (weights, m, v, steps) and hyper-parameters."""
    w, m, v, steps = state[:4]
    na = len(twin.actor.shapes)
    twin.actor.set_flat(w[:n_actor])
    twin.critic.set_flat(w[n_actor:])
    twin.actor.set_adam(m[:n_actor], v[:n_actor], steps[:na])
    twin.critic.set_adam(m[n_actor:], v[n_actor:], steps[na:])
    twin.set_hyperparams(type(hp).from_buffer_copy(hp))


def train_pop(gpu, pop, pairs, seed, epochs=3):
    """One wb_population_train_dev call with device draws: pairs [(agent, trajectory)], one ring column each."""
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    R, Cols = max(len(t.States) for _, t in pairs), len(pairs)
    dev = [torch.from_numpy(x).cuda() for x in ring_from([t for _, t in pairs], [(c, 0) for c in range(Cols)], R, Cols)]
    out = [torch.zeros(R, Cols, device="cuda") for _ in range(3)]
    items = np.array([[a, c, 0, len(t.States)] for c, (a, t) in enumerate(pairs)], np.int32)
    check(lib().wb_population_train_dev(pop._h, len(items), ptr(items), R, Cols, epochs, seed, *[ptr(x) for x in dev], None,
                                        *[ptr(x) for x in out], None, None))
    pop.sync()


def train_twin(gpu, twin, agent, traj, episode, seed, epochs=3):
    """The same episode on a twin, with the documented device draw of `agent`'s `episode`-th episode."""
    train_replay(gpu, twin, fresh(traj), device_draw(len(traj.States), twin.hp.batch_size, epochs, episode, agent, seed), epochs)


def get_hp(gpu, pop, a):
    from ppo_bipedalwalker_b200._lib import check, lib
    out = gpu.Hyperparams()
    check(lib().wb_population_get_hyperparams(pop._h, a, C.byref(out)))
    return out


def same_hp(x, y):
    return bytes(x) == bytes(y)


@pytest.mark.parametrize("net", list(NETS))
def test_setters_round_trip_and_an_agent_given_a_twins_state_trains_like_it(gpu, net):
    pop = population(gpu, net, 3, hp=hp_sweep(gpu, 3, batch_sizes=(32, 48)), seed=4)
    ref = make_twin(gpu, pop, 0, hp=hp_sweep(gpu, 5, batch_sizes=(40,))[4])
    trajs = trajectories(gpu, 12, 4, [150, 90, 200, 120], seed=1)
    ref.TrainTrajectories([fresh(trajs[0]), fresh(trajs[1])], epochs=2)  # a twin with Adam state of its own
    w, m, v, steps, _ = agent_state(ref)
    assert steps.min() > 0 and np.abs(m).max() > 0
    pop.set_weights(1, w)
    pop.set_adam(1, m, v, steps)
    pop.set_hyperparams(1, ref.hp)
    got = pop_state(pop, 1)
    assert_same(got[:4], (w, m, v, steps), "round trip")
    assert same_hp(get_hp(gpu, pop, 1), ref.hp) and same_hp(pop.hp[1], ref.hp)
    untouched = [pop_state(pop, a) for a in (0, 2)]
    # agent 1 has trained no episode: its device draws are keyed (episode 0, agent 1)
    train_pop(gpu, pop, [(1, trajs[2]), (1, trajs[3])], seed=17)
    train_twin(gpu, ref, 1, trajs[2], 0, 17)
    train_twin(gpu, ref, 1, trajs[3], 1, 17)
    assert_same(pop_state(pop, 1), agent_state(ref), "trained after the setters")
    for a, before in zip((0, 2), untouched):
        assert_same(pop_state(pop, a), before, a)


@pytest.mark.parametrize("net", list(NETS))
def test_copy_agents_copies_rows_bit_for_bit_in_one_launch(gpu, net):
    n = 40
    pop = population(gpu, net, n, hp=hp_sweep(gpu, n, batch_sizes=(32, 48, 64)), seed=6)
    trajs = trajectories(gpu, 12, 4, [100 + 7 * a for a in range(n)], seed=2)
    train_pop(gpu, pop, [(a, trajs[a]) for a in range(n) if a % 5 != 4], seed=3)  # agents 4, 9, ... have never trained
    episodes = [0 if a % 5 == 4 else 1 for a in range(n)]
    before = [pop_state(pop, a) for a in range(n)]
    hp_before = [gpu.Hyperparams.from_buffer_copy(h) for h in pop.hp]
    rng = np.random.default_rng(0)
    order = rng.permutation(n)
    dst, src = order[:15], order[15:30][rng.integers(0, 15, 15)]  # several dst may share a src
    new_hp = []
    for k in range(15):
        h = gpu.Hyperparams.from_buffer_copy(hp_before[src[k]])
        h.alpha, h.epsilon, h.log_std = h.alpha * 1.2, 0.25 + 0.01 * k, -0.5 - 0.1 * k
        h.batch_size = 16 + k
        new_hp.append(h)
    launches = pop.launch_count()
    pop.copy_agents(list(zip(dst, src)), new_hp)
    pop.sync()
    assert pop.launch_count() == launches + 1
    for k, (d, s) in enumerate(zip(dst, src)):
        w, m, v, steps, g = pop_state(pop, d)
        assert_same((w, m, v, steps), before[s][:4], (d, s))
        assert np.array_equal(bits(g), bits(before[d][4])), "dst keeps its gradient buffer"
        assert same_hp(get_hp(gpu, pop, d), new_hp[k]) and same_hp(pop.hp[d], new_hp[k])
    for a in set(range(n)) - set(dst):
        assert_same(pop_state(pop, a), before[a], a)
        assert same_hp(get_hp(gpu, pop, a), hp_before[a])
    # hp None: dst takes src's hyper-parameters
    pop.copy_agents([(order[30], order[0])])
    assert same_hp(get_hp(gpu, pop, order[30]), new_hp[0]) and same_hp(pop.hp[order[30]], new_hp[0])
    # training dst afterwards equals a twin given src's state, the new hyper-parameters and dst's own episode counter
    more = trajectories(gpu, 12, 4, [120 + 11 * k for k in range(6)], seed=3)
    picked = [int(d) for d in dst[:6]]
    twins = {}
    for k, d in enumerate(picked):
        twins[d] = make_twin(gpu, pop, d)
        give(twins[d], before[src[k]], new_hp[k], pop.N_ACTOR)
    train_pop(gpu, pop, [(d, more[k]) for k, d in enumerate(picked)], seed=29)
    for k, d in enumerate(picked):
        train_twin(gpu, twins[d], d, more[k], episodes[d], 29)
        assert_same(pop_state(pop, d), agent_state(twins[d]), d)


def test_refused_arguments_change_nothing(gpu):
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    n = 6
    pop = gpu.PPOPopulation(n, hp=hp_sweep(gpu, n), seed=2)
    train_pop(gpu, pop, [(a, t) for a, t in enumerate(trajectories(gpu, 12, 4, [130] * n, seed=4))], seed=1)
    before = [pop_state(pop, a) for a in range(n)]
    hp_before = [bytes(get_hp(gpu, pop, a)) for a in range(n)]
    launches = pop.launch_count()
    bad_hp = gpu.default_hyperparams()
    bad_hp.batch_size = 0
    good = gpu.default_hyperparams()
    cases = [([], [], None),                        # n_pairs < 1
             ([6], [0], None), ([-1], [0], None),   # dst out of range
             ([1], [6], None), ([1], [-2], None),   # src out of range
             ([2], [2], None),                      # dst == src
             ([1, 1], [0, 2], None),                # a dst listed twice
             ([1, 2], [0, 1], None),                # an agent both a src and a dst
             ([3, 4], [0, 0], [good, bad_hp])]      # batch_size < 1
    for dst, src, hps in cases:
        d, s = np.array(dst + [0], np.int32), np.array(src + [0], np.int32)
        arr = (gpu.Hyperparams * len(hps))(*hps) if hps else None
        assert lib().wb_population_copy_agents(pop._h, len(dst), ptr(d), ptr(s), arr) == 1, (dst, src)
    m, v, steps = pop.adam(0)
    assert lib().wb_population_set_adam(pop._h, n, ptr(m), ptr(v), ptr(steps)) == 1
    assert lib().wb_population_set_adam(pop._h, -1, ptr(m), ptr(v), ptr(steps)) == 1
    assert lib().wb_population_set_hyperparams(pop._h, 1, C.byref(bad_hp)) == 1
    assert lib().wb_population_set_hyperparams(pop._h, n, C.byref(good)) == 1
    assert lib().wb_population_get_hyperparams(pop._h, n, C.byref(good)) == 1
    with pytest.raises(gpu.WalkerB200Error):
        pop.copy_agents([(1, 0), (1, 2)])
    pop.sync()
    assert pop.launch_count() == launches
    for a in range(n):
        assert_same(pop_state(pop, a), before[a], a)
        assert bytes(get_hp(gpu, pop, a)) == hp_before[a] and bytes(pop.hp[a]) == hp_before[a]


def replay_with_copies(gpu, loop, rec, hp0, xlog):
    """One PPOAgent twin per agent, in lockstep: each acts with wb_policy_act_dev of its current weights, trains on each of its
    episodes with the restated device draw (keyed by its own episode counter), and at the end of every step takes the logged
    copies with set_flat / set_adam / set_hyperparams.  Asserts every step's actions and log-probabilities; returns the twins."""
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    pop = loop.pop
    twins = [make_twin(gpu, pop, a, hp=hp0[a]) for a in range(loop.n)]
    steps, n = rec["dones"].shape
    states = torch.from_numpy(rec["states"]).cuda()
    acts, logp = torch.empty(steps, n, 4, device="cuda"), torch.empty(steps, n, 4, device="cuda")
    ta, tl = torch.empty(n, 4, device="cuda"), torch.empty(n, 4, device="cuda")
    start, episode = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for t in range(steps):
        for a in range(n):
            check(lib().wb_policy_act_dev(twins[a]._h, a + 1, ptr(states[t]), loop.act_seed, t, ptr(ta), ptr(tl), None, None))
            acts[t, a], logp[t, a] = ta[a], tl[a]
        for a in np.flatnonzero(rec["dones"][t]):
            rows = slice(start[a], t + 1)
            tr = gpu.Trajectory(States=list(rec["states"][rows, a]), Actions=list(rec["actions"][rows, a]),
                                LogProbabilities=list(rec["logp"][rows, a]), Rewards=list(rec["rewards"][rows, a]))
            train_replay(gpu, twins[a], tr, device_draw(t + 1 - start[a], twins[a].hp.batch_size, loop.epochs, episode[a], a,
                                                        loop.train_seed), loop.epochs)
            start[a], episode[a] = t + 1, episode[a] + 1
        for x in xlog[xlog["step"] == t]:
            d, s = int(x["dst"]), int(x["src"])
            src_state = agent_state(twins[s])
            h = gpu.Hyperparams(*[x[name].item() for name, _ in gpu.Hyperparams._fields_])
            give(twins[d], src_state, h, pop.N_ACTOR)
    torch.cuda.synchronize()
    assert np.array_equal(bits(acts.cpu().numpy()), bits(rec["actions"]))
    assert np.array_equal(bits(logp.cpu().numpy()), bits(rec["logp"]))
    return twins


# (64 walkers, short episodes, a short window and a quarter of the ranked agents copying: dozens of copies in a few hundred steps)
@pytest.mark.parametrize("rough,net", [(False, "default"), (True, "default"), (False, "wide128")])
def test_independent_ppo_with_pbt_replays_in_lockstep(gpu, rough, net):
    n, steps, interval, fraction, window = 64, 240, 30, 0.25, 2
    hp = hp_sweep(gpu, n, batch_sizes=(16, 24))
    for h in hp:
        h.max_timesteps, h.use_gae, h.normalize_advantages = 40, 0, 0
    terrain = None
    if rough:
        rng = np.random.default_rng(4)
        terrain = [gpu.CreateRoughFloor(rng.integers(0, 100, 11)) for _ in range(n)]
    kw = {} if NETS[net] is None else dict(actor=NETS[net][0], critic=NETS[net][1])
    perturb = {"alpha": (1e-5, 1e-2), "gamma": (0.8, 0.99), "epsilon": (0.05, 0.5), "log_std": (-3.0, 0.0)}
    pbt = gpu.PBT(interval, fraction=fraction, window=window, perturb=perturb, seed=7)
    loop = gpu.IndependentPPO(n, hp=hp, seed=21, epochs=2, terrain=terrain, pbt=pbt, **kw)
    hp0 = [gpu.Hyperparams.from_buffer_copy(h) for h in loop.pop.hp]
    before = loop.pop.launch_count()
    rec = record_loop(gpu, loop, steps)
    log, xlog = loop.episode_log(), loop.exploit_log()
    assert len(xlog) >= 10 and len(set(xlog["step"])) >= 3
    copy_steps = len(set(xlog["step"].tolist()))
    assert loop.pop.launch_count() - before == steps + int(rec["dones"].any(1).sum()) + copy_steps
    want = restate(n, [(int(e["step"]), int(e["agent"]), float(e["reward"])) for e in log], steps, [hp_dict(h) for h in hp0], interval,
                   fraction, window, perturb=perturb, seed=7)
    assert [(int(x["step"]), int(x["dst"]), int(x["src"])) for x in xlog] == [(t, d, s) for t, d, s, _ in want]
    for x, (_, _, _, h) in zip(xlog, want):
        assert all(np.float32(x[name]).view(np.uint32) == np.float32(h[name]).view(np.uint32) for name in FLOATS)
        assert all(x[name] == h[name] for name in ("iterations", "max_timesteps", "batch_size"))
    twins = replay_with_copies(gpu, loop, rec, hp0, xlog)
    for a in range(n):
        assert_same(pop_state(loop.pop, a), agent_state(twins[a]), a)
        assert same_hp(loop.pop.hp[a], twins[a].hp) and same_hp(get_hp(gpu, loop.pop, a), twins[a].hp)


def test_fraction_zero_equals_no_pbt(gpu):
    n, steps = 64, 150
    hp = gpu.default_hyperparams()
    hp.max_timesteps, hp.batch_size = 40, 16
    loops = [gpu.IndependentPPO(n, hp=hp, seed=5, epochs=2, pbt=p) for p in (None, gpu.PBT(10, fraction=0.0, window=1))]
    recs = [record_loop(gpu, loop, steps) for loop in loops]
    assert loops[0].pop.launch_count() == loops[1].pop.launch_count()
    assert len(loops[1].exploit_log()) == 0
    for k in recs[0]:
        assert np.array_equal(recs[0][k], recs[1][k]), k
    for a in range(n):
        assert_same(pop_state(loops[0].pop, a), pop_state(loops[1].pop, a), a)


def test_two_populations_copying_and_training_on_two_streams(gpu):
    import torch
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    n, R = 8, 260
    trajs = trajectories(gpu, 12, 4, [130, 200, 90, 256, 160, 70, 110, 240], seed=9)
    ring = ring_from(trajs, [(c, 0) for c in range(n)], R, n)
    items = np.array([[c, c, 0, len(t.States)] for c, t in enumerate(trajs)], np.int32)
    dst, src = np.array([1, 4, 6], np.int32), np.array([0, 3, 0], np.int32)
    hps = (gpu.Hyperparams * 3)(*hp_sweep(gpu, 3, batch_sizes=(32,)))

    def calls(pop, dev, outs):
        check(lib().wb_population_train_dev(pop._h, n, ptr(items), R, n, 3, 5, *[ptr(x) for x in dev], None, *[ptr(x) for x in outs[0]],
                                            None, None))
        check(lib().wb_population_copy_agents(pop._h, 3, ptr(dst), ptr(src), hps))
        check(lib().wb_population_train_dev(pop._h, n, ptr(items), R, n, 3, 6, *[ptr(x) for x in dev], None, *[ptr(x) for x in outs[1]],
                                            None, None))

    def buffers():
        return [torch.from_numpy(x).cuda() for x in ring], [[torch.zeros(R, n, device="cuda") for _ in range(3)] for _ in range(2)]

    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    paired = [gpu.PPOPopulation(n, seed=1, stream=s1.cuda_stream), gpu.PPOPopulation(n, seed=2, stream=s2.cuda_stream)]
    bufs = [buffers() for _ in paired]
    torch.cuda.synchronize()
    for p, (dev, outs) in zip(paired, bufs):  # both streams enqueued before either finishes
        calls(p, dev, outs)
    torch.cuda.synchronize()
    for seed, (dev, outs), p in zip((1, 2), bufs, paired):
        ref = gpu.PPOPopulation(n, seed=seed)
        rdev, routs = buffers()
        calls(ref, rdev, routs)
        ref.sync()
        for x, y in zip(sum(outs, []), sum(routs, [])):
            assert torch.equal(x, y)
        for a in range(n):
            assert_same(pop_state(p, a), pop_state(ref, a), a)

"""PPOAgent.Train(Trajectory) for a list of finished episodes in one device call (wb_ppo_train_trajectories): against the
per-mini-batch path (PPOAgent.Train per trajectory), against a restatement of PPOAgent.cs:147-172 on the CPU oracle, and its
entries, streams and edge cases."""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# below B, not a multiple of 64, empty, the max_timesteps cap, exactly B, longer than the kernel's shared-memory returns (1 024 rows)
LENGTHS = [37, 130, 0, 1001, 64, 200, 63, 1500]


def rollout(gpu, lengths, seed=0, sdim=12):
    """Real walker steps from the library's Environment under a seeded random policy (auto-reset), cut into trajectories."""
    env = gpu.Environment(1)
    roller = gpu.PPOAgent(seed=seed)
    state = env.InitialState()
    trajs = []
    for T in lengths:
        t = gpu.Trajectory()
        for _ in range(T):
            a, lp, _, _ = roller.SampleActions(state)
            t.States.append(state[0][:sdim].copy())
            state, reward, _ = env.Update(gpu.DT_FRAME, a, auto_reset=True)
            t.Actions.append(a[0].copy())
            t.LogProbabilities.append(lp[0].copy())
            t.Rewards.append(float(reward[0]))
        trajs.append(t)
    return trajs


def keep_clear_of_leaky_kinks(states, actor_flat, critic_flat, margin=1e-5):
    """A sample whose hidden pre-activation is within rounding distance of 0 may take either LeakyReLU slope: replace it."""
    s = states.astype(np.float64)
    a, c = np.asarray(actor_flat, np.float64), np.asarray(critic_flat, np.float64)
    z1 = s @ a[:768].reshape(64, 12).T + a[768:832]
    z2 = np.maximum(0.2 * z1, z1) @ a[832:4928].reshape(64, 64).T + a[4928:4992]
    zc = s @ c[:768].reshape(64, 12).T + c[768:832]
    tight = np.minimum(np.minimum(np.abs(z1).min(1), np.abs(z2).min(1)), np.abs(zc).min(1)) < margin
    if tight.any():
        states[tight] = states[np.flatnonzero(~tight)[0]]
    return states


def clear_of_boundaries(trajs, agent, perturb_rng=None):
    """Keep samples clear of the LeakyReLU kinks and the clip boundaries under the initial weights (see test_ppo_gpu.py)."""
    af, cf = agent.actor.get_flat(), agent.critic.get_flat()
    std = np.exp(np.float32(agent.hp.log_std))
    for t in trajs:
        if not t.States:
            continue
        s = keep_clear_of_leaky_kinks(np.array(t.States, np.float32), af, cf)
        t.States = list(s)
        mean, _ = agent.FeedForward(s)
        a = np.array(t.Actions, np.float32)
        logp = (-np.log(std) - np.log(np.sqrt(2 * np.pi)) - 0.5 * ((a - mean) / std) ** 2).astype(np.float32)
        old = logp if perturb_rng is None else (logp + 0.25 * perturb_rng.normal(size=logp.shape)).astype(np.float32)
        ratio = np.exp(logp.astype(np.float64) - old)
        old[(np.abs(ratio - 1.3) < 1e-3) | (np.abs(ratio - 0.7) < 1e-3)] += np.float32(0.01)
        t.LogProbabilities = list(old)
    return trajs


def fresh(trajs):
    return [type(t)(States=list(t.States), Actions=list(t.Actions), LogProbabilities=list(t.LogProbabilities), Rewards=list(t.Rewards))
            for t in trajs]


def bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def agent_state(agent):
    out = {}
    for which in ("actor", "critic"):
        net = getattr(agent, which)
        m, v, it = net.get_adam()
        out[which] = (net.get_flat(), m, v, it, net.get_grads())
    return out


def assert_same_state(a, b):
    for which in ("actor", "critic"):
        for x, y, name in zip(a[which], b[which], ("weights", "adam m", "adam v", "step counters", "gradient buffer")):
            assert np.array_equal(bits(x) if x.dtype == np.float32 else x, bits(y) if y.dtype == np.float32 else y), (which, name)


def make_agent(gpu, seed, batch_size=64, use_gae=0, normalize=0, variant=0, **kw):
    hp = gpu.default_hyperparams()
    hp.batch_size, hp.use_gae, hp.normalize_advantages = batch_size, use_gae, normalize
    agent = gpu.PPOAgent(hp=hp, seed=seed, **kw)
    agent.set_variant(variant)
    return agent


@pytest.mark.parametrize("use_gae", [0, 1])
@pytest.mark.parametrize("normalize", [0, 1])
def test_one_call_equals_train_per_trajectory_bit_for_bit(gpu, use_gae, normalize):
    """Same seed, same mini-batches: the one-launch kernel and PPOAgent.Train on the CUDA-core kernel (variant 1) run the same tile
    code, the same single-CTA reduction and the same Adam with the same host corrections -- weights, Adam state, the gradient
    buffer, losses, skipped counts and Values / Returns / Advantages agree to the bit."""
    trajs = rollout(gpu, LENGTHS, seed=1)
    ref = make_agent(gpu, 3, use_gae=use_gae, normalize=normalize, variant=1)
    new = make_agent(gpu, 3, use_gae=use_gae, normalize=normalize, variant=0)
    t_ref, t_new = fresh(trajs), fresh(trajs)
    ref_losses = [ref.Train(t) for t in t_ref]
    new_losses = new.TrainTrajectories(t_new)
    assert_same_state(agent_state(ref), agent_state(new))
    assert np.array_equal(np.array(ref_losses, np.float32).view(np.uint32), np.array(new_losses, np.float32).view(np.uint32))
    for a, b in zip(t_ref, t_new):
        for attr in ("Values", "Returns", "Advantages"):
            assert np.array_equal(bits(getattr(a, attr)), bits(getattr(b, attr))), attr
    _, _, it = new.actor.get_adam()
    assert list(it) == [5 * sum(T // 64 for T in LENGTHS)] * 3
    assert ref.rng.random() == new.rng.random()  # the same number of draws


def oracle_train(O, actor, critic, ohp, hp, trajs, rng, epochs, B):
    """PPOAgent.Train(Trajectory) restated on the oracle: CalculateValues, MC return / GAE, Normalize, shuffled mini-batches."""
    out = []
    for t in trajs:
        T = len(t.States)
        if T == 0:
            out.append(None)
            continue
        S = np.array(t.States, np.float32)
        values = critic.forward(S)[:, 0].copy()
        r = np.array(t.Rewards, np.float32)
        G, A = O.gae(r, values, hp.gamma, hp.lambda_) if hp.use_gae else O.mc_returns(r, values, hp.gamma)
        if hp.normalize_advantages:
            A = O.normalize(A, hp.epsilon)
        acts, lp = np.array(t.Actions, np.float32), np.array(t.LogProbabilities, np.float32)
        for _ in range(epochs):
            perm = rng.permutation(T)
            for j in range(T // B):
                idx = perm[j * B:(j + 1) * B]
                O.ppo_train_batch(actor, critic, ohp, S[idx], acts[idx], lp[idx], A[idx], G[idx], optimise=True)
        out.append(values)
    return out


def oracle_pair(gpu, O, agent, actor_layers=None, critic_layers=None):
    actor = O.Net(agent.stateSize, actor_layers or O.ACTOR_LAYERS)
    critic = O.Net(agent.stateSize, critic_layers or O.CRITIC_LAYERS)
    actor.set_params(agent.actor.get_flat())
    critic.set_params(agent.critic.get_flat())
    ohp = O.hyper_defaults()
    ohp.batch_size = agent.hp.batch_size
    return actor, critic, ohp


def check_against_oracle(gpu, O, agent, trajs, actor, critic, ohp, epochs=5):
    rng = copy.deepcopy(agent.rng)
    agent.TrainTrajectories(trajs, epochs)
    ref_values = oracle_train(O, actor, critic, ohp, agent.hp, trajs, rng, epochs, agent.hp.batch_size)
    hp = agent.hp
    for t, rv in zip(trajs, ref_values):
        if rv is None:
            continue
        v = np.array(t.Values, np.float32)
        np.testing.assert_allclose(v, rv, rtol=0, atol=1e-5)
        r = np.array(t.Rewards, np.float32)
        G, A = O.gae(r, v, hp.gamma, hp.lambda_) if hp.use_gae else O.mc_returns(r, v, hp.gamma)
        if hp.normalize_advantages:
            A = O.normalize(A, hp.epsilon)
        assert np.array_equal(bits(t.Returns), bits(G)) and np.array_equal(bits(t.Advantages), bits(A))
    np.testing.assert_allclose(agent.actor.get_flat(), actor.get_params(), rtol=0, atol=2e-5)
    np.testing.assert_allclose(agent.critic.get_flat(), critic.get_params(), rtol=0, atol=2e-5)


@pytest.mark.parametrize("batch_size", [64, 100])
def test_one_call_tracks_the_oracle(gpu, O, batch_size):
    """B = 64 (one tile per mini-batch) and B = 100 (a partial second tile), 5 epochs, GAE + Normalize."""
    agent = make_agent(gpu, 5, batch_size=batch_size, use_gae=1, normalize=1)
    trajs = clear_of_boundaries(rollout(gpu, [70, 130, 40, 0, 210], seed=2), agent, np.random.default_rng(5))
    actor, critic, ohp = oracle_pair(gpu, O, agent)
    check_against_oracle(gpu, O, agent, trajs, actor, critic, ohp)


def test_non_default_network_runs_the_sequenced_path(gpu, O):
    """A user-edited DSL network: the same entry enqueues the per-trajectory / per-mini-batch kernels; against the restatement and
    against PPOAgent.Train on the same network (same kernels: bit for bit)."""
    actor_dsl, critic_dsl = "Input |32| (ReLU) |4| (TanH) Output", "Input |16| (ReLU) |16| (TanH) |1| Output"
    agent = make_agent(gpu, 7, batch_size=64, actor=actor_dsl, critic=critic_dsl, variant=2)
    twin = make_agent(gpu, 7, batch_size=64, actor=actor_dsl, critic=critic_dsl, variant=2)
    trajs = rollout(gpu, [70, 130, 0, 40], seed=3)
    perturb = np.random.default_rng(7)
    for t in trajs:
        t.LogProbabilities = [lp + np.float32(0.2) * perturb.normal(size=4).astype(np.float32) for lp in t.LogProbabilities]
    actor, critic, ohp = oracle_pair(gpu, O, agent, gpu.ParseLayers(actor_dsl), gpu.ParseLayers(critic_dsl))
    t_twin = fresh(trajs)
    for t in t_twin:
        twin.Train(t)
    check_against_oracle(gpu, O, agent, trajs, actor, critic, ohp)
    assert_same_state(agent_state(twin), agent_state(agent))


@pytest.mark.parametrize("variant", [0, 1])
def test_one_launch_per_call_on_the_default_networks(gpu, variant):
    agent = make_agent(gpu, 9, variant=variant)
    trajs = rollout(gpu, [130, 70], seed=4)
    before = agent.launch_count()
    agent.TrainTrajectories(trajs)
    assert agent.launch_count() == before + 1
    agent.TrainTrajectories(trajs[:1])
    assert agent.launch_count() == before + 2


def flat_inputs(agent, trajs, epochs=5):
    """What TrainTrajectories passes to the C entry (draws from agent.rng)."""
    B = agent.hp.batch_size
    lengths = [len(t.States) for t in trajs]
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    blocks = []
    for T in lengths:
        if T:
            for _ in range(epochs):
                perm = agent.rng.permutation(T)
                blocks.extend(perm[j * B:(j + 1) * B] for j in range(T // B))
    index = np.concatenate(blocks).astype(np.int32)
    cat = lambda attr, w: np.ascontiguousarray(np.concatenate([np.array(getattr(t, attr), np.float32).reshape(-1, w) for t in trajs if len(t.States)]))
    return offsets, index, cat("States", 12), cat("Actions", 4), cat("LogProbabilities", 4), cat("Rewards", 1).ravel()


def to_device(offsets, index, S, A, L, R):
    import torch
    n = len(offsets) - 1
    dev = [torch.from_numpy(x).cuda() for x in (S, A, L, R, index)]
    out = [torch.zeros(R.size, device="cuda") for _ in range(3)] + [torch.zeros(2 * n, device="cuda"),
                                                                     torch.zeros(n, dtype=torch.int32, device="cuda")]
    return offsets, dev, out


def train_dev(agent, offsets, dev, out):
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    check(lib().wb_ppo_train_trajectories_dev(agent._h, len(offsets) - 1, ptr(offsets), 5, *[ptr(t) for t in dev], *[ptr(t) for t in out]))


def test_dev_entry_equals_host_entry_and_two_streams_run_concurrently(gpu):
    import torch
    trajs = rollout(gpu, [130, 70, 1001], seed=5)
    host = make_agent(gpu, 11)
    alone = [make_agent(gpu, 11), make_agent(gpu, 12)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    paired = [make_agent(gpu, 11, stream=s1.cuda_stream), make_agent(gpu, 12, stream=s2.cuda_stream)]
    host_losses = host.TrainTrajectories(fresh(trajs))
    bufs = [to_device(*flat_inputs(a, trajs)) for a in alone]
    pbufs = [to_device(*flat_inputs(a, trajs)) for a in paired]  # (the same draws: same seeds)
    torch.cuda.synchronize()
    for a, b in zip(alone, bufs):
        train_dev(a, *b)
        a.sync()
    for a, b in zip(paired, pbufs):  # both enqueued before either finishes
        train_dev(a, *b)
    torch.cuda.synchronize()
    assert_same_state(agent_state(host), agent_state(alone[0]))
    assert np.array_equal(np.array(host_losses, np.float32).ravel().view(np.uint32), bufs[0][2][3].cpu().numpy().view(np.uint32))
    for x, y in zip(bufs[0][2][:3], pbufs[0][2][:3]):
        assert torch.equal(x, y)
    for a, b in zip(alone, paired):
        assert_same_state(agent_state(a), agent_state(b))


def test_short_trajectory_fills_values_and_takes_no_adam_step(gpu, O):
    agent = make_agent(gpu, 13, variant=1)
    trajs = rollout(gpu, [40], seed=6)
    w0 = agent.actor.get_flat()
    losses = agent.TrainTrajectories(trajs)
    assert losses == [(0.0, 0.0)]
    _, _, it = agent.actor.get_adam()
    assert list(it) == [0, 0, 0] and np.array_equal(agent.actor.get_flat(), w0)
    assert np.array_equal(bits(trajs[0].Values), bits(agent.FeedForward(np.array(trajs[0].States))[1]))


def test_underflowing_old_probability_is_skipped_like_the_twin(gpu):
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    trajs = rollout(gpu, [130, 70], seed=7)
    trajs[0].LogProbabilities[5] = np.array([0.0, -200.0, 0.0, 0.0], np.float32)  # exp underflows: the sample is skipped
    ref, new = make_agent(gpu, 15, variant=1), make_agent(gpu, 15)
    ref_skipped = []
    for t in fresh(trajs):  # PPOAgent.Train per trajectory, counting skipped samples per mini-batch
        ref.CalculateValues(t)
        T, B = len(t.States), 64
        S, A, L = (np.array(getattr(t, k), np.float32) for k in ("States", "Actions", "LogProbabilities"))
        G, Adv = np.array(t.Returns, np.float32), np.array(t.Advantages, np.float32)
        total = 0
        for _ in range(5):
            perm = ref.rng.permutation(T)
            for j in range(T // B):
                idx = perm[j * B:(j + 1) * B]
                total += ref.TrainBatch(S[idx], A[idx], L[idx], Adv[idx], G[idx])[2]
        ref_skipped.append(total)
    offsets, index, S, A, L, R = flat_inputs(new, trajs)
    losses = np.zeros(4, np.float32)
    skipped = np.zeros(2, np.int32)
    check(lib().wb_ppo_train_trajectories(new._h, 2, ptr(offsets), 5, ptr(S), ptr(A), ptr(L), ptr(R), ptr(index), None, None, None,
                                          ptr(losses), ptr(skipped)))
    assert list(skipped) == ref_skipped and ref_skipped[0] == 5  # once per epoch
    assert_same_state(agent_state(ref), agent_state(new))


def test_bad_arguments_are_refused_and_change_nothing(gpu):
    from ppo_bipedalwalker_b200._lib import check, lib, ptr
    agent = make_agent(gpu, 17)
    trajs = rollout(gpu, [130, 70], seed=8)
    offsets, index, S, A, L, R = flat_inputs(agent, trajs)
    before = agent_state(agent)
    bad_index = index.copy()
    bad_index[-1] = 70  # trajectory 1 has rows 0..69
    cases = [(2, offsets, 5, bad_index), (2, np.array([0, 130, 100], np.int32), 5, index), (2, offsets, -1, index),
             (0, offsets, 5, index)]
    for n, off, epochs, idx in cases:
        with pytest.raises(gpu.WalkerB200Error):
            check(lib().wb_ppo_train_trajectories(agent._h, n, ptr(off), epochs, ptr(S), ptr(A), ptr(L), ptr(R), ptr(idx), None, None, None,
                                                  None, None))
        assert_same_state(before, agent_state(agent))

"""The population-based training schedule (PBT, host only) against a plain restatement of the rule its docstring states, on
synthetic episode streams: ties, short histories, fraction 0 and 0.5, dropped bottom agents, perturbation bounds, seeds and refused
arguments.  tests/test_population_pbt_gpu.py reuses restate() on the episodes of a real IndependentPPO run."""
import numpy as np
import pytest

FLOATS = ("alpha", "beta1", "beta2", "adam_epsilon", "gamma", "lambda_", "epsilon", "log_std")  # wb_hyperparams order


def restate(n, episodes, steps, hp, interval, fraction=0.2, window=5, perturb=None, seed=0):
    """The rule, restated.  episodes: (step, agent, reward sum) of every finished episode; hp: every agent's starting
    hyper-parameters as {field: value}.  Returns the copies [(step, dst, src, dst's new {field: value})] in order."""
    if perturb is None:
        perturb = {"alpha": (1e-5, 1e-2), "epsilon": (0.05, 0.5), "log_std": (-3.0, 0.0)}
    g = np.random.default_rng(seed)
    hp = [dict(h) for h in hp]
    hist = [[] for _ in range(n)]
    top, waiting, out = [], [], []
    for t in range(steps):
        ended = sorted((int(a), r) for s, a, r in episodes if s == t)
        for a, r in ended:
            hist[a].append(np.float64(np.float32(r)))
        for a, _ in ended:
            if a not in waiting:
                continue
            src = top[g.integers(len(top))]
            new = dict(hp[src])
            for name in FLOATS:
                if name in perturb:
                    lo, hi = perturb[name]
                    f = 0.8 if g.random() < 0.5 else 1.2
                    new[name] = np.float32(min(max(np.float32(np.float64(new[name]) * f), lo), hi))
            hp[a] = new
            hist[a] = []
            waiting.remove(a)
            out.append((t, a, src, new))
        if (t + 1) % interval == 0:
            ranked = [a for a in range(n) if len(hist[a]) >= window]
            score = {a: np.mean(np.array(hist[a][-window:], np.float64)) for a in ranked}
            ranked.sort(key=lambda a: (-score[a], a))
            k = int(np.floor(fraction * len(ranked)))
            top, waiting = ranked[:k], ranked[len(ranked) - k:] if k else []
    return out


def hp_dict(h):
    return {name: getattr(h, name) for name, _ in type(h)._fields_}


def run_schedule(wb, n, episodes, steps, hps, **kw):
    """PBT.step driven as IndependentPPO drives it, with the copies applied to the hyper-parameter list."""
    pbt = wb.PBT(**kw)
    hps = [wb.Hyperparams.from_buffer_copy(h) for h in hps]
    out = []
    for t in range(steps):
        ended = [(a, r) for s, a, r in episodes if s == t]
        for dst, src, h in pbt.step(t, [a for a, _ in ended], [r for _, r in ended], hps):
            hps[dst] = h
            out.append((t, dst, src, hp_dict(h)))
    return out


def synthetic(n, steps, seed, levels=None):
    """Episodes of random lengths per agent; rewards from `levels` values (ties) or continuous."""
    rng = np.random.default_rng(seed)
    episodes = []
    for a in range(n):
        t = int(rng.integers(0, 8))
        while t < steps:
            r = float(rng.choice(levels)) if levels is not None else float(np.float32(rng.normal(a * 0.1, 1.0)))
            episodes.append((t, a, r))
            t += int(rng.integers(1, 12))
    return sorted(episodes, key=lambda e: (e[0], e[1]))


def assert_same_copies(got, want):
    assert [(t, d, s) for t, d, s, _ in got] == [(t, d, s) for t, d, s, _ in want]
    for (_, _, _, h), (_, _, _, r) in zip(got, want):
        for name in FLOATS:
            assert np.float32(h[name]).view(np.uint32) == np.float32(r[name]).view(np.uint32), name
        for name in ("iterations", "max_timesteps", "batch_size", "use_gae", "normalize_advantages"):
            assert h[name] == r[name], name


def sweep(wb, n):
    out = []
    for a in range(n):
        h = wb.default_hyperparams()
        h.alpha, h.gamma, h.log_std, h.batch_size = 1e-3 * (1 + a % 4), 0.9 + 0.01 * (a % 3), -1.0 + 0.1 * (a % 5), 16 + a
        out.append(h)
    return out


@pytest.mark.parametrize("interval,fraction,window,levels", [(10, 0.2, 3, None), (7, 0.5, 1, [0.0, 1.0]), (5, 0.34, 4, [0.0, 1.0, 2.0]),
                                                             (13, 0.25, 8, None), (1, 0.5, 2, [1.0])])
def test_schedule_equals_the_restated_rule(wb, interval, fraction, window, levels):
    n, steps = 23, 300
    episodes = synthetic(n, steps, seed=interval, levels=levels)
    hps = sweep(wb, n)
    got = run_schedule(wb, n, episodes, steps, hps, interval=interval, fraction=fraction, window=window, seed=5)
    want = restate(n, episodes, steps, [hp_dict(h) for h in hps], interval, fraction, window, seed=5)
    assert len(want) > 5
    assert_same_copies(got, want)


def test_ties_go_to_the_lower_agent_index(wb):
    """Every agent scores the same: the top set is the lowest indices, the bottom set the highest."""
    n = 10
    episodes = [(t, a, 1.0) for t in range(0, 40, 2) for a in range(n)] + [(t, a, 1.0) for t in range(1, 40, 2) for a in range(n)]
    pbt = wb.PBT(interval=4, fraction=0.3, window=2)
    hps = [wb.default_hyperparams() for _ in range(n)]
    for t in range(4):
        pbt.step(t, list(range(n)), [1.0] * n, hps)
    assert pbt.top == [0, 1, 2] and set(np.flatnonzero(pbt.bottom)) == {7, 8, 9}
    copies = pbt.step(4, list(range(n)), [1.0] * n, hps)
    assert [d for d, _, _ in copies] == [7, 8, 9] and all(s in (0, 1, 2) for _, s, _ in copies)
    want = restate(n, sorted(episodes), 5, [hp_dict(h) for h in hps], 4, 0.3, 2)
    assert [(d, s) for _, d, s, _ in want] == [(d, s) for d, s, _ in copies]


def test_short_histories_are_unranked_and_fraction_zero_copies_nothing(wb):
    n = 6
    hps = [wb.default_hyperparams() for _ in range(n)]
    pbt = wb.PBT(interval=1, fraction=0.5, window=3)
    for t in range(2):  # agents 0..2 finish three episodes, 3..5 two
        pbt.step(t, list(range(n)), [float(a) for a in range(n)], hps)
    pbt.step(2, [0, 1, 2], [0.0, 1.0, 2.0], hps)
    assert pbt.top == [2] and set(np.flatnonzero(pbt.bottom)) == {0} and set(pbt.scores()) == {0, 1, 2}
    episodes = synthetic(n, 200, seed=3)
    assert run_schedule(wb, n, episodes, 200, hps, interval=5, fraction=0.0, window=1) == []


def test_a_bottom_agent_whose_episode_does_not_end_before_the_next_snapshot_is_dropped(wb):
    n = 4
    hps = [wb.default_hyperparams() for _ in range(n)]
    # window 1, interval 3: the snapshot after t = 2 ranks 3 > 2 > 1 > 0: top [3, 2], bottom {1, 0}.  Agent 0 ends at t = 4 and
    # copies.  Agent 1's episode runs on past the next snapshot (after t = 5: 3 > 1 > 2, with agent 0 unranked since its copy),
    # whose bottom set is {2}: agent 1 is dropped and does not copy when its episode ends at t = 6.
    episodes = [(0, 0, 0.0), (0, 1, 1.0), (1, 2, 2.0), (1, 3, 3.0), (4, 0, 9.0), (5, 2, -5.0), (6, 1, 0.5)]
    got = run_schedule(wb, n, episodes, 9, hps, interval=3, fraction=0.5, window=1)
    assert [(t, d) for t, d, _, _ in got] == [(4, 0)] and got[0][2] in (2, 3)
    assert_same_copies(got, restate(n, episodes, 9, [hp_dict(h) for h in hps], 3, 0.5, 1))
    got = run_schedule(wb, n, episodes + [(7, 2, 0.0)], 9, hps, interval=3, fraction=0.5, window=1)
    assert [(t, d, s) for t, d, s, _ in got][1:] == [(7, 2, 3)]


def test_perturbation_stays_in_bounds_and_touches_only_the_listed_fields(wb):
    n, steps = 16, 400
    bounds = {"alpha": (1e-4, 2e-3), "beta1": (0.85, 0.95), "beta2": (0.99, 0.9995), "adam_epsilon": (1e-9, 1e-7), "gamma": (0.8, 0.99),
              "lambda_": (0.9, 0.99), "epsilon": (0.1, 0.35), "log_std": (-2.0, -0.5)}
    episodes = synthetic(n, steps, seed=11)
    hps = sweep(wb, n)
    got = run_schedule(wb, n, episodes, steps, hps, interval=9, fraction=0.5, window=2, perturb=bounds, seed=2)
    assert len(got) > 20
    assert_same_copies(got, restate(n, episodes, steps, [hp_dict(h) for h in hps], 9, 0.5, 2, perturb=bounds, seed=2))
    clipped = 0
    for _, _, _, h in got:
        for name, (lo, hi) in bounds.items():
            assert np.float32(lo) <= np.float32(h[name]) <= np.float32(hi), name
            clipped += np.float32(h[name]) in (np.float32(lo), np.float32(hi))
    assert clipped > 0
    only_alpha = run_schedule(wb, n, episodes, steps, hps, interval=9, fraction=0.5, window=2, perturb={"alpha": (0.0, 1.0)}, seed=2)
    start = {tuple(np.float32(h[name]) for name in FLOATS[1:]) for h in (hp_dict(x) for x in hps)}
    assert only_alpha and all(tuple(np.float32(h[name]) for name in FLOATS[1:]) in start for *_, h in only_alpha)


def test_the_same_seed_gives_the_same_pairs(wb):
    n, steps = 20, 300
    episodes = synthetic(n, steps, seed=4)
    hps = sweep(wb, n)
    runs = [run_schedule(wb, n, episodes, steps, hps, interval=6, fraction=0.4, window=2, seed=s) for s in (8, 8, 9)]
    assert_same_copies(runs[0], runs[1])
    assert [(t, d, s) for t, d, s, _ in runs[0]] != [(t, d, s) for t, d, s, _ in runs[2]] or \
        [h["alpha"] for *_, h in runs[0]] != [h["alpha"] for *_, h in runs[2]]


@pytest.mark.parametrize("kw", [dict(interval=0), dict(interval=5, fraction=-0.1), dict(interval=5, fraction=0.51),
                                dict(interval=5, window=0), dict(interval=5, perturb={"batch_size": (1, 64)}),
                                dict(interval=5, perturb={"iterations": (1, 10)}), dict(interval=5, perturb={"alpha": (1e-2, 1e-5)}),
                                dict(interval=5, perturb={"lambda": (0.9, 0.99)})])
def test_bad_arguments_are_refused(wb, kw):
    with pytest.raises(ValueError):
        wb.PBT(**kw)

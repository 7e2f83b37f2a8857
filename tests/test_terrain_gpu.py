"""GPU tests of the walker on arbitrary terrain (wb_terrain_env_*, TerrainEnvBatch, VectorPPO(terrain=...)): against the specialised
walker kernel on the flat floor, and against the NumPy restatement (tests/terrain_restatement.py over oracle/np_oracle.py) on rough floors and
with a loose obstacle, bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DT = np.float32(0.0166667)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _np_oracle():
    import terrain_restatement
    return terrain_restatement.P


def restated_env(terrain, **kwargs):
    """The walker on `terrain` (restatement bodies) in the NumPy restatement."""
    import terrain_restatement
    return terrain_restatement.TerrainEnvironment(terrain, **kwargs)


def oracle_bodies(gpu, P, objs):
    """The same IObjects as restatement RigidBodies (vertices, material, flags, acceleration, inertia override)."""
    out = []
    for i, o in enumerate(objs):
        m = gpu.MATERIALS[o.material]
        b = P._body_from((m.InverseMass, m.Restitution, m.Friction), [P.Vec(x, y) for x, y in o.vertices], o.isStatic, o.isFloor, f"t{i}")
        b.acceleration = P.Vec(*o.acceleration)
        if o.inverseInertia >= 0 and not o.isStatic:
            b.inverse_inertia = np.float32(o.inverseInertia)
        out.append(b)
    return out


def rough_heights(rng, lo, n):
    return [[int(h) for h in rng.integers(lo, 100, 11)] for _ in range(n)]


@pytest.mark.parametrize("n", [256, 37])
def test_flat_floor_equals_the_walker_kernel(gpu, n):
    """CreateFloor("Metal") as terrain through terrain_step_kernel against physics_lanes_kernel (EnvBatch): two independent CUDA
    implementations of Environment.Update, bit for bit on obs / reward / done at every env-step and on the walker record, with
    NaN / +-inf actions, auto-reset on and (for a stretch) off, a masked reset and a first-episode reset."""
    hp = gpu.default_hyperparams()
    hp.max_timesteps = 60
    env = gpu.EnvBatch(n, floor_materials="Metal", hp=hp)
    ter = gpu.TerrainEnvBatch(n, gpu.CreateFloor("Metal"), hp=hp)
    f, iv = env.get_state()
    g, jv = ter.walker_state()
    assert np.array_equal(bits(f), bits(g)) and np.array_equal(iv, jv)
    assert np.array_equal(bits(env.get_obs()), bits(ter.get_obs()))
    rng = np.random.default_rng(n)
    steps = np.zeros(n, np.int64)
    ended_early = timed_out = 0
    specials = np.array([np.nan, np.inf, -np.inf], np.float32)
    for step in range(400):
        a = rng.uniform(-1.3, 1.3, (n, 4)).astype(np.float32)
        hit = rng.random((n, 4)) < 0.002
        a[hit] = rng.choice(specials, hit.sum())
        if step == 100:
            mask = (rng.random(n) < 0.5).astype(np.uint8)
            env.reset(mask)
            ter.reset(mask)
            steps[mask != 0] = 0
        if step == 300:
            env.reset(None, first_episode=True)
            ter.reset(None, first_episode=True)
            steps[:] = 0
        auto = not (150 <= step < 190)
        o1, r1, d1 = env.step(a, auto_reset=auto)
        o2, r2, d2 = ter.step(a, auto_reset=auto)
        assert np.array_equal(bits(o1), bits(o2)), f"obs differ at env-step {step}"
        assert np.array_equal(bits(r1), bits(r2)), f"reward differs at env-step {step}"
        assert np.array_equal(d1, d2), f"done differs at env-step {step}"
        steps += 1
        d = d1 != 0
        timed_out += int((d & (steps > hp.max_timesteps)).sum())
        ended_early += int((d & (steps <= hp.max_timesteps)).sum())
        if auto:
            steps[d] = 0
        if step % 25 == 24:
            f, iv = env.get_state()
            g, jv = ter.walker_state()
            assert np.array_equal(bits(f), bits(g)), f"walker record differs at env-step {step}"
            assert np.array_equal(iv, jv), f"flags / steps differ at env-step {step}"
            assert np.array_equal(iv[:, 1], steps)
    assert ended_early > 0 and timed_out > 0
    assert ter.launch_count() > 400


def _rough_run(gpu, P, heights, n_steps, seed):
    n = len(heights)
    floors = [gpu.CreateRoughFloor(h) for h in heights]
    ter = gpu.TerrainEnvBatch(n, floors)
    refs = [restated_env(oracle_bodies(gpu, P, fl)) for fl in floors]
    rng = np.random.default_rng(seed)
    dones = np.zeros(n, np.int64)
    for step in range(n_steps):
        a = rng.uniform(-1.2, 1.2, (n, 4)).astype(np.float32)
        obs, rew, done = ter.step(a)
        g, jv = ter.get_state()
        for c in range(n):
            ro, rr, rd = refs[c].step(a[c], DT, auto_reset=True)
            assert np.array_equal(bits(obs[c]), bits(ro)), f"obs differ: copy {c}, env-step {step}"
            assert bits(rew[c]) == bits(rr) and bool(done[c]) == rd, f"reward / done differ: copy {c}, env-step {step}"
            rf, ri = refs[c].terrain_state()
            assert np.array_equal(bits(g[c]), bits(rf)), f"record differs: copy {c}, env-step {step}"
            assert np.array_equal(jv[c], ri), f"collided / flags / steps differ: copy {c}, env-step {step}"
            dones[c] += int(rd)
    return dones


def test_rough_floor_matches_the_restatement(gpu):
    """Environment.CreateRoughFloor with injected heights, each of 4 copies on its own floor (set_terrain), against its own
    restatement: heights over the full range (the walker spawns into the floor and episodes end at once) and heights in
    [87, 100), where every floor top is below the feet (y = 886.25) and the episodes run on."""
    P = _np_oracle()
    rng = np.random.default_rng(31)
    full = rough_heights(rng, 0, 4)
    dones = _rough_run(gpu, P, full, 40, 1)
    assert dones.sum() > 10
    high = rough_heights(rng, 87, 4)
    # on the restatement alone: no episode ends in the first 10 env-steps on these floors
    for h in high:
        ref = restated_env(oracle_bodies(gpu, P, gpu.CreateRoughFloor(h)))
        for _ in range(10):
            assert not ref.step(np.zeros(4, np.float32), DT)[2]
    dones = _rough_run(gpu, P, high, 40, 2)
    assert dones.sum() < 4 * 10


def test_loose_obstacle_persists_across_resets(gpu):
    """A dynamic Square (gravity on) in front of the walker on the flat floor: it falls, settles, is pushed; a Reset re-creates the
    walker only, so the square stays where the last step left it -- as in the restatement."""
    P = _np_oracle()
    sq = gpu.Square.FromSize("Wood", (175, 860), 30)
    sq.acceleration = (0.0, 980.0)
    terrain = gpu.CreateFloor("Metal") + [sq]
    hp = gpu.default_hyperparams()
    hp.max_timesteps = 15
    ter = gpu.TerrainEnvBatch(2, terrain, hp=hp)
    ref = restated_env(oracle_bodies(gpu, P, terrain), max_timesteps=15)
    rng = np.random.default_rng(8)
    tv = ter.total_verts
    sq_rows = slice(2 * (tv - 4), 2 * tv)
    for step in range(36):
        a = np.tile(rng.uniform(-1.2, 1.2, 4).astype(np.float32), (2, 1))
        if step == 25:
            before, _ = ter.get_state()
            ter.reset()
            ref.reset()
            after, _ = ter.get_state()
            assert np.array_equal(bits(before[:, sq_rows]), bits(after[:, sq_rows]))
        obs, rew, done = ter.step(a)
        ro, rr, rd = ref.step(a[0], DT, auto_reset=True)
        g, jv = ter.get_state()
        rf, ri = ref.terrain_state()
        for c in range(2):
            assert np.array_equal(bits(obs[c]), bits(ro)) and bits(rew[c]) == bits(rr) and bool(done[c]) == rd, f"env-step {step}"
            assert np.array_equal(bits(g[c]), bits(rf)) and np.array_equal(jv[c], ri), f"record differs at env-step {step}"
    moved = g[0, sq_rows].reshape(4, 2) - sq.vertices
    assert np.abs(moved).max() > 1.0  # the square really moved (it fell onto the floor)


def test_bad_descriptions_are_rejected(gpu):
    tri = gpu.Triangle.FromSize("Wood", (0, 0), 10, isStatic=True)
    with pytest.raises(gpu.WalkerB200Error) as ei:
        gpu.TerrainEnvBatch(4, [gpu.Triangle.FromSize("Wood", (10 * i, 0), 10, isStatic=True) for i in range(12)])
    assert ei.value.code == 4  # WB_ERR_UNSUPPORTED: 5 + 12 bodies exceed a scene
    gpu.TerrainEnvBatch(4, [gpu.Triangle.FromSize("Wood", (10 * i, 0), 10, isStatic=True) for i in range(11)]).close()
    with pytest.raises(gpu.WalkerB200Error) as ei:
        gpu.TerrainEnvBatch(4, [tri, gpu.IObject(np.zeros((2, 2), np.float32), isStatic=True)])
    assert ei.value.code == 1
    ter = gpu.TerrainEnvBatch(4, gpu.CreateRoughFloor([50] * 11))
    with pytest.raises(ValueError):
        ter.set_terrain(np.zeros((4, 2 * 40 - 2), np.float32))
    with pytest.raises(ValueError):
        ter.set_terrain(np.zeros((3, 2 * 40), np.float32))
    with pytest.raises(ValueError):  # per-copy lists of different topology
        gpu.TerrainEnvBatch(2, [gpu.CreateRoughFloor([50] * 11), gpu.CreateFloor()])
    for n in (0, -3):
        with pytest.raises(gpu.WalkerB200Error) as ei:
            gpu.TerrainEnvBatch(n, gpu.CreateFloor())
        assert ei.value.code == 1


def _dev_buffers(torch, n):
    return (torch.empty(n, 12, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, device="cuda", dtype=torch.uint8))


def test_one_launch_per_step_dev(gpu):
    import torch
    n = 300
    ter = gpu.TerrainEnvBatch(n, gpu.CreateRoughFloor([90] * 11), stream=torch.cuda.current_stream().cuda_stream)
    a = torch.zeros(n, 4, device="cuda")
    obs, rew, done = _dev_buffers(torch, n)
    before = ter.launch_count()
    for k in range(5):
        ter.step_dev(a, obs, rew, done)
        assert ter.launch_count() == before + k + 1
    torch.cuda.synchronize()


def test_two_environments_on_two_streams(gpu):
    """Different terrains stepped concurrently on two streams give what stepping them one after the other gives: the topology is a
    kernel parameter, never a shared __constant__ symbol."""
    import torch
    n, T = 512, 12
    terrains = [gpu.CreateFloor("Metal"), gpu.CreateRoughFloor([88, 95, 91, 99, 87, 93, 90, 96, 89, 94, 92])]
    acts = torch.from_numpy(np.random.default_rng(3).uniform(-1.2, 1.2, (T, n, 4)).astype(np.float32)).cuda()

    def run(concurrent):
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        envs = [gpu.TerrainEnvBatch(n, t, stream=s.cuda_stream) for t, s in zip(terrains, streams)]
        outs = [[_dev_buffers(torch, n) for _ in range(T)] for _ in envs]
        torch.cuda.synchronize()
        order = [(t, e) for t in range(T) for e in range(2)] if concurrent else [(t, e) for e in range(2) for t in range(T)]
        for t, e in order:
            with torch.cuda.stream(streams[e]):
                envs[e].step_dev(acts[t], *outs[e][t])
            if not concurrent and t == T - 1:
                streams[e].synchronize()
        torch.cuda.synchronize()
        res = [[torch.cat([o.view(n, -1).float() for o in outs[e][t]], 1).cpu().numpy() for t in range(T)] for e in range(2)]
        states = [env.get_state() for env in envs]
        return res, states

    r1, s1 = run(True)
    r2, s2 = run(False)
    for e in range(2):
        for t in range(T):
            assert np.array_equal(bits(r1[e][t]), bits(r2[e][t])), (e, t)
        assert np.array_equal(bits(s1[e][0]), bits(s2[e][0])) and np.array_equal(s1[e][1], s2[e][1])
    assert not np.array_equal(bits(r1[0][T - 1]), bits(r1[1][T - 1]))  # the two terrains really differ


def _ppo_snapshot(vp):
    return (vp.rewards.cpu().numpy().copy(), vp.dones.cpu().numpy().copy(), vp.states.cpu().numpy().copy(),
            vp.agent.actor.get_flat().copy(), vp.agent.critic.get_flat().copy())


def test_vector_ppo_on_the_flat_floor_terrain_equals_the_default(gpu):
    import torch
    snaps = []
    for terrain in (None, gpu.CreateFloor()):
        vp = gpu.VectorPPO(1024, horizon=16, minibatch_global=4096, seed=5, terrain=terrain)
        out = []
        for _ in range(2):
            vp.iterate()
            out.append(_ppo_snapshot(vp))
        torch.cuda.synchronize()
        snaps.append(out)
        del vp
    for it in range(2):
        for k, (x, y) in enumerate(zip(snaps[0][it], snaps[1][it])):
            assert np.array_equal(np.ascontiguousarray(x).view(np.uint8), np.ascontiguousarray(y).view(np.uint8)), (it, k)


def test_vector_ppo_trains_on_a_per_walker_rough_floor(gpu):
    """One iteration on a rough floor of its own per walker: the weights change and stay finite, and the rewards / dones of 8
    walkers replay bit for bit through the restatement from the recorded (unclipped) actions."""
    P = _np_oracle()
    n, T = 1024, 16
    rng = np.random.default_rng(12)
    heights = rough_heights(rng, 80, n)
    floors = [gpu.CreateRoughFloor(h) for h in heights]
    vp = gpu.VectorPPO(n, horizon=T, minibatch_global=4096, seed=9, terrain=floors)
    w0 = (vp.agent.actor.get_flat().copy(), vp.agent.critic.get_flat().copy())
    vp.iterate()
    w1 = (vp.agent.actor.get_flat(), vp.agent.critic.get_flat())
    for a, b in zip(w0, w1):
        assert np.isfinite(b).all() and not np.array_equal(a, b)
    acts = vp.actions.cpu().numpy()
    rews = vp.rewards.cpu().numpy()
    dones = vp.dones.cpu().numpy()
    for w in np.linspace(0, n - 1, 8).astype(int):
        ref = restated_env(oracle_bodies(gpu, P, floors[w]))
        for t in range(T):
            _, rr, rd = ref.step(acts[t, w], DT, auto_reset=True)
            assert bits(rews[t, w]) == bits(rr) and bool(dones[t, w]) == rd, f"walker {w}, env-step {t}"

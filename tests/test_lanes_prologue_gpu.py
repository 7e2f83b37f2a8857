"""The lanes physics kernel's prologue and write-back for every lanes layout, bit for bit against the CPU oracle.

The kernel stages each CTA's walker records as whole aligned pieces of the padded SoA rows, with the walkers' flags, step
counters, positions, material ids, joint torques and actions in the same batch, and writes the records back as whole
pieces where every walker of the CTA is live.  These tests cover what that can get wrong: batch sizes that end inside a
CTA for each layout (columns past n must never be stored and must not change the live walkers' results), mixed walker
and floor materials (the material bytes are fetched as the aligned word that holds them), Walker.TakeActions with NaN,
+-inf and out-of-range actions (the torques are read before any is written), masked resets, and a contact-heavy start
with per-substep pair and joint traces."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MATS = ["Ice", "Wood", "Paper", "Titanium", "Carpet", "Rubber", "Metal", "SuperRubber"]
LAYOUTS = [2, 4, 8, 16, 32]


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_state_equal(env, ref, what):
    f, iv = env.get_state()
    rf, riv = ref.get_state()
    bad = np.argwhere(bits(f) != bits(rf))
    assert bad.size == 0, f"{what}: {len(bad)} state words differ, first (env,field)={bad[0]} gpu={f[tuple(bad[0])]!r} ref={rf[tuple(bad[0])]!r}"
    assert np.array_equal(iv, riv), f"{what}: flags/steps differ"


def mixed(n):
    return [MATS[i % 8] for i in range(n)], [MATS[(3 * i + 1) % 8] for i in range(n)]


@pytest.mark.parametrize("variant", LAYOUTS)
def test_ragged_batches_mixed_materials(gpu, O, variant):
    """Sizes that end at every offset inside a CTA of 32 / L walkers, and inside a 256-walker row padding block."""
    for n in (2, 3, 5, 6, 11, 15, 17, 31, 63, 255, 257, 1003):
        floors, walkers = mixed(n)
        env = gpu.EnvBatch(n, floor_materials=floors, walker_materials=walkers)
        env.set_variant(variant)
        ref = O.EnvBatch(n, floor=floors, walker=walkers)
        rng = np.random.default_rng(n)
        for t in range(4):
            a = rng.uniform(-1.3, 1.3, (n, 4)).astype(np.float32)
            if t == 2:
                mask = (rng.random(n) < 0.5).astype(np.uint8)
                env.reset(mask)
                for i in np.flatnonzero(mask):
                    ref.reset(int(i))
            obs, rew, done = env.step(a)
            robs, rrew, rdone = ref.step(a)
            assert np.array_equal(bits(obs), bits(robs)) and np.array_equal(bits(rew), bits(rrew)) and np.array_equal(done, rdone), \
                f"n={n} variant={variant} env-step {t}: obs / reward / done differ"
        assert_state_equal(env, ref, f"n={n} variant={variant}")


def _special_actions(rng, n):
    a = rng.uniform(-3, 3, (n, 4)).astype(np.float32)
    special = np.array([np.nan, np.inf, -np.inf, 1.0, -1.0, 2.5, -7.0, 0.999], np.float32)
    hit = rng.random((n, 4)) < 0.3
    a[hit] = rng.choice(special, int(hit.sum()))
    return a


@pytest.mark.parametrize("variant", LAYOUTS)
def test_take_actions_nonfinite_and_out_of_range(gpu, O, variant):
    """Matrix.Clip + Walker.TakeActions with NaN / +-inf / out-of-range actions over several env-steps (each step's torque
    change is taken against the torque the previous step stored).  Bit for bit against the compacting kernel, which stages
    the torques its own way, and against the oracle with NaN equal to NaN (the CPU and the GPU produce different NaN bits)."""
    n = 45
    floors, walkers = mixed(n)
    env = gpu.EnvBatch(n, floor_materials=floors, walker_materials=walkers)
    env.set_variant(variant)
    other = gpu.EnvBatch(n, floor_materials=floors, walker_materials=walkers)
    other.set_variant(1001)
    ref = O.EnvBatch(n, floor=floors, walker=walkers)
    rng = np.random.default_rng(variant)
    for t in range(6):
        a = _special_actions(rng, n)
        obs, rew, done = env.step(a)
        oobs, orew, odone = other.step(a)
        ref.step(a)
        assert np.array_equal(bits(obs), bits(oobs)) and np.array_equal(bits(rew), bits(orew)) and np.array_equal(done, odone), \
            f"variant {variant} against 1001 at env-step {t}"
        f, iv = env.get_state()
        of, oiv = other.get_state()
        rf, riv = ref.get_state()
        assert np.array_equal(bits(f), bits(of)) and np.array_equal(iv, oiv), f"state against 1001 at env-step {t}"
        assert np.array_equal(f, rf, equal_nan=True) and np.array_equal(iv, riv), f"state against the oracle at env-step {t}"
        finite = np.isfinite(rf).all(axis=1)
        assert np.array_equal(bits(f[finite]), bits(rf[finite])), f"finite walkers against the oracle at env-step {t}"
    assert not np.isfinite(f).all(), "no walker took a non-finite action"


@pytest.mark.parametrize("variant", [8, 16, 32])
def test_contact_stress_start_traces(gpu, O, variant):
    """workloads.contact_stress_start (every body spinning at up to 5 rad/s): leg pole pairs collide in the first substeps,
    so the joints' and pairs' impulses change angular velocities mid-sweep.  Pair traces, joint traces, observations and
    state bit for bit, with the traced and the fused (untraced) kernel of the layout."""
    import workloads
    n, per, steps = 72, 9, 8
    rng = np.random.default_rng(variant)
    f0, iv0 = O.EnvBatch(n).get_state()
    floors = workloads.contact_stress_start(n, per, f0, rng)
    traced, fused = gpu.EnvBatch(n, floor_materials=floors), gpu.EnvBatch(n, floor_materials=floors)
    traced.set_variant(variant)
    fused.set_variant(variant)
    tref, fref = O.EnvBatch(n, floor=floors), O.EnvBatch(n, floor=floors)
    for e in (traced, fused, tref, fref):
        e.set_state(f0.copy(), iv0.copy())
    sat = 0
    for t in range(steps):
        a = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
        traced.take_actions(a)
        tref.take_actions(a)
        pt, jt = traced.debug_contacts(gpu.DT_FRAME)
        rpt, rjt = tref.step_objects(O.DT_FRAME, 50, trace=True)
        for name in pt.dtype.names:
            assert np.array_equal(pt[name].view(np.uint32), rpt[name].view(np.uint32)), f"pair trace field {name} differs at env-step {t}"
        for name in jt.dtype.names:
            assert np.array_equal(jt[name].view(np.uint32), rjt[name].view(np.uint32)), f"joint trace field {name} differs at env-step {t}"
        sat += int(rpt["sat"].sum())
        traced.observe()
        tref.observe()
        obs, rew, done = fused.step(a, auto_reset=False)
        robs, rrew, rdone = fref.step(a, auto_reset=False)
        assert np.array_equal(bits(obs), bits(robs)) and np.array_equal(bits(rew), bits(rrew)) and np.array_equal(done, rdone), \
            f"fused step differs at env-step {t}"
    assert_state_equal(traced, tref, f"traced, variant {variant}")
    assert_state_equal(fused, fref, f"fused, variant {variant}")
    assert sat > 10 * n * steps, "the start is not contact-heavy"

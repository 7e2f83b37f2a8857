"""The leg-split lanes kernels with 8, 16 and 32 lanes per walker step the Body beside the first leg segments and test its
floor bounding box in the same pass; the Body-floor pair is resolved only in a warp where that test hits (4 lanes per walker
keep the Body's own slot and are checked the same way).  These tests put Bodies onto the floor in chosen columns of a warp
-- the first, the last, a middle one, all of them, and one walker beside empty columns -- and compare pair traces, joint
traces, state and observations with the oracle bit for bit, over the substeps in which the Body comes down and the ones
after."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MATS = ["Ice", "Wood", "Paper", "Titanium", "Carpet", "Rubber", "Metal", "SuperRubber"]
FLOOR_FIRST = 1 << 6
BODY_TRACE_SLOT = 4  # the Body's one candidate, the floor


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def tipped(f, gap, vy, turn):
    """The record `f` turned by `turn` rad about the Body's centroid and lowered until the Body's lowest vertex is `gap` above
    the floor (y = 900), every body moving down at `vy`."""
    f = f.copy()
    pts = np.concatenate([f[:58].reshape(29, 2), f[58:68].reshape(5, 2)]).astype(np.float64)
    c = pts[29 + 2]
    rot = np.array([[np.cos(turn), -np.sin(turn)], [np.sin(turn), np.cos(turn)]])
    pts = (pts - c) @ rot.T + c
    pts[:, 1] += 900.0 - gap - pts[12:17, 1].max()
    f[:58] = pts[:29].reshape(-1).astype(np.float32)
    f[58:68] = pts[29:].reshape(-1).astype(np.float32)
    f[68:78] = np.tile(np.float32([0.0, vy]), 5)
    f[83:88] = np.float32(turn)
    return f


# the Body comes down onto the floor after 13-37 substeps / is on it from the first substep; the legs land first and hold the
# Body up (for an env-step or two: random actions tip most of these walkers over later)
FALLING = [(1.0, 150.0, np.pi / 2), (0.5, 50.0, 2.0)]
STANDING = [(3.0, 150.0, 1.2), (2.0, 120.0, -1.4)]


@pytest.mark.parametrize("lanes", [4, 8, 16, 32])
def test_body_on_the_floor_in_chosen_columns(gpu, O, lanes):
    E = 32 // lanes  # walkers per warp
    # warp 0: first column falls, warp 1: last column, warp 2: a middle column, warp 3: every column, warp 4: one walker alone
    falls = [[0], [E - 1], [E // 2], list(range(E))]
    n = 4 * E + 1
    falling = np.zeros(n, bool)
    for w, cols in enumerate(falls):
        falling[[w * E + c for c in cols]] = True
    falling[4 * E] = True
    floors = [MATS[i % 8] for i in range(n)]
    ref = O.EnvBatch(n, floor=floors)
    f, iv = ref.get_state()
    for i in range(n):
        kind = FALLING if falling[i] else STANDING
        f[i] = tipped(f[i], *kind[i % 2])
    iv[1::2, 0] |= FLOOR_FIRST
    ref.set_state(f, iv)
    env = gpu.EnvBatch(n, floor_materials=floors)
    env.set_variant(lanes)
    env.set_state(f, iv)
    rng = np.random.default_rng(lanes)
    for t in range(3):
        a = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
        env.take_actions(a)
        ref.take_actions(a)
        pt, jt = env.debug_contacts(gpu.DT_FRAME)
        rpt, rjt = ref.step_objects(O.DT_FRAME, 50, trace=True)
        assert np.array_equal(jt.view(np.uint8), rjt.view(np.uint8)), f"joint trace differs at step {t}"
        for name in pt.dtype.names:
            bad = np.argwhere(pt[name].view(np.uint32) != rpt[name].view(np.uint32))
            assert bad.size == 0, f"pair trace field {name} differs at step {t}, first (walker, substep, slot) {bad[0]}"
        gf, giv = env.get_state()
        rf, riv = ref.get_state()
        assert np.array_equal(bits(gf), bits(rf)), f"state differs after step {t}"
        assert np.array_equal(giv, riv), f"flags / steps differ after step {t}"
        obs, rew, done = env.observe()
        robs, rrew, rdone = ref.observe()
        assert np.array_equal(bits(obs), bits(robs)) and np.array_equal(bits(rew), bits(rrew)) and np.array_equal(done, rdone)
        assert (rpt["other"][:, :, BODY_TRACE_SLOT] == 5).all()
        if t == 0:
            # the workload does what it is meant to: in the first env-step Bodies meet the floor only in the chosen columns,
            # some of them after coming down (later env-steps go on from there, with more walkers tipping over)
            hit = rpt["aabb"][:, :, BODY_TRACE_SLOT] != 0
            assert np.array_equal(hit.any(axis=1), falling) and np.array_equal(done.astype(bool), falling)
            first_hit = hit.argmax(axis=1)[falling]
            assert (first_hit > 0).any() and (first_hit == 0).any()

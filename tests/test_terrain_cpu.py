"""The walker-on-terrain restatement (tests/terrain_restatement.py over oracle/np_oracle.py) and the wb_terrain_env_* entry points
without a GPU."""
import ctypes as C

import numpy as np
import pytest


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _restatement():
    import terrain_restatement
    return terrain_restatement


def test_restatement_with_the_default_floor_as_terrain_equals_the_default():
    """TerrainEnvironment([the CreateFloor body]) and np_oracle.Environment() step bit for bit alike, through terminals, resets and
    the list-order switch a Reset makes (the floor-first flag read from where the walker sits in the list)."""
    T = _restatement()
    a = T.P.Environment(max_timesteps=8)
    b = T.TerrainEnvironment([T.default_floor()], max_timesteps=8)
    rng = np.random.default_rng(4)
    dones = 0
    for step in range(30):
        act = rng.uniform(-1.3, 1.3, 4).astype(np.float32)
        if step == 20:
            a.reset()
            b.reset()
        oa, ra, da = a.step(act, np.float32(0.0166667), auto_reset=True)
        ob, rb, db = b.step(act, np.float32(0.0166667), auto_reset=True)
        assert np.array_equal(bits(oa), bits(ob)) and bits(ra) == bits(rb) and da == db, f"step {step}"
        fa, ia = a.flat_state()
        fb, ib = b.flat_state()
        assert np.array_equal(bits(fa), bits(fb)) and np.array_equal(ia, ib), f"record differs at step {step}"
        dones += int(da)
    assert dones >= 2 and (ia[0] & (1 << 6))  # episodes ended; the floor is first after the resets


def test_restatement_terrain_record_lists_bodies_in_index_order():
    """terrain_state() keeps the walker's five bodies first whatever the list order, so it lines up with wb_terrain_env_get_state."""
    T = _restatement()
    env = T.TerrainEnvironment([T.default_floor()], max_timesteps=3)
    f0, i0 = env.terrain_state()
    for _ in range(4):  # the 4th step times out and auto-resets
        env.step(np.zeros(4, np.float32), np.float32(0.0166667), auto_reset=True)
    f1, i1 = env.terrain_state()
    assert f0.shape == f1.shape == (2 * 33 + 6 * 6 + 4,)
    assert np.array_equal(bits(f1[:58]), bits(f0[:58]))  # a fresh walker again, in the same slots
    assert i0[1] == 0 and i1[1] == (1 << 6) and i1[2] == 0


def test_terrain_env_create_fails_without_a_device(wb):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    floor = wb.CreateFloor("Metal")
    desc = (wb._lib.BodyDesc * 1)(wb._lib.BodyDesc(4, 1, 1, 6, 0, 0.0, 0.0, -1.0))
    verts = np.ascontiguousarray(floor[0].vertices.reshape(-1), np.float32)
    h = C.c_void_p()
    rc = wb.lib().wb_terrain_env_create(8, desc, 1, verts.ctypes.data_as(C.c_void_p), 4, None, C.byref(h))
    assert rc == 2 and not h.value
    with pytest.raises(wb.WalkerB200Error) as ei:
        wb.TerrainEnvBatch(8, floor)
    assert ei.value.code == 2

"""The walker on arbitrary terrain in the NumPy restatement (oracle/np_oracle.py), the checker of the wb_terrain_env_* path.

np_oracle.Environment builds the walker and Environment.CreateFloor; TerrainEnvironment replaces that one floor body with any list
of restatement RigidBodies (Environment.CreateRoughFloor, Environment.cs:230-261, or anything else).  Nothing else needs to
change: the Collided / terminal logic reads the walker's own bodies, and Reset removes the walker and appends a new one after the
terrain (Environment.cs:167-173), exactly as it does after the flat floor.  Only the floor-first flag of the record is re-read:
it is set whenever the walker is no longer first in Environment._rigidBodies.
"""
from __future__ import annotations

import numpy as np

import __graft_entry__ as ge

ge.load_oracle()
import np_oracle as P  # noqa: E402

FLOOR_FIRST = 1 << 6
TERMINAL = 1 << 5


class TerrainEnvironment(P.Environment):
    def __init__(self, terrain, **kwargs):
        super().__init__(**kwargs)
        self.rigid_bodies.remove(self.floor)
        self.terrain = list(terrain)
        self.rigid_bodies.extend(self.terrain)

    def flat_state(self):
        """The canonical 92-float + 2-int walker record (as wb_env_get_state / TerrainEnvBatch.walker_state)."""
        f, iv = super().flat_state()
        iv[0] = (iv[0] & ~FLOOR_FIRST) | (FLOOR_FIRST if self.rigid_bodies[0] is not self.lll else 0)
        return f, iv

    def terrain_state(self):
        """Record of wb_terrain_env_get_state: the wb_scene_* record over [LLL, LLU, Body, RLL, RLU, terrain...] in index order
        (whatever the list order) + the 4 joint torques; ints [Collided bit per body index, Terminal | floor-first, steps]."""
        f, collided = P.Scene(self.dyn() + self.terrain, self.joints).flat_state()
        _, iv = self.flat_state()
        return f, np.array([collided, int(iv[0]) & (TERMINAL | FLOOR_FIRST), self.steps], np.int32)


def default_floor():
    """Environment.CreateFloor (Environment.cs:211-226) as a restatement body."""
    return P.hull_from_positions((15, 0.3, 1.0), [(-50, 1050), (-50, 900), (1050, 900), (1050, 1050)], is_static=True, is_floor=True,
                                 name="floor")

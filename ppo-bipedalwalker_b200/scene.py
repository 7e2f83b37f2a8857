"""General scenes: the reference's IObject plugin surface (Objects/IObject.cs:7-10) for N lockstep copies.

Host-side mirror of the shape factories -- `Square.FromSize` (Square.cs:18-32), `Triangle.FromSize` (Triangle.cs:18-31),
`Hexagon.FromSize` (Hexagon.cs:18-34), `Pole.FromSize` (Pole.cs:18-34), `Hull.FromPositions` (Hull.cs:18-29),
`Skeleton.SmoothCorners` (Skeleton.cs:33-53) -- and of `Joint` (Joint.cs), plus `Scene`, which hands the lists to
libwalker_b200 (`wb_scene_*`) and runs `Environment.StepObjects` (Environment.cs:126-143) on the GPU, and `TerrainEnvBatch`, the
walker environment on any such list in place of the flat floor (`wb_terrain_env_*`).  Vertex templates are
computed here in float32 with the reference's formulas; all stepping happens in csrc/physics_scene.cu (no CPU path).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from ._lib import ACT, OBS, BodyDesc, Hyperparams, JointDesc, check, lib, ptr
from .env import DT_FRAME, IMaterial, MATERIALS, default_hyperparams

f32 = np.float32


def _material_id(m) -> int:
    if isinstance(m, IMaterial):
        return m.register().id
    if isinstance(m, str):
        return MATERIALS[m].id
    return int(m)


@dataclass(eq=False)  # bodies are compared by identity (like the reference's object references), never by vertex values
class IObject:
    """One rigid body of a scene: RigidBody ctor arguments (RigidBody.cs:36-50) + its vertex list (Skeleton.AddVectors)."""
    vertices: np.ndarray  # [n, 2] float32
    material: object = "Metal"
    isStatic: bool = False
    isFloor: bool = False
    acceleration: tuple = (0.0, 0.0)      # RigidBody.AddAcceleration
    inverseInertia: float = -1.0          # < 0: 0.001f * inverse mass; >= 0: RigidBody.SetInverseInertia-style override
    associated: list = field(default_factory=list)  # RigidBody.AddAssociatedBodies: IObjects this body never collides with

    def SmoothCorners(self, count: int = 1) -> "IObject":  # Skeleton.cs:33-53 (the cached centroid is NOT refreshed there either:
        v = self.vertices                                  # smooth before the body enters a scene)
        for _ in range(count):
            n = len(v)
            new = []
            for j in range(n):
                ab = ((v[(j + 1) % n] - v[j]).astype(f32) * f32(0.2)).astype(f32)
                ac = ((v[(j - 1) % n] - v[j]).astype(f32) * f32(0.2)).astype(f32)
                new.append((v[j] + ac).astype(f32))
                new.append((v[j] + ab).astype(f32))
            v = np.array(new, f32)
        self.vertices = v
        return self


def _obj(verts, material, isStatic=False, isFloor=False) -> IObject:
    return IObject(np.array(verts, f32), material, isStatic, isFloor)


class Square:
    @staticmethod
    def FromSize(material, centroid, size, isStatic=False) -> IObject:  # Square.cs:18-32
        cx, cy = f32(centroid[0]), f32(centroid[1])
        a = f32(f32(0.5) * f32(size))
        return _obj([(cx + a, cy + a), (cx - a, cy + a), (cx - a, cy - a), (cx + a, cy - a)], material, isStatic)


class Triangle:
    @staticmethod
    def FromSize(material, centroid, size, isStatic=False) -> IObject:  # Triangle.cs:18-31
        cx, cy = f32(centroid[0]), f32(centroid[1])
        a = f32(f32(0.5) * f32(size))
        return _obj([(cx, cy + a), (cx - a, cy - a), (cx + a, cy - a)], material, isStatic)


class Hexagon:
    @staticmethod
    def FromSize(material, centroid, size, isStatic=False) -> IObject:  # Hexagon.cs:18-34
        cx, cy = f32(centroid[0]), f32(centroid[1])
        a = f32(f32(0.5) * f32(size))
        h = f32(a * f32(0.5))
        return _obj([(cx + h, cy + a), (cx - h, cy + a), (cx - a, cy), (cx - h, cy - a), (cx + h, cy - a), (cx + a, cy)], material, isStatic)


class Pole:
    @staticmethod
    def FromSize(material, centroid, size, isStatic=False) -> IObject:  # Pole.cs:18-34
        cx, cy = f32(centroid[0]), f32(centroid[1])
        a = f32(f32(0.1) * f32(size))
        h = f32(a * f32(3.5))
        return _obj([(cx + a, cy + h), (cx, cy + h), (cx - a, cy + h), (cx - a, cy - h), (cx, cy - h), (cx + a, cy - h)], material, isStatic)


class Hull:
    @staticmethod
    def FromPositions(material, positions, isStatic=False, isFloor=False) -> IObject:  # Hull.cs:18-29
        return _obj(positions, material, isStatic, isFloor)


@dataclass(eq=False)
class Joint:
    """new Joint(bodyA, bodyB, indexA, indexB), Joint.cs:20-28 (bodies given as IObjects of the scene)."""
    bodyA: IObject
    bodyB: IObject
    indexA: int
    indexB: int


def _body_desc(o: IObject, index: dict) -> BodyDesc:
    mask = 0
    for a in o.associated:
        mask |= 1 << index[id(a)]
    return BodyDesc(len(o.vertices), int(o.isStatic), int(o.isFloor), _material_id(o.material), mask, float(o.acceleration[0]),
                    float(o.acceleration[1]), float(o.inverseInertia))


def _describe(objects):
    """IObject list -> (wb_body_desc array, all vertices concatenated (x, y) float32); associations index the list."""
    index = {id(o): i for i, o in enumerate(objects)}
    descs = (BodyDesc * len(objects))()
    for i, o in enumerate(objects):
        descs[i] = _body_desc(o, index)
    vflat = np.ascontiguousarray(np.concatenate([np.asarray(o.vertices, f32).reshape(-1) for o in objects]), f32)
    return descs, vflat


class Scene:
    """N lockstep copies of `objects` (+ `joints`): Environment._rigidBodies in list order."""

    def __init__(self, n: int, objects, joints=(), iterations: int = 50, stream: int | None = None):
        self.n = n
        self.objects = list(objects)
        self.joints = list(joints)
        B, J = len(self.objects), len(self.joints)
        index = {id(o): i for i, o in enumerate(self.objects)}
        descs, vflat = _describe(self.objects)
        self.vertex_counts = [len(o.vertices) for o in self.objects]
        jd = (JointDesc * max(J, 1))()
        for k, j in enumerate(self.joints):
            jd[k] = JointDesc(index[id(j.bodyA)], j.indexA, index[id(j.bodyB)], j.indexB)
        h = C.c_void_p()
        check(lib().wb_scene_create(n, descs, B, ptr(vflat), jd if J else None, J, iterations, C.byref(h)))
        self._h = h
        if stream is not None:
            check(lib().wb_scene_set_stream(self._h, C.c_void_p(stream)))
        k = C.c_int32(0)
        check(lib().wb_scene_state_floats(self._h, C.byref(k)))
        self.state_floats = k.value

    def close(self):
        if getattr(self, "_h", None) and lib is not None:
            lib().wb_scene_destroy(self._h)
            self._h = None

    __del__ = close

    def get_state(self):
        """-> (state [n, floats], collided [n]); per copy: vertices body by body, centroids, velocities, omega, angle, torques."""
        f = np.empty((self.state_floats, self.n), np.float32)
        c = np.empty(self.n, np.int32)
        check(lib().wb_scene_get_state(self._h, ptr(f), ptr(c)))
        return np.ascontiguousarray(f.T), c

    def set_state(self, f, collided=None):
        ft = np.ascontiguousarray(np.asarray(f, np.float32).reshape(self.n, self.state_floats).T)
        check(lib().wb_scene_set_state(self._h, ptr(ft), None if collided is None else ptr(np.ascontiguousarray(collided, np.int32))))

    def SetTorques(self, torques):  # Joint.SetTorque on every joint, Joint.cs:56-61
        t = np.ascontiguousarray(torques, np.float32).reshape(self.n, len(self.joints))
        check(lib().wb_scene_set_torques(self._h, ptr(t)))

    def StepObjects(self, deltaTime: float = DT_FRAME):  # Environment.cs:126-143
        check(lib().wb_scene_step_objects(self._h, C.c_float(deltaTime)))


def _signature(objects) -> list:
    index = {id(o): i for i, o in enumerate(objects)}
    return [tuple(getattr(_body_desc(o, index), k) for k, _ in BodyDesc._fields_) for o in objects]


class TerrainEnvBatch:
    """N walkers, each on its own copy of a terrain (wb_terrain_env handle): Environment.Update (Environment.cs:64-92) with the
    IObject list `terrain` in place of Environment.CreateFloor -- e.g. CreateRoughFloor(heights) for Hyperparameters.RoughFloor.

    `terrain` is one IObject list shared by every walker, or a list of n such lists with the same topology (vertex counts, flags,
    materials, associations); their vertices are loaded per copy with set_terrain.  The methods follow EnvBatch; get_state
    returns the full record ([n, state_floats] floats over [LLL, LLU, Body, RLL, RLU, terrain...] in index order + 4 joint
    torques, [n, 3] ints: Collided bits per body index, flags, steps) and walker_state() the walker's part as EnvBatch.get_state
    has it."""

    def __init__(self, n: int, terrain, walker_material="Carpet", hp: Hyperparams | None = None, stream: int | None = None):
        self.n = int(n)
        self.hp = hp if hp is not None else default_hyperparams()
        terrain = list(terrain)
        per_copy = len(terrain) > 0 and not isinstance(terrain[0], IObject)
        if per_copy:
            if len(terrain) != self.n:
                raise ValueError(f"a per-copy terrain needs {self.n} IObject lists, got {len(terrain)}")
            first = list(terrain[0])
            sig = _signature(first)
            for t in terrain[1:]:
                if _signature(list(t)) != sig:
                    raise ValueError("every copy's terrain must have the same topology as the first")
        else:
            first = terrain
        self.objects = first
        descs, vflat = _describe(first) if first else ((BodyDesc * 0)(), np.zeros(0, f32))
        self.vertex_counts = [len(o.vertices) for o in first]
        h = C.c_void_p()
        check(lib().wb_terrain_env_create(self.n, descs, len(first), ptr(vflat), _material_id(walker_material), C.byref(self.hp),
                                          C.byref(h)))
        self._h = h
        if stream is not None:
            self.set_stream(stream)
        k = C.c_int32(0)
        check(lib().wb_terrain_env_state_floats(self._h, C.byref(k)))
        self.state_floats = k.value
        self.n_bodies = 5 + len(first)
        self.total_verts = 29 + sum(self.vertex_counts)
        if per_copy:
            self.set_terrain(np.stack([np.concatenate([np.asarray(o.vertices, f32).reshape(-1) for o in t]) for t in terrain]))

    def close(self):
        if getattr(self, "_h", None) and lib is not None:
            lib().wb_terrain_env_destroy(self._h)
            self._h = None

    __del__ = close

    def set_stream(self, cuda_stream: int):
        check(lib().wb_terrain_env_set_stream(self._h, C.c_void_p(cuda_stream)))

    def launch_count(self) -> int:
        out = C.c_int64(0)
        check(lib().wb_terrain_env_launch_count(self._h, C.byref(out)))
        return out.value

    def set_terrain(self, vertices):
        """Per-copy terrain vertices [n, 2 * terrain vertices] (x, y interleaved, body by body); the walkers are not touched."""
        v = np.asarray(vertices, f32)
        want = 2 * sum(self.vertex_counts)
        if v.ndim != 2 or v.shape != (self.n, want):
            raise ValueError(f"terrain vertices must have shape ({self.n}, {want}), got {v.shape}")
        check(lib().wb_terrain_env_set_terrain(self._h, ptr(np.ascontiguousarray(v))))

    def get_state(self):
        f = np.empty((self.state_floats, self.n), np.float32)
        iv = np.empty((3, self.n), np.int32)
        check(lib().wb_terrain_env_get_state(self._h, ptr(f), ptr(iv)))
        return np.ascontiguousarray(f.T), np.ascontiguousarray(iv.T)

    def set_state(self, f, iv):
        f = np.ascontiguousarray(np.asarray(f, np.float32).reshape(self.n, self.state_floats).T)
        iv = np.ascontiguousarray(np.asarray(iv, np.int32).reshape(self.n, 3).T)
        check(lib().wb_terrain_env_set_state(self._h, ptr(f), ptr(iv)))

    def walker_state(self):
        """The walker's part of the record as EnvBatch.get_state returns it: ([n, 92] floats, [n, 2] ints: flags, steps)."""
        g, iv = self.get_state()
        tv, B = self.total_verts, self.n_bodies
        f = np.concatenate([g[:, 0:58], g[:, 2 * tv:2 * tv + 10], g[:, 2 * tv + 2 * B:2 * tv + 2 * B + 10],
                            g[:, 2 * tv + 4 * B:2 * tv + 4 * B + 5], g[:, 2 * tv + 5 * B:2 * tv + 5 * B + 5],
                            g[:, 2 * tv + 6 * B:2 * tv + 6 * B + 4]], axis=1)
        ints = np.stack([(iv[:, 0] & 0x1F) | iv[:, 1], iv[:, 2]], axis=1).astype(np.int32)
        return np.ascontiguousarray(f), ints

    def reset(self, mask=None, first_episode: bool = False):
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        check(lib().wb_terrain_env_reset(self._h, ptr(m), int(first_episode)))

    def get_obs(self):
        obs = np.empty((self.n, OBS), np.float32)
        check(lib().wb_terrain_env_get_obs(self._h, ptr(obs)))
        return obs

    def step(self, actions, delta_time: float = DT_FRAME, auto_reset: bool = True, out=None):
        """actions [n, 4] -> (obs [n, 12], reward [n], done [n]) host arrays; one kernel launch."""
        a = np.ascontiguousarray(actions, np.float32).reshape(self.n, ACT)
        if out is None:
            out = (np.empty((self.n, OBS), np.float32), np.empty(self.n, np.float32), np.empty(self.n, np.uint8))
        obs, rew, done = out
        check(lib().wb_terrain_env_step(self._h, ptr(a), delta_time, int(auto_reset), ptr(obs), ptr(rew), ptr(done)))
        return obs, rew, done

    def step_dev(self, actions_dev, obs_dev, reward_dev, done_dev, delta_time: float = DT_FRAME, auto_reset: bool = True):
        """Device pointers (ints or torch CUDA tensors); enqueues on the handle's stream, no sync."""
        check(lib().wb_terrain_env_step_dev(self._h, ptr(actions_dev), delta_time, int(auto_reset), ptr(obs_dev), ptr(reward_dev),
                                            ptr(done_dev)))


# ---------------------------------------------------------------- the reference's own scene pieces as IObject lists
def CreateFloor(material="Metal") -> list:
    """Environment.CreateFloor, flat branch (Environment.cs:211-226): one static floor hull."""
    return [Hull.FromPositions(material, [(-50, 1050), (-50, 900), (1050, 900), (1050, 1050)], isStatic=True, isFloor=True)]


def CreateRoughFloor(heights, segments: int = 10, roughness: int = 100, material="Metal") -> list:
    """Environment.CreateRoughFloor (Environment.cs:230-261): `segments` static floor hulls whose tops follow random heights.
    The reference draws them from an UNSEEDED System.Random (`random.Next(0, roughness)`, :242,:249), so the draws are an
    argument here: heights[0] is the draw for the first `previousVector`, heights[1 + i] the draw of segment i (integers in
    [0, roughness)).  The reference's invalid-argument branch (segments <= 0 or roughness < 0: log and retry with the
    defaults) becomes a ValueError."""
    if segments <= 0 or roughness < 0:
        raise ValueError("Invalid floor segments/roughness values.")
    heights = [int(h) for h in heights]
    if len(heights) != segments + 1 or any(h < 0 or h >= max(roughness, 1) for h in heights):
        raise ValueError("heights must hold segments + 1 integers in [0, roughness)")
    initial_y, initial_x = 800, -50
    prev = (initial_x, initial_y + heights[0])
    movement = 1200 // segments  # C# integer division
    out = []
    for i in range(segments):
        x = initial_x + i * movement
        y = 800 + heights[1 + i]
        out.append(Hull.FromPositions(material, [(x, 1050), prev, (x, y), (x + movement, 1050)], isStatic=True, isFloor=True))
        prev = (x, y)
    return out


def CreateCreature(position=(125, 800), material="Carpet"):
    """Walker.CreateCreature (Walker.cs:40-46): CreateBodies (:155-178), CreateJoints (:181-189), AddAssociatedBodies (:204-209)
    and AddAcceleration((0, 980)).  Returns (objects in the order they join Environment._rigidBodies -- LLL, LLU, Body, RLL,
    RLU --, joints in creation order)."""
    px, py = f32(position[0]), f32(position[1])
    body = Hull.FromPositions(material, [(px + f32(20), py + f32(20)), (px, py + f32(20)), (px - f32(20), py + f32(20)),
                                         (px - f32(20), py - f32(20)), (px + f32(20), py - f32(20))])
    body.inverseInertia = 0.0003  # Body.SetInverseInertia(0.0003f), Walker.cs:168
    llu = Pole.FromSize(material, (px, py + f32(30)), 75)
    lll = Pole.FromSize(material, (px, py + f32(60)), 75)
    rlu = Pole.FromSize(material, (px, py + f32(30)), 75)
    rll = Pole.FromSize(material, (px, py + f32(60)), 75)
    joints = [Joint(body, llu, 1, 4), Joint(body, rlu, 1, 4), Joint(llu, lll, 2, 3), Joint(rlu, rll, 2, 3)]
    llu.associated = [rlu, rll, body]
    lll.associated = [rlu, rll, body]
    rlu.associated = [llu, lll, body]
    rll.associated = [llu, lll, body]
    body.associated = [llu, rlu, lll, rll]
    objs = [lll, llu, body, rll, rlu]
    for o in objs:
        o.acceleration = (0.0, 980.0)
    return objs, joints


__all__ = ["IObject", "Square", "Triangle", "Hexagon", "Pole", "Hull", "Joint", "Scene", "TerrainEnvBatch", "CreateFloor", "CreateRoughFloor", "CreateCreature"]

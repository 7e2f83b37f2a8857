// physics_scene.cu -- the reference's rigid-body engine for ARBITRARY scenes (sm_100a): any list of convex polygons
// (IObject plugins: Square / Triangle / Hexagon / Pole / Hull, smoothed or not, Objects/RigidBodies/*.cs), static or dynamic,
// floor or not, any IMaterial, association ("no collide") lists and pseudo-revolute joints -- N independent copies of the
// scene stepped in lockstep.  SURVEY.md section 8f row 4; the walker-specialised kernels in physics_lanes.cu cover the default
// scene much faster, this one covers everything Environment.StepObjects (Environment.cs:126-143) can be asked to do:
//   for each substep: every Joint.Step in list order (Joint.cs:31-41), then every body's IObject.Update in list order
//   (RigidBody.Step, RigidBody.cs:54-61: integrate, rotate unless static, then ResolveCollisions :66-96 against every other
//   body in list order except itself and its associated bodies: AABB, Collided latch, SAT, contact points, MoveObjects, impulses).
// One thread per scene copy; the copy's state lives in shared memory as columns ([slot][copy]); vertex counts are runtime
// values (<= 16 per polygon), so everything is a loop over shared memory -- general, not fast.  Same arithmetic contract as the
// walker kernels (IEEE binary32, no FMA, correctly rounded 1/x, sqrt, division, (float)cos/sin((double)theta)).
#include "physics.cuh"
#include "physics_math.cuh"

namespace wb {
namespace sc {

__constant__ SceneConst c_scene;

struct Ctx {
  const SceneConst* s;  // topology: &c_scene (scene_step_kernel) or the terrain kernel's __grid_constant__ parameter
  float2* v2;  // column of float2 slots: vertices [total_verts], centroids [B], velocities [B]
  float* f;    // column of float slots: omega [B], angle [B]
  int stride;  // copies per CTA
  int collided;
  int rot;     // Environment._rigidBodies order: list position k holds body index (k + rot) mod B (0: index order)
  bool static_fixed;  // never write a static body's velocities (see resolve_collisions)
};

// body index at list position k (the body sweep of StepObjects and the candidate loop of ResolveCollisions both follow it)
__device__ __forceinline__ int list_body(const Ctx& c, int k) {
  const int b = k + c.rot;
  return b >= c.s->n_bodies ? b - c.s->n_bodies : b;
}

__device__ __forceinline__ float2& VX(const Ctx& c, int b, int i) { return c.v2[(c.s->vert_offset[b] + i) * c.stride]; }
__device__ __forceinline__ float2& CEN(const Ctx& c, int b) { return c.v2[(c.s->total_verts + b) * c.stride]; }
__device__ __forceinline__ float2& VEL(const Ctx& c, int b) { return c.v2[(c.s->total_verts + c.s->n_bodies + b) * c.stride]; }
__device__ __forceinline__ float& OMEGA(const Ctx& c, int b) { return c.f[b * c.stride]; }
__device__ __forceinline__ float& ANGLE(const Ctx& c, int b) { return c.f[(c.s->n_bodies + b) * c.stride]; }

// Skeleton.Move, Skeleton.cs:76-85
__device__ void move_body(const Ctx& c, int b, float2 d) {
  const int n = c.s->n_verts[b];
  for (int i = 0; i < n; i++) VX(c, b, i) = vadd(VX(c, b, i), d);
  CEN(c, b) = vadd(CEN(c, b), d);
}

struct Dyn {
  float2 c, v;
  float w, im, ii;
};
__device__ __forceinline__ Dyn load_dyn(const Ctx& c, int b) {
  Dyn d;
  d.c = CEN(c, b);
  d.v = VEL(c, b);
  d.w = OMEGA(c, b);
  d.im = c.s->inv_mass[b];
  d.ii = c.s->inv_inertia[b];
  return d;
}
__device__ __forceinline__ void store_dyn(const Ctx& c, int b, const Dyn& d) {
  VEL(c, b) = d.v;
  OMEGA(c, b) = d.w;
}

// Impulses.CalculateImpulse, Impulses.cs:86-115
__device__ void calculate_impulse(const Dyn& A, const Dyn& B, float2 contact, float force, float2 n, float2& rA, float2& rB, float& impulse) {
  rA = vsub(contact, A.c);
  const float2 perpA = mk2(-rA.y, rA.x);
  const float kA = vdot(n, perpA);
  rB = vsub(contact, B.c);
  const float2 perpB = mk2(-rB.y, rB.x);
  const float kB = vdot(n, perpB);
  const float2 va = vadd(A.v, vmul(perpA, A.w));
  const float2 vb = vadd(B.v, vmul(perpB, B.w));
  const float2 vrel = vsub(vb, va);
  const float vn = vdot(vrel, n);
  const float j = fmul(-force, vn);
  const float denom = fadd(fadd(fadd(A.im, B.im), fmul(fmul(kA, kA), A.ii)), fmul(fmul(kB, kB), B.ii));
  impulse = fdiv(j, denom);
}

// Impulses.ApplyImpulses, Impulses.cs:57-82
__device__ void apply_impulses(Dyn& A, Dyn& B, float2 n, float impulse, float2 rA, float2 rB) {
  const float2 J = vmul(n, impulse);
  const float2 velA = vsub(A.v, vmul(J, A.im));
  const float2 velB = vadd(B.v, vmul(J, B.im));
  const float2 perpA = mk2(-rA.y, rA.x);
  const float wA = fsub(A.w, fmul(vdot(perpA, J), A.ii));
  const float2 perpB = mk2(-rB.y, rB.x);
  const float wB = fadd(B.w, fmul(vdot(perpB, J), B.ii));
  A.v = velA;
  B.v = velB;
  A.w = wA;
  B.w = wB;
}

// Joint.Step, Joint.cs:31-41
__device__ void joint_step(const Ctx& c, int k) {
  const int A = c.s->joint_a[k], ia = c.s->joint_ia[k], B = c.s->joint_b[k], ib = c.s->joint_ib[k];
  float2 ab = vsub(VX(c, B, ib), VX(c, A, ia));
  const float depth = fsqrt(fadd(fmul(ab.x, ab.x), fmul(ab.y, ab.y)));
  if (depth < 0.1f) return;
  ab = vnormalize(ab);
  move_body(c, A, vhalf(vmul(ab, depth)));
  move_body(c, B, vhalf(vmul(vneg(ab), depth)));
  Dyn X = load_dyn(c, B);  // Manifold(bodyA := joint._bodyB, bodyB := joint._bodyA)
  Dyn Y = load_dyn(c, A);
  const float2 contact = vhalf(vadd(VX(c, A, ia), VX(c, B, ib)));
  float2 rX, rY;
  float j;
  calculate_impulse(X, Y, contact, fadd(1.0f, 1.0f), ab, rX, rY, j);
  apply_impulses(X, Y, ab, j, rX, rY);
  store_dyn(c, B, X);
  store_dyn(c, A, Y);
}

// BoundingBox.FindSignificantCorners, Skeleton.cs:144-176
__device__ void aabb_of(const Ctx& c, int b, float2& mn, float2& mx) {
  const int n = c.s->n_verts[b];
  mn = mk2(FLT_MAX, FLT_MAX);
  mx = mk2(-FLT_MAX, -FLT_MAX);
  for (int i = 0; i < n; i++) {
    const float2 p = VX(c, b, i);
    mn.x = fminf(mn.x, p.x);
    mn.y = fminf(mn.y, p.y);
    mx.x = fmaxf(mx.x, p.x);
    mx.y = fmaxf(mx.y, p.y);
  }
}

// SATCollision.ProjectPoints, SATCollision.cs:63-76
__device__ void project(const Ctx& c, int b, float2 axis, float& mn, float& mx) {
  const int n = c.s->n_verts[b];
  mn = FLT_MAX;
  mx = -FLT_MAX;
  for (int i = 0; i < n; i++) {
    const float t = vdot(axis, VX(c, b, i));
    mn = fminf(mn, t);
    mx = fmaxf(mx, t);
  }
}

// SATCollision.AxisChecks, SATCollision.cs:39-59 (own = the polygon whose edges give the axes)
__device__ bool axis_checks(const Ctx& c, int own, int other, float2& normal, float& depth) {
  const int n = c.s->n_verts[own];
  for (int i = 0; i < n; i++) {
    const float2 edge = vsub(VX(c, own, i + 1 == n ? 0 : i + 1), VX(c, own, i));
    float2 axis = mk2(-edge.y, edge.x);
    if (axis.x == 0.0f && axis.y == 0.0f) continue;
    axis = vnormalize(axis);
    float omin, omax, tmin, tmax;
    project(c, own, axis, omin, omax);
    project(c, other, axis, tmin, tmax);
    const float temp = fminf(fsub(tmax, omin), fsub(omax, tmin));
    if (!((omin < tmax) && (tmin < omax))) return false;
    if (temp >= depth) continue;
    depth = temp;
    normal = axis;
  }
  return true;
}

struct Face {
  float2 a, b, max;
};

// ContactPoints.GetSignificantVertex + GetSignificantFace, ContactPoints.cs:79-113
__device__ Face significant_face(const Ctx& c, int b, float2 nrm) {
  const int n = c.s->n_verts[b];
  float best = FLT_MAX;
  int k = 0;
  for (int i = 0; i < n; i++) {
    const float pr = vdot(VX(c, b, i), nrm);
    if (pr < best) {
      best = pr;
      k = i;
    }
  }
  const float2 sv = VX(c, b, k), next = VX(c, b, k + 1 == n ? 0 : k + 1), prev = VX(c, b, k == 0 ? n - 1 : k - 1);
  const float2 after = vnormalize(vsub(sv, next));
  const float2 before = vnormalize(vsub(sv, prev));
  Face f;
  if (vdot(nrm, before) >= vdot(nrm, after)) {
    f.a = sv;
    f.b = prev;
  } else {
    f.a = next;
    f.b = sv;
  }
  f.max = sv;
  return f;
}

// ContactPoints.ClipVectors, ContactPoints.cs:56-76
__device__ int clip_vectors(float2 a, float2 b, float2 nrm, float offset, float2& o0, float2& o1) {
  int cnt = 0;
  const float da = fsub(vdot(a, nrm), offset);
  const float db = fsub(vdot(b, nrm), offset);
  if (da >= 0.0f) {
    o0 = a;
    cnt = 1;
  }
  if (db >= 0.0f) {
    if (cnt == 0) o0 = b; else o1 = b;
    cnt++;
  }
  if (fmul(da, db) < 0.0f) {
    float2 ed = vsub(b, a);
    const float location = fdiv(da, fsub(da, db));
    ed = vmul(ed, location);
    ed = vadd(ed, a);
    if (cnt == 0) o0 = ed; else if (cnt == 1) o1 = ed;
    cnt++;
  }
  return cnt;
}

// ContactPoints.GetContactPoints, ContactPoints.cs:13-53
__device__ int contact_points(const Ctx& c, int A, int B, float2 normal, float2& c0, float2& c1) {
  Face ref = significant_face(c, A, normal);
  Face inc = significant_face(c, B, vneg(normal));
  float2 rf = vsub(ref.b, ref.a);
  const float2 ifv = vsub(inc.b, inc.a);
  if (fabsf(vdot(rf, normal)) > fabsf(vdot(ifv, normal))) {
    const Face t = ref;
    ref = inc;
    inc = t;
    rf = vsub(ref.b, ref.a);
  }
  rf = vnormalize(rf);
  float offset = vdot(rf, ref.a);
  float2 p0 = mk2(0.f, 0.f), p1 = mk2(0.f, 0.f);
  int cnt = clip_vectors(inc.a, inc.b, rf, offset, p0, p1);
  if (cnt < 2) return 0;
  offset = vdot(rf, ref.b);
  float2 q0 = mk2(0.f, 0.f), q1 = mk2(0.f, 0.f);
  cnt = clip_vectors(p0, p1, vneg(rf), -offset, q0, q1);
  if (cnt < 2) return 0;
  cnt = 2;
  const float2 rn = mk2(rf.y, -rf.x);
  const float maximum = vdot(rn, ref.max);
  if (fsub(vdot(rn, q0), maximum) < 0.0f) {  // List.Remove(First())
    q0 = q1;
    cnt = 1;
  }
  const float2 last = (cnt == 2) ? q1 : q0;
  if (fsub(vdot(rn, last), maximum) < 0.0f) {  // List.Remove(Last()): deletes the first element EQUAL to the value
    if (cnt == 2) {
      if (q0.x == q1.x && q0.y == q1.y) q0 = q1;
      cnt = 1;
    } else {
      cnt = 0;
    }
  }
  c0 = q0;
  c1 = q1;
  return cnt;
}

// RigidBody.ResolveCollisions for body A, RigidBody.cs:66-96
__device__ void resolve_collisions(Ctx& c, int A) {
  const int nb = c.s->n_bodies;
  for (int k = 0; k < nb; k++) {
    const int B = list_body(c, k);
    if (B == A) continue;
    if ((c.s->assoc[A] >> B) & 1u) continue;
    float2 amin, amax, bmin, bmax;
    aabb_of(c, A, amin, amax);
    aabb_of(c, B, bmin, bmax);
    if (!(amin.x < bmax.x && amax.x > bmin.x && amin.y < bmax.y && amax.y > bmin.y)) continue;
    if (c.s->is_floor[B]) c.collided |= (1 << A);
    if (c.s->is_floor[A]) c.collided |= (1 << B);
    // SATCollision.IsColliding, SATCollision.cs:15-35
    float2 normal = mk2(0.0f, 0.0f);
    float depth = FLT_MAX;
    if (!(axis_checks(c, A, B, normal, depth) && axis_checks(c, B, A, normal, depth))) continue;
    if (vdot(vsub(CEN(c, B), CEN(c, A)), normal) > 0.0f) normal = vmul(normal, -1.0f);
    float2 c0 = mk2(0.f, 0.f), c1 = mk2(0.f, 0.f);
    const int ncp = contact_points(c, A, B, normal, c0, c1);
    // RigidBody.MoveObjects, RigidBody.cs:99-113
    if (c.s->is_static[A]) {
      move_body(c, B, vmul(vneg(normal), depth));
    } else if (c.s->is_static[B]) {
      move_body(c, A, vmul(normal, depth));
    } else {
      move_body(c, A, vhalf(vmul(normal, depth)));
      move_body(c, B, vhalf(vmul(vneg(normal), depth)));
    }
    if (ncp == 0) continue;
    // Impulses.ResolveCollisions, Impulses.cs:12-28
    Dyn X = load_dyn(c, A), Y = load_dyn(c, B);
    const float e = net_max(c.s->restitution[A], c.s->restitution[B]);
    const float mu = net_min(c.s->friction[A], c.s->friction[B]);
    const float2 contact = (ncp == 2) ? vhalf(vadd(c0, c1)) : c0;
    const float2 tangent = mk2(-normal.y, normal.x);
    float2 rA, rB, rAf, rBf;
    float j, jf;
    calculate_impulse(X, Y, contact, fadd(1.0f, e), normal, rA, rB, j);
    calculate_impulse(X, Y, contact, mu, tangent, rAf, rBf, jf);
    apply_impulses(X, Y, normal, j, rA, rB);
    apply_impulses(X, Y, tangent, jf, rAf, rBf);
    store_dyn(c, A, X);
    // a static body has inverse mass / inertia 0: finite impulses leave it unchanged.  A NaN impulse (a walker driven by NaN
    // actions) would leave NaN in it, as in the reference; with static_fixed (the terrain kernel) static bodies are never written,
    // like the walker kernels' floor, so one bad episode cannot wreck terrain that outlives the walker's resets
    if (!(c.static_fixed && c.s->is_static[B])) store_dyn(c, B, Y);
  }
}

// RigidBody.Step, RigidBody.cs:54-61,116-140
__device__ void body_step(Ctx& c, int b, float dt) {
  float2 v = VEL(c, b);
  v = vadd(v, vmul(mk2(c.s->accel_x[b], c.s->accel_y[b]), dt));
  VEL(c, b) = v;
  move_body(c, b, vmul(v, dt));
  if (c.s->is_static[b]) return;
  const float theta = fmul(OMEGA(c, b), dt);
  float ang = fadd(ANGLE(c, b), theta);
  const float PI_F = 3.14159274f, TAU_F = 6.28318548f;
  if (ang > PI_F) ang = fsub(ang, TAU_F);
  else if (ang < -PI_F) ang = fadd(ang, TAU_F);
  ANGLE(c, b) = ang;
  float m11, m12;
  rotz(theta, m11, m12);
  const float2 cen = CEN(c, b);
  const int n = c.s->n_verts[b];
  for (int i = 0; i < n; i++) {  // Skeleton.Rotate, Skeleton.cs:89-97
    const float2 p = vsub(VX(c, b, i), cen);
    const float2 t = vrotate(p, m11, m12);
    VX(c, b, i) = vadd(t, cen);
  }
  resolve_collisions(c, b);
}

// state rows (per copy): 2*total_verts vertex floats, 2B centroids, 2B velocities, B omega, B angle  (+ J torques kept in HBM)
__global__ void __launch_bounds__(32) scene_step_kernel(const SceneParams p) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x;
  const int copy = blockIdx.x * 32 + lane;
  if (copy >= p.n) return;  // no synchronisation anywhere: each thread owns its column
  const int nv2 = c_scene.total_verts + 2 * c_scene.n_bodies;
  const int nf = 2 * c_scene.n_bodies;
  Ctx c;
  c.s = &c_scene;
  c.v2 = reinterpret_cast<float2*>(smem) + lane;
  c.f = smem + nv2 * 2 * 32 + lane;
  c.stride = 32;
  c.collided = p.collided[copy];
  c.rot = 0;
  c.static_fixed = false;
  float* col = reinterpret_cast<float*>(c.v2);
  for (int r = 0; r < nv2 * 2; r++) col[(r >> 1) * 64 + (r & 1)] = p.state[(size_t)r * p.n_pad + copy];
  for (int r = 0; r < nf; r++) c.f[r * 32] = p.state[(size_t)(nv2 * 2 + r) * p.n_pad + copy];

  if (p.torques) {  // Joint.SetTorque, Joint.cs:56-61 (row of _currentTorque per joint follows the body rows)
    for (int k = 0; k < c_scene.n_joints; k++) {
      float* cur = p.state + (size_t)(nv2 * 2 + nf + k) * p.n_pad + copy;
      const float amount = p.torques[(size_t)copy * c_scene.n_joints + k];
      const float change = fsub(amount, *cur);
      *cur = amount;
      OMEGA(c, c_scene.joint_b[k]) = fadd(OMEGA(c, c_scene.joint_b[k]), fmul(change, 5.0f));
    }
  }
  if (p.iterations > 0) {  // Environment.StepObjects, Environment.cs:126-143
    const float dt = fdiv(p.dt, (float)p.iterations);
    for (int it = 0; it < p.iterations; it++) {
      for (int k = 0; k < c_scene.n_joints; k++) joint_step(c, k);
      for (int b = 0; b < c_scene.n_bodies; b++) body_step(c, b, dt);
    }
  }
  for (int r = 0; r < nv2 * 2; r++) p.state[(size_t)r * p.n_pad + copy] = col[(r >> 1) * 64 + (r & 1)];
  for (int r = 0; r < nf; r++) p.state[(size_t)(nv2 * 2 + r) * p.n_pad + copy] = c.f[r * 32];
  p.collided[copy] = c.collided;
}

// ---- the walker on arbitrary terrain: Environment.Update minus the policy (Environment.cs:64-92) over the scene
// [LLL, LLU, Body, RLL, RLU, terrain...] (Walker.CreateCreature, Walker.cs:40-46,155-209, + the caller's IObjects).
// Phases as physics_lanes_kernel; the list order is walker first as constructed (Environment.cs:46-48) and terrain first after
// a Reset, which re-creates the walker and appends it (Environment.cs:167-173): a rotation of the body indices by 5.
constexpr int kWalkerBodies = 5, kBody = 2, kLLU = 1, kRLU = 4;

__global__ void __launch_bounds__(32) terrain_step_kernel(const __grid_constant__ TerrainConst tc, const TerrainParams p) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x;
  const int copy = blockIdx.x * 32 + lane;
  if (copy >= p.n) return;  // one thread per copy, no synchronisation
  const SceneConst& s = tc.topo;
  const int nb = s.n_bodies, tv = s.total_verts;
  const int nv2 = tv + 2 * nb;
  const int nf = 2 * nb;
  Ctx c;
  c.s = &s;
  c.v2 = reinterpret_cast<float2*>(smem) + lane;
  c.f = smem + nv2 * 2 * 32 + lane;
  c.stride = 32;
  c.static_fixed = true;
  float* col = reinterpret_cast<float*>(c.v2);
  for (int r = 0; r < nv2 * 2; r++) col[(r >> 1) * 64 + (r & 1)] = p.state[(size_t)r * p.n_pad + copy];
  for (int r = 0; r < nf; r++) c.f[r * 32] = p.state[(size_t)(nv2 * 2 + r) * p.n_pad + copy];
  float* torque_rows = p.state + (size_t)(nv2 * 2 + nf) * p.n_pad + copy;
  c.collided = p.ints[copy];
  int flags = p.ints[p.n_pad + copy];
  int steps = p.ints[2 * (size_t)p.n_pad + copy];

  // Walker.Reset + CreateCreature (Walker.cs:212-236): the walker's five bodies as wb_env_create builds them, torques zero,
  // Collided cleared; the terrain bodies are left as they are (the reference keeps them in _rigidBodies)
  auto fresh_walker = [&]() {
    const int wv = s.vert_offset[kWalkerBodies - 1] + s.n_verts[kWalkerBodies - 1];
    for (int i = 0; i < wv; i++) c.v2[i * 32] = make_float2(tc.walker_init[2 * i], tc.walker_init[2 * i + 1]);
    for (int b = 0; b < kWalkerBodies; b++) {
      CEN(c, b) = make_float2(tc.walker_init[2 * wv + 2 * b], tc.walker_init[2 * wv + 2 * b + 1]);
      VEL(c, b) = make_float2(0.0f, 0.0f);
      OMEGA(c, b) = 0.0f;
      ANGLE(c, b) = 0.0f;
    }
    for (int k = 0; k < s.n_joints; k++) torque_rows[(size_t)k * p.n_pad] = 0.0f;
    c.collided &= ~((1 << kWalkerBodies) - 1);
  };

  if ((p.phases & kPhaseResetMasked) && (p.reset_mask == nullptr || p.reset_mask[copy])) {
    fresh_walker();
    flags = (p.phases & kPhaseFirstEpisode) ? 0 : WB_FLAG_FLOOR_FIRST;
    steps = 0;
  }
  if (p.phases & kPhaseIncSteps) steps++;
  if (p.phases & kPhaseTakeActions) {
    // Matrix.Clip (Matrix.cs:377-405; NaN passes, +-inf clip), Walker.TakeActions (Walker.cs:66-75), Joint.SetTorque (Joint.cs:56-61)
    for (int k = 0; k < s.n_joints; k++) {
      float a = p.actions[(size_t)copy * s.n_joints + k];
      if (a >= 1.0f) a = 1.0f;
      else if (a <= -1.0f) a = -1.0f;
      const float change = fsub(a, torque_rows[(size_t)k * p.n_pad]);
      torque_rows[(size_t)k * p.n_pad] = a;
      OMEGA(c, s.joint_b[k]) = fadd(OMEGA(c, s.joint_b[k]), fmul(change, 5.0f));
    }
  }
  // Walker._position (Walker.cs:19) is the Body's cached centroid at the last Walker.Update: the centroid this launch starts from
  const float2 prev = CEN(c, kBody);
  if (p.phases & kPhaseStepObjects) {  // Environment.StepObjects, Environment.cs:126-143, in the copy's list order
    c.rot = (flags & WB_FLAG_FLOOR_FIRST) ? kWalkerBodies : 0;
    const float dt = fdiv(p.dt, (float)p.iterations);
    for (int it = 0; it < p.iterations; it++) {
      for (int k = 0; k < s.n_joints; k++) joint_step(c, k);
      for (int k = 0; k < nb; k++) body_step(c, list_body(c, k), dt);
    }
  }
  if (p.phases & kPhaseObserve) {
    // Walker.Update (Walker.cs:49-54): Terminal latches on the Collided of Body, LLU or RLU (any is_floor body)
    const float2 pos = CEN(c, kBody);
    if (c.collided & ((1 << kBody) | (1 << kLLU) | (1 << kRLU))) flags |= WB_FLAG_TERMINAL;
    // CalculateReward, Environment.cs:148-154 (incl. the "-= -0.1f" sign quirk)
    const float dx = fsub(pos.x, prev.x);
    const float h = fdiv(VX(c, kBody, 1).y, 500.0f);
    float r = 0.0f;
    r = fadd(r, (dx > 0.0f && h < 1.6f) ? dx : 0.0f);
    r = fsub(r, (h > 1.65f) ? -0.1f : 0.0f);
    bool terminal = false;
    if ((flags & WB_FLAG_TERMINAL) || steps > p.max_timesteps) {  // Environment.cs:106-110
      if (flags & WB_FLAG_TERMINAL) r = fsub(r, 40.0f);
      terminal = true;
    }
    if (pos.x > 900.0f) {  // :113-117
      r = fadd(r, 80.0f);
      terminal = true;
    }
    if (terminal && (p.phases & kPhaseAutoReset)) {  // Reset + InitialState, Environment.cs:91,157-180
      fresh_walker();
      flags = WB_FLAG_FLOOR_FIRST;
      steps = 0;
    }
    p.reward[copy] = r;
    p.done[copy] = terminal ? 1 : 0;
  }
  if (p.phases & (kPhaseObserve | kPhaseObsOnly)) {  // Walker.GetState, Walker.cs:132-152
    const float2 j0 = VX(c, kBody, 1), j2 = VX(c, kLLU, 2), j3 = VX(c, kRLU, 2), bv = VEL(c, kBody);
    float* o = p.obs + (size_t)copy * WB_OBS;
    o[0] = fdiv(j0.x, 900.0f);
    o[1] = fdiv(j0.y, 500.0f);
    o[2] = fdiv(j2.x, 900.0f);
    o[3] = fdiv(j2.y, 500.0f);
    o[4] = fdiv(j3.x, 900.0f);
    o[5] = fdiv(j3.y, 500.0f);
    o[6] = fdiv(bv.x, 60.0f);
    o[7] = fdiv(bv.y, 60.0f);
    o[8] = ANGLE(c, 0);
    o[9] = ANGLE(c, kLLU);
    o[10] = ANGLE(c, 3);
    o[11] = ANGLE(c, kRLU);
  }
  for (int r = 0; r < nv2 * 2; r++) p.state[(size_t)r * p.n_pad + copy] = col[(r >> 1) * 64 + (r & 1)];
  for (int r = 0; r < nf; r++) p.state[(size_t)(nv2 * 2 + r) * p.n_pad + copy] = c.f[r * 32];
  p.ints[copy] = c.collided;
  p.ints[p.n_pad + copy] = flags;
  p.ints[2 * (size_t)p.n_pad + copy] = steps;
}

}  // namespace sc

size_t scene_smem_bytes(const SceneConst& s) { return (size_t)32 * ((size_t)(s.total_verts + 2 * s.n_bodies) * 8 + (size_t)2 * s.n_bodies * 4); }

cudaError_t launch_scene(const SceneParams& p, const SceneConst& s, cudaStream_t stream) {
  const size_t smem = scene_smem_bytes(s);
  // the topology lives in constant memory; a process may hold several scenes, so it is (re)sent with every launch (~1.5 KB)
  cudaError_t e = cudaMemcpyToSymbolAsync(sc::c_scene, &s, sizeof(SceneConst), 0, cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(sc::scene_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  sc::scene_step_kernel<<<(p.n + 31) / 32, 32, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t terrain_kernel_setup() {
  // one value for every handle (the largest scene the kernel accepts), so handles created later never lower it under a
  // launch of an earlier one
  SceneConst worst{};
  worst.n_bodies = kSceneMaxBodies;
  worst.total_verts = kSceneMaxBodies * kSceneMaxVerts;
  return cudaFuncSetAttribute(sc::terrain_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scene_smem_bytes(worst));
}

cudaError_t launch_terrain(const TerrainConst& tc, const TerrainParams& p, cudaStream_t stream) {
  // the topology travels as a kernel parameter: handles on different streams never share a __constant__ symbol
  sc::terrain_step_kernel<<<(p.n + 31) / 32, 32, scene_smem_bytes(tc.topo), stream>>>(tc, p);
  return cudaGetLastError();
}

}  // namespace wb

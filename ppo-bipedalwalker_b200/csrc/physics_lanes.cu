// physics_lanes.cu -- lockstep rigid-body step for N independent BipedalWalker environments (sm_100a),
// L lanes per environment (L = 1, 2, 4, 8, 16), one warp per CTA.
//
// Replaces, for a whole batch per launch, the reference's Environment.StepObjects and everything under it
// (Environment.cs:126-143; Joint.cs:31-61; RigidBody.cs:54-140; Skeleton.cs:76-176; SATCollision.cs:15-104;
// ContactPoints.cs:13-134; Impulses.cs:12-115) plus the walker glue around it (Walker.cs:49-75,132-152,
// Environment.cs:96-122,148-154,167-180).
//
// The reference's step is a strictly sequential Gauss-Seidel sweep per environment (4 joints, then 5 bodies in list
// order, every candidate pair resolved in place), so the unlimited parallelism is ACROSS environments; inside one, only
// the 12 SAT axes of a pair and the vertices of a Move/Rotate are independent.
//   L = 1  (throughput): every lane of a warp advances a different walker.  No redundant work, no shuffles.
//   L > 1  (latency, few walkers per SM): the lanes of a walker first split by LEG -- during the body sweep the left leg
//          {LLL, LLU}, the Body and the right leg {RLL, RLU} never touch each other's state (association lists,
//          Walker.cs:204-208; the floor is immutable), so {LLL, LLU, Body} and {RLL, RLU} are swept concurrently by the two
//          halves of the walker's lanes with bit-identical results -- and inside a half the G = L/2 lanes split the SAT axes
//          (axis i on lane i mod G, then a lexicographic (depth, index) min over the G lanes = the reference's "first
//          minimal axis wins") and the vertices of every Move / Rotate; the scalar parts are computed redundantly and
//          written by lane 0 of the group.  Fewer walkers share a warp, so the warp also follows the reference's early
//          exits more closely (a warp executes the union of its walkers' branches: with 32 walkers per warp some walker
//          always collides).
// State: the 92-float record is read once from the SoA arrays in HBM (coalesced), kept in shared memory as COLUMNS
// ([slot][env]: any data-dependent access -- support vertex k, its neighbours, runtime body ids -- is conflict free and
// lanes of one walker read by broadcast), advanced by all `iterations` substeps on chip and written back once.
// Control flow is WARP-UNIFORM: every branch is taken on a __any_sync vote and lanes are predicated inside, so all
// warp-level primitives use the full mask (plain SHFL / VOTE / WARPSYNC).  There are no block-level barriers.
//
// Arithmetic contract: IEEE binary32, every multiply/add individually rounded (never FMA; TU compiled with -fmad=false),
// correctly rounded 1/x, sqrt and division, (float)cos/sin((double)theta) for Skeleton.Rotate -- the same operation order
// as the reference's C# (SURVEY.md Appendix A/C).  Bit-exact against the oracle.  There is no CPU path.
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include "physics.cuh"
#include "physics_math.cuh"

namespace wb {
namespace pl {
constexpr unsigned kFull = 0xFFFFFFFFu;

#ifdef WB_PHASE_PROFILE
// experiment builds only (scripts/build_variant.sh prof -DWB_PHASE_PROFILE): cycle accounting of the compacting kernel
// (scripts/phase_profile.py) and of the lanes kernel (scripts/lanes_profile.py)
__device__ unsigned long long g_prof[24];
__device__ __forceinline__ long long prof_clock() {
  long long t;
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(t)::"memory");
  return t;
}
// lanes kernel: clock64 cycles of each CTA (one warp) of the last launch: entry to the first substep, the substep loop,
// observe + write-back (3 per CTA, CTAs beyond kLanesProfCtas are not recorded); read with wb_lanes_prof_read
constexpr int kLanesProfCtas = 1 << 16;
__device__ unsigned long long g_lanes_prof[3 * kLanesProfCtas];
#endif


__constant__ Material c_materials[WB_MAX_MATERIALS];
__constant__ float c_init_state[kStateFloats];  // state record of a freshly created walker
__constant__ FloorConst c_floor;

enum { LLL = 0, LLU = 1, BODY = 2, RLL = 3, RLU = 4, FLOOR = 5 };

// ---------------------------------------------------------------- shared-memory columns of one env
// float2 slots: vertices body*6 + i (Body's 6th slot mirrors its vertex 0, see below), centroids, velocities
constexpr int kV2Cen = 30;
constexpr int kV2Vel = 35;
constexpr int kV2Count = 40;
// float slots
constexpr int kFOmega = 0;
constexpr int kFAngle = 5;
constexpr int kFCount = 10;

// The Body hull has 5 vertices; its 6th slot holds a COPY of vertex 0 that goes through the same Move/Rotate operations
// (so it stays bit-identical to vertex 0).  Every polygon is then a 6-gon for the kernels: the duplicate never changes a
// min/max projection, never wins the strict "first smallest" support-vertex scan, edge 4 (P5 - P4) equals the hull's closing
// edge P0 - P4, and edge 5 (P0 - P5) is the zero vector, which SATCollision.AxisChecks itself skips (SATCollision.cs:45).
__device__ __forceinline__ int nverts(int b) { return b == BODY ? 5 : 6; }

template <int L_, int E_>
struct Env {
  static constexpr int L = L_;  // lanes per environment
  static constexpr int E = E_;  // environments (columns) per CTA
  float2* v2;   // this env's column of float2 slots: slot s at v2[s * E]
  float* f;     // this env's column of float slots
  const FloorConst* fl;  // the floor's constants (shared-memory copy: lanes index it with different runtime indices)
  int sub;      // lane inside the env's L lanes
  int gsub;     // lane inside the current working group (the whole env for joints, one leg's half during the body sweep)
  int gshift;   // first lane of the current working group inside the warp
  bool live;    // env < n
  int flags;    // Collided bits, Terminal, floor-first (identical on the L lanes)
  // material-derived constants (RigidBody ctor, RigidBody.cs:36-50; Impulses.cs:16-17)
  float im_w;     // walker inverse mass
  float ii_pole;  // 0.001f * inverse mass
  float e_ww, mu_ww, e_wf, mu_wf;
};

template <class EV> __device__ __forceinline__ float2& V2(const EV& e, int slot) { return e.v2[slot * EV::E]; }
template <class EV> __device__ __forceinline__ float& F1(const EV& e, int slot) { return e.f[slot * EV::E]; }
template <class EV> __device__ __forceinline__ float inv_inertia(const EV& e, int b) { return b == BODY ? 0.0003f : e.ii_pole; }  // Walker.cs:168
// material-derived constants of one walker (RigidBody ctor, RigidBody.cs:36-50; Impulses.cs:16-17)
template <class EV> __device__ __forceinline__ void set_materials(EV& e, const Material& mw, const Material& mf) {
  e.im_w = mw.inverse_mass;
  e.ii_pole = fmul(0.001f, mw.inverse_mass);
  e.e_ww = net_max(mw.restitution, mw.restitution);
  e.mu_ww = net_min(mw.friction, mw.friction);
  e.e_wf = net_max(mw.restitution, mf.restitution);
  e.mu_wf = net_min(mw.friction, mf.friction);
}
template <int L> __device__ __forceinline__ void lanes_sync() { if (L > 1) __syncwarp(); }
// true when `pred` holds on any lane of my env's group (full-mask vote: control flow is warp-uniform)
template <class EV, int G> __device__ __forceinline__ bool group_any(const EV& e, bool pred) {
  if (EV::L == 1) return pred;
  const unsigned b = __ballot_sync(kFull, pred);
  return ((b >> e.gshift) & ((1u << G) - 1u)) != 0u;
}

struct BodyDyn {
  float2 c, v;
  float w, im, ii;
};

template <class EV> __device__ __forceinline__ BodyDyn load_dyn(const EV& e, int b) {
  BodyDyn d;
  d.c = V2(e, kV2Cen + b);
  d.v = V2(e, kV2Vel + b);
  d.w = F1(e, kFOmega + b);
  d.im = e.im_w;
  d.ii = inv_inertia(e, b);
  return d;
}
template <class EV> __device__ __forceinline__ BodyDyn floor_dyn(const EV& e) {
  BodyDyn d;
  d.c = e.fl->cen;
  d.v = mk2(0.0f, 0.0f);
  d.w = 0.0f;
  d.im = 0.0f;
  d.ii = 0.0f;
  return d;
}
template <class EV> __device__ __forceinline__ void store_dyn(const EV& e, int b, const BodyDyn& d) {
  V2(e, kV2Vel + b) = d.v;
  F1(e, kFOmega + b) = d.w;
}

// Impulses.CalculateImpulse, Impulses.cs:86-115
__device__ __forceinline__ void calculate_impulse(const BodyDyn& A, const BodyDyn& B, float2 contact, float force, float2 n,
                                                  float2& rA, float2& rB, float& impulse) {
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
  const float2 k = mk2(kA, kB);
  const float2 kki = vmul2_nosum(vmul2_nosum(k, k), mk2(A.ii, B.ii));  // (kA*kA*A.ii, kB*kB*B.ii)
  const float denom = fadd(fadd(fadd(A.im, B.im), kki.x), kki.y);
  impulse = fdiv(j, denom);
}

// Impulses.ApplyImpulses, Impulses.cs:57-82
__device__ __forceinline__ void apply_impulses(BodyDyn& A, BodyDyn& B, float2 n, float impulse, float2 rA, float2 rB) {
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

// Skeleton.Move (Skeleton.cs:76-85) of up to two bodies, split over the G lanes of the working group: items 0..5 = A's six
// vertex slots (the Body's mirror slot moves with its vertex 0), 6 = A's centroid, 7..13 the same for B.  Predicated by `on`.
template <class EV, int G>
__device__ __forceinline__ void move_bodies(const EV& e, bool on, int A, float2 dA, bool moveB, int B, float2 dB) {
#pragma unroll
  for (int it0 = 0; it0 < 14; it0 += G) {
    const int it = it0 + e.gsub;
    const bool second = it >= 7;
    const int k = second ? it - 7 : it;
    const int b = second ? B : A;
    if (on && it < 14 && (!second || moveB)) {
      const int slot = (k < 6) ? b * 6 + k : kV2Cen + b;
      V2(e, slot) = vadd(V2(e, slot), second ? dB : dA);
    }
  }
}

// ---------------------------------------------------------------- Joint.Step, Joint.cs:31-41
// G = EV::L: the env's lanes step one joint; G < EV::L: the working group of G lanes (e.gsub, e.gshift) steps its own joint
template <class EV, bool TRACE, int G = EV::L>
__device__ __forceinline__ void joint_step(const EV& e, int A, int ia, int B, int ib, wb_joint_trace* tr) {
  const bool leader = (G == EV::L) ? e.sub == 0 : e.gsub == 0;
  const float2 pA = V2(e, A * 6 + ia);
  const float2 pB = V2(e, B * 6 + ib);
  float2 ab = vsub(pB, pA);
  const float depth = fsqrt(vdot(ab, ab));  // Vector2.Length
  if (TRACE) {
    if (tr && e.live && leader) {
      tr->active = !(depth < 0.1f);
      tr->depth = depth;
    }
  }
  const bool active = e.live && !(depth < 0.1f);
  if (!__any_sync(kFull, active)) return;
  ab = vnormalize_fast(ab);
  const float2 dA = vhalf(vmul(ab, depth));
  const float2 dB = vhalf(vmul(vneg(ab), depth));
  BodyDyn X = load_dyn(e, B);  // Manifold(bodyA := joint._bodyB, bodyB := joint._bodyA), Joint.cs:40
  BodyDyn Y = load_dyn(e, A);
  lanes_sync<EV::L>();  // every lane has read the pre-move points, centroids and velocities
  move_bodies<EV, G>(e, active, A, dA, true, B, dB);
  X.c = vadd(X.c, dB);  // the impulse sees the POST-move centroids and joint points
  Y.c = vadd(Y.c, dA);
  const float2 contact = vhalf(vadd(vadd(pA, dA), vadd(pB, dB)));  // Vector2.Divide(p0 + p1, 2), Impulses.cs:35
  float2 rX, rY;
  float j;
  calculate_impulse(X, Y, contact, fadd(1.0f, 1.0f), ab, rX, rY, j);
  apply_impulses(X, Y, ab, j, rX, rY);
  if (active && leader) {
    store_dyn(e, B, X);
    store_dyn(e, A, Y);
  }
  lanes_sync<EV::L>();
}

// ---------------------------------------------------------------- SAT, SATCollision.cs:15-104
// float.MaxValue / float.MinValue seeds take part in the min/max exactly like the reference's "if (t < min) min = t"
__device__ __forceinline__ void project6(const float2 (&P)[6], float2 ax, float& mn, float& mx) {
  const float t0 = vdot(ax, P[0]), t1 = vdot(ax, P[1]), t2 = vdot(ax, P[2]);
  const float t3 = vdot(ax, P[3]), t4 = vdot(ax, P[4]), t5 = vdot(ax, P[5]);
  mn = fminf(fminf(fminf(FLT_MAX, t0), fminf(t1, t2)), fminf(fminf(t3, t4), t5));
  mx = fmaxf(fmaxf(fmaxf(-FLT_MAX, t0), fmaxf(t1, t2)), fmaxf(fmaxf(t3, t4), t5));
}
__device__ __forceinline__ void project4(const float2* P, float2 ax, float& mn, float& mx) {
  const float t0 = vdot(ax, P[0]), t1 = vdot(ax, P[1]), t2 = vdot(ax, P[2]), t3 = vdot(ax, P[3]);
  mn = fminf(fminf(fminf(FLT_MAX, t0), t1), fminf(t2, t3));
  mx = fmaxf(fmaxf(fmaxf(-FLT_MAX, t0), t1), fmaxf(t2, t3));
}

// ---------------------------------------------------------------- contact points, ContactPoints.cs:13-134
struct Face {
  float2 a, b, max;
};

// GetSignificantFace given the support vertex sv = P[k] and its neighbours (ContactPoints.cs:79-94)
__device__ __forceinline__ Face face_from(float2 sv, float2 next, float2 prev, float2 nrm) {
  const float2 after = vnormalize_fast(vsub(sv, next));
  const float2 before = vnormalize_fast(vsub(sv, prev));
  const bool use_before = vdot(nrm, before) >= vdot(nrm, after);
  Face f;
  f.a = use_before ? sv : next;
  f.b = use_before ? prev : sv;
  f.max = sv;
  return f;
}

// GetSignificantVertex (ContactPoints.cs:97-113): first index with the strictly smallest projection
__device__ __forceinline__ int support_index6(const float2 (&P)[6], float2 nrm) {
  float best = FLT_MAX;
  int k = 0;  // (k stays 0 only if no projection is below float.MaxValue: non-finite state)
#pragma unroll
  for (int i = 0; i < 6; i++) {
    const float pr = vdot(P[i], nrm);
    const bool lt = pr < best;
    k = lt ? i : k;
    best = lt ? pr : best;
  }
  return k;
}

template <class EV>
__device__ __forceinline__ Face significant_face_body(const EV& e, int b, const float2 (&P)[6], float2 nrm) {
  const int n = nverts(b);
  const int k = support_index6(P, nrm);
  const int kn = (k + 1 == n) ? 0 : k + 1;
  const int kp = (k == 0) ? n - 1 : k - 1;
  return face_from(V2(e, b * 6 + k), V2(e, b * 6 + kn), V2(e, b * 6 + kp), nrm);
}

template <class EV>
__device__ __forceinline__ Face significant_face_floor(const EV& e, float2 nrm) {
  float best = FLT_MAX;
  int k = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const float pr = vdot(e.fl->v[i], nrm);
    const bool lt = pr < best;
    k = lt ? i : k;
    best = lt ? pr : best;
  }
  return face_from(e.fl->v[k], e.fl->v[(k + 1) & 3], e.fl->v[(k + 3) & 3], nrm);
}

// ClipVectors, ContactPoints.cs:56-76: appends up to 3 points; only the first two are ever used
__device__ __forceinline__ int clip_vectors(float2 a, float2 b, float2 nrm, float offset, float2& o0, float2& o1) {
  int cnt = 0;
  const float2 dab = vsub(mk2(vdot(a, nrm), vdot(b, nrm)), mk2(offset, offset));
  const float da = dab.x, db = dab.y;
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

__device__ __forceinline__ bool veq(float2 a, float2 b) { return a.x == b.x && a.y == b.y; }

// GetContactPoints after the two significant faces are known, ContactPoints.cs:13-53
__device__ __forceinline__ int contact_points(Face ref, Face inc, float2 normal, float2& c0, float2& c1) {
  float2 rf = vsub(ref.b, ref.a);
  const float2 ifv = vsub(inc.b, inc.a);
  if (fabsf(vdot(rf, normal)) > fabsf(vdot(ifv, normal))) {
    const Face t = ref;
    ref = inc;
    inc = t;
    rf = vsub(ref.b, ref.a);
  }
  rf = vnormalize_fast(rf);
  float offset = vdot(rf, ref.a);
  float2 p0 = mk2(0.f, 0.f), p1 = mk2(0.f, 0.f);
  int cnt = clip_vectors(inc.a, inc.b, rf, offset, p0, p1);
  if (cnt < 2) return 0;
  offset = vdot(rf, ref.b);
  float2 q0 = mk2(0.f, 0.f), q1 = mk2(0.f, 0.f);
  cnt = clip_vectors(p0, p1, vneg(rf), -offset, q0, q1);
  if (cnt < 2) return 0;
  cnt = 2;  // ClipVectors returns 3 points only if da >= 0, db >= 0 and da*db < 0 at once, which is impossible
  const float2 rn = mk2(rf.y, -rf.x);
  const float maximum = vdot(rn, ref.max);
  // List.Remove(First()) then List.Remove(Last()): Remove deletes the first element EQUAL to the value
  if (fsub(vdot(rn, q0), maximum) < 0.0f) {
    q0 = q1;
    cnt = 1;
  }
  const float2 last = (cnt == 2) ? q1 : q0;
  if (fsub(vdot(rn, last), maximum) < 0.0f) {
    if (cnt == 2) {
      if (veq(q0, q1)) q0 = q1;  // removes index 0 when both points are equal (same value survives)
      cnt = 1;
    } else {
      cnt = 0;
    }
  }
  c0 = q0;
  c1 = q1;
  return cnt;
}

// Impulses.ResolveCollisions, Impulses.cs:12-28: both impulses come from the PRE-impulse velocities (:23-24), then both are applied (:26-27)
__device__ __forceinline__ void resolve_impulses(BodyDyn& X, BodyDyn& Y, int ncp, float2 c0, float2 c1, float2 normal, float e, float mu) {
  const float2 contact = (ncp == 2) ? vhalf(vadd(c0, c1)) : c0;
  const float2 tangent = mk2(-normal.y, normal.x);
  float2 rA, rB, rAf, rBf;
  float j, jf;
  calculate_impulse(X, Y, contact, fadd(1.0f, e), normal, rA, rB, j);
  calculate_impulse(X, Y, contact, mu, tangent, rAf, rBf, jf);
  apply_impulses(X, Y, normal, j, rA, rB);
  apply_impulses(X, Y, tangent, jf, rAf, rBf);
}

// the same with two or more lanes per pair: even lanes compute the normal impulse, odd lanes the "friction" impulse (both from
// the PRE-impulse velocities, so they are independent), the lanes swap the two scalars and every lane applies both in order
__device__ __forceinline__ void resolve_impulses_split(BodyDyn& X, BodyDyn& Y, int ncp, float2 c0, float2 c1, float2 normal, float e, float mu,
                                                       bool odd) {
  const float2 contact = (ncp == 2) ? vhalf(vadd(c0, c1)) : c0;
  const float2 tangent = mk2(-normal.y, normal.x);
  float2 rA, rB;
  float mine;
  calculate_impulse(X, Y, contact, odd ? mu : fadd(1.0f, e), odd ? tangent : normal, rA, rB, mine);  // rA, rB do not depend on the direction
  const float other = __shfl_xor_sync(kFull, mine, 1);
  apply_impulses(X, Y, normal, odd ? other : mine, rA, rB);
  apply_impulses(X, Y, tangent, odd ? mine : other, rA, rB);
}

__device__ __forceinline__ void aabb6(const float2 (&P)[6], float2& mn, float2& mx) {
  mn.x = fminf(fminf(fminf(P[0].x, P[1].x), fminf(P[2].x, P[3].x)), fminf(P[4].x, P[5].x));
  mn.y = fminf(fminf(fminf(P[0].y, P[1].y), fminf(P[2].y, P[3].y)), fminf(P[4].y, P[5].y));
  mx.x = fmaxf(fmaxf(fmaxf(P[0].x, P[1].x), fmaxf(P[2].x, P[3].x)), fmaxf(P[4].x, P[5].x));
  mx.y = fmaxf(fmaxf(fmaxf(P[0].y, P[1].y), fmaxf(P[2].y, P[3].y)), fmaxf(P[4].y, P[5].y));
}
// BoundingBox.IsColliding, Skeleton.cs:133-140
__device__ __forceinline__ bool aabb_hit(float2 amin, float2 amax, float2 bmin, float2 bmax) {
  return amin.x < bmax.x && amax.x > bmin.x && amin.y < bmax.y && amax.y > bmin.y;
}

// pair-trace record of a candidate whose SAT has not found a collision (yet)
__device__ __forceinline__ wb_pair_trace pair_trace_no_sat(int other, bool aabb) {
  wb_pair_trace rec;
  rec.other = other;
  rec.aabb = aabb ? 1 : 0;
  rec.sat = 0;
  rec.axis = -1;
  rec.nx = rec.ny = rec.depth = 0.0f;
  rec.ncontacts = 0;
  rec.c0x = rec.c0y = rec.c1x = rec.c1y = 0.0f;
  return rec;
}

// ---------------------------------------------------------------- one candidate of RigidBody.ResolveCollisions (RigidBody.cs:66-96)
// FLOORB = false: a leg segment A against the other segment B of its own leg (both dynamic poles)
// FLOORB = true : a walker body A against the static floor (scene constants)
// `want`: this env takes part (candidate exists at this position of its list order).
// `sep_axis` (may be null): receives the index (0..11, A's edges then B's) of the first separating axis this lane found
// BY_LAYOUT: true = the SAT rounds vote or not by layout (see kVote), false = straight-line rounds and one vote at the end
// KNOWN_HIT: the caller has already established that the bounding boxes overlap (stage 1 of the compacting kernel)
template <class EV, int G, bool TRACE, bool FLOORB, bool BY_LAYOUT = true, bool KNOWN_HIT = false>
__device__ __forceinline__ void resolve_pair(EV& e, bool want, int A, int B, wb_pair_trace* tr, int* sep_axis = nullptr) {
  const FloorConst& fl = *e.fl;
  float2 PA[6], PB[6];
#pragma unroll
  for (int i = 0; i < 6; i++) PA[i] = V2(e, A * 6 + i);
  if (!FLOORB) {
#pragma unroll
    for (int i = 0; i < 6; i++) PB[i] = V2(e, B * 6 + i);
  }
  bool hit = want;
  if (!KNOWN_HIT) {
    float2 amin, amax, bmin, bmax;
    aabb6(PA, amin, amax);
    if (FLOORB) {
      bmin = fl.bb_min;
      bmax = fl.bb_max;
    } else {
      aabb6(PB, bmin, bmax);
    }
    hit = want && aabb_hit(amin, amax, bmin, bmax);
  }
  if (FLOORB && hit) e.flags |= (1 << A);  // if (body._isFloor) Collided = true  (before SAT: RigidBody.cs:75)
  wb_pair_trace rec;
  if (TRACE) rec = pair_trace_no_sat(FLOORB ? FLOOR : B, hit);
#ifdef WB_PHASE_PROFILE
  const long long rp_t0 = prof_clock();
  long long rp_t1 = rp_t0;
#endif
  bool colliding = false;
  if (__any_sync(kFull, hit)) {
    // AxisChecks(A, B) then AxisChecks(B, A) (SATCollision.cs:19-29,39-59): axis i of the 12 (10 against the floor) goes to
    // lane i mod G.  Once an axis separates, the reference returns false and nothing computed afterwards is used, so the
    // rounds simply stop for an env as soon as any of its lanes saw a separating axis; a skipped (zero) axis has NaN
    // projections and must not touch anything.  "tempDepth >= depth -> continue" keeps the FIRST minimal axis: each lane
    // updates only on a strictly smaller depth (its axes come in increasing order) and the lanes are then combined by a
    // lexicographic (depth, index) minimum.
    const int nA = nverts(A);
    float depth = FLT_MAX;
    float2 normal = mk2(0.0f, 0.0f);
    int idx = 0x7FFFFFFF;
    bool sep = false;
    // Projection.IsOverlapping + depth (SATCollision.cs:47-50,100-104): symmetric in the two projections.  Returns true when
    // no env of the warp needs another axis.
    // kVote: normally the rounds stop as soon as no walker of the warp needs another axis (one vote per round).  With G == 4
    // (the 8-lanes-per-walker layout of the 4096-walker case: latency bound, 8 pairs in flight per warp, so an early stop is
    // rare) the three rounds are fully unrolled WITHOUT votes: a straight-line block lets the rounds' long dependency chains
    // (edge -> 1/sqrt -> 12 dot products -> min/max tree) overlap; the separation flags meet in one vote after the last round.
    // Measured at 4096 walkers: G = 4 0.472 -> 0.452 ms per env-step; G = 8 (throughput bound) 0.474 -> 0.596, so it keeps the votes.
    constexpr bool kVote = BY_LAYOUT && G != 4;
    bool my_sep = false;
    auto accumulate = [&](bool use, float2 axis, int axis_idx, float omin, float omax, float tmin, float tmax) {
      const float2 dd = vsub(mk2(tmax, omax), mk2(omin, tmin));  // (tmax - omin, omax - tmin)
      const float temp = fminf(dd.x, dd.y);
      const bool overlapping = (omin < tmax) && (tmin < omax);
      if (use && temp < depth) {
        depth = temp;
        normal = axis;
        idx = axis_idx;
      }
      if (sep_axis != nullptr && use && !overlapping && !sep && !my_sep) *sep_axis = axis_idx;
      if (!kVote) {
        my_sep = my_sep || (use && !overlapping);
        return false;
      }
      const bool separated = group_any<EV, G>(e, use && !overlapping);  // (a vote: every lane takes part, no short-circuit)
      sep = sep || separated;
      return !__any_sync(kFull, hit && !sep);
    };
    // left normal of edge k of polygon `own`, zero test, Vector2.Normalize (SATCollision.cs:43-46)
    auto edge_axis = [&](int own, int k, bool& skip) {
      const float2 p0 = V2(e, own * 6 + k), p1 = V2(e, own * 6 + (k == 5 ? 0 : k + 1));
      const float2 edge = vsub(p1, p0);
      const float2 axis = mk2(-edge.y, edge.x);
      skip = (axis.x == 0.0f) && (axis.y == 0.0f);
      return vnormalize_fast(axis);
    };
    // the same from the registers that already hold both polygons (two lanes per pair: lane parity picks between two static
    // edges, so no shared-memory access with a runtime index is needed); r is a compile-time round index
    auto edge_axis_reg = [&](const float2 (&P)[6], int r, bool odd, bool& skip) {
      const float2 p0 = odd ? P[(r + 1) % 6] : P[r % 6], p1 = odd ? P[(r + 2) % 6] : P[(r + 1) % 6];
      const float2 edge = vsub(p1, p0);
      const float2 axis = mk2(-edge.y, edge.x);
      skip = (axis.x == 0.0f) && (axis.y == 0.0f);
      return vnormalize_fast(axis);
    };
    auto round_a_vs_floor = [&](int r) {  // AxisChecks(A, floor): A's 6 edges
      const int i = r + e.gsub;
      const bool valid = i < 6;
      bool skip;
      const float2 axis = (G == 2 && !kVote) ? edge_axis_reg(PA, r, e.gsub != 0, skip) : edge_axis(A, valid ? i : 0, skip);
      float omin, omax, tmin, tmax;
      project6(PA, axis, omin, omax);
      project4(fl.v, axis, tmin, tmax);
      return accumulate(valid && !skip, axis, i, omin, omax, tmin, tmax);
    };
    auto round_floor_vs_a = [&](int r) {  // AxisChecks(floor, A): constant axes and constant own projection
      const int i = r + e.gsub;
      const bool valid = i < 4;
      const int k = valid ? i : 0;
      const float2 axis = fl.axis[k];
      float tmin, tmax;
      project6(PA, axis, tmin, tmax);
      return accumulate(valid && fl.skip[k] == 0, axis, nA + k, fl.pmin[k], fl.pmax[k], tmin, tmax);
    };
    auto round_pole = [&](int r) {  // AxisChecks(A, B) then AxisChecks(B, A)
      const int i = r + e.gsub;
      const bool valid = i < 12;
      const bool ownA = i < 6;
      const int k = ownA ? i : (valid ? i - 6 : 0);
      bool skip;
      float2 axis;
      if (G == 2 && !kVote) {  // (r is even and known at compile time after unrolling: r < 6 <=> the edge belongs to A)
        axis = (r < 6) ? edge_axis_reg(PA, r, e.gsub != 0, skip) : edge_axis_reg(PB, r - 6, e.gsub != 0, skip);
      } else {
        axis = edge_axis(ownA ? A : B, k, skip);
      }
      float amn, amx, bmn, bmx;
      project6(PA, axis, amn, amx);
      project6(PB, axis, bmn, bmx);
      return accumulate(valid && !skip, axis, ownA ? i : nA + k, amn, amx, bmn, bmx);
    };
    if (kVote) {
      if (FLOORB) {
        bool done = false;
#pragma unroll 1
        for (int r = 0; r < 6 && !done; r += G) done = round_a_vs_floor(r);
#pragma unroll 1
        for (int r = 0; r < 4 && !done; r += G) done = round_floor_vs_a(r);
      } else {
#pragma unroll 1
        for (int r = 0; r < 12; r += G)
          if (round_pole(r)) break;
      }
    } else {  // (unrolled by 6, not fully: G = 1 gives the pole loop 12 trips; rolled rounds measured slower, DESIGN §4.1)
      if (FLOORB) {
#pragma unroll 6
        for (int r = 0; r < 6; r += G) round_a_vs_floor(r);
#pragma unroll 6
        for (int r = 0; r < 4; r += G) round_floor_vs_a(r);
      } else {
#pragma unroll 6
        for (int r = 0; r < 12; r += G) round_pole(r);
      }
      sep = group_any<EV, G>(e, my_sep);
    }
    colliding = hit && !sep;
#ifdef WB_PHASE_PROFILE
    rp_t1 = prof_clock();
#endif
    // the contact stage stays inlined in every caller: one shared non-inlined copy for the compacting kernel's two drains
    // measured slower, DESIGN §4.2
    if (__any_sync(kFull, colliding)) {
      if (G > 1) {
#pragma unroll
        for (int m = 1; m < G; m <<= 1) {
          const float od = __shfl_xor_sync(kFull, depth, m);
          const int oi = __shfl_xor_sync(kFull, idx, m);
          const float ox = __shfl_xor_sync(kFull, normal.x, m);
          const float oy = __shfl_xor_sync(kFull, normal.y, m);
          if (od < depth || (od == depth && oi < idx)) {
            depth = od;
            idx = oi;
            normal = mk2(ox, oy);
          }
        }
      }
      // orient: normal points from B towards A (SATCollision.cs:31-32, cached centroids)
      BodyDyn X = load_dyn(e, A);
      BodyDyn Y = FLOORB ? floor_dyn(e) : load_dyn(e, B);
      if (vdot(vsub(Y.c, X.c), normal) > 0.0f) normal = vmul(normal, -1.0f);
      // GetSignificantFace of A (along the normal) and of B (against it), ContactPoints.cs:15-16.  With two or more lanes per
      // pair the even lanes take A and the odd lanes B through ONE code path (the floor is padded to a 6-gon with copies of
      // its vertex 0, which never win the strict "first smallest" scan), then the lanes swap faces.
      Face ref, inc;
      if (G == 1) {
        ref = significant_face_body(e, A, PA, normal);
        inc = FLOORB ? significant_face_floor(e, vneg(normal)) : significant_face_body(e, B, PB, vneg(normal));
      } else {
        const bool odd = (e.gsub & 1) != 0;
        const float2 nn = odd ? vneg(normal) : normal;
        float2 P[6];
        int n, stride;
        const float2* vb;
        if (FLOORB) {
#pragma unroll
          for (int i = 0; i < 6; i++) {
            const float2 f = fl.v[i < 4 ? i : 0];
            P[i] = odd ? f : PA[i];
          }
          n = odd ? 4 : nA;
          vb = odd ? fl.v : &V2(e, A * 6);
          stride = odd ? 1 : EV::E;
        } else {
#pragma unroll
          for (int i = 0; i < 6; i++) P[i] = odd ? PB[i] : PA[i];
          n = nverts(odd ? B : A);
          vb = &V2(e, (odd ? B : A) * 6);
          stride = EV::E;
        }
        const int k = support_index6(P, nn);
        const int kn = (k + 1 == n) ? 0 : k + 1;
        const int kp = (k == 0) ? n - 1 : k - 1;
        const Face mine = face_from(vb[k * stride], vb[kn * stride], vb[kp * stride], nn);
        Face other;
        other.a.x = __shfl_xor_sync(kFull, mine.a.x, 1);
        other.a.y = __shfl_xor_sync(kFull, mine.a.y, 1);
        other.b.x = __shfl_xor_sync(kFull, mine.b.x, 1);
        other.b.y = __shfl_xor_sync(kFull, mine.b.y, 1);
        other.max.x = __shfl_xor_sync(kFull, mine.max.x, 1);
        other.max.y = __shfl_xor_sync(kFull, mine.max.y, 1);
        ref = odd ? other : mine;
        inc = odd ? mine : other;
      }
      float2 c0 = mk2(0.f, 0.f), c1 = mk2(0.f, 0.f);
      const int ncp = contact_points(ref, inc, normal, c0, c1);
      if (TRACE) {
        if (colliding) {
          rec.sat = 1;
          rec.axis = idx;
          rec.nx = normal.x;
          rec.ny = normal.y;
          rec.depth = depth;
          rec.ncontacts = ncp;
          if (ncp > 0) {
            rec.c0x = c0.x;
            rec.c0y = c0.y;
          }
          if (ncp > 1) {
            rec.c1x = c1.x;
            rec.c1y = c1.y;
          }
        }
      }
      // RigidBody.MoveObjects, RigidBody.cs:99-113, applied even with 0 contact points: static B -> A.Move(normal * depth),
      // both dynamic -> A.Move(normal * depth / 2), B.Move(-normal * depth / 2)
      const float2 dA = FLOORB ? vmul(normal, depth) : vhalf(vmul(normal, depth));
      const float2 dB = FLOORB ? mk2(0.f, 0.f) : vhalf(vmul(vneg(normal), depth));
      lanes_sync<EV::L>();  // every lane has read the pre-move vertices, centroids and velocities
      move_bodies<EV, G>(e, colliding, A, dA, !FLOORB, B, dB);
      // impulses (only with contact points) read the PRE-move velocities but the POST-move centroids
      X.c = vadd(X.c, dA);
      if (!FLOORB) Y.c = vadd(Y.c, dB);
      if (G == 1) {
        if (ncp > 0) resolve_impulses(X, Y, ncp, c0, c1, normal, FLOORB ? e.e_wf : e.e_ww, FLOORB ? e.mu_wf : e.mu_ww);
      } else {  // warp-uniform: every lane takes part in the exchange, the result is used only where ncp > 0
        resolve_impulses_split(X, Y, ncp, c0, c1, normal, FLOORB ? e.e_wf : e.e_ww, FLOORB ? e.mu_wf : e.mu_ww, (e.gsub & 1) != 0);
      }
      if (ncp > 0 && colliding && e.gsub == 0) {
        store_dyn(e, A, X);
        if (!FLOORB) store_dyn(e, B, Y);  // the floor is never written (inverse mass/inertia 0)
      }
      lanes_sync<EV::L>();
    }
  }
  if (TRACE) {
    if (tr && want && e.gsub == 0) *tr = rec;
  }
#ifdef WB_PHASE_PROFILE
  const unsigned prof_want = __ballot_sync(kFull, want), prof_coll = __ballot_sync(kFull, colliding);
  if (!TRACE && (threadIdx.x & 31) == 0) {
    const long long rp_t2 = prof_clock();
    const int k = FLOORB ? 1 : 0;
    atomicAdd(&g_prof[8 + 4 * k + 0], (unsigned long long)(rp_t1 - rp_t0));   // AABB + SAT
    atomicAdd(&g_prof[8 + 4 * k + 1], (unsigned long long)(rp_t2 - rp_t1));   // contact pipeline + moves + impulses
    atomicAdd(&g_prof[8 + 4 * k + 2], 1ull);                                  // warp-level calls
    atomicAdd(&g_prof[8 + 4 * k + 3], (unsigned long long)__popc(prof_want) | ((unsigned long long)__popc(prof_coll) << 32));
  }
#endif
}


// ---------------------------------------------------------------- RigidBody.Step, RigidBody.cs:54-61,116-140
// The integration half: StepLinearVelocity, StepAngularVelocity, Skeleton.Move + Rotate of body b by the nq lanes that step it
// (this lane is number q of them); round r moves vertex slot r * nq + q and also leaves the new vertex in P[r].
// `on`: this lane really steps body b (false for the right-leg half while the left-leg half steps the Body)
template <class EV, int R>
__device__ __forceinline__ void integrate_step(const EV& e, bool on, int b, int q, int nq, float dt, float2 (&P)[R]) {
  // StepLinearVelocity: v += a * dt (gravity (0, 980), Walker.cs:45); Skeleton.Move(v * dt)
  float2 v = V2(e, kV2Vel + b);
  v = vadd(v, vmul(mk2(0.0f, 980.0f), dt));
  const float2 d = vmul(v, dt);
  // StepAngularVelocity: angle = WrapAngle(angle + w * dt); Skeleton.Rotate(w * dt)
  const float w = F1(e, kFOmega + b);
  const float theta = fmul(w, dt);
  float ang = fadd(F1(e, kFAngle + b), theta);
  const float PI_F = 3.14159274f, TAU_F = 6.28318548f;
  if (ang > PI_F) ang = fsub(ang, TAU_F);
  else if (ang < -PI_F) ang = fadd(ang, TAU_F);
  float m11, m12;
  rotz(theta, m11, m12);
  const float2 cen = vadd(V2(e, kV2Cen + b), d);
  lanes_sync<EV::L>();  // all reads of the old centroid / velocity / angle are done
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int i = r * nq + q;
    P[r] = mk2(0.0f, 0.0f);
    if (i < 6 && on) {
      // Move then Rotate (Vector2.Transform(p - centroid, R) + centroid, Skeleton.cs:93)
      float2 p = vadd(V2(e, b * 6 + i), d);
      p = vsub(p, cen);
      const float2 t = vrotate(p, m11, m12);
      P[r] = vadd(t, cen);
      V2(e, b * 6 + i) = P[r];
    }
  }
  if (q == 0 && on) {
    V2(e, kV2Cen + b) = cen;
    V2(e, kV2Vel + b) = v;
    F1(e, kFAngle + b) = ang;
  }
  lanes_sync<EV::L>();
}

// The collision half: RigidBody.ResolveCollisions of body b
template <class EV, int G, bool TRACE>
__device__ __forceinline__ void resolve_candidates(EV& e, bool on, int b, wb_pair_trace* tr_base) {
  // ResolveCollisions: candidates in Environment._rigidBodies order, skipping self and associated bodies (Walker.cs:204-208):
  // a leg segment meets the other segment of its own leg and the floor; the Body only the floor.  The floor comes first in the
  // list after the first Reset (Walker.cs:212-223).  Three uniform phases keep a warp whose environments disagree on the list
  // order from running the pole-pole pair twice: [floor if floor-first] [leg partner] [floor if floor-last].
  const int slot = (0x75420 >> (4 * b)) & 0xF;     // trace slot base {0,2,4,5,7}
  const int partner = (0x34F01 >> (4 * b)) & 0xF;  // {LLU, LLL, -, RLU, RLL}
  const bool floor_first = (e.flags & WB_FLAG_FLOOR_FIRST) != 0;
#pragma unroll 1
  for (int phase = 0; phase < 3; phase++) {
    if (phase == 1) {
      const bool want = on && b != BODY;
      if (__any_sync(kFull, want))
        resolve_pair<EV, G, TRACE, false>(e, want, b, b == BODY ? LLL : partner, (TRACE && tr_base) ? tr_base + slot + (floor_first ? 1 : 0) : nullptr);
    } else {
      const bool want = on && ((b == BODY) ? (phase == 0) : ((phase == 0) == floor_first));
      if (__any_sync(kFull, want))
        resolve_pair<EV, G, TRACE, true>(e, want, b, FLOOR, (TRACE && tr_base) ? tr_base + slot + ((b == BODY || floor_first) ? 0 : 1) : nullptr);
    }
  }
}

template <class EV, int G, bool TRACE>
__device__ __forceinline__ void body_step(EV& e, bool on, int b, float dt, wb_pair_trace* tr_base) {
  float2 P[(6 + G - 1) / G];
  integrate_step(e, on, b, e.gsub, G, dt, P);
  resolve_candidates<EV, G, TRACE>(e, on, b, tr_base);
}

// The body sweep of the leg split (LEGS = 2) with G >= 4 lanes per half in TWO slots instead of three: the Body shares no
// mutable state with either leg during the sweep (it only meets the floor), so it needs no slot of its own.
//   slot 0  integrate LLL on lanes 0..H-1 of the left half, the Body on lanes H..G-1 and RLL on the right half in ONE pass (one
//           rotz on the chain); test the Body's bounding box against the floor on its new vertices; resolve the Body-floor
//           pair only in a warp where that test hits (a Body on the floor ends the episode, so this is rare); then LLL's and
//           RLL's candidates
//   slot 1  LLU on the left half, RLU on the right half
// Every body still meets its candidates in list order with the values the sequential sweep gives it, so the result is the
// sequential one bit for bit.  With G = 2 (4 lanes per walker) the left half would move each of LLL and the Body on one lane
// in six rounds instead of three: measured slower (contact_stress +2 %), so that layout keeps the three-slot sweep.
template <class EV, int G, bool TRACE>
__device__ __forceinline__ void legs_sweep(EV& e, bool left, float dt, wb_pair_trace* tr_base) {
  static_assert(G >= 4, "two or more lanes per body in slot 0");
  constexpr int H = G / 2;            // lanes per body on the left half in slot 0
  constexpr int R = (6 + H - 1) / H;  // vertex rounds
  const int base = e.gshift - (left ? 0 : G);  // the walker's first lane
#pragma unroll 1
  for (int k = 0; k < 2; k++) {
    const bool body_lane = k == 0 && left && e.gsub >= H;
    const int seg = left ? (k == 0 ? LLL : LLU) : (k == 0 ? RLL : RLU);
    float2 P[R];
    integrate_step(e, e.live, body_lane ? BODY : seg, body_lane ? e.gsub - H : e.gsub, (k == 0 && left) ? H : G, dt, P);
    if (k == 0) {
      // BoundingBox.IsColliding(Body, floor) (Skeleton.cs:133-140) on the new vertices: slot i is P[i / H] of body lane i mod H
      float2 Q[6];
#pragma unroll
      for (int i = 0; i < 6; i++) {
        Q[i].x = __shfl_sync(kFull, P[i / H].x, base + H + i % H);
        Q[i].y = __shfl_sync(kFull, P[i / H].y, base + H + i % H);
      }
      float2 mn, mx;
      aabb6(Q, mn, mx);
      const unsigned hits = __ballot_sync(kFull, body_lane && e.live && aabb_hit(mn, mx, e.fl->bb_min, e.fl->bb_max));
      const bool body_hit = ((hits >> base) & ((1u << G) - 1u)) != 0u;  // on every lane of the walker
      if (body_hit) e.flags |= 1 << BODY;  // if (body._isFloor) Collided = true  (before SAT: RigidBody.cs:75)
      wb_pair_trace* tr = (TRACE && tr_base) ? tr_base + 4 : nullptr;  // the Body's one candidate, the floor
      if (TRACE) {
        if (tr && e.live && left && e.gsub == 0 && !body_hit) *tr = pair_trace_no_sat(FLOOR, false);
      }
      if (hits != 0u) resolve_pair<EV, G, TRACE, true, true, true>(e, left && body_hit, left ? BODY : RLL, FLOOR, tr);
    }
    resolve_candidates<EV, G, TRACE>(e, e.live, seg, tr_base);
  }
}

// Walker.GetState, Walker.cs:132-152
template <class EV>
__device__ __forceinline__ void store_observation(const EV& e, float* dst) {  // dst is 16-byte aligned (48 B per env)
  const float2 j0 = V2(e, BODY * 6 + 1), j2 = V2(e, LLU * 6 + 2), j3 = V2(e, RLU * 6 + 2), bv = V2(e, kV2Vel + BODY);
  float4* d4 = reinterpret_cast<float4*>(dst);
  d4[0] = make_float4(fdiv(j0.x, 900.0f), fdiv(j0.y, 500.0f), fdiv(j2.x, 900.0f), fdiv(j2.y, 500.0f));
  d4[1] = make_float4(fdiv(j3.x, 900.0f), fdiv(j3.y, 500.0f), fdiv(bv.x, 60.0f), fdiv(bv.y, 60.0f));
  d4[2] = make_float4(F1(e, kFAngle + LLL), F1(e, kFAngle + LLU), F1(e, kFAngle + RLL), F1(e, kFAngle + RLU));
}

// canonical record index f < 88 (walker_b200.h) -> word index inside a column set of E environments (env column 0);
// rows 88..91 (joint torques) stay in HBM.  The float2 slots come first, then the float slots.
template <int E>
__device__ __forceinline__ int record_word(int f) {
  if (f < 58) {
    const int vtx = f >> 1, slot = vtx + (vtx >= 17 ? 1 : 0);
    return slot * E * 2 + (f & 1);
  }
  if (f < 78) return (kV2Cen + ((f - 58) >> 1)) * E * 2 + (f & 1);
  return kV2Count * E * 2 + (f - 78) * E;
}

// a walker's inputs besides its record, staged in shared memory with the record (physics_lanes_kernel)
struct __align__(16) WalkerInputs {
  float4 actions;
  float torque[4];
  float2 pos;
  int32_t flags, steps;
  uint32_t mat_words[2];  // the aligned words of walker_mat / floor_mat that hold this walker's bytes
};

template <int V> struct FloatVec;
template <> struct FloatVec<1> { using T = float; };
template <> struct FloatVec<2> { using T = float2; };
template <> struct FloatVec<4> { using T = float4; };

// The CTA's E records as whole aligned pieces: each of the 39 float2 slot rows is one run of 2E floats in HBM
// (state_index) and in s_state (record_word), each of the 10 float rows (78..87) one run of E floats.  Calls
// fn(HBM float offset, s_state float offset, first column, floats per column, std::integral_constant<int, V>) for the
// pieces of this lane: V = 4 floats (16 B) where the run allows it.  Every piece of the CTA lies inside the padded rows
// (kEnvPad is a multiple of E).  The loops have compile-time trip counts, so they unroll and every piece is in flight
// before any is consumed.
template <int E, class F>
__device__ __forceinline__ void for_record_pieces(int lane, int env0, int n_pad, F&& fn) {
  constexpr int VA = 2 * E < 4 ? 2 * E : 4, PA = 2 * E / VA, NA = kStateSlots2 * PA;
  constexpr int VB = E < 4 ? E : 4, PB = E / VB, NB = kFCount * PB;
#pragma unroll
  for (int j = 0; j < (NA + 31) / 32; j++) {
    const int i = j * 32 + lane, s2 = i / PA, k = i % PA;
    if (NA % 32 == 0 || i < NA)
      fn(((size_t)s2 * n_pad + env0) * 2 + k * VA, (s2 + (s2 >= 17 ? 1 : 0)) * 2 * E + k * VA, k * VA / 2, 2,
         std::integral_constant<int, VA>());
  }
#pragma unroll
  for (int j = 0; j < (NB + 31) / 32; j++) {
    const int i = j * 32 + lane, r = i / PB, k = i % PB;
    if (NB % 32 == 0 || i < NB)
      fn((size_t)(78 + r) * n_pad + env0 + k * VB, kV2Count * 2 * E + r * E + k * VB, k * VB, 1, std::integral_constant<int, VB>());
  }
}

// cp.async of one aligned piece of B = 4, 8 or 16 bytes, global -> shared; complete for this thread after cp_async_wait_all
template <int B>
__device__ __forceinline__ void cp_async(float* smem, const float* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem), "n"(B)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// 16 resident warps per SM for L = 16 as well (at most 128 registers): a warp's registers come from ONE of the four SM
// sub-partitions (16 K each), so 129-160 registers leave 3 warps per sub-partition, and 4096 walkers with 16 lanes (2048
// warps) no longer fit one wave
template <int L, int LEGS, bool TRACE>
__global__ void __launch_bounds__(32, (L <= 4 || L == 16) ? 16 : 8) physics_lanes_kernel(const PhysicsParams p) {
  static_assert(LEGS == 1 || (LEGS == 2 && L >= 2), "the leg split needs at least two lanes per environment");
  constexpr int E = 32 / L;
  __shared__ __align__(16) float s_state[(kV2Count * 2 + kFCount) * E];
  __shared__ FloorConst s_floor;
  __shared__ WalkerInputs s_in[E];
  const int lane = threadIdx.x;
  const int env0 = blockIdx.x * E;
#ifdef WB_PHASE_PROFILE
  const long long t_entry = prof_clock();
#endif

  using EV = Env<L, E>;
  EV e;
  const int col = lane / L;
  const int env = env0 + col;
  e.v2 = reinterpret_cast<float2*>(s_state) + col;
  e.f = s_state + kV2Count * E * 2 + col;
  e.fl = &s_floor;
  e.sub = lane % L;
  e.gsub = e.sub;
  e.gshift = col * L;
  e.live = env < p.n;
  const int envc = e.live ? env : 0;  // dead lanes shadow env 0 read-only (they never store)
  float* torque_rows = p.state + (size_t)88 * p.n_pad + envc;

  // ---- stage the E records and each walker's inputs with every load in flight at once, so that this prologue costs one
  // memory round trip before the first substep rather than one per load.  Everything goes to shared memory by cp.async and
  // is waited for once (plain loads issued here would be scheduled behind the wait).  The record's rows are shared by all
  // 32 lanes (SoA rows are contiguous over envs); lane 0 of each walker fetches that walker's scalars, and Walker.TakeActions'
  // four joint torques (they stay in HBM) and actions.
  for_record_pieces<E>(lane, env0, p.n_pad, [&](size_t g, int s, int, int, auto v) {
    cp_async<decltype(v)::value * 4>(s_state + s, p.state + g);
  });
  WalkerInputs& in = s_in[col];
  if (e.sub == 0) {
    cp_async<4>(reinterpret_cast<float*>(&in.flags), reinterpret_cast<const float*>(p.flags + envc));
    cp_async<4>(reinterpret_cast<float*>(&in.steps), reinterpret_cast<const float*>(p.steps + envc));
    cp_async<4>(&in.pos.x, p.pos + envc);
    cp_async<4>(&in.pos.y, p.pos + p.n_pad + envc);
    // the material bytes arrive as the aligned word that holds them (the rows are padded to kEnvPad walkers)
    cp_async<4>(reinterpret_cast<float*>(&in.mat_words[0]), reinterpret_cast<const float*>(p.walker_mat + (envc & ~3)));
    cp_async<4>(reinterpret_cast<float*>(&in.mat_words[1]), reinterpret_cast<const float*>(p.floor_mat + (envc & ~3)));
    if (p.phases & kPhaseTakeActions) {
#pragma unroll
      for (int k = 0; k < 4; k++) cp_async<4>(&in.torque[k], torque_rows + (size_t)k * p.n_pad);
      if (e.live) cp_async<16>(reinterpret_cast<float*>(&in.actions), p.actions + (size_t)env * 4);
    }
  }
  constexpr int kFloorWords = sizeof(FloorConst) / 4;
#pragma unroll
  for (int j = 0; j < (kFloorWords + 31) / 32; j++) {
    const int w = j * 32 + lane;
    if (w < kFloorWords) reinterpret_cast<uint32_t*>(&s_floor)[w] = reinterpret_cast<const uint32_t*>(&c_floor)[w];
  }
  cp_async_wait_all();
  __syncwarp();
  e.flags = in.flags;
  int steps = in.steps;
  float2 pos = in.pos;
  {
    const int byte = 8 * (envc & 3);
    set_materials(e, c_materials[(in.mat_words[0] >> byte) & 0xFFu], c_materials[(in.mat_words[1] >> byte) & 0xFFu]);
  }

  // the fresh walker record into this lane's column, shared by the walker's L lanes (88 / L words per lane instead of 88 on
  // one lane; the loop stays rolled to keep the register count); the caller syncs the warp before the column is read
  auto write_initial_column = [&]() {
#pragma unroll 1
    for (int j = 0; j < (88 + L - 1) / L; j++) {
      const int f = j * L + e.sub;
      if (88 % L == 0 || f < 88) s_state[record_word<E>(f) + (f < 78 ? 2 * col : col)] = c_init_state[f];
    }
  };
  // the columns of walkers past n (the last CTA only) hold the fresh walker record, as a reset would leave it
  if (!e.live) write_initial_column();
  __syncwarp();
  if (e.sub == 0) V2(e, BODY * 6 + 5) = V2(e, BODY * 6);
  __syncwarp();

  // Walker.Reset + CreateCreature: fresh walker record (constants computed on the host with the reference's formulas)
  auto write_initial_record = [&](bool on) {
    if (!__any_sync(kFull, on)) return;
    __syncwarp();
    if (on) write_initial_column();
    __syncwarp();
    if (on && e.sub == 0) {
      V2(e, BODY * 6 + 5) = V2(e, BODY * 6);
#pragma unroll
      for (int k = 0; k < 4; k++) torque_rows[(size_t)k * p.n_pad] = in.torque[k] = c_init_state[88 + k];
    }
    __syncwarp();
  };

  if (p.phases & kPhaseResetMasked) {
    const bool on = e.live && (p.reset_mask == nullptr || p.reset_mask[envc]);
    write_initial_record(on);
    if (on) {
      e.flags = (p.phases & kPhaseFirstEpisode) ? 0 : WB_FLAG_FLOOR_FIRST;
      steps = 0;
      pos = V2(e, kV2Cen + BODY);  // InitialState -> Walker.Update
    }
  }
  if (p.phases & kPhaseIncSteps) steps++;

  if (p.phases & kPhaseTakeActions) {
    // Matrix.Clip (Matrix.cs:377-405), Walker.TakeActions (Walker.cs:66-75), Joint.SetTorque (Joint.cs:56-61)
    if (e.live && e.sub == 0) {
      const float act[4] = {in.actions.x, in.actions.y, in.actions.z, in.actions.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        float a = act[k];
        if (a >= 1.0f) a = 1.0f;
        else if (a <= -1.0f) a = -1.0f;
        const float change = fsub(a, in.torque[k]);
        torque_rows[(size_t)k * p.n_pad] = a;
        const int bodyB = (k == 0) ? LLU : (k == 1) ? RLU : (k == 2) ? LLL : RLL;  // Walker.cs:182-185
        F1(e, kFOmega + bodyB) = fadd(F1(e, kFOmega + bodyB), fmul(change, 5.0f));
      }
    }
    __syncwarp();
  }

#ifdef WB_PHASE_PROFILE
  const long long t_substeps = prof_clock();
#endif
  if (p.phases & kPhaseStepObjects) {
    const float dt = fdiv(p.dt, (float)p.iterations);  // deltaTime /= Hyperparameters.Iterations
#pragma unroll 1
    for (int it = 0; it < p.iterations; it++) {
      wb_joint_trace* jt = nullptr;
      wb_pair_trace* pt = nullptr;
      if (TRACE) {
        if (p.joint_trace) jt = p.joint_trace + ((size_t)envc * p.iterations + it) * 4;
        if (p.pair_trace) pt = p.pair_trace + ((size_t)envc * p.iterations + it) * WB_PAIR_SLOTS;  // all 9 slots are written every substep
      }
      // joints in creation order (Walker.cs:182-187): (Body v1, LLU v4) (Body v1, RLU v4) (LLU v2, LLL v3) (RLU v2, RLL v3)
      if (LEGS == 1) {
#pragma unroll 1
        for (int k = 0; k < 4; k++) {
          const int A = (0x4122 >> (4 * k)) & 0xF, B = (0x3041 >> (4 * k)) & 0xF;
          joint_step<EV, TRACE>(e, A, k < 2 ? 1 : 2, B, k < 2 ? 4 : 3, jt ? jt + k : nullptr);
        }
      } else {
        // joint 1 (Body, RLU) and joint 2 (LLU, LLL) share no body: each body still sees its joints in creation order
        // (Body: 0, 1; LLU: 0, 2; RLU: 1, 3), so stepping 1 and 2 side by side on the two halves of the env's lanes gives the
        // sequential result bit for bit with three joint steps on the walker's chain instead of four
        constexpr int G = L / LEGS;
        joint_step<EV, TRACE>(e, BODY, 1, LLU, 4, jt ? jt + 0 : nullptr);
        const int leg = e.sub / G;
        e.gsub = e.sub % G;
        e.gshift = col * L + leg * G;
        const bool left = leg == 0;  // (one call with per-lane bodies: control flow stays warp-uniform)
        joint_step<EV, TRACE, G>(e, left ? LLU : BODY, left ? 2 : 1, left ? LLL : RLU, left ? 3 : 4, jt ? jt + (left ? 2 : 1) : nullptr);
        e.gsub = e.sub;
        e.gshift = col * L;
        joint_step<EV, TRACE>(e, RLU, 2, RLL, 3, jt ? jt + 3 : nullptr);
      }
      // bodies in list order; the static floor's Update is a no-op (a = v = 0, returns before rotation/collisions)
      if (LEGS == 1) {
#pragma unroll 1
        for (int b = 0; b < 5; b++) body_step<EV, L, TRACE>(e, e.live, b, dt, pt);
      } else {
        // {LLL, LLU, Body} on the first half of the env's lanes, {RLL, RLU} on the second: the three subsystems share no
        // mutable state during the sweep, so any interleaving reproduces the sequential list-order result bit for bit
        constexpr int G = L / LEGS;
        const int leg = e.sub / G;
        e.gsub = e.sub % G;
        e.gshift = col * L + leg * G;
        if constexpr (G >= 4) {
          legs_sweep<EV, G, TRACE>(e, leg == 0, dt, pt);
        } else {  // three slots: (LLL | RLL), (LLU | RLU), (Body | idle)
#pragma unroll 1
          for (int k = 0; k < 3; k++) {
            const bool on = e.live && (leg == 0 || k < 2);
            body_step<EV, G, TRACE>(e, on, leg == 0 ? k : (k < 2 ? RLL + k : RLU), dt, pt);
          }
        }
        e.gsub = e.sub;
        e.gshift = col * L;
      }
    }
    if (LEGS == 2) e.flags |= __shfl_xor_sync(kFull, e.flags, L / LEGS);  // each half latched its own bodies' Collided bits
  }
#ifdef WB_PHASE_PROFILE
  const long long t_observe = prof_clock();
#endif

  if (p.phases & kPhaseObserve) {
    // Walker.Update, Walker.cs:49-54
    const float2 prev = pos;
    pos = V2(e, kV2Cen + BODY);
    if (e.flags & ((1 << BODY) | (1 << LLU) | (1 << RLU))) e.flags |= WB_FLAG_TERMINAL;
    // CalculateReward, Environment.cs:148-154 (incl. the "-= -0.1f" sign quirk)
    const float dx = fsub(pos.x, prev.x);
    const float h = fdiv(V2(e, BODY * 6 + 1).y, 500.0f);
    float r = 0.0f;
    r = fadd(r, (dx > 0.0f && h < 1.6f) ? dx : 0.0f);
    r = fsub(r, (h > 1.65f) ? -0.1f : 0.0f);
    bool terminal = false;
    if ((e.flags & WB_FLAG_TERMINAL) || steps > p.max_timesteps) {  // Environment.cs:106-110
      if (e.flags & WB_FLAG_TERMINAL) r = fsub(r, 40.0f);
      terminal = true;
    }
    if (pos.x > 900.0f) {  // :113-117
      r = fadd(r, 80.0f);
      terminal = true;
    }
    const bool reset_now = e.live && terminal && (p.phases & kPhaseAutoReset);
    write_initial_record(reset_now);
    if (reset_now) {
      e.flags = WB_FLAG_FLOOR_FIRST;
      steps = 0;
      pos = V2(e, kV2Cen + BODY);
    }
    if (e.live && e.sub == 0) {
      store_observation(e, p.obs + (size_t)env * WB_OBS);
      p.reward[env] = r;
      p.done[env] = terminal ? 1 : 0;
    }
  } else if (p.phases & kPhaseObsOnly) {
    if (e.live && e.sub == 0) store_observation(e, p.obs + (size_t)env * WB_OBS);
  }

  if (e.live && e.sub == 0) {
    p.flags[env] = e.flags;
    p.steps[env] = steps;
    p.pos[env] = pos.x;
    p.pos[p.n_pad + env] = pos.y;
  }
  __syncwarp();
  // ---- write the records back in the same pieces; a piece that reaches past n (the last CTA only) stores float by float
  const bool all_live = env0 + E <= p.n;
  for_record_pieces<E>(lane, env0, p.n_pad, [&](size_t g, int s, int c0, int per_col, auto v) {
    constexpr int V = decltype(v)::value;
    using T = typename FloatVec<V>::T;
    if (all_live) {
      *reinterpret_cast<T*>(p.state + g) = *reinterpret_cast<const T*>(s_state + s);
    } else {
#pragma unroll
      for (int j = 0; j < V; j++)
        if (env0 + c0 + j / per_col < p.n) p.state[g + j] = s_state[s + j];
    }
  });
#ifdef WB_PHASE_PROFILE
  if (lane == 0 && blockIdx.x < kLanesProfCtas) {
    const long long t_end = prof_clock();
    g_lanes_prof[3 * blockIdx.x + 0] = t_substeps - t_entry;
    g_lanes_prof[3 * blockIdx.x + 1] = t_observe - t_substeps;
    g_lanes_prof[3 * blockIdx.x + 2] = t_end - t_observe;
  }
#endif
}

// test hook: compares rcp_sqrt_rn(s) with __frcp_rn(__fsqrt_rn(s)) for every bit pattern in [first, first + count)
__global__ void rcp_sqrt_check_kernel(uint32_t first, uint64_t count, unsigned long long* mismatches, uint32_t* first_bad) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  unsigned long long bad = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
    const uint32_t bits = first + (uint32_t)i;
    const float s = __uint_as_float(bits);
    const uint32_t a = __float_as_uint(rcp_sqrt_rn(s));
    const uint32_t b = __float_as_uint(__frcp_rn(__fsqrt_rn(s)));
    const bool both_nan = ((a & 0x7FFFFFFFu) > 0x7F800000u) && ((b & 0x7FFFFFFFu) > 0x7F800000u);
    if (a != b && !both_nan) {
      bad++;
      atomicMin(first_bad, bits);
    }
  }
  if (bad) atomicAdd(mismatches, bad);
}

// test hook: evaluates the rotation coefficients for an array of angles (mode 0: production path, 1: force the
// double-double slow path, 2: force the libm-style sincos path)
__global__ void rotz_debug_kernel(const float* radians, int n, int mode, float* c_out, float* s_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float c, s;
  if (mode == 1) {
    sincos_dd_small((double)radians[i], c, s);
  } else if (mode == 2) {
    double sd, cd;
    sincos((double)radians[i], &sd, &cd);
    c = (float)cd;
    s = (float)sd;
  } else {
    rotz(radians[i], c, s);
  }
  c_out[i] = c;
  s_out[i] = s;
}

template <int L, int LEGS>
static cudaError_t launch_l(const PhysicsParams& p, bool trace, cudaStream_t stream) {
  constexpr int E = 32 / L;
  const int grid = (p.n + E - 1) / E;
  if (trace)
    physics_lanes_kernel<L, LEGS, true><<<grid, 32, 0, stream>>>(p);
  else
    physics_lanes_kernel<L, LEGS, false><<<grid, 32, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace pl

// ================================================================ throughput kernel with CTA-level work compaction
// One thread per environment (as L = 1 above), but a warp of the plain kernel executes the UNION of its 32 walkers' branches,
// and in a decorrelated rollout the expensive branches are rare per walker yet almost always present in some lane: a leg
// pair's AABBs overlap 85 % of the time but SAT finds a collision in only ~10 % of the substeps, the floor is touched in ~5 %,
// a joint needs correcting in ~20 % (profiles/hotspots_r1.md, r1d: 31 % of the executed lane-slots did useful work).
// Here a CTA of kE walkers (256 by default) advances in lockstep PHASES, and each phase has two stages:
//   stage 1  every thread, for ITS walker: the cheap, common part -- integrate the body; for a leg pair test the separating
//            axis that separated this pair last time (temporal coherence; any order of the axis tests gives the reference's
//            result: if one axis separates, SATCollision.IsColliding is false whatever the others say), then the AABBs; for
//            a floor pair the AABBs (and the Collided latch).  Walkers that need the expensive part push an item (walker,
//            body) onto a queue in shared memory.  (Joints run whole in the owning thread, see joint_in_thread.)
//   stage 2  after a CTA barrier, the queued items are processed DENSELY: thread t takes item t (any thread can work on any
//            walker: the state columns live in shared memory), runs the full resolve_pair of the plain kernel
//            on that walker's columns and records the separating axis it found, if any, for the next substep (the hints
//            also survive from launch to launch: PhysicsParams::axis_cache).
// Left and right leg are swept in the same phase (they share no mutable state, see the leg split above), which halves the
// number of barriers and doubles the queue density.  Arithmetic and order per walker are those of the plain kernel: the
// results are bit-identical (tests/test_physics_gpu.py runs every variant against the oracle).
// ---- cp.async.bulk (the TMA engine's 1-D form): contiguous global <-> shared copies issued by one thread
namespace bulk {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void load(void* smem_dst, const void* gmem_src, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void store(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void commit_and_wait_reads() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
}  // namespace bulk

namespace pc {
using namespace pl;

// -DWB_PHASE_PROFILE (experiment builds only, scripts/build_variant.sh): cycles per warp spent in stage 1, at the barrier before
// the drain, in the drain and at the barrier after it, summed over all warps of all CTAs; read with wb_prof_read (below)
#ifdef WB_PHASE_PROFILE
#define WB_PROF_DECL long long prof_t = prof_clock(); unsigned long long prof_acc[4] = {0, 0, 0, 0}; unsigned long long prof_items = 0, prof_rounds = 0
#define WB_PROF_MARK(k) do { const long long now_ = prof_clock(); prof_acc[k] += (unsigned long long)(now_ - prof_t); prof_t = now_; } while (0)
#else
#define WB_PROF_DECL
#define WB_PROF_MARK(k)
#endif

// kE walkers (= threads) share one queue and advance in lockstep.  Measured at 262144 walkers (ms per env-step): kE = 32 (ONE
// WARP per CTA, rounds separated by __syncwarp only, no block barrier anywhere) 8.86 -- sparse per-warp queues execute the
// expensive stage once per warp however few items it has; 64: 7.35; 128: 5.93; 256: 5.45 (default; 4.79 today); 512: 6.06 (one CTA
// per SM: nothing overlaps its barriers); 192 walkers x 3 CTAs per SM needs <= 96 registers per thread: 6.3.  Aggregation beats
// barrier cost up to the point where CTAs stop overlapping each other.  Shared memory (360 B per walker) and registers both cap
// residency at 512 walkers per SM.
template <int kE>
struct Shared {
  float state[(kV2Count * 2 + kFCount) * kE];
  Material mtab[WB_MAX_MATERIALS];      // copy of the material table (stage 2 works on other walkers: divergent indices)
  unsigned char wmat[kE], fmat[kE];     // walker / floor material id per walker
  FloorConst floor;
  unsigned char axis[4 * kE];   // last separating axis per ordered leg pair {LLL->LLU, LLU->LLL, RLL->RLU, RLU->RLL}
  unsigned short queue[3 * kE];  // a floor round holds at most three items per walker (two leg segments + the Body)
  int count[2];  // ping-pong: the counter of the next round is cleared while the current one drains
  unsigned long long stage_bar;  // mbarrier of the bulk-copy staging
#ifdef WB_PHASE_PROFILE
  long long prof_arrive[2][2][32];  // [round parity][barrier][warp]: arrival time at the barrier
#endif
};
// The noinline stages below rebuild their shared-memory pointers from this array instead of receiving pointers as arguments:
// an argument is a generic 64-bit address (LD / ST through the generic path), a pointer derived here stays LDS / STS.
extern __shared__ __align__(16) unsigned char smem_pc[];
template <int kE> __device__ __forceinline__ Shared<kE>& shm() { return *reinterpret_cast<Shared<kE>*>(smem_pc); }

template <int kE> __device__ __forceinline__ void scope_sync() {
  if (kE == 32) __syncwarp(); else __syncthreads();
}
template <int kE> __device__ __forceinline__ bool scope_any(bool pred) {
  if (kE == 32) return __any_sync(kFull, pred) != 0;
  return __syncthreads_or(pred) != 0;
}

template <int kE>
__device__ __forceinline__ void env_for_column(Env<1, kE>& e, Shared<kE>& S, int col, bool live) {
  e.v2 = reinterpret_cast<float2*>(S.state) + col;
  e.f = S.state + kV2Count * kE * 2 + col;
  e.fl = &S.floor;
  e.sub = 0;
  e.gsub = 0;
  e.gshift = 0;
  e.live = live;
  e.flags = 0;
  set_materials(e, S.mtab[S.wmat[col]], S.mtab[S.fmat[col]]);
}

// queue push: one shared-memory atomic per warp
template <int kE>
__device__ __forceinline__ void push(Shared<kE>& S, int parity, bool want, int item) {
  const unsigned m = __ballot_sync(kFull, want);
  if (m == 0) return;
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == 0) base = atomicAdd(&S.count[parity], __popc(m));
  base = __shfl_sync(kFull, base, 0);
  if (want) S.queue[base + __popc(m & ((1u << lane) - 1u))] = (unsigned short)item;
}

__device__ __forceinline__ int pair_slot(int b) { return b == LLL ? 0 : b == LLU ? 1 : b == RLL ? 2 : 3; }
__device__ __forceinline__ int partner_of(int b) { return (0x34F01 >> (4 * b)) & 0xF; }  // {LLU, LLL, -, RLU, RLL}

// stage 1 of a leg pair: true when the pair needs the full narrow phase.  Tests the cached axis first (a separating axis
// settles the pair: no collision, nothing else to do), then the bounding boxes.
template <int kE>
__device__ __noinline__ bool pole_pair_needs_work(int col, int A, int B) {
  Env<1, kE> e;
  env_for_column(e, shm<kE>(), col, true);
  const int cached = shm<kE>().axis[pair_slot(A) * kE + col];
  float2 PA[6], PB[6];
#pragma unroll
  for (int i = 0; i < 6; i++) PA[i] = V2(e, A * 6 + i);
#pragma unroll
  for (int i = 0; i < 6; i++) PB[i] = V2(e, B * 6 + i);
  const int own = cached < 6 ? A : B;
  const int k = cached < 6 ? cached : cached - 6;
  const float2 p0 = V2(e, own * 6 + k), p1 = V2(e, own * 6 + (k == 5 ? 0 : k + 1));
  const float2 edge = vsub(p1, p0);
  float2 axis = mk2(-edge.y, edge.x);
  const bool skip = (axis.x == 0.0f) && (axis.y == 0.0f);
  axis = vnormalize_fast(axis);
  float amn, amx, bmn, bmx;
  project6(PA, axis, amn, amx);
  project6(PB, axis, bmn, bmx);
  const bool overlapping = (amn < bmx) && (bmn < amx);
  if (!skip && !overlapping) return false;  // AxisChecks would return false at this axis
  float2 amin, amax, bmin, bmax;
  aabb6(PA, amin, amax);
  aabb6(PB, bmin, bmax);
  return aabb_hit(amin, amax, bmin, bmax);
}

// stage 1 of a floor pair: bounding boxes (the caller latches Collided, RigidBody.cs:73-76)
template <int kE>
__device__ __noinline__ bool floor_pair_needs_work(int col, int A) {
  Env<1, kE> e;
  env_for_column(e, shm<kE>(), col, true);
  float2 PA[6];
#pragma unroll
  for (int i = 0; i < 6; i++) PA[i] = V2(e, A * 6 + i);
  float2 amin, amax;
  aabb6(PA, amin, amax);
  return aabb_hit(amin, amax, e.fl->bb_min, e.fl->bb_max);
}

// RigidBody.StepLinearVelocity / StepAngularVelocity / Skeleton.Move / Rotate of one body (the first half of body_step), and
// the bounding-box test against the floor on the NEW vertices while they are still in registers (what floor_pair_needs_work
// would reload and recompute right afterwards for a floor-first walker)
template <int kE>
__device__ __noinline__ bool integrate_body_floor_test(int col, int b, float dt) {
  Env<1, kE> e;
  env_for_column(e, shm<kE>(), col, true);
  float2 v = V2(e, kV2Vel + b);
  v = vadd(v, vmul(mk2(0.0f, 980.0f), dt));
  const float2 d = vmul(v, dt);
  const float w = F1(e, kFOmega + b);
  const float theta = fmul(w, dt);
  float ang = fadd(F1(e, kFAngle + b), theta);
  const float PI_F = 3.14159274f, TAU_F = 6.28318548f;
  if (ang > PI_F) ang = fsub(ang, TAU_F);
  else if (ang < -PI_F) ang = fadd(ang, TAU_F);
  float m11, m12;
  rotz(theta, m11, m12);
  const float2 cen = vadd(V2(e, kV2Cen + b), d);
  float2 P[6];
#pragma unroll
  for (int i = 0; i < 6; i++) {
    float2 p = vadd(V2(e, b * 6 + i), d);
    p = vsub(p, cen);
    const float2 t = vrotate(p, m11, m12);
    P[i] = vadd(t, cen);
    V2(e, b * 6 + i) = P[i];
  }
  V2(e, kV2Cen + b) = cen;
  V2(e, kV2Vel + b) = v;
  F1(e, kFAngle + b) = ang;
  float2 amin, amax;
  aabb6(P, amin, amax);
  return aabb_hit(amin, amax, e.fl->bb_min, e.fl->bb_max);
}

// Joints: every thread runs Joint.Step for its OWN walker's four joints, in creation order, instead of three queue rounds.  A joint
// needs correcting in ~20 % of the substeps and its chain is short (~120 instructions), so a warp executes all four chains at
// 20 % lane density -- more issued instructions than the dense drain (+6 %), but three rounds (six barriers, three waits for
// the slowest warp) fewer per substep: 262144 walkers 4.26 -> 4.05 ms per env-step (profiles/ab_experiments_r2.log).  Two joints
// merged into one function, static joint indices and warp-level joint passes all measured slower, DESIGN §4.2.
template <int kE>
__device__ __noinline__ void joint_in_thread(int col, int k) {
  Env<1, kE> e;
  env_for_column(e, shm<kE>(), col, true);
  const int A = (0x4122 >> (4 * k)) & 0xF, B = (0x3041 >> (4 * k)) & 0xF;
  joint_step<Env<1, kE>, false>(e, A, k < 2 ? 1 : 2, B, k < 2 ? 4 : 3, nullptr);
}

enum { kItemPole = 0, kItemFloor = 1 };

// stage 2: the queued items, densely, kG lanes per item (the lanes split the SAT axes and the vertices of the moves exactly
// like the L > 1 layouts of the plain kernel; with ~15-20 % of the walkers queued per round this keeps most warps of the CTA
// busy and roughly halves the latency of the round).  Item = walker column | payload << 10.  Four lanes per floor item
// measured slower, DESIGN §4.2.
constexpr int kG = 2;

template <int G, int kE>
__device__ __forceinline__ void group_env_for_column(Env<G, kE>& e, Shared<kE>& S, int col, bool live) {
  e.v2 = reinterpret_cast<float2*>(S.state) + col;
  e.f = S.state + kV2Count * kE * 2 + col;
  e.fl = &S.floor;
  e.sub = threadIdx.x % G;
  e.gsub = e.sub;
  e.gshift = ((threadIdx.x & 31) / G) * G;
  e.live = live;
  e.flags = 0;
  set_materials(e, S.mtab[S.wmat[col]], S.mtab[S.fmat[col]]);
}

template <int KIND, int kE>
__device__ __noinline__ void drain(int parity) {
  Shared<kE>& S = shm<kE>();
  using EVG = Env<kG, kE>;
  const int count = S.count[parity];
  const int warp_base = (threadIdx.x >> 5) * (32 / kG), lane = threadIdx.x & 31;
#pragma unroll 1
  for (int base = warp_base; base < count; base += kE / kG) {
    const int slot = base + lane / kG;
    const bool valid = slot < count;
    const int item = valid ? S.queue[slot] : 0;
    const int col = item & 1023, payload = item >> 10;
    EVG q;
    group_env_for_column<kG, kE>(q, S, col, valid);
    // straight-line SAT rounds (BY_LAYOUT = false): 16 items share a warp, so an early stop (all of them separated) practically
    // never happens
    if (KIND == kItemPole) {
      int sep_axis = -1;
      resolve_pair<EVG, kG, false, false, false, true>(q, valid, payload, partner_of(payload), nullptr, &sep_axis);
      // the lane that saw the lowest separating axis of the group records it (any separating axis is a valid cache entry)
      if (valid && sep_axis >= 0) S.axis[pair_slot(payload) * kE + col] = (unsigned char)sep_axis;
    } else {
      resolve_pair<EVG, kG, false, true, false, true>(q, valid, payload, FLOOR, nullptr);
    }
  }
}

template <int kE>
__global__ void __launch_bounds__(kE, kE == 192 ? 3 : (kE == 160 ? 3 : 512 / kE)) physics_compact_kernel(const PhysicsParams p) {
  using EV = Env<1, kE>;
  Shared<kE>& S = shm<kE>();
  const int tid = threadIdx.x;
  const int env0 = blockIdx.x * kE;
  const int env = env0 + tid;
  const bool live = env < p.n;
  const int envc = live ? env : 0;

  for (int w = tid; w < (int)(sizeof(FloorConst) / 4); w += kE)
    reinterpret_cast<uint32_t*>(&S.floor)[w] = reinterpret_cast<const uint32_t*>(&c_floor)[w];
  // stage the CTA's records: every float2 slot of the device layout is ONE contiguous run of kE * 8 bytes (every float row kE * 4)
  // that lands in its shared-memory column as it is -- 49 bulk copies (cp.async.bulk, completion counted on an mbarrier) issued by
  // one thread, no register staging.  The rows are padded to whole CTAs (kEnvPad), so the runs are always complete.
  constexpr bool kBulk = (kE % 32 == 0) && (kEnvPad % kE == 0);
  if (kBulk) {
    if (tid == 0) {
      bulk::mbar_init(&S.stage_bar, 1);
      bulk::fence_mbar_init();
    }
    scope_sync<kE>();
    if (tid == 0) {
      bulk::mbar_expect_tx(&S.stage_bar, (uint32_t)(kStateSlots2 * kE * 8 + 10 * kE * 4));
#pragma unroll 1
      for (int s2 = 0; s2 < kStateSlots2; s2++) {  // record slot -> column slot (the Body's mirror slot, then centroids / velocities)
        const int col_slot = s2 < 17 ? s2 : (s2 < 29 ? s2 + 1 : (s2 < 34 ? kV2Cen + (s2 - 29) : kV2Vel + (s2 - 34)));
        bulk::load(S.state + (size_t)col_slot * kE * 2, p.state + ((size_t)s2 * p.n_pad + env0) * 2, kE * 8, &S.stage_bar);
      }
#pragma unroll 1
      for (int r = 0; r < 10; r++)
        bulk::load(S.state + (size_t)kV2Count * kE * 2 + (size_t)r * kE, p.state + (size_t)(78 + r) * p.n_pad + env0, kE * 4, &S.stage_bar);
    }
  } else {
#pragma unroll 1
    for (int f = 0; f < 88; f++)
      S.state[record_word<kE>(f) + (f < 78 ? 2 * tid : tid)] = live ? p.state[state_index(f, envc, p.n_pad)] : c_init_state[f];
  }
  for (int w = tid; w < (int)(sizeof(Material) * WB_MAX_MATERIALS / 4); w += kE)
    reinterpret_cast<uint32_t*>(S.mtab)[w] = reinterpret_cast<const uint32_t*>(c_materials)[w];
  S.wmat[tid] = p.walker_mat[envc];
  S.fmat[tid] = p.floor_mat[envc];
  {
    const uint32_t packed = (p.axis_cache != nullptr && live) ? p.axis_cache[env] : 0u;
#pragma unroll
    for (int s = 0; s < 4; s++) {
      const uint32_t a = (packed >> (8 * s)) & 0xFFu;
      S.axis[s * kE + tid] = (unsigned char)(a < 12u ? a : 0u);
    }
  }
  if (tid == 0) S.count[0] = S.count[1] = 0;
  if (kBulk) bulk::mbar_wait(&S.stage_bar, 0);  // the bulk copies have landed (the async proxy's writes are visible after the wait)
  scope_sync<kE>();  // the floor constants / counters written above are read by every thread of the scope
  EV e;
  env_for_column(e, S, tid, live);
  V2(e, BODY * 6 + 5) = V2(e, BODY * 6);
  float* torque_rows = p.state + (size_t)88 * p.n_pad + envc;
  e.flags = p.flags[envc];
  int steps = p.steps[envc];
  float2 pos = mk2(p.pos[envc], p.pos[p.n_pad + envc]);

  auto write_initial_record = [&]() {  // Walker.Reset + CreateCreature (own walker only: no synchronisation needed)
#pragma unroll 1
    for (int f = 0; f < 88; f++) S.state[record_word<kE>(f) + (f < 78 ? 2 * tid : tid)] = c_init_state[f];
    V2(e, BODY * 6 + 5) = V2(e, BODY * 6);
    for (int k = 0; k < 4; k++) torque_rows[(size_t)k * p.n_pad] = c_init_state[88 + k];
  };

  if (p.phases & kPhaseResetMasked) {
    if (live && (p.reset_mask == nullptr || p.reset_mask[envc])) {
      write_initial_record();
      e.flags = (p.phases & kPhaseFirstEpisode) ? 0 : WB_FLAG_FLOOR_FIRST;
      steps = 0;
      pos = V2(e, kV2Cen + BODY);
    }
  }
  if (p.phases & kPhaseIncSteps) steps++;
  if ((p.phases & kPhaseTakeActions) && live) {
    const float4 a4 = *reinterpret_cast<const float4*>(p.actions + (size_t)env * 4);
    const float act[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      float a = act[k];
      if (a >= 1.0f) a = 1.0f;
      else if (a <= -1.0f) a = -1.0f;
      const float change = fsub(a, torque_rows[(size_t)k * p.n_pad]);
      torque_rows[(size_t)k * p.n_pad] = a;
      const int bodyB = (k == 0) ? LLU : (k == 1) ? RLU : (k == 2) ? LLL : RLL;
      F1(e, kFOmega + bodyB) = fadd(F1(e, kFOmega + bodyB), fmul(change, 5.0f));
    }
  }

  if (p.phases & kPhaseStepObjects) {
    const float dt = fdiv(p.dt, (float)p.iterations);
    const bool floor_first = (e.flags & WB_FLAG_FLOOR_FIRST) != 0;
    // which floor sub-phases this CTA needs at all (the list order only changes at a reset, never inside the sweep)
    // padding threads (env >= n) sweep a scratch copy of the initial walker like everybody else -- no thread of the CTA ever
    // leaves the lockstep -- and simply never store anything to global memory
    const bool any_first = scope_any<kE>(floor_first);
    const bool any_last = scope_any<kE>(!floor_first);

    // one queue round: (stage 1 already pushed) barrier, drain, barrier; the other counter is cleared in between
    int parity = 0;
    WB_PROF_DECL;
    // (the clock read after a BAR.SYNC.DEFER_BLOCKING can issue before the warp really blocks, so waits are not measured around
    //  the barrier: every warp publishes its ARRIVAL time and afterwards charges (latest arrival - own arrival) as its wait)
    auto round = [&](auto drain_fn) {
#ifdef WB_PHASE_PROFILE
      const int pw = tid >> 5, nw = kE >> 5;
      long long t_arr0 = prof_clock();
      if ((tid & 31) == 0) S.prof_arrive[parity][0][pw] = t_arr0;
#endif
      // (the other counter was last read by the previous round's drain, which ended behind that round's second barrier: it can be
      //  cleared before this round's first barrier, and the next round's pushes find it cleared whether or not the second one runs)
      if (tid == 0) S.count[parity ^ 1] = 0;
      scope_sync<kE>();
#ifdef WB_PHASE_PROFILE
      long long last0 = 0;
      for (int w = 0; w < nw; w++) last0 = max(last0, S.prof_arrive[parity][0][w]);
      prof_acc[0] += (unsigned long long)(t_arr0 - prof_t);  // stage 1: from the end of the previous round to my arrival
      prof_acc[1] += (unsigned long long)(last0 - t_arr0);   // wait before the drain
      prof_items += S.count[parity];
      prof_rounds++;
#else
      if (S.count[parity] == 0) {  // nothing queued (the upper legs' floor round, most of the time): no drain, no second barrier
        parity ^= 1;
        return;
      }
#endif
      drain_fn();
#ifdef WB_PHASE_PROFILE
      long long t_arr1 = prof_clock();
      if ((tid & 31) == 0) S.prof_arrive[parity][1][pw] = t_arr1;
#endif
      scope_sync<kE>();
#ifdef WB_PHASE_PROFILE
      long long last1 = 0;
      for (int w = 0; w < nw; w++) last1 = max(last1, S.prof_arrive[parity][1][w]);
      prof_acc[2] += (unsigned long long)(t_arr1 - last0);  // drain: from the release of the first barrier to my arrival
      prof_acc[3] += (unsigned long long)(last1 - t_arr1);  // wait after the drain
      prof_t = last1;
#endif
      parity ^= 1;
    };

#pragma unroll 1
    for (int it = 0; it < p.iterations; it++) {
      for (int k = 0; k < 4; k++) joint_in_thread<kE>(tid, k);
      // ---- body sweep: {LLL, RLL, Body}, then {LLU, RLU}; per leg segment [floor if floor-first] [leg partner] [floor if
      //      floor-last].  The Body only ever meets the floor (Walker.cs:204-209), so its step is independent of both legs during
      //      the sweep: it is integrated with the first pair and its floor item rides in that pair's first floor round instead
      //      of costing a round of its own.
#pragma unroll 1
      for (int ph = 0; ph < 2; ph++) {
        const int b0 = ph == 0 ? LLL : LLU;
        const int b1 = ph == 0 ? RLL : RLU;
        bool body_pending = ph == 0;
        const bool hit0 = integrate_body_floor_test<kE>(tid, b0, dt);
        const bool hit1 = integrate_body_floor_test<kE>(tid, b1, dt);
        const bool hitb = body_pending && integrate_body_floor_test<kE>(tid, BODY, dt);  // (ph is uniform: no divergent call)
        if (any_first) {
          // (the upper legs' sparse floor round stays a queue round: resolving it in the owning warp measured slower, DESIGN §4.2)
          const bool f0 = floor_first && hit0, f1 = floor_first && hit1;
          e.flags |= (f0 ? 1 << b0 : 0) | (f1 ? 1 << b1 : 0);
          push(S, parity, f0, tid | (b0 << 10));
          push(S, parity, f1, tid | (b1 << 10));
          if (body_pending) {
            if (hitb) e.flags |= 1 << BODY;
            push(S, parity, hitb, tid | (BODY << 10));
            body_pending = false;
          }
          round([&] { drain<kItemFloor, kE>(parity); });
        }
        push(S, parity, pole_pair_needs_work<kE>(tid, b0, partner_of(b0)), tid | (b0 << 10));
        push(S, parity, pole_pair_needs_work<kE>(tid, b1, partner_of(b1)), tid | (b1 << 10));
        round([&] { drain<kItemPole, kE>(parity); });
        if (any_last) {
          const bool f0 = !floor_first && floor_pair_needs_work<kE>(tid, b0), f1 = !floor_first && floor_pair_needs_work<kE>(tid, b1);
          e.flags |= (f0 ? 1 << b0 : 0) | (f1 ? 1 << b1 : 0);
          push(S, parity, f0, tid | (b0 << 10));
          push(S, parity, f1, tid | (b1 << 10));
          if (body_pending) {  // (a CTA whose walkers are all floor-last)
            const bool fb = floor_pair_needs_work<kE>(tid, BODY);
            if (fb) e.flags |= 1 << BODY;
            push(S, parity, fb, tid | (BODY << 10));
            body_pending = false;
          }
          round([&] { drain<kItemFloor, kE>(parity); });
        }
      }
    }
#ifdef WB_PHASE_PROFILE
    if ((tid & 31) == 0) {
      for (int k = 0; k < 4; k++) atomicAdd(&g_prof[k], prof_acc[k]);
      atomicAdd(&g_prof[4], 1ull);
      if (tid == 0) {
        atomicAdd(&g_prof[5], prof_items);
        atomicAdd(&g_prof[6], prof_rounds);
      }
    }
#endif
  }

  if (p.phases & kPhaseObserve) {
    const float2 prev = pos;
    pos = V2(e, kV2Cen + BODY);
    if (e.flags & ((1 << BODY) | (1 << LLU) | (1 << RLU))) e.flags |= WB_FLAG_TERMINAL;
    const float dx = fsub(pos.x, prev.x);
    const float h = fdiv(V2(e, BODY * 6 + 1).y, 500.0f);
    float r = 0.0f;
    r = fadd(r, (dx > 0.0f && h < 1.6f) ? dx : 0.0f);
    r = fsub(r, (h > 1.65f) ? -0.1f : 0.0f);
    bool terminal = false;
    if ((e.flags & WB_FLAG_TERMINAL) || steps > p.max_timesteps) {
      if (e.flags & WB_FLAG_TERMINAL) r = fsub(r, 40.0f);
      terminal = true;
    }
    if (pos.x > 900.0f) {
      r = fadd(r, 80.0f);
      terminal = true;
    }
    if (live && terminal && (p.phases & kPhaseAutoReset)) {
      write_initial_record();
      e.flags = WB_FLAG_FLOOR_FIRST;
      steps = 0;
      pos = V2(e, kV2Cen + BODY);
    }
    if (live) {
      store_observation(e, p.obs + (size_t)env * WB_OBS);
      p.reward[env] = r;
      p.done[env] = terminal ? 1 : 0;
    }
  } else if (p.phases & kPhaseObsOnly) {
    if (live) store_observation(e, p.obs + (size_t)env * WB_OBS);
  }

  if (live) {
    p.flags[env] = e.flags;
    p.steps[env] = steps;
    p.pos[env] = pos.x;
    p.pos[p.n_pad + env] = pos.y;
    if (p.axis_cache != nullptr)
      p.axis_cache[env] = (uint32_t)S.axis[tid] | ((uint32_t)S.axis[kE + tid] << 8) | ((uint32_t)S.axis[2 * kE + tid] << 16) |
                          ((uint32_t)S.axis[3 * kE + tid] << 24);
    if (!kBulk) {
#pragma unroll 8
      for (int f = 0; f < 88; f++) p.state[state_index(f, env, p.n_pad)] = S.state[record_word<kE>(f) + (f < 78 ? 2 * tid : tid)];
    }
  }
  if (kBulk) {
    // write the records back the way they came: bulk stores shared -> global (the pad walkers of a ragged last CTA are real
    // walkers in the padding of the rows; they never receive actions and are never read)
    bulk::fence_proxy_async();  // this thread's generic-proxy writes to the columns -> visible to the async proxy
    scope_sync<kE>();
    if (tid == 0) {
#pragma unroll 1
      for (int s2 = 0; s2 < kStateSlots2; s2++) {
        const int col_slot = s2 < 17 ? s2 : (s2 < 29 ? s2 + 1 : (s2 < 34 ? kV2Cen + (s2 - 29) : kV2Vel + (s2 - 34)));
        bulk::store(p.state + ((size_t)s2 * p.n_pad + env0) * 2, S.state + (size_t)col_slot * kE * 2, kE * 8);
      }
#pragma unroll 1
      for (int r = 0; r < 10; r++)
        bulk::store(p.state + (size_t)(78 + r) * p.n_pad + env0, S.state + (size_t)kV2Count * kE * 2 + (size_t)r * kE, kE * 4);
      bulk::commit_and_wait_reads();  // shared memory must outlive the reads of the bulk stores
    }
  }
}

template <int kE>
static cudaError_t launch_compact(const PhysicsParams& p, cudaStream_t stream) {
  // opt in to > 48 KB of dynamic shared memory: a per-DEVICE function attribute (a process may drive several GPUs)
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(physics_compact_kernel<kE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Shared<kE>));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(physics_compact_kernel<kE>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    if (getenv("WB_DEBUG_OCCUPANCY")) {
      int nb = 0;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, physics_compact_kernel<kE>, kE, sizeof(Shared<kE>));
      fprintf(stderr, "physics_compact_kernel<%d>: %d CTAs/SM, %zu B shared per CTA\n", kE, nb, sizeof(Shared<kE>));
    }
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  physics_compact_kernel<kE><<<(p.n + kE - 1) / kE, kE, sizeof(Shared<kE>), stream>>>(p);
  return cudaGetLastError();
}

}  // namespace pc

#ifdef WB_PHASE_PROFILE
extern "C" int wb_prof_read(unsigned long long* out24, int reset) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out24, pl::g_prof, sizeof(unsigned long long) * 24) != cudaSuccess) return 1;
  if (reset) {
    unsigned long long z[24] = {};
    cudaMemcpyToSymbol(pl::g_prof, z, sizeof(z));
  }
  return 0;
}
// the lanes kernel's last launch: 3 cycle counts per CTA for the first `ctas` CTAs (pl::g_lanes_prof)
extern "C" int wb_lanes_prof_read(unsigned long long* out, int ctas) {
  if (ctas < 0 || ctas > pl::kLanesProfCtas) return 1;
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(out, pl::g_lanes_prof, sizeof(unsigned long long) * 3 * ctas) != cudaSuccess;
}
#endif

// ---------------------------------------------------------------- host side
cudaError_t upload_materials(const Material* table, int count) {
  return cudaMemcpyToSymbol(pl::c_materials, table, sizeof(Material) * count);
}

cudaError_t upload_scene_constants(const float* init_state92, const FloorConst* floor) {
  cudaError_t e = cudaMemcpyToSymbol(pl::c_init_state, init_state92, sizeof(float) * kStateFloats);
  if (e != cudaSuccess) return e;
  return cudaMemcpyToSymbol(pl::c_floor, floor, sizeof(FloorConst));
}

// variant code = lanes per environment (1, 2, 4, 8, 16; for >= 2 the lanes split by leg first), 100 + lanes (4, 8, 16) for
// the measured-for-comparison layout without the leg split (all lanes of a walker work on one pair), or 1001 = one thread
// per walker with work compaction over a lockstep scope of 256 walkers (the throughput kernel; 1002 / 1003: scope of one warp /
// of 128 walkers, kept for comparison)
bool physics_lanes_supported(int variant) {
  switch (variant) {
    case 1: case 2: case 4: case 8: case 16: case 32: case 104: case 108: case 116: case 1001: case 1002: case 1003: case 1004: case 1005: return true;
    default: return false;
  }
}

cudaError_t launch_physics(const PhysicsParams& p, int variant, bool trace, cudaStream_t stream) {
  switch (variant) {
    case 1: return pl::launch_l<1, 1>(p, trace, stream);
    case 2: return pl::launch_l<2, 2>(p, trace, stream);
    case 4: return pl::launch_l<4, 2>(p, trace, stream);
    case 8: return pl::launch_l<8, 2>(p, trace, stream);
    case 16: return pl::launch_l<16, 2>(p, trace, stream);
    case 32: return pl::launch_l<32, 2>(p, trace, stream);
    case 104: return pl::launch_l<4, 1>(p, trace, stream);
    case 108: return pl::launch_l<8, 1>(p, trace, stream);
    case 116: return pl::launch_l<16, 1>(p, trace, stream);
    // compacting kernels (the trace hook uses the plain kernel): lockstep scope of 256 walkers (default), one warp, 128 walkers
    case 1001: return trace ? pl::launch_l<1, 1>(p, true, stream) : pc::launch_compact<256>(p, stream);
    case 1002: return trace ? pl::launch_l<1, 1>(p, true, stream) : pc::launch_compact<32>(p, stream);
    case 1003: return trace ? pl::launch_l<1, 1>(p, true, stream) : pc::launch_compact<128>(p, stream);
    case 1004: return trace ? pl::launch_l<1, 1>(p, true, stream) : pc::launch_compact<192>(p, stream);
    case 1005: return trace ? pl::launch_l<1, 1>(p, true, stream) : pc::launch_compact<160>(p, stream);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_rcp_sqrt_check(uint32_t first, uint64_t count, unsigned long long* mismatches_dev, uint32_t* first_bad_dev,
                                  cudaStream_t stream) {
  pl::rcp_sqrt_check_kernel<<<148 * 8, 256, 0, stream>>>(first, count, mismatches_dev, first_bad_dev);
  return cudaGetLastError();
}

cudaError_t launch_rotz_debug(const float* radians, int n, int mode, float* c_out, float* s_out, cudaStream_t stream) {
  pl::rotz_debug_kernel<<<(n + 255) / 256, 256, 0, stream>>>(radians, n, mode, c_out, s_out);
  return cudaGetLastError();
}

}  // namespace wb

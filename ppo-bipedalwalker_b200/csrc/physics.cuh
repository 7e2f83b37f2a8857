// physics.cuh -- shared declarations between the physics kernel (physics_lanes.cu) and the C ABI (api_env.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/walker_b200.h"

namespace wb {

constexpr int kEnvPad = 256;      // the SoA rows are padded to a multiple of 256 environments: one lockstep CTA of the compacting
                                  // kernel always moves whole 2 KB / 1 KB row segments with bulk copies (pad walkers are real, idle walkers)
constexpr int kStateFloats = WB_STATE_FLOATS;

// Device layout of the state record (structure of arrays over walkers, x/y of one point adjacent):
//   float2 slot s = 0..38 (29 vertices, 5 cached centroids, 5 linear velocities = record floats 2s, 2s+1):  state2[s][n_pad]
//   float rows 78..91 (angular velocities, tracked angles, joint torques):                                state[f][n_pad]
// A walker's (x, y) pairs sit next to each other, so a row segment of a CTA's walkers lands in the kernels' shared-memory
// columns ([slot][walker] float2) with ONE contiguous copy -- cp.async.bulk in the compacting kernel.
__host__ __device__ inline size_t state_index(int f, size_t env, size_t n_pad) {
  return f < 78 ? ((size_t)(f >> 1) * n_pad + env) * 2 + (size_t)(f & 1) : (size_t)f * n_pad + env;
}
constexpr int kStateSlots2 = 39;  // float2 slots of the record

struct Material {
  float inverse_mass, restitution, friction;
};

// phases of one launch (a fused env-step sets all of the first five)
enum : int {
  kPhaseIncSteps = 1,      // Environment.Update: _steps++            (Environment.cs:72)
  kPhaseTakeActions = 2,   // Matrix.Clip + Walker.TakeActions         (Environment.cs:78)
  kPhaseStepObjects = 4,   // Environment.StepObjects                  (Environment.cs:126-143)
  kPhaseObserve = 8,       // Walker.Update + reward/terminal/GetState (Environment.cs:101-121)
  kPhaseAutoReset = 16,    // Reset + InitialState after a terminal    (Environment.cs:91,157-180)
  kPhaseObsOnly = 32,      // Walker.GetState only
  kPhaseResetMasked = 64,  // wb_env_reset: reset envs with mask != 0
  kPhaseFirstEpisode = 128 // with kPhaseResetMasked: constructor list order (floor last)
};

struct PhysicsParams {
  float* state;        // the record in the device layout above (state_index)
  int32_t* flags;      // [n_pad]
  int32_t* steps;      // [n_pad]
  float* pos;          // [2][n_pad]  Walker._position (Walker.cs:19)
  const uint8_t* floor_mat;   // [n_pad]
  const uint8_t* walker_mat;  // [n_pad]
  uint32_t* axis_cache;       // [n_pad] or null: the compacting kernel's last separating axis per ordered leg pair (4 x 8 bits),
                              // carried from launch to launch (a hint only: any value 0..11 is a legal first axis to test)
  const float* actions;       // [n][4]
  const uint8_t* reset_mask;  // [n] or null
  float* obs;          // [n][12]
  float* reward;       // [n]
  uint8_t* done;       // [n]
  wb_pair_trace* pair_trace;   // [n][iterations][9] or null
  wb_joint_trace* joint_trace; // [n][iterations][4] or null
  int32_t n, n_pad;
  float dt;            // frame delta (divided by iterations inside, Environment.cs:128)
  int32_t iterations;
  int32_t max_timesteps;
  int32_t phases;
};

// Environment.CreateFloor (Environment.cs:211-226) and everything about the static floor that never changes, computed once
// on the host with the reference's formulas (strict fp32): vertices, cached centroid, bounding box, the normalised left
// normals of its edges (SATCollision.cs:43-46) and its own projection onto each of them (SATCollision.cs:63-76)
struct FloorConst {
  float2 v[4];
  float2 cen;
  float2 bb_min, bb_max;
  float2 axis[4];
  float pmin[4], pmax[4];
  int32_t skip[4];  // axis == Vector2.Zero: skipped by AxisChecks
};

// host-side helpers implemented in physics_lanes.cu
cudaError_t upload_materials(const Material* table, int count);
cudaError_t upload_scene_constants(const float* init_state92, const FloorConst* floor);
bool physics_lanes_supported(int lanes_per_env);
cudaError_t launch_physics(const PhysicsParams& p, int lanes_per_env, bool trace, cudaStream_t stream);
cudaError_t launch_rotz_debug(const float* radians, int n, int mode, float* c_out, float* s_out, cudaStream_t stream);
cudaError_t launch_rcp_sqrt_check(uint32_t first, uint64_t count, unsigned long long* mismatches_dev, uint32_t* first_bad_dev,
                                  cudaStream_t stream);

// ---- general scenes (physics_scene.cu): any list of convex polygons + joints, N lockstep copies
constexpr int kSceneMaxBodies = 16, kSceneMaxVerts = 16, kSceneMaxJoints = 16;
struct SceneConst {
  int32_t n_bodies, n_joints, total_verts, pad;
  int32_t n_verts[kSceneMaxBodies], vert_offset[kSceneMaxBodies], is_static[kSceneMaxBodies], is_floor[kSceneMaxBodies];
  uint32_t assoc[kSceneMaxBodies];  // bit j: body j is on this body's "no collide" list (RigidBody.cs:143-152)
  float inv_mass[kSceneMaxBodies], inv_inertia[kSceneMaxBodies], restitution[kSceneMaxBodies], friction[kSceneMaxBodies];
  float accel_x[kSceneMaxBodies], accel_y[kSceneMaxBodies];
  int32_t joint_a[kSceneMaxJoints], joint_ia[kSceneMaxJoints], joint_b[kSceneMaxJoints], joint_ib[kSceneMaxJoints];
};
struct SceneParams {
  float* state;          // [rows][n_pad]: 2*total_verts vertex floats, 2B centroids, 2B velocities, B omega, B angle, J torques
  int32_t* collided;     // [n_pad] bit per body
  const float* torques;  // [n][J] or null
  int32_t n, n_pad;
  float dt;
  int32_t iterations;    // 0: no StepObjects (SetTorque only)
};
size_t scene_smem_bytes(const SceneConst& s);
cudaError_t launch_scene(const SceneParams& p, const SceneConst& s, cudaStream_t stream);

// ---- the walker on arbitrary terrain (physics_scene.cu: terrain_step_kernel): bodies [LLL, LLU, Body, RLL, RLU, terrain...]
constexpr int kWalkerRecordInit = 68;  // the fresh walker's 29 vertices + 5 cached centroids (floats 0..67 of the 92-float record)
struct TerrainConst {
  SceneConst topo;
  float walker_init[kWalkerRecordInit];
};
struct TerrainParams {
  float* state;               // [rows][n_pad]: the SceneParams record over all bodies, then the 4 joint torques
  int32_t* ints;              // [3][n_pad]: Collided bit per body index, flags (WB_FLAG_TERMINAL, WB_FLAG_FLOOR_FIRST), steps
  const float* actions;       // [n][4]
  const uint8_t* reset_mask;  // [n] or null
  float* obs;                 // [n][12]
  float* reward;              // [n]
  uint8_t* done;              // [n]
  int32_t n, n_pad;
  float dt;
  int32_t iterations, max_timesteps;
  int32_t phases;             // kPhase* as PhysicsParams
};
cudaError_t terrain_kernel_setup();
cudaError_t launch_terrain(const TerrainConst& tc, const TerrainParams& p, cudaStream_t stream);
// Walker ctor + CreateCreature (api_env.cu): the 92-float record wb_env_create starts every walker from
void walker_initial_record(float* init92);

}  // namespace wb

// api_scene.cu -- C ABI for general scenes (include/walker_b200.h, wb_scene_*): the reference's IObject plugin surface
// (Objects/IObject.cs:7-10; Objects/RigidBodies/{Square,Triangle,Hexagon,Pole,Hull,Joint}.cs) for N lockstep copies of an
// arbitrary list of convex polygons and joints.  All compute is in physics_scene.cu; there is no CPU path.
#include <new>
#include <vector>

#include "common.h"
#include "physics.cuh"

using namespace wb;

struct wb_scene {
  int32_t n = 0, n_pad = 0;
  int32_t iterations = 50;
  int32_t rows = 0;  // state floats per copy
  SceneConst sc{};
  cudaStream_t stream = nullptr;
  float* d_state = nullptr;     // [rows][n_pad]
  int32_t* d_collided = nullptr;
  float* d_torques = nullptr;   // [n][J]
  int64_t launches = 0;
};

// strict-fp32 host arithmetic (volatile stores keep every intermediate in binary32)
static inline float f_add(float a, float b) { volatile float r = a + b; return r; }
static inline float f_mul(float a, float b) { volatile float r = a * b; return r; }
static inline float f_div(float a, float b) { volatile float r = a / b; return r; }

extern "C" {

// wb_body_desc / wb_joint_desc lists -> the kernels' topology (RigidBody ctor, RigidBody.cs:36-50; Joint ctor, Joint.cs:20-28)
static int32_t build_topology(const wb_body_desc* bodies, int32_t n_bodies, const wb_joint_desc* joints, int32_t n_joints, SceneConst& c) {
  c = SceneConst{};
  c.n_bodies = n_bodies;
  c.n_joints = n_joints;
  int off = 0;
  for (int b = 0; b < n_bodies; b++) {
    const wb_body_desc& d = bodies[b];
    if (d.n_vertices < 3 || d.n_vertices > kSceneMaxVerts) return fail(WB_ERR_INVALID, "body %d: a polygon has 3..16 vertices", b);
    float im, e, mu;
    if (wb_material_get(d.material, &im, &e, &mu) != WB_OK)
      return fail(WB_ERR_INVALID, "body %d uses an unregistered material id %d", b, d.material);
    c.n_verts[b] = d.n_vertices;
    c.vert_offset[b] = off;
    off += d.n_vertices;
    c.is_static[b] = d.is_static != 0;
    c.is_floor[b] = d.is_floor != 0;
    c.assoc[b] = d.associated_mask;
    // RigidBody ctor, RigidBody.cs:36-50: static => inverse mass = inverse inertia = 0; else 0.001 * inverse mass (or the override)
    c.inv_mass[b] = d.is_static ? 0.0f : im;
    c.inv_inertia[b] = d.is_static ? 0.0f : (d.inverse_inertia >= 0.0f ? d.inverse_inertia : f_mul(0.001f, im));
    c.restitution[b] = e;
    c.friction[b] = mu;
    c.accel_x[b] = d.accel_x;
    c.accel_y[b] = d.accel_y;
  }
  c.total_verts = off;
  for (int k = 0; k < n_joints; k++) {
    const wb_joint_desc& j = joints[k];
    const bool ok = j.body_a >= 0 && j.body_a < n_bodies && j.body_b >= 0 && j.body_b < n_bodies && j.vertex_a >= 0 &&
                    j.vertex_a < c.n_verts[j.body_a] && j.vertex_b >= 0 && j.vertex_b < c.n_verts[j.body_b];
    if (!ok) return fail(WB_ERR_INVALID, "joint %d references a body / vertex that does not exist", k);
    c.joint_a[k] = j.body_a;
    c.joint_ia[k] = j.vertex_a;
    c.joint_b[k] = j.body_b;
    c.joint_ib[k] = j.vertex_b;
  }
  return WB_OK;
}

// Skeleton.FindCentroid (sum, then multiply by 1f / count, Skeleton.cs:100-113) of bodies [b0, b1) -> out[2 * (b - b0) ...]
static void centroids_of(const SceneConst& c, const float* vertices_xy, int b0, int b1, float* out) {
  for (int b = b0; b < b1; b++) {
    float sx = 0.0f, sy = 0.0f;
    for (int i = 0; i < c.n_verts[b]; i++) {
      sx = f_add(sx, vertices_xy[2 * (c.vert_offset[b] - c.vert_offset[b0] + i)]);
      sy = f_add(sy, vertices_xy[2 * (c.vert_offset[b] - c.vert_offset[b0] + i) + 1]);
    }
    const float factor = f_div(1.0f, (float)c.n_verts[b]);
    out[2 * (b - b0)] = f_mul(sx, factor);
    out[2 * (b - b0) + 1] = f_mul(sy, factor);
  }
}

int32_t wb_scene_create(int32_t n_envs, const wb_body_desc* bodies, int32_t n_bodies, const float* vertices_xy, const wb_joint_desc* joints,
                        int32_t n_joints, int32_t iterations, wb_scene** out) {
  WB_REQUIRE(out, "out is null");
  *out = nullptr;
  WB_REQUIRE(n_envs > 0 && bodies && vertices_xy, "bad argument");
  WB_REQUIRE(n_bodies > 0 && n_bodies <= kSceneMaxBodies, "a scene holds 1..16 bodies");
  WB_REQUIRE(n_joints >= 0 && n_joints <= kSceneMaxJoints && (n_joints == 0 || joints), "a scene holds 0..16 joints");
  WB_REQUIRE(iterations > 0 && iterations < 200, "iterations must be in (0, 200)");  // Hyperparameters.cs:189-217
  if (int32_t rc = require_device()) return rc;
  wb_scene* s = new (std::nothrow) wb_scene();
  WB_REQUIRE(s, "out of host memory");
  s->n = n_envs;
  s->n_pad = (n_envs + kEnvPad - 1) / kEnvPad * kEnvPad;
  s->iterations = iterations;
  SceneConst& c = s->sc;
  if (int32_t rc = build_topology(bodies, n_bodies, joints, n_joints, c)) {
    delete s;
    return rc;
  }
  if (scene_smem_bytes(c) > 200 * 1024) {
    delete s;
    return fail(WB_ERR_UNSUPPORTED, "scene too large for one SM's shared memory (%zu bytes per 32 copies)", scene_smem_bytes(c));
  }
  s->rows = 2 * c.total_verts + 4 * n_bodies + 2 * n_bodies + n_joints;
  // one copy of the initial state: vertices, cached centroids, zeros
  std::vector<float> one((size_t)s->rows, 0.0f);
  for (int i = 0; i < 2 * c.total_verts; i++) one[i] = vertices_xy[i];
  centroids_of(c, vertices_xy, 0, n_bodies, one.data() + 2 * c.total_verts);
  std::vector<float> all((size_t)s->rows * s->n_pad);
  for (int r = 0; r < s->rows; r++)
    for (int i = 0; i < s->n_pad; i++) all[(size_t)r * s->n_pad + i] = one[r];
  cudaError_t e = cudaMalloc(&s->d_state, sizeof(float) * all.size());
  if (e == cudaSuccess) e = cudaMalloc(&s->d_collided, sizeof(int32_t) * s->n_pad);
  if (e == cudaSuccess) e = cudaMalloc(&s->d_torques, sizeof(float) * (size_t)s->n * (n_joints > 0 ? n_joints : 1));
  if (e == cudaSuccess) e = cudaMemcpy(s->d_state, all.data(), sizeof(float) * all.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(s->d_collided, 0, sizeof(int32_t) * s->n_pad);
  if (e != cudaSuccess) {  // nothing leaks behind a failed create
    wb_scene_destroy(s);
    return fail(WB_ERR_CUDA, "wb_scene_create: %s", cudaGetErrorString(e));
  }
  *out = s;
  return WB_OK;
}

int32_t wb_scene_destroy(wb_scene* s) {
  if (!s) return WB_OK;
  cudaFree(s->d_state);
  cudaFree(s->d_collided);
  cudaFree(s->d_torques);
  delete s;
  return WB_OK;
}

int32_t wb_scene_set_stream(wb_scene* s, void* cuda_stream) {
  WB_REQUIRE(s, "scene is null");
  s->stream = (cudaStream_t)cuda_stream;
  return WB_OK;
}

int32_t wb_scene_state_floats(const wb_scene* s, int32_t* per_copy_out) {
  WB_REQUIRE(s && per_copy_out, "null argument");
  *per_copy_out = s->rows;
  return WB_OK;
}

int32_t wb_scene_set_state(wb_scene* s, const float* state_host, const int32_t* collided_host) {
  WB_REQUIRE(s && state_host, "null argument");
  WB_CUDA(cudaMemcpy2DAsync(s->d_state, sizeof(float) * s->n_pad, state_host, sizeof(float) * s->n, sizeof(float) * s->n, s->rows,
                            cudaMemcpyHostToDevice, s->stream));
  if (collided_host) WB_CUDA(cudaMemcpyAsync(s->d_collided, collided_host, sizeof(int32_t) * s->n, cudaMemcpyHostToDevice, s->stream));
  WB_CUDA(cudaStreamSynchronize(s->stream));
  return WB_OK;
}

int32_t wb_scene_get_state(wb_scene* s, float* state_host, int32_t* collided_host) {
  WB_REQUIRE(s && state_host, "null argument");
  WB_CUDA(cudaMemcpy2DAsync(state_host, sizeof(float) * s->n, s->d_state, sizeof(float) * s->n_pad, sizeof(float) * s->n, s->rows,
                            cudaMemcpyDeviceToHost, s->stream));
  if (collided_host) WB_CUDA(cudaMemcpyAsync(collided_host, s->d_collided, sizeof(int32_t) * s->n, cudaMemcpyDeviceToHost, s->stream));
  WB_CUDA(cudaStreamSynchronize(s->stream));
  return WB_OK;
}

static int32_t scene_launch(wb_scene* s, const float* d_torques, float dt, int iterations) {
  SceneParams p{};
  p.state = s->d_state;
  p.collided = s->d_collided;
  p.torques = d_torques;
  p.n = s->n;
  p.n_pad = s->n_pad;
  p.dt = dt;
  p.iterations = iterations;
  WB_CUDA(launch_scene(p, s->sc, s->stream));
  s->launches++;
  return WB_OK;
}

int32_t wb_scene_set_torques(wb_scene* s, const float* torques_host) {
  WB_REQUIRE(s && torques_host, "null argument");
  WB_REQUIRE(s->sc.n_joints > 0, "the scene has no joints");
  WB_CUDA(cudaMemcpyAsync(s->d_torques, torques_host, sizeof(float) * (size_t)s->n * s->sc.n_joints, cudaMemcpyHostToDevice, s->stream));
  if (int32_t rc = scene_launch(s, s->d_torques, 0.0f, 0)) return rc;
  WB_CUDA(cudaStreamSynchronize(s->stream));
  return WB_OK;
}

int32_t wb_scene_step_objects(wb_scene* s, float delta_time) {
  WB_REQUIRE(s, "scene is null");
  if (int32_t rc = scene_launch(s, nullptr, delta_time, s->iterations)) return rc;
  WB_CUDA(cudaStreamSynchronize(s->stream));
  return WB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ the walker on arbitrary terrain (wb_terrain_env_*)
// Environment with Hyperparameters.RoughFloor (Hyperparameters.cs:88, Environment.CreateRoughFloor, Environment.cs:230-261) or any
// other list of IObjects in place of the flat floor: scene = [LLL, LLU, Body, RLL, RLU] (Walker.CreateCreature) + terrain bodies,
// stepped by terrain_step_kernel (physics_scene.cu), one launch per env-step.
namespace {
constexpr int kTerrainMax = kSceneMaxBodies - 5;
constexpr int kTerrainInts = 3;
}  // namespace

struct wb_terrain_env {
  int32_t n = 0, n_pad = 0;
  int32_t rows = 0;           // state floats per copy
  int32_t terrain_verts = 0;  // vertices of all terrain bodies
  wb_hyperparams hp{};
  TerrainConst tc{};
  cudaStream_t stream = nullptr;
  float* d_state = nullptr;   // [rows][n_pad]
  int32_t* d_ints = nullptr;  // [3][n_pad]
  float* d_actions = nullptr;
  float* d_obs = nullptr;
  float* d_reward = nullptr;
  uint8_t* d_done = nullptr;
  uint8_t* d_mask = nullptr;
  int64_t launches = 0;
};

static int32_t terrain_launch(wb_terrain_env* env, int phases, float dt, const float* d_actions, const uint8_t* d_mask, float* d_obs,
                              float* d_reward, uint8_t* d_done) {
  TerrainParams p{};
  p.state = env->d_state;
  p.ints = env->d_ints;
  p.actions = d_actions;
  p.reset_mask = d_mask;
  p.obs = d_obs;
  p.reward = d_reward;
  p.done = d_done;
  p.n = env->n;
  p.n_pad = env->n_pad;
  p.dt = dt;
  p.iterations = env->hp.iterations;
  p.max_timesteps = env->hp.max_timesteps;
  p.phases = phases;
  WB_CUDA(launch_terrain(env->tc, p, env->stream));
  env->launches++;
  return WB_OK;
}

extern "C" {

int32_t wb_terrain_env_create(int32_t n_envs, const wb_body_desc* terrain, int32_t n_terrain, const float* vertices_xy,
                              int32_t walker_material, const wb_hyperparams* hp, wb_terrain_env** out) {
  WB_REQUIRE(out, "out is null");
  *out = nullptr;
  WB_REQUIRE(n_envs > 0 && terrain && vertices_xy, "bad argument");
  WB_REQUIRE(n_terrain > 0, "a terrain holds at least one body");
  if (n_terrain > kTerrainMax)
    return fail(WB_ERR_UNSUPPORTED, "the walker's 5 bodies plus %d terrain bodies exceed the %d bodies of a scene", n_terrain, kSceneMaxBodies);
  if (int32_t rc = require_device()) return rc;
  wb_hyperparams h{};
  if (hp) h = *hp; else wb_hyperparams_default(&h);
  WB_REQUIRE(h.iterations > 0 && h.iterations < 200, "iterations must be in (0, 200)");  // Hyperparameters.cs:189-217
  // Walker.CreateBodies / CreateJoints / AddAssociatedBodies / AddAcceleration (Walker.cs:155-209): bodies in the order they join
  // Environment._rigidBodies, association masks over those indices; the terrain's masks are over the terrain list
  const wb_body_desc walker[5] = {
      {6, 0, 0, walker_material, 0x1Cu, 0.0f, 980.0f, -1.0f},     // LLL: {RLU, RLL, Body}
      {6, 0, 0, walker_material, 0x1Cu, 0.0f, 980.0f, -1.0f},     // LLU: {RLU, RLL, Body}
      {5, 0, 0, walker_material, 0x1Bu, 0.0f, 980.0f, 0.0003f},   // Body: {LLU, RLU, LLL, RLL}; SetInverseInertia(0.0003f), Walker.cs:168
      {6, 0, 0, walker_material, 0x07u, 0.0f, 980.0f, -1.0f},     // RLL: {LLU, LLL, Body}
      {6, 0, 0, walker_material, 0x07u, 0.0f, 980.0f, -1.0f}};    // RLU: {LLU, LLL, Body}
  const wb_joint_desc joints[4] = {{2, 1, 1, 4}, {2, 1, 4, 4}, {1, 2, 0, 3}, {4, 2, 3, 3}};  // Walker.cs:182-187
  wb_body_desc all[kSceneMaxBodies];
  for (int b = 0; b < 5; b++) all[b] = walker[b];
  for (int t = 0; t < n_terrain; t++) {
    if (terrain[t].associated_mask >> n_terrain)
      return fail(WB_ERR_INVALID, "terrain body %d is associated with a body outside the terrain list", t);
    all[5 + t] = terrain[t];
    all[5 + t].associated_mask = terrain[t].associated_mask << 5;
  }
  wb_terrain_env* env = new (std::nothrow) wb_terrain_env();
  WB_REQUIRE(env, "out of host memory");
  env->n = n_envs;
  env->n_pad = (n_envs + kEnvPad - 1) / kEnvPad * kEnvPad;
  env->hp = h;
  SceneConst& c = env->tc.topo;
  const int nb = 5 + n_terrain;
  if (int32_t rc = build_topology(all, nb, joints, 4, c)) {
    delete env;
    return rc;
  }
  float init92[WB_STATE_FLOATS];
  walker_initial_record(init92);
  for (int i = 0; i < kWalkerRecordInit; i++) env->tc.walker_init[i] = init92[i];
  const int wv = c.vert_offset[5];  // 29
  env->terrain_verts = c.total_verts - wv;
  env->rows = 2 * c.total_verts + 6 * nb + 4;
  // one copy of the constructor state (Environment.cs:39-51): walker as wb_env_create builds it, terrain as given
  std::vector<float> one((size_t)env->rows, 0.0f);
  for (int i = 0; i < 2 * wv; i++) one[i] = init92[i];
  for (int i = 0; i < 2 * env->terrain_verts; i++) one[2 * wv + i] = vertices_xy[i];
  for (int i = 0; i < 10; i++) one[2 * c.total_verts + i] = init92[2 * wv + i];
  centroids_of(c, vertices_xy, 5, nb, one.data() + 2 * c.total_verts + 10);
  std::vector<float> rep((size_t)env->rows * env->n_pad);
  for (int r = 0; r < env->rows; r++)
    for (int i = 0; i < env->n_pad; i++) rep[(size_t)r * env->n_pad + i] = one[r];
  const size_t np = (size_t)env->n_pad;
  cudaError_t e = terrain_kernel_setup();
  if (e == cudaSuccess) e = cudaMalloc(&env->d_state, sizeof(float) * rep.size());
  if (e == cudaSuccess) e = cudaMalloc(&env->d_ints, sizeof(int32_t) * kTerrainInts * np);
  if (e == cudaSuccess) e = cudaMalloc(&env->d_actions, sizeof(float) * WB_ACT * np);
  if (e == cudaSuccess) e = cudaMalloc(&env->d_obs, sizeof(float) * WB_OBS * np);
  if (e == cudaSuccess) e = cudaMalloc(&env->d_reward, sizeof(float) * np);
  if (e == cudaSuccess) e = cudaMalloc(&env->d_done, np);
  if (e == cudaSuccess) e = cudaMalloc(&env->d_mask, np);
  if (e == cudaSuccess) e = cudaMemcpy(env->d_state, rep.data(), sizeof(float) * rep.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(env->d_ints, 0, sizeof(int32_t) * kTerrainInts * np);  // walker first, nothing collided, steps 0
  if (e != cudaSuccess) {
    wb_terrain_env_destroy(env);
    return fail(WB_ERR_CUDA, "wb_terrain_env_create: %s", cudaGetErrorString(e));
  }
  *out = env;
  return WB_OK;
}

int32_t wb_terrain_env_destroy(wb_terrain_env* env) {
  if (!env) return WB_OK;
  cudaFree(env->d_state);
  cudaFree(env->d_ints);
  cudaFree(env->d_actions);
  cudaFree(env->d_obs);
  cudaFree(env->d_reward);
  cudaFree(env->d_done);
  cudaFree(env->d_mask);
  delete env;
  return WB_OK;
}

int32_t wb_terrain_env_set_stream(wb_terrain_env* env, void* cuda_stream) {
  WB_REQUIRE(env, "env is null");
  env->stream = (cudaStream_t)cuda_stream;
  return WB_OK;
}

int32_t wb_terrain_env_state_floats(const wb_terrain_env* env, int32_t* per_copy_out) {
  WB_REQUIRE(env && per_copy_out, "null argument");
  *per_copy_out = env->rows;
  return WB_OK;
}

int32_t wb_terrain_env_set_terrain(wb_terrain_env* env, const float* vertices_host) {
  WB_REQUIRE(env && vertices_host, "null argument");
  const SceneConst& c = env->tc.topo;
  const int n = env->n, nb = c.n_bodies, K = nb - 5, tvt = env->terrain_verts, wv = c.vert_offset[5];
  const size_t np = (size_t)env->n_pad;
  // SoA blocks of the terrain's rows: vertices [2 tvt][n], cached centroids [2K][n]; velocities, omega and angle are zero
  std::vector<float> verts((size_t)2 * tvt * n), cen((size_t)2 * K * n), zeros((size_t)2 * K * n, 0.0f), one(2 * K);
  for (int i = 0; i < n; i++) {
    const float* v = vertices_host + (size_t)i * 2 * tvt;
    for (int r = 0; r < 2 * tvt; r++) verts[(size_t)r * n + i] = v[r];
    centroids_of(c, v, 5, nb, one.data());
    for (int r = 0; r < 2 * K; r++) cen[(size_t)r * n + i] = one[r];
  }
  const int tv = c.total_verts;
  struct Block {
    int row, count;
    const float* src;
  } blocks[5] = {{2 * wv, 2 * tvt, verts.data()}, {2 * tv + 10, 2 * K, cen.data()}, {2 * tv + 2 * nb + 10, 2 * K, zeros.data()},
                 {2 * tv + 4 * nb + 5, K, zeros.data()}, {2 * tv + 5 * nb + 5, K, zeros.data()}};
  for (const Block& b : blocks)
    WB_CUDA(cudaMemcpy2DAsync(env->d_state + (size_t)b.row * np, sizeof(float) * np, b.src, sizeof(float) * n, sizeof(float) * n, b.count,
                              cudaMemcpyHostToDevice, env->stream));
  // new bodies: their Collided latches start cleared, the walker's stay
  std::vector<int32_t> col(n);
  WB_CUDA(cudaMemcpyAsync(col.data(), env->d_ints, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  for (int i = 0; i < n; i++) col[i] &= 0x1F;
  WB_CUDA(cudaMemcpyAsync(env->d_ints, col.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_terrain_env_reset(wb_terrain_env* env, const uint8_t* mask_host, int32_t first_episode) {
  WB_REQUIRE(env, "env is null");
  const uint8_t* d_mask = nullptr;
  if (mask_host) {
    WB_CUDA(cudaMemcpyAsync(env->d_mask, mask_host, env->n, cudaMemcpyHostToDevice, env->stream));
    d_mask = env->d_mask;
  }
  if (int32_t rc = terrain_launch(env, kPhaseResetMasked | (first_episode ? kPhaseFirstEpisode : 0), 0.0f, nullptr, d_mask, nullptr,
                                  nullptr, nullptr))
    return rc;
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_terrain_env_get_state(wb_terrain_env* env, float* state_f_host, int32_t* state_i_host) {
  WB_REQUIRE(env && state_f_host && state_i_host, "null argument");
  const size_t n = env->n, np = env->n_pad;
  WB_CUDA(cudaMemcpy2DAsync(state_f_host, sizeof(float) * n, env->d_state, sizeof(float) * np, sizeof(float) * n, env->rows,
                            cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaMemcpy2DAsync(state_i_host, sizeof(int32_t) * n, env->d_ints, sizeof(int32_t) * np, sizeof(int32_t) * n, kTerrainInts,
                            cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_terrain_env_set_state(wb_terrain_env* env, const float* state_f_host, const int32_t* state_i_host) {
  WB_REQUIRE(env && state_f_host && state_i_host, "null argument");
  const size_t n = env->n, np = env->n_pad;
  WB_CUDA(cudaMemcpy2DAsync(env->d_state, sizeof(float) * np, state_f_host, sizeof(float) * n, sizeof(float) * n, env->rows,
                            cudaMemcpyHostToDevice, env->stream));
  WB_CUDA(cudaMemcpy2DAsync(env->d_ints, sizeof(int32_t) * np, state_i_host, sizeof(int32_t) * n, sizeof(int32_t) * n, kTerrainInts,
                            cudaMemcpyHostToDevice, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

static int32_t terrain_copy_out(wb_terrain_env* env, float* obs_host, float* reward_host, uint8_t* done_host) {
  if (obs_host) WB_CUDA(cudaMemcpyAsync(obs_host, env->d_obs, sizeof(float) * WB_OBS * env->n, cudaMemcpyDeviceToHost, env->stream));
  if (reward_host) WB_CUDA(cudaMemcpyAsync(reward_host, env->d_reward, sizeof(float) * env->n, cudaMemcpyDeviceToHost, env->stream));
  if (done_host) WB_CUDA(cudaMemcpyAsync(done_host, env->d_done, env->n, cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_terrain_env_get_obs(wb_terrain_env* env, float* obs_host) {
  WB_REQUIRE(env && obs_host, "null argument");
  if (int32_t rc = terrain_launch(env, kPhaseObsOnly, 0.0f, nullptr, nullptr, env->d_obs, nullptr, nullptr)) return rc;
  return terrain_copy_out(env, obs_host, nullptr, nullptr);
}

static int terrain_step_phases(int32_t auto_reset) {
  return kPhaseIncSteps | kPhaseTakeActions | kPhaseStepObjects | kPhaseObserve | (auto_reset ? kPhaseAutoReset : 0);
}

int32_t wb_terrain_env_step(wb_terrain_env* env, const float* actions_host, float delta_time, int32_t auto_reset, float* obs_host,
                            float* reward_host, uint8_t* done_host) {
  WB_REQUIRE(env && actions_host, "null argument");
  WB_CUDA(cudaMemcpyAsync(env->d_actions, actions_host, sizeof(float) * WB_ACT * env->n, cudaMemcpyHostToDevice, env->stream));
  if (int32_t rc = terrain_launch(env, terrain_step_phases(auto_reset), delta_time, env->d_actions, nullptr, env->d_obs, env->d_reward,
                                  env->d_done))
    return rc;
  return terrain_copy_out(env, obs_host, reward_host, done_host);
}

int32_t wb_terrain_env_step_dev(wb_terrain_env* env, const float* actions_dev, float delta_time, int32_t auto_reset, float* obs_dev,
                                float* reward_dev, uint8_t* done_dev) {
  WB_REQUIRE(env && actions_dev && obs_dev && reward_dev && done_dev, "null argument");
  return terrain_launch(env, terrain_step_phases(auto_reset), delta_time, actions_dev, nullptr, obs_dev, reward_dev, done_dev);
}

int32_t wb_terrain_env_launch_count(const wb_terrain_env* env, int64_t* count_out) {
  WB_REQUIRE(env && count_out, "null argument");
  *count_out = env->launches;
  return WB_OK;
}

}  // extern "C"

// api_env.cu -- C ABI for the environment batch (include/walker_b200.h): handles, materials, scene construction,
// host<->device staging.  All compute is in physics.cu; there is no CPU path.
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <new>
#include <unordered_map>
#include <vector>

#include "common.h"
#include "physics.cuh"

namespace wb {

static thread_local char g_err[512] = "";
char* last_error_buffer() { return g_err; }

int32_t fail(int32_t code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int32_t require_device() {
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(WB_ERR_NO_DEVICE, "no CUDA device: %s (libwalker_b200 has no CPU fallback)", cudaGetErrorString(e));
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return fail(WB_ERR_NO_DEVICE, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(WB_ERR_NO_DEVICE, "device %d is sm_%d%d; libwalker_b200 is built for sm_100a only", dev, prop.major, prop.minor);
  return WB_OK;
}

// ------------------------------------------------------------------ materials (Materials/*.cs, IMaterial.cs:6-11)
static std::mutex g_mat_mutex;
static Material g_materials[WB_MAX_MATERIALS] = {
    {11.0f, 0.3f, 0.0f},   // Ice
    {20.0f, 0.3f, 0.01f},  // Wood
    {1.0f, 0.3f, 0.1f},    // Paper
    {0.01f, 0.1f, 0.2f},   // Titanium
    {5.0f, 0.3f, 0.8f},    // Carpet
    {11.0f, 0.7f, 0.5f},   // Rubber
    {15.0f, 0.3f, 1.0f},   // Metal
    {11.0f, 1.0f, 1.0f},   // SuperRubber
};
static int g_material_count = WB_NUM_BUILTIN_MATERIALS;

// ------------------------------------------------------------------ scene constants, host restatement in strict fp32
// (volatile stores keep every intermediate in binary32 and stop the host compiler from contracting)
static inline float f_add(float a, float b) { volatile float r = a + b; return r; }
static inline float f_sub(float a, float b) { volatile float r = a - b; return r; }
static inline float f_mul(float a, float b) { volatile float r = a * b; return r; }
static inline float f_div(float a, float b) { volatile float r = a / b; return r; }

// Skeleton.FindCentroid (Skeleton.cs:100-113): sum, then Vector2 / count = multiply by (1f / count)
static void centroid_of(const float* v, int n, float* out) {
  float sx = 0.0f, sy = 0.0f;
  for (int i = 0; i < n; i++) {
    sx = f_add(sx, v[2 * i]);
    sy = f_add(sy, v[2 * i + 1]);
  }
  const float factor = f_div(1.0f, (float)n);
  out[0] = f_mul(sx, factor);
  out[1] = f_mul(sy, factor);
}

// Pole.FromSize (Pole.cs:18-34)
static void pole_from_size(float cx, float cy, float size, float* v12) {
  const float adjustment = f_mul((float)0.1, size);
  const float h = f_mul(adjustment, 3.5f);
  const float xs[6] = {f_add(cx, adjustment), cx, f_sub(cx, adjustment), f_sub(cx, adjustment), cx, f_add(cx, adjustment)};
  const float ys[6] = {f_add(cy, h), f_add(cy, h), f_add(cy, h), f_sub(cy, h), f_sub(cy, h), f_sub(cy, h)};
  for (int i = 0; i < 6; i++) {
    v12[2 * i] = xs[i];
    v12[2 * i + 1] = ys[i];
  }
}

// Walker ctor + CreateBodies (Walker.cs:25-34,155-177) and Environment.CreateFloor (Environment.cs:211-226)
static void build_scene_constants(float* init92, float* floor10) {
  const float px = 125.0f, py = 800.0f;  // Walker._position, Walker.cs:31
  float verts[58];
  float* lll = verts;
  float* llu = verts + 12;
  float* body = verts + 24;
  float* rll = verts + 34;
  float* rlu = verts + 46;
  const float hull[10] = {f_add(px, 20.f), f_add(py, 20.f), px, f_add(py, 20.f), f_sub(px, 20.f), f_add(py, 20.f),
                          f_sub(px, 20.f), f_sub(py, 20.f), f_add(px, 20.f), f_sub(py, 20.f)};
  memcpy(body, hull, sizeof(hull));
  pole_from_size(f_add(px, 0.f), f_add(py, 30.f), 75.f, llu);
  pole_from_size(f_add(px, 0.f), f_add(py, 60.f), 75.f, lll);
  pole_from_size(f_add(px, 0.f), f_add(py, 30.f), 75.f, rlu);
  pole_from_size(f_add(px, 0.f), f_add(py, 60.f), 75.f, rll);
  memset(init92, 0, sizeof(float) * kStateFloats);
  memcpy(init92, verts, sizeof(verts));
  centroid_of(lll, 6, init92 + 58);
  centroid_of(llu, 6, init92 + 60);
  centroid_of(body, 5, init92 + 62);
  centroid_of(rll, 6, init92 + 64);
  centroid_of(rlu, 6, init92 + 66);
  const float fl[8] = {-50.f, 1050.f, -50.f, 900.f, 1050.f, 900.f, 1050.f, 1050.f};
  memcpy(floor10, fl, sizeof(fl));
  centroid_of(fl, 4, floor10 + 8);
}

// the floor's derived constants (see FloorConst): bounding box, edge normals, own projections -- same operation order as
// BoundingBox.FindSignificantCorners (Skeleton.cs:144-176), SATCollision.AxisChecks/ProjectPoints (SATCollision.cs:39-76)
static void build_floor_constants(const float* floor10, FloorConst* fc) {
  memset(fc, 0, sizeof(*fc));
  float minx = 3.402823466e+38f, miny = 3.402823466e+38f, maxx = -3.402823466e+38f, maxy = -3.402823466e+38f;
  for (int i = 0; i < 4; i++) {
    fc->v[i] = make_float2(floor10[2 * i], floor10[2 * i + 1]);
    if (fc->v[i].x > maxx) maxx = fc->v[i].x;
    if (fc->v[i].y > maxy) maxy = fc->v[i].y;
    if (fc->v[i].x < minx) minx = fc->v[i].x;
    if (fc->v[i].y < miny) miny = fc->v[i].y;
  }
  fc->cen = make_float2(floor10[8], floor10[9]);
  fc->bb_min = make_float2(minx, miny);
  fc->bb_max = make_float2(maxx, maxy);
  for (int i = 0; i < 4; i++) {
    const float2 p0 = fc->v[i], p1 = fc->v[(i + 1) % 4];
    const float ex = f_sub(p1.x, p0.x), ey = f_sub(p1.y, p0.y);
    float ax = -ey, ay = ex;
    fc->skip[i] = (ax == 0.0f && ay == 0.0f) ? 1 : 0;
    const float val = f_div(1.0f, sqrtf(f_add(f_mul(ax, ax), f_mul(ay, ay))));  // Vector2.Normalize
    ax = f_mul(ax, val);
    ay = f_mul(ay, val);
    fc->axis[i] = make_float2(ax, ay);
    float mn = 3.402823466e+38f, mx = -3.402823466e+38f;
    for (int j = 0; j < 4; j++) {
      const float t = f_add(f_mul(ax, fc->v[j].x), f_mul(ay, fc->v[j].y));
      if (t < mn) mn = t;
      if (t > mx) mx = t;
    }
    fc->pmin[i] = mn;
    fc->pmax[i] = mx;
  }
}

void walker_initial_record(float* init92) {
  float floor10[10];
  build_scene_constants(init92, floor10);
}

}  // namespace wb

using namespace wb;

// Lanes per environment when the caller does not choose: with few walkers per SM the step is latency bound and the lanes of
// a walker split its SAT axes and vertices; with many, one lane per walker does no redundant work (see physics_lanes.cu).
// The boundaries are read off profiles/variant_sweep_r2.log (scripts/variant_sweep.sh: every candidate variant timed from one
// snapshot 512 env-steps into a random-action rollout, 1 ... 262 144 walkers on a 148-SM B200); each is where the faster variant
// changes -- mostly where the narrower layout's warps stop fitting one wave (8 lanes: 12 warps per SM = 48 walkers; 4 lanes:
// 19 warps per SM = 152 walkers).
static int default_lanes(int n_envs, int sm_count) {
  const long per_sm = ((long)n_envs + sm_count - 1) / sm_count;
  if (per_sm <= 10) return 32;   // a handful of walkers (the reference's single-walker case): all 32 lanes on one walker
  if (per_sm <= 22) return 16;   // 2048 walkers: 0.315 ms (16) vs 0.325 (8) / 0.345 (32); 3072: 0.359 vs 0.366
  if (per_sm <= 48) return 8;    // 4096: 0.375 (8) vs 0.416 (16) / 0.446 (4); 7104: 0.438 vs 0.510 (4)
  // (second sweep of round 2, after the compacting kernel lost its joint rounds -- appended to profiles/variant_sweep_r2.log: the
  //  2-lane layout no longer wins anywhere, and between ~125 and ~375 walkers per SM four CTAs of 128 walkers beat two of 256)
  if (per_sm <= 124) return 4;   // 8192: 0.508 (4) vs 0.688 (8); 16384: 0.727 (4) vs 0.782 (1003) / 0.784 (2)
  if (per_sm <= 375) return 1003;  // 20480: 0.843 (1003) vs 0.895 (2) / 1.027 (4); 32768: 0.912 vs 0.948 (1001); 53248: 1.073 vs 1.134 (1001)
  return 1001;  // GPU full: scopes of 256 walkers, two CTAs per SM (57344: 1.142 vs 1.172 (1003); 262144: 3.98 vs 4.38)
}

struct wb_env_batch {
  int32_t n = 0, n_pad = 0;
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  wb_hyperparams hp{};
  int lanes = 0;  // kernel variant: lanes per environment (1, 2, 4, 8, 16) or 1001 (compacting); chosen from the batch size at creation
  int64_t launches = 0;
  // device state (structure of arrays)
  float* d_state = nullptr;    // 92 floats per walker in the device layout of physics.cuh (state_index), rows padded to n_pad
  int32_t* d_flags = nullptr;  // [n_pad]
  int32_t* d_steps = nullptr;  // [n_pad]
  float* d_pos = nullptr;      // [2][n_pad]
  uint8_t* d_floor_mat = nullptr;
  uint8_t* d_walker_mat = nullptr;
  uint32_t* d_axis_cache = nullptr;  // [n_pad] separating-axis hints of the compacting kernel, carried across launches
  // device I/O staging for the host-pointer entry points
  float* d_actions = nullptr;  // [n][4]
  float* d_obs = nullptr;      // [n][12]
  float* d_reward = nullptr;   // [n]
  uint8_t* d_done = nullptr;   // [n]
  uint8_t* d_mask = nullptr;   // [n]
  float init92[WB_STATE_FLOATS];
};

extern "C" {

const char* wb_version(void) { return "walker_b200 0.1.0 (sm_100a)"; }

int32_t wb_last_error(char* buf, size_t buf_len) {
  if (!buf || buf_len == 0) return WB_ERR_INVALID;
  strncpy(buf, last_error_buffer(), buf_len - 1);
  buf[buf_len - 1] = 0;
  return WB_OK;
}

int32_t wb_init(int32_t device) {
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(WB_ERR_NO_DEVICE, "cudaSetDevice(%d): %s (libwalker_b200 has no CPU fallback)", device, cudaGetErrorString(e));
  }
  return require_device();
}

int32_t wb_hyperparams_default(wb_hyperparams* hp) {
  WB_REQUIRE(hp, "hp is null");
  hp->iterations = 50;
  hp->max_timesteps = 1000;
  hp->batch_size = 64;
  hp->use_gae = 0;
  hp->normalize_advantages = 0;
  hp->alpha = 0.001f;
  hp->beta1 = 0.9f;
  hp->beta2 = 0.999f;
  hp->adam_epsilon = 1e-8f;
  hp->gamma = 0.9f;
  hp->lambda = 0.95f;
  hp->epsilon = 0.3f;
  hp->log_std = -1.0f;
  return WB_OK;
}

int32_t wb_material_register(float inverse_mass, float restitution, float friction, int32_t* id_out) {
  WB_REQUIRE(id_out, "id_out is null");
  std::lock_guard<std::mutex> lock(g_mat_mutex);
  if (g_material_count >= WB_MAX_MATERIALS) return fail(WB_ERR_INVALID, "material table full (%d)", WB_MAX_MATERIALS);
  g_materials[g_material_count] = Material{inverse_mass, restitution, friction};
  *id_out = g_material_count++;
  return WB_OK;
}

int32_t wb_material_get(int32_t id, float* inverse_mass, float* restitution, float* friction) {
  std::lock_guard<std::mutex> lock(g_mat_mutex);
  if (id < 0 || id >= g_material_count) return fail(WB_ERR_INVALID, "unknown material id %d", id);
  if (inverse_mass) *inverse_mass = g_materials[id].inverse_mass;
  if (restitution) *restitution = g_materials[id].restitution;
  if (friction) *friction = g_materials[id].friction;
  return WB_OK;
}

static int32_t launch(wb_env_batch* env, int phases, float dt, const float* d_actions, float* d_obs, float* d_reward,
                      uint8_t* d_done, const uint8_t* d_mask, wb_pair_trace* d_pt, wb_joint_trace* d_jt, int n_override = 0) {
  PhysicsParams p{};
  p.state = env->d_state;
  p.flags = env->d_flags;
  p.steps = env->d_steps;
  p.pos = env->d_pos;
  p.floor_mat = env->d_floor_mat;
  p.walker_mat = env->d_walker_mat;
  p.axis_cache = env->d_axis_cache;
  p.actions = d_actions;
  p.reset_mask = d_mask;
  p.obs = d_obs;
  p.reward = d_reward;
  p.done = d_done;
  p.pair_trace = d_pt;
  p.joint_trace = d_jt;
  p.n = n_override > 0 ? n_override : env->n;
  p.n_pad = env->n_pad;
  p.dt = dt;
  p.iterations = env->hp.iterations;
  p.max_timesteps = env->hp.max_timesteps;
  p.phases = phases;
  WB_CUDA(launch_physics(p, env->lanes, d_pt != nullptr || d_jt != nullptr, env->stream));
  env->launches++;
  return WB_OK;
}

int32_t wb_env_create(int32_t n_envs, const uint8_t* floor_material_ids, const uint8_t* walker_material_ids,
                      const wb_hyperparams* hp, wb_env_batch** out) {
  WB_REQUIRE(out, "out is null");
  *out = nullptr;
  WB_REQUIRE(n_envs > 0, "n_envs must be positive");
  if (int32_t rc = require_device()) return rc;
  wb_env_batch* env = new (std::nothrow) wb_env_batch();
  WB_REQUIRE(env, "out of host memory");
  cudaGetDevice(&env->device);
  cudaDeviceGetAttribute(&env->sm_count, cudaDevAttrMultiProcessorCount, env->device);
  env->n = n_envs;
  env->lanes = default_lanes(n_envs, env->sm_count);
  env->n_pad = (n_envs + kEnvPad - 1) / kEnvPad * kEnvPad;
  if (hp) env->hp = *hp; else wb_hyperparams_default(&env->hp);
  if (env->hp.iterations <= 0 || env->hp.iterations >= 200) {  // Hyperparameters.cs:189-217 range check
    delete env;
    return fail(WB_ERR_INVALID, "iterations must be in (0, 200)");
  }
  const size_t np = (size_t)env->n_pad;
  std::vector<uint8_t> fm(np, (uint8_t)WB_METAL), wm(np, (uint8_t)WB_CARPET);
  Material table[WB_MAX_MATERIALS];
  {
    std::lock_guard<std::mutex> lock(g_mat_mutex);  // held only for the table snapshot, not across the upload
    for (int i = 0; i < n_envs; i++) {
      if (floor_material_ids) fm[i] = floor_material_ids[i];
      if (walker_material_ids) wm[i] = walker_material_ids[i];
      if (fm[i] >= g_material_count || wm[i] >= g_material_count) {
        delete env;
        return fail(WB_ERR_INVALID, "env %d uses an unregistered material id", i);
      }
    }
    memcpy(table, g_materials, sizeof(table));
  }
  // any failure from here on releases everything allocated so far (wb_env_destroy) before returning
#define WB_ENV_TRY(expr)                                                                    \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      wb_env_destroy(env);                                                                  \
      return wb::fail(WB_ERR_CUDA, "wb_env_create: %s: %s", #expr, cudaGetErrorString(_e)); \
    }                                                                                       \
  } while (0)
  WB_ENV_TRY(upload_materials(table, WB_MAX_MATERIALS));
  float floor10[10];
  FloorConst floor_const;
  build_scene_constants(env->init92, floor10);
  build_floor_constants(floor10, &floor_const);
  WB_ENV_TRY(upload_scene_constants(env->init92, &floor_const));
  WB_ENV_TRY(cudaMalloc(&env->d_state, sizeof(float) * kStateFloats * np));
  WB_ENV_TRY(cudaMalloc(&env->d_flags, sizeof(int32_t) * np));
  WB_ENV_TRY(cudaMalloc(&env->d_steps, sizeof(int32_t) * np));
  WB_ENV_TRY(cudaMalloc(&env->d_pos, sizeof(float) * 2 * np));
  WB_ENV_TRY(cudaMalloc(&env->d_floor_mat, np));
  WB_ENV_TRY(cudaMalloc(&env->d_walker_mat, np));
  WB_ENV_TRY(cudaMalloc(&env->d_axis_cache, sizeof(uint32_t) * np));
  WB_ENV_TRY(cudaMemset(env->d_axis_cache, 0, sizeof(uint32_t) * np));
  WB_ENV_TRY(cudaMalloc(&env->d_actions, sizeof(float) * WB_ACT * np));
  WB_ENV_TRY(cudaMalloc(&env->d_obs, sizeof(float) * WB_OBS * np));
  WB_ENV_TRY(cudaMalloc(&env->d_reward, sizeof(float) * np));
  WB_ENV_TRY(cudaMalloc(&env->d_done, np));
  WB_ENV_TRY(cudaMalloc(&env->d_mask, np));
  WB_ENV_TRY(cudaMemset(env->d_state, 0, sizeof(float) * kStateFloats * np));
  WB_ENV_TRY(cudaMemset(env->d_flags, 0, sizeof(int32_t) * np));
  WB_ENV_TRY(cudaMemset(env->d_steps, 0, sizeof(int32_t) * np));
  WB_ENV_TRY(cudaMemset(env->d_pos, 0, sizeof(float) * 2 * np));
  WB_ENV_TRY(cudaMemcpy(env->d_floor_mat, fm.data(), np, cudaMemcpyHostToDevice));
  WB_ENV_TRY(cudaMemcpy(env->d_walker_mat, wm.data(), np, cudaMemcpyHostToDevice));
  // constructor state: walker first, floor last (Environment.cs:46-48), then InitialState -- for the padding of the rows too:
  // the pad walkers are real, idle walkers (they never receive actions and are never read), so a lockstep CTA of the compacting
  // kernel can always move whole row segments
  if (int32_t rc = launch(env, kPhaseResetMasked | kPhaseFirstEpisode, 0.f, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                          env->n_pad)) {
    wb_env_destroy(env);
    return rc;
  }
  WB_ENV_TRY(cudaStreamSynchronize(env->stream));
#undef WB_ENV_TRY
  *out = env;
  return WB_OK;
}

int32_t wb_env_destroy(wb_env_batch* env) {
  if (!env) return WB_OK;
  cudaFree(env->d_state);
  cudaFree(env->d_flags);
  cudaFree(env->d_steps);
  cudaFree(env->d_pos);
  cudaFree(env->d_floor_mat);
  cudaFree(env->d_walker_mat);
  cudaFree(env->d_axis_cache);
  cudaFree(env->d_actions);
  cudaFree(env->d_obs);
  cudaFree(env->d_reward);
  cudaFree(env->d_done);
  cudaFree(env->d_mask);
  delete env;
  return WB_OK;
}

int32_t wb_env_count(const wb_env_batch* env, int32_t* n_out) {
  WB_REQUIRE(env && n_out, "null argument");
  *n_out = env->n;
  return WB_OK;
}

int32_t wb_env_set_stream(wb_env_batch* env, void* cuda_stream) {
  WB_REQUIRE(env, "env is null");
  env->stream = (cudaStream_t)cuda_stream;
  return WB_OK;
}

int32_t wb_env_sync(wb_env_batch* env) {
  WB_REQUIRE(env, "env is null");
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_env_launch_count(const wb_env_batch* env, int64_t* count_out) {
  WB_REQUIRE(env && count_out, "null argument");
  *count_out = env->launches;
  return WB_OK;
}

int32_t wb_env_set_variant(wb_env_batch* env, int32_t lanes_per_env) {
  WB_REQUIRE(env, "env is null");
  if (lanes_per_env == 0) lanes_per_env = default_lanes(env->n, env->sm_count);
  if (!physics_lanes_supported(lanes_per_env)) return fail(WB_ERR_INVALID, "variant must be 1, 2, 4, 8 or 16 lanes per walker, 104 / 108 / 116 (no leg split) or 1001 / 1002 / 1003 (compacting throughput kernels)");
  env->lanes = lanes_per_env;
  return WB_OK;
}

int32_t wb_env_get_variant(const wb_env_batch* env, int32_t* lanes_per_env_out) {
  WB_REQUIRE(env && lanes_per_env_out, "null argument");
  *lanes_per_env_out = env->lanes;
  return WB_OK;
}

int32_t wb_env_reset(wb_env_batch* env, const uint8_t* mask_host, int32_t first_episode) {
  WB_REQUIRE(env, "env is null");
  const uint8_t* d_mask = nullptr;
  if (mask_host) {
    WB_CUDA(cudaMemcpyAsync(env->d_mask, mask_host, env->n, cudaMemcpyHostToDevice, env->stream));
    d_mask = env->d_mask;
  }
  if (int32_t rc = launch(env, kPhaseResetMasked | (first_episode ? kPhaseFirstEpisode : 0), 0.f, nullptr, nullptr, nullptr,
                          nullptr, d_mask, nullptr, nullptr))
    return rc;
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

// canonical host blob [92][n] <-> the device layout (physics.cuh: state_index); also fills Walker._position on the way in
__global__ void state_layout_kernel(float* __restrict__ canonical, float* __restrict__ dev_state, float* __restrict__ pos, int n, int n_pad,
                                    int to_device) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)kStateFloats * n) return;
  const int f = (int)(i / n);
  const size_t env = i % n;
  if (to_device) {
    const float v = canonical[i];
    dev_state[state_index(f, env, n_pad)] = v;
    // Walker._position == Body centroid at every step boundary (Walker.cs:52): floats 62 / 63 of the record
    if (f == 62) pos[env] = v;
    if (f == 63) pos[n_pad + env] = v;
  } else {
    canonical[i] = dev_state[state_index(f, env, n_pad)];
  }
}

static int32_t convert_state(wb_env_batch* env, float* host_blob, bool to_device) {
  const size_t n = env->n, bytes = sizeof(float) * kStateFloats * n;
  float* d_tmp = nullptr;
  WB_CUDA(cudaMalloc(&d_tmp, bytes));
  cudaError_t e = cudaSuccess;
  if (to_device) e = cudaMemcpyAsync(d_tmp, host_blob, bytes, cudaMemcpyHostToDevice, env->stream);
  if (e == cudaSuccess) {
    const size_t total = (size_t)kStateFloats * n;
    state_layout_kernel<<<(unsigned)((total + 255) / 256), 256, 0, env->stream>>>(d_tmp, env->d_state, env->d_pos, (int)n, env->n_pad,
                                                                                 to_device ? 1 : 0);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess && !to_device) e = cudaMemcpyAsync(host_blob, d_tmp, bytes, cudaMemcpyDeviceToHost, env->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(env->stream);
  cudaFree(d_tmp);
  if (e != cudaSuccess) return fail(WB_ERR_CUDA, "state layout conversion: %s", cudaGetErrorString(e));
  return WB_OK;
}

int32_t wb_env_set_state(wb_env_batch* env, const float* state_f_host, const int32_t* state_i_host) {
  WB_REQUIRE(env && state_f_host && state_i_host, "null argument");
  const size_t n = env->n;
  if (int32_t rc = convert_state(env, const_cast<float*>(state_f_host), true)) return rc;
  WB_CUDA(cudaMemcpyAsync(env->d_flags, state_i_host, n * sizeof(int32_t), cudaMemcpyHostToDevice, env->stream));
  WB_CUDA(cudaMemcpyAsync(env->d_steps, state_i_host + n, n * sizeof(int32_t), cudaMemcpyHostToDevice, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_env_get_state(wb_env_batch* env, float* state_f_host, int32_t* state_i_host) {
  WB_REQUIRE(env && state_f_host && state_i_host, "null argument");
  const size_t n = env->n;
  if (int32_t rc = convert_state(env, state_f_host, false)) return rc;
  WB_CUDA(cudaMemcpyAsync(state_i_host, env->d_flags, n * sizeof(int32_t), cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaMemcpyAsync(state_i_host + n, env->d_steps, n * sizeof(int32_t), cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_env_take_actions(wb_env_batch* env, const float* actions_host) {
  WB_REQUIRE(env && actions_host, "null argument");
  WB_CUDA(cudaMemcpyAsync(env->d_actions, actions_host, sizeof(float) * WB_ACT * env->n, cudaMemcpyHostToDevice, env->stream));
  if (int32_t rc = launch(env, kPhaseTakeActions, 0.f, env->d_actions, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr)) return rc;
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_env_step_objects(wb_env_batch* env, float delta_time) {
  WB_REQUIRE(env, "env is null");
  if (int32_t rc = launch(env, kPhaseStepObjects, delta_time, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr)) return rc;
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_env_debug_contacts(wb_env_batch* env, float delta_time, wb_pair_trace* pair_trace_host,
                              wb_joint_trace* joint_trace_host) {
  WB_REQUIRE(env && pair_trace_host && joint_trace_host, "null argument");
  const size_t npair = (size_t)env->n * env->hp.iterations * WB_PAIR_SLOTS;
  const size_t njoint = (size_t)env->n * env->hp.iterations * 4;
  wb_pair_trace* d_pt = nullptr;
  wb_joint_trace* d_jt = nullptr;
  WB_CUDA(cudaMalloc(&d_pt, npair * sizeof(wb_pair_trace)));
  cudaError_t e = cudaMalloc(&d_jt, njoint * sizeof(wb_joint_trace));
  if (e != cudaSuccess) {
    cudaFree(d_pt);
    return fail(WB_ERR_CUDA, "cudaMalloc(joint trace): %s", cudaGetErrorString(e));
  }
  int32_t rc = launch(env, kPhaseStepObjects, delta_time, nullptr, nullptr, nullptr, nullptr, nullptr, d_pt, d_jt);
  if (rc == WB_OK) {
    e = cudaMemcpyAsync(pair_trace_host, d_pt, npair * sizeof(wb_pair_trace), cudaMemcpyDeviceToHost, env->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(joint_trace_host, d_jt, njoint * sizeof(wb_joint_trace), cudaMemcpyDeviceToHost, env->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(env->stream);
    if (e != cudaSuccess) rc = fail(WB_ERR_CUDA, "trace copy: %s", cudaGetErrorString(e));
  }
  cudaFree(d_pt);
  cudaFree(d_jt);
  return rc;
}

static int32_t copy_out(wb_env_batch* env, float* obs_host, float* reward_host, uint8_t* done_host) {
  if (obs_host) WB_CUDA(cudaMemcpyAsync(obs_host, env->d_obs, sizeof(float) * WB_OBS * env->n, cudaMemcpyDeviceToHost, env->stream));
  if (reward_host) WB_CUDA(cudaMemcpyAsync(reward_host, env->d_reward, sizeof(float) * env->n, cudaMemcpyDeviceToHost, env->stream));
  if (done_host) WB_CUDA(cudaMemcpyAsync(done_host, env->d_done, env->n, cudaMemcpyDeviceToHost, env->stream));
  WB_CUDA(cudaStreamSynchronize(env->stream));
  return WB_OK;
}

int32_t wb_env_observe(wb_env_batch* env, float* obs_host, float* reward_host, uint8_t* done_host) {
  WB_REQUIRE(env, "env is null");
  if (int32_t rc = launch(env, kPhaseObserve, 0.f, nullptr, env->d_obs, env->d_reward, env->d_done, nullptr, nullptr, nullptr)) return rc;
  return copy_out(env, obs_host, reward_host, done_host);
}

int32_t wb_env_get_obs(wb_env_batch* env, float* obs_host) {
  WB_REQUIRE(env && obs_host, "null argument");
  if (int32_t rc = launch(env, kPhaseObsOnly, 0.f, nullptr, env->d_obs, nullptr, nullptr, nullptr, nullptr, nullptr)) return rc;
  return copy_out(env, obs_host, nullptr, nullptr);
}

static int step_phases(int32_t auto_reset) {
  return kPhaseIncSteps | kPhaseTakeActions | kPhaseStepObjects | kPhaseObserve | (auto_reset ? kPhaseAutoReset : 0);
}

int32_t wb_env_step(wb_env_batch* env, const float* actions_host, float delta_time, int32_t auto_reset, float* obs_host,
                    float* reward_host, uint8_t* done_host) {
  WB_REQUIRE(env && actions_host, "null argument");
  // Zero-copy path: when every host buffer of the call is pinned, the kernel reads the actions and writes the observations,
  // rewards and done flags straight through the device-side aliases of the caller's buffers (16 B / 53 B per walker over
  // PCIe, issued by the kernel itself) -- no staging copies, one launch and one synchronisation per env-step.  Pageable
  // buffers (or WB_NO_ZERO_COPY=1) take the staged path: H2D copy, launch, three D2H copies.
  static const bool zero_copy_enabled = getenv("WB_NO_ZERO_COPY") == nullptr;
  if (zero_copy_enabled) {
    const size_t n = (size_t)env->n;
    const float* a = static_cast<const float*>(wb::device_alias_of_pinned(actions_host, sizeof(float) * WB_ACT * n));
    float* o = obs_host ? static_cast<float*>(wb::device_alias_of_pinned(obs_host, sizeof(float) * WB_OBS * n)) : env->d_obs;
    float* r = reward_host ? static_cast<float*>(wb::device_alias_of_pinned(reward_host, sizeof(float) * n)) : env->d_reward;
    uint8_t* d = done_host ? static_cast<uint8_t*>(wb::device_alias_of_pinned(done_host, n)) : env->d_done;
    if (a && o && r && d && (reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(o) & 15) == 0) {
      if (int32_t rc = launch(env, step_phases(auto_reset), delta_time, a, o, r, d, nullptr, nullptr, nullptr)) return rc;
      WB_CUDA(cudaStreamSynchronize(env->stream));
      return WB_OK;
    }
  }
  WB_CUDA(cudaMemcpyAsync(env->d_actions, actions_host, sizeof(float) * WB_ACT * env->n, cudaMemcpyHostToDevice, env->stream));
  if (int32_t rc = launch(env, step_phases(auto_reset), delta_time, env->d_actions, env->d_obs, env->d_reward, env->d_done, nullptr,
                          nullptr, nullptr))
    return rc;
  return copy_out(env, obs_host, reward_host, done_host);
}

// Small managed arrays (the reference's 12-float observation, 4-float action ...) usually SHARE a page, and cudaHostRegister
// refuses a range that touches an already registered page.  wb_host_pin therefore registers the page-rounded range in one call
// and, if that is refused, page by page, skipping the pages some earlier call registered; what THIS call registered is
// remembered per caller pointer so that wb_host_unpin releases exactly that.
static std::mutex g_pin_mutex;
static std::unordered_map<void*, std::vector<void*>> g_pins;   // caller pointer -> base addresses this call registered
constexpr uintptr_t kHostPage = 4096;

int32_t wb_host_pin(void* host_ptr, size_t bytes) {
  WB_REQUIRE(host_ptr && bytes > 0, "bad argument");
  if (int32_t rc = require_device()) return rc;
  const uintptr_t first = reinterpret_cast<uintptr_t>(host_ptr) & ~(kHostPage - 1);
  const uintptr_t last = (reinterpret_cast<uintptr_t>(host_ptr) + bytes + kHostPage - 1) & ~(kHostPage - 1);
  std::lock_guard<std::mutex> lock(g_pin_mutex);
  WB_REQUIRE(g_pins.find(host_ptr) == g_pins.end(), "wb_host_pin: this buffer is already pinned");
  std::vector<void*> mine;
  cudaError_t e = cudaHostRegister(reinterpret_cast<void*>(first), last - first, cudaHostRegisterDefault);
  if (e == cudaSuccess) {
    mine.push_back(reinterpret_cast<void*>(first));
  } else if (e == cudaErrorHostMemoryAlreadyRegistered) {
    cudaGetLastError();
    for (uintptr_t page = first; page < last; page += kHostPage) {
      e = cudaHostRegister(reinterpret_cast<void*>(page), kHostPage, cudaHostRegisterDefault);
      if (e == cudaSuccess) {
        mine.push_back(reinterpret_cast<void*>(page));
      } else if (e == cudaErrorHostMemoryAlreadyRegistered) {
        cudaGetLastError();  // an earlier wb_host_pin (or the caller) page-locked it: nothing to do
      } else {
        cudaGetLastError();
        for (void* q : mine) cudaHostUnregister(q);
        return fail(WB_ERR_CUDA, "wb_host_pin: cudaHostRegister: %s", cudaGetErrorString(e));
      }
    }
  } else {
    cudaGetLastError();
    return fail(WB_ERR_CUDA, "wb_host_pin: cudaHostRegister: %s", cudaGetErrorString(e));
  }
  g_pins.emplace(host_ptr, std::move(mine));
  return WB_OK;
}

int32_t wb_host_unpin(void* host_ptr) {
  WB_REQUIRE(host_ptr, "null argument");
  if (int32_t rc = require_device()) return rc;
  std::lock_guard<std::mutex> lock(g_pin_mutex);
  auto it = g_pins.find(host_ptr);
  WB_REQUIRE(it != g_pins.end(), "wb_host_unpin: this buffer was not pinned with wb_host_pin");
  cudaError_t first_error = cudaSuccess;
  for (void* q : it->second) {
    const cudaError_t e = cudaHostUnregister(q);
    if (e != cudaSuccess && first_error == cudaSuccess) first_error = e;
  }
  g_pins.erase(it);
  if (first_error != cudaSuccess) {
    cudaGetLastError();
    return fail(WB_ERR_CUDA, "wb_host_unpin: cudaHostUnregister: %s", cudaGetErrorString(first_error));
  }
  return WB_OK;
}

int32_t wb_env_step_dev(wb_env_batch* env, const float* actions_dev, float delta_time, int32_t auto_reset, float* obs_dev,
                        float* reward_dev, uint8_t* done_dev) {
  WB_REQUIRE(env && actions_dev && obs_dev && reward_dev && done_dev, "null argument");
  return launch(env, step_phases(auto_reset), delta_time, actions_dev, obs_dev, reward_dev, done_dev, nullptr, nullptr, nullptr);
}

int32_t wb_debug_rotz(int32_t n, const float* radians_host, int32_t mode, float* cos_host, float* sin_host) {
  WB_REQUIRE(n > 0 && radians_host && cos_host && sin_host, "bad argument");
  if (int32_t rc = require_device()) return rc;
  float *d_in = nullptr, *d_c = nullptr, *d_s = nullptr;
  WB_CUDA(cudaMalloc(&d_in, sizeof(float) * 3 * (size_t)n));
  d_c = d_in + n;
  d_s = d_c + n;
  cudaError_t e = cudaMemcpy(d_in, radians_host, sizeof(float) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = launch_rotz_debug(d_in, n, mode, d_c, d_s, nullptr);
  if (e == cudaSuccess) e = cudaMemcpy(cos_host, d_c, sizeof(float) * n, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(sin_host, d_s, sizeof(float) * n, cudaMemcpyDeviceToHost);
  cudaFree(d_in);
  if (e != cudaSuccess) return fail(WB_ERR_CUDA, "wb_debug_rotz: %s", cudaGetErrorString(e));
  return WB_OK;
}

int32_t wb_debug_rcp_sqrt_check(uint32_t first_bits, uint64_t count, uint64_t* mismatches_out, uint32_t* first_bad_bits_out) {
  WB_REQUIRE(mismatches_out && first_bad_bits_out, "null argument");
  if (int32_t rc = require_device()) return rc;
  unsigned long long* d_cnt = nullptr;
  uint32_t* d_bad = nullptr;
  WB_CUDA(cudaMalloc(&d_cnt, sizeof(unsigned long long)));
  WB_CUDA(cudaMalloc(&d_bad, sizeof(uint32_t)));
  cudaError_t e = cudaMemset(d_cnt, 0, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemset(d_bad, 0xFF, sizeof(uint32_t));
  if (e == cudaSuccess) e = launch_rcp_sqrt_check(first_bits, count, d_cnt, d_bad, nullptr);
  unsigned long long cnt = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(first_bad_bits_out, d_bad, sizeof(uint32_t), cudaMemcpyDeviceToHost);
  cudaFree(d_cnt);
  cudaFree(d_bad);
  if (e != cudaSuccess) return fail(WB_ERR_CUDA, "wb_debug_rcp_sqrt_check: %s", cudaGetErrorString(e));
  *mismatches_out = cnt;
  return WB_OK;
}

}  // extern "C"

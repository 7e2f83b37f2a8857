// api_policy.cu -- C ABI for the PPO policy/value networks (include/walker_b200.h).  Compute is in mlp.cu.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.h"
#include "mlp.cuh"

using namespace wb;

struct wb_policy {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  wb_hyperparams hp{};
  int64_t launches = 0;
  int variant = 0;  // 0: tcgen05 tensor-core kernel (default), 1: fp32 CUDA-core kernel, 2: the any-topology kernel (mlp_generic.cu)
  bool default_topology = true;  // the reference's default networks: the specialised kernels apply
  GenNet actor{}, critic{};      // both networks as parsed layer tables
  int n_actor = kActorParams, n_critic = kCriticParams, n_total = kTotalParams;
  int grad_floats = kGradFloats;  // n_total + {sum g_V, sum mean_k g_mu, skipped}, padded to a float4 multiple
  int gen_ts = 0;                 // samples per tile of the generic kernel (from the shared-memory budget)
  int32_t iterations[kGenMaxDense] = {};  // DenseLayer._iteration per dense layer: actor layers, then critic layers
  float* d_params = nullptr;    // [n_total] actor | critic
  float* d_grads = nullptr;     // [grad_floats]
  float* d_m = nullptr;         // Adam first moment
  float* d_v = nullptr;         // Adam second moment
  float* d_partials = nullptr;  // [2 * sm_count][grad_floats]
  // staging for the host-pointer entry points (grown on demand)
  float* d_stage = nullptr;
  size_t stage_floats = 0;
  // fused reduce + all-reduce over NVLink peer memory (wb_comm_*)
  float* d_exch = nullptr;       // this rank's exchange buffer (kExchBytes), exported through CUDA IPC
  uint32_t* h_comm_status = nullptr;  // mapped pinned host word: set by reduce_exchange_kernel when a peer never arrived
  uint32_t* d_comm_status = nullptr;  // its device alias
  uint32_t* d_comm_dead = nullptr;    // device-memory copy of the status word (what the kernels check at launch)
  double* d_norm_stats = nullptr;     // [2][kNormCtas] partial sums of PPOAgent.Normalize (wb_normalize_advantages_dev)
  uint32_t* d_grid_sync = nullptr;    // arrival counter of the gradient kernel's grid barrier (fused single-process tail)
  uint32_t grid_sync_target = 0;
  ExchPeers peers{};
  void* opened[kExchMaxWorld] = {};  // IPC mappings to close
  int comm_rank = -1, comm_world = 0;
  uint32_t comm_epoch = 0;
  // wb_ppo_train_trajectories: device offsets + Adam correction table (uploaded from a pinned host copy), scratch rows
  char* h_episode_tab = nullptr;
  char* d_episode_tab = nullptr;
  size_t episode_tab_bytes = 0;
  cudaEvent_t episode_tab_copied = nullptr;  // the previous upload has left the pinned copy
  float* d_episode_scratch = nullptr;
  size_t episode_scratch_floats = 0;
};

static int32_t ensure_stage(wb_policy* p, size_t floats) {
  if (floats <= p->stage_floats) return WB_OK;
  if (p->d_stage) cudaFree(p->d_stage);
  p->d_stage = nullptr;
  p->stage_floats = 0;
  WB_CUDA(cudaMalloc(&p->d_stage, floats * sizeof(float)));
  p->stage_floats = floats;
  return WB_OK;
}

static bool use_generic(const wb_policy* p) { return !p->default_topology || p->variant == 2; }

static cudaError_t run_mlp(wb_policy* p, const MlpParams& m) {
  if (use_generic(p)) {
    GenParams g{};
    g.actor = p->actor;
    g.critic = p->critic;
    g.params = m.params;
    g.n = m.n;
    g.mode = m.mode;
    g.ts = p->gen_ts;
    g.grad_floats = p->grad_floats;
    g.states = m.states;
    g.actions = m.actions;
    g.old_logp = m.old_logp;
    g.advantages = m.advantages;
    g.returns = m.returns;
    g.uniforms = m.uniforms;
    g.seed = m.seed;
    g.step = m.step;
    g.mean = m.mean;
    g.value = m.value;
    g.out_actions = m.out_actions;
    g.out_logp = m.out_logp;
    g.partials = m.partials;
    g.log_std = m.log_std;
    g.epsilon = m.epsilon;
    g.batch_size = m.batch_size;
    return launch_mlp_generic(g, generic_grid_for(m.n, p->gen_ts, p->sm_count), p->stream);
  }
  if (p->variant == 1) return launch_mlp(m, mlp_grid_for(m.n, p->sm_count), p->stream);
  return launch_mlp_tc(m, tc_grid_for(m.n, p->sm_count), p->stream);
}
static int grid_of(const wb_policy* p, int n) {
  if (use_generic(p)) return generic_grid_for(n, p->gen_ts, p->sm_count);
  return p->variant == 1 ? mlp_grid_for(n, p->sm_count) : tc_grid_for(n, p->sm_count);
}
// per-CTA partials -> the gradient buffer (fixed order); also NeuralNetwork.Zero(): the buffer is overwritten
static cudaError_t reduce_grads(wb_policy* p, int grid) {
  if (use_generic(p)) return launch_reduce_partials_n(p->d_partials, grid, p->d_grads, p->grad_floats, p->stream);
  return launch_reduce_partials(p->d_partials, grid, p->d_grads, p->stream);
}

static void fill_mlp_common(const wb_policy* p, MlpParams& m, int n, int mode) {
  m = MlpParams{};
  m.params = p->d_params;
  m.n = n;
  m.mode = mode;
  m.log_std = p->hp.log_std;
  m.epsilon = p->hp.epsilon;
  m.batch_size = (float)p->hp.batch_size;
}

// a timed-out exchange leaves the ranks' weights out of step: refuse every later data-parallel update of this handle
static int32_t comm_healthy(const wb_policy* p) {
  if (*reinterpret_cast<volatile uint32_t*>(p->h_comm_status) != 0u)
    return fail(WB_ERR_COMM, "a gradient exchange timed out (a peer never arrived): gradients were not applied for the affected slices "
                             "and the replicas may have diverged; recreate the policy handles on every rank");
  return WB_OK;
}

extern "C" {

int32_t wb_policy_create(int32_t state_size, int32_t action_size, const int32_t* actor_kinds, const int32_t* actor_sizes,
                         int32_t actor_layers, const int32_t* critic_kinds, const int32_t* critic_sizes, int32_t critic_layers,
                         const wb_hyperparams* hp, wb_policy** out) {
  WB_REQUIRE(out, "out is null");
  *out = nullptr;
  Networks nets;
  if (int32_t rc = build_networks(state_size, action_size, actor_kinds, actor_sizes, actor_layers, critic_kinds, critic_sizes, critic_layers, &nets))
    return rc;
  const GenNet& actor = nets.actor;
  const GenNet& critic = nets.critic;
  if (int32_t rc = require_device()) return rc;
  wb_policy* p = new (std::nothrow) wb_policy();
  WB_REQUIRE(p, "out of host memory");
  p->default_topology = nets.default_topology;
  p->actor = actor;
  p->critic = critic;
  p->n_actor = actor.n_params;
  p->n_critic = critic.n_params;
  p->n_total = actor.n_params + critic.n_params;
  p->grad_floats = (p->n_total + 3 + 3) / 4 * 4;
  p->gen_ts = nets.gen_ts;
  cudaGetDevice(&p->device);
  cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, p->device);
  if (hp) p->hp = *hp; else wb_hyperparams_default(&p->hp);
  // (any failure below releases what was allocated so far: nothing leaks behind a failed create)
  cudaError_t e = cudaMalloc(&p->d_params, sizeof(float) * p->n_total);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_grads, sizeof(float) * p->grad_floats);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_m, sizeof(float) * p->n_total);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_v, sizeof(float) * p->n_total);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_partials, sizeof(float) * p->grad_floats * (size_t)(2 * p->sm_count));
  if (e == cudaSuccess) e = cudaMalloc(&p->d_norm_stats, sizeof(double) * 2 * kNormCtas);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_grid_sync, sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMemset(p->d_grid_sync, 0, sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc(&p->d_comm_dead, sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMemset(p->d_comm_dead, 0, sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaHostAlloc(&p->h_comm_status, sizeof(uint32_t), cudaHostAllocMapped);
  if (e == cudaSuccess) {
    *p->h_comm_status = 0;
    e = cudaHostGetDevicePointer(&p->d_comm_status, p->h_comm_status, 0);
  }
  if (e == cudaSuccess) e = cudaMemset(p->d_params, 0, sizeof(float) * p->n_total);
  if (e == cudaSuccess) e = cudaMemset(p->d_grads, 0, sizeof(float) * p->grad_floats);
  if (e == cudaSuccess) e = cudaMemset(p->d_m, 0, sizeof(float) * p->n_total);
  if (e == cudaSuccess) e = cudaMemset(p->d_v, 0, sizeof(float) * p->n_total);
  if (e != cudaSuccess) {
    wb_policy_destroy(p);
    return fail(WB_ERR_CUDA, "wb_policy_create: %s", cudaGetErrorString(e));
  }
  *out = p;
  return WB_OK;
}

int32_t wb_policy_destroy(wb_policy* p) {
  if (!p) return WB_OK;
  cudaFree(p->d_params);
  cudaFree(p->d_grads);
  cudaFree(p->d_m);
  cudaFree(p->d_v);
  for (int r = 0; r < kExchMaxWorld; r++)
    if (p->opened[r]) cudaIpcCloseMemHandle(p->opened[r]);
  cudaFree(p->d_exch);
  if (p->h_comm_status) cudaFreeHost(p->h_comm_status);
  cudaFree(p->d_norm_stats);
  cudaFree(p->d_grid_sync);
  cudaFree(p->d_comm_dead);
  cudaFree(p->d_partials);
  cudaFree(p->d_stage);
  if (p->h_episode_tab) cudaFreeHost(p->h_episode_tab);
  cudaFree(p->d_episode_tab);
  if (p->episode_tab_copied) cudaEventDestroy(p->episode_tab_copied);
  cudaFree(p->d_episode_scratch);
  delete p;
  return WB_OK;
}

int32_t wb_policy_set_stream(wb_policy* p, void* cuda_stream) {
  WB_REQUIRE(p, "policy is null");
  p->stream = (cudaStream_t)cuda_stream;
  return WB_OK;
}

int32_t wb_policy_set_variant(wb_policy* p, int32_t variant) {
  WB_REQUIRE(p, "policy is null");
  WB_REQUIRE(variant == 0 || variant == 1 || variant == 2, "variant must be 0 (tensor-core), 1 (CUDA-core) or 2 (any-topology kernel)");
  if (!p->default_topology && variant != 2)
    return fail(WB_ERR_UNSUPPORTED, "variants 0 and 1 are specialised for the reference's default networks; this policy runs the any-topology kernel");
  p->variant = variant;
  return WB_OK;
}

int32_t wb_policy_sync(wb_policy* p) {
  WB_REQUIRE(p, "policy is null");
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

int32_t wb_policy_set_hyperparams(wb_policy* p, const wb_hyperparams* hp) {
  WB_REQUIRE(p && hp, "null argument");
  p->hp = *hp;
  return WB_OK;
}

static int32_t which_range(const wb_policy* p, int32_t which, int* off, int* count) {
  if (which == 0) {
    *off = 0;
    *count = p->n_actor;
  } else if (which == 1) {
    *off = p->n_actor;
    *count = p->n_critic;
  } else {
    return fail(WB_ERR_INVALID, "which must be 0 (actor) or 1 (critic)");
  }
  return WB_OK;
}

int32_t wb_policy_num_params(const wb_policy* p, int32_t which, int32_t* n_out) {
  WB_REQUIRE(p && n_out, "null argument");
  int off, count;
  if (int32_t rc = which_range(p, which, &off, &count)) return rc;
  *n_out = count;
  return WB_OK;
}

static int32_t copy_range(wb_policy* p, float* dev_base, int32_t which, const float* src_host, float* dst_host) {
  int off, count;
  if (int32_t rc = which_range(p, which, &off, &count)) return rc;
  if (src_host) WB_CUDA(cudaMemcpyAsync(dev_base + off, src_host, sizeof(float) * count, cudaMemcpyHostToDevice, p->stream));
  if (dst_host) WB_CUDA(cudaMemcpyAsync(dst_host, dev_base + off, sizeof(float) * count, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

int32_t wb_policy_set_weights(wb_policy* p, int32_t which, const float* flat_host) {
  WB_REQUIRE(p && flat_host, "null argument");
  return copy_range(p, p->d_params, which, flat_host, nullptr);
}
int32_t wb_policy_get_weights(wb_policy* p, int32_t which, float* flat_host) {
  WB_REQUIRE(p && flat_host, "null argument");
  return copy_range(p, p->d_params, which, nullptr, flat_host);
}
int32_t wb_policy_get_grads(wb_policy* p, int32_t which, float* flat_host) {
  WB_REQUIRE(p && flat_host, "null argument");
  return copy_range(p, p->d_grads, which, nullptr, flat_host);
}

int32_t wb_policy_get_adam(wb_policy* p, int32_t which, float* m_host, float* v_host, int32_t* iterations_host) {
  WB_REQUIRE(p && m_host && v_host && iterations_host, "null argument");
  if (int32_t rc = copy_range(p, p->d_m, which, nullptr, m_host)) return rc;
  if (int32_t rc = copy_range(p, p->d_v, which, nullptr, v_host)) return rc;
  const int first = which == 0 ? 0 : p->actor.n_dense, cnt = which == 0 ? p->actor.n_dense : p->critic.n_dense;
  for (int i = 0; i < cnt; i++) iterations_host[i] = p->iterations[first + i];
  return WB_OK;
}

int32_t wb_policy_set_adam(wb_policy* p, int32_t which, const float* m_host, const float* v_host, const int32_t* iterations_host) {
  WB_REQUIRE(p && m_host && v_host && iterations_host, "null argument");
  if (int32_t rc = copy_range(p, p->d_m, which, m_host, nullptr)) return rc;
  if (int32_t rc = copy_range(p, p->d_v, which, v_host, nullptr)) return rc;
  const int first = which == 0 ? 0 : p->actor.n_dense, cnt = which == 0 ? p->actor.n_dense : p->critic.n_dense;
  for (int i = 0; i < cnt; i++) p->iterations[first + i] = iterations_host[i];
  return WB_OK;
}

// ---- forward / sample
int32_t wb_policy_forward_dev(wb_policy* p, int32_t n, const float* states_dev, float* mean_dev, float* value_dev) {
  WB_REQUIRE(p && states_dev, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  MlpParams m;
  fill_mlp_common(p, m, n, kModeForward);
  m.states = states_dev;
  m.mean = mean_dev;
  m.value = value_dev;
  WB_CUDA(run_mlp(p, m));
  p->launches++;
  return WB_OK;
}

int32_t wb_policy_forward(wb_policy* p, int32_t n, const float* states_host, float* mean_host, float* value_host) {
  WB_REQUIRE(p && states_host, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  const size_t IN = (size_t)p->actor.input, ACT = (size_t)p->actor.output;
  const size_t N = (size_t)n;
  if (int32_t rc = ensure_stage(p, N * (IN + ACT + 1))) return rc;
  float* d_states = p->d_stage;
  float* d_mean = d_states + N * IN;
  float* d_value = d_mean + N * ACT;
  WB_CUDA(cudaMemcpyAsync(d_states, states_host, sizeof(float) * N * IN, cudaMemcpyHostToDevice, p->stream));
  if (int32_t rc = wb_policy_forward_dev(p, n, d_states, d_mean, d_value)) return rc;
  if (mean_host) WB_CUDA(cudaMemcpyAsync(mean_host, d_mean, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  if (value_host) WB_CUDA(cudaMemcpyAsync(value_host, d_value, sizeof(float) * N, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

int32_t wb_policy_sample_dev(wb_policy* p, int32_t n, const float* states_dev, const float* uniforms_dev, float* actions_dev,
                             float* logp_dev, float* mean_dev) {
  WB_REQUIRE(p && states_dev && uniforms_dev && actions_dev && logp_dev, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  MlpParams m;
  fill_mlp_common(p, m, n, kModeSample);
  m.states = states_dev;
  m.uniforms = uniforms_dev;
  m.out_actions = actions_dev;
  m.out_logp = logp_dev;
  m.mean = mean_dev;
  WB_CUDA(run_mlp(p, m));
  p->launches++;
  return WB_OK;
}

int32_t wb_policy_sample_philox_dev(wb_policy* p, int32_t n, const float* states_dev, uint64_t seed, uint64_t step,
                                    float* actions_dev, float* logp_dev, float* mean_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && logp_dev, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  MlpParams m;
  fill_mlp_common(p, m, n, kModeSamplePhilox);
  m.states = states_dev;
  m.seed = seed;
  m.step = step;
  m.out_actions = actions_dev;
  m.out_logp = logp_dev;
  m.mean = mean_dev;
  WB_CUDA(run_mlp(p, m));
  p->launches++;
  return WB_OK;
}

int32_t wb_policy_act_dev(wb_policy* p, int32_t n, const float* states_dev, uint64_t seed, uint64_t step, float* actions_dev,
                          float* logp_dev, float* mean_dev, float* value_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && logp_dev, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  MlpParams m;
  fill_mlp_common(p, m, n, kModeSamplePhilox);
  m.states = states_dev;
  m.seed = seed;
  m.step = step;
  m.out_actions = actions_dev;
  m.out_logp = logp_dev;
  m.mean = mean_dev;
  m.value = value_dev;
  WB_CUDA(run_mlp(p, m));
  p->launches++;
  return WB_OK;
}

int32_t wb_segment_returns_dev(wb_policy* p, int32_t n_envs, int32_t horizon, const float* rewards_dev, const float* values_dev,
                               const uint8_t* dones_dev, const float* last_values_dev, float* returns_dev, float* advantages_dev) {
  WB_REQUIRE(p && rewards_dev && values_dev && dones_dev && returns_dev && advantages_dev, "null argument");
  WB_REQUIRE(n_envs > 0 && horizon > 0, "n_envs and horizon must be positive");
  WB_CUDA(launch_segment_returns(rewards_dev, values_dev, dones_dev, last_values_dev, n_envs, horizon, p->hp.gamma, p->hp.lambda,
                                 p->hp.use_gae, returns_dev, advantages_dev, p->stream));
  p->launches++;
  if (p->hp.normalize_advantages) return wb_normalize_advantages_dev(p, -1, (int64_t)n_envs * horizon, (int64_t)n_envs * horizon, advantages_dev);
  return WB_OK;
}

int32_t wb_normalize_advantages_dev(wb_policy* p, int32_t stage, int64_t n_local, int64_t n_global, float* advantages_dev) {
  WB_REQUIRE(p && advantages_dev, "null argument");
  WB_REQUIRE(stage >= -1 && stage <= 2, "stage must be -1 (all), 0, 1 or 2");
  WB_REQUIRE(n_local > 0 && n_global >= n_local, "n_local must be positive and n_global >= n_local");
  const int first = stage < 0 ? 0 : stage, last = stage < 0 ? 2 : stage;
  for (int st = first; st <= last; st++) {
    WB_CUDA(launch_normalize_stage(advantages_dev, (long)n_local, (double)n_global, st, p->hp.epsilon, p->d_norm_stats, p->stream));
    p->launches++;
  }
  return WB_OK;
}

int32_t wb_normalize_stats_buffer(wb_policy* p, void** dev_ptr_out, int32_t* n_doubles_out) {
  WB_REQUIRE(p && dev_ptr_out && n_doubles_out, "null argument");
  *dev_ptr_out = p->d_norm_stats;
  *n_doubles_out = 2 * kNormCtas;
  return WB_OK;
}

int32_t wb_gather_minibatch_dev(wb_policy* p, int32_t batch, const int32_t* index_dev, const float* states_pool, const float* actions_pool,
                                const float* logp_pool, const float* advantages_pool, const float* returns_pool, float* states_out,
                                float* actions_out, float* logp_out, float* advantages_out, float* returns_out) {
  WB_REQUIRE(p && index_dev && states_pool && actions_pool && logp_pool && advantages_pool && returns_pool, "null argument");
  WB_REQUIRE(states_out && actions_out && logp_out && advantages_out && returns_out, "null argument");
  WB_REQUIRE(batch > 0, "batch must be positive");
  if (p->actor.input != kIn || p->actor.output != kAct) return fail(WB_ERR_UNSUPPORTED, "the minibatch gather is laid out for 12 observations and 4 actions");
  WB_CUDA(launch_gather_minibatch(index_dev, batch, states_pool, actions_pool, logp_pool, advantages_pool, returns_pool, states_out,
                                  actions_out, logp_out, advantages_out, returns_out, p->stream));
  p->launches++;
  return WB_OK;
}

int32_t wb_policy_sample(wb_policy* p, int32_t n, const float* states_host, const float* uniforms_host, float* actions_host,
                         float* logp_host, float* mean_host) {
  WB_REQUIRE(p && states_host && uniforms_host && actions_host && logp_host, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  const size_t IN = (size_t)p->actor.input, ACT = (size_t)p->actor.output;
  const size_t N = (size_t)n;
  if (int32_t rc = ensure_stage(p, N * (IN + ACT * 2 + ACT * 3))) return rc;
  float* d_states = p->d_stage;
  float* d_uni = d_states + N * IN;
  float* d_act = d_uni + N * ACT * 2;
  float* d_logp = d_act + N * ACT;
  float* d_mean = d_logp + N * ACT;
  WB_CUDA(cudaMemcpyAsync(d_states, states_host, sizeof(float) * N * IN, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_uni, uniforms_host, sizeof(float) * N * ACT * 2, cudaMemcpyHostToDevice, p->stream));
  if (int32_t rc = wb_policy_sample_dev(p, n, d_states, d_uni, d_act, d_logp, d_mean)) return rc;
  WB_CUDA(cudaMemcpyAsync(actions_host, d_act, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaMemcpyAsync(logp_host, d_logp, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  if (mean_host) WB_CUDA(cudaMemcpyAsync(mean_host, d_mean, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

// ---- gradient
int32_t wb_ppo_grad_dev(wb_policy* p, int32_t n, const float* states_dev, const float* actions_dev, const float* old_logp_dev,
                        const float* advantages_dev, const float* returns_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && old_logp_dev && advantages_dev && returns_dev, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  WB_REQUIRE(p->hp.batch_size > 0, "batch_size must be positive");
  MlpParams m;
  fill_mlp_common(p, m, n, kModeGrad);
  m.states = states_dev;
  m.actions = actions_dev;
  m.old_logp = old_logp_dev;
  m.advantages = advantages_dev;
  m.returns = returns_dev;
  m.partials = p->d_partials;
  const int grid = grid_of(p, n);
  WB_CUDA(run_mlp(p, m));
  WB_CUDA(reduce_grads(p, grid));
  p->launches += 2;
  return WB_OK;
}

/* ---- fused gradient reduction + all-reduce over NVLink peer memory ---- */
int32_t wb_comm_local_handle(wb_policy* p, void* handle64_out) {
  WB_REQUIRE(p && handle64_out, "null argument");
  if (use_generic(p))
    return fail(WB_ERR_UNSUPPORTED, "the fused NVLink gradient exchange is built for the default networks' 6152-float buffer; other topologies "
                                    "all-reduce wb_policy_grad_buffer with NCCL (wb_ppo_grad_dev + all-reduce + wb_adam_step)");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  if (!p->d_exch) {
    WB_CUDA(cudaMalloc(&p->d_exch, kExchBytes));
    WB_CUDA(cudaMemset(p->d_exch, 0, kExchBytes));
    WB_CUDA(cudaDeviceSynchronize());
  }
  cudaIpcMemHandle_t h;
  WB_CUDA(cudaIpcGetMemHandle(&h, p->d_exch));
  memcpy(handle64_out, &h, sizeof(h));
  return WB_OK;
}

int32_t wb_comm_connect(wb_policy* p, int32_t rank, int32_t world, const void* all_handles64) {
  WB_REQUIRE(p && all_handles64, "null argument");
  WB_REQUIRE(world >= 1 && world <= kExchMaxWorld && rank >= 0 && rank < world, "world must be 1..8 and 0 <= rank < world");
  WB_REQUIRE(p->d_exch, "call wb_comm_local_handle first");
  for (int r = 0; r < world; r++) {
    if (r == rank) {
      p->peers.base[r] = p->d_exch;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)all_handles64 + (size_t)r * sizeof(h), sizeof(h));
    void* ptr = nullptr;
    WB_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    p->opened[r] = ptr;
    p->peers.base[r] = (float*)ptr;
  }
  p->comm_rank = rank;
  p->comm_world = world;
  p->comm_epoch = 0;
  return WB_OK;
}

int32_t wb_comm_status(wb_policy* p, int32_t* connected_world_out, int32_t* failed_out) {
  WB_REQUIRE(p && connected_world_out && failed_out, "null argument");
  *connected_world_out = p->comm_world;
  WB_CUDA(cudaStreamSynchronize(p->stream));
  *failed_out = (int32_t)*reinterpret_cast<volatile uint32_t*>(p->h_comm_status);
  return WB_OK;
}

int32_t wb_ppo_grad_allreduce_dev(wb_policy* p, int32_t n, const float* states_dev, const float* actions_dev, const float* old_logp_dev,
                                  const float* advantages_dev, const float* returns_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && old_logp_dev && advantages_dev && returns_dev, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  WB_REQUIRE(p->hp.batch_size > 0, "batch_size must be positive");
  WB_REQUIRE(p->comm_world >= 1, "not connected: call wb_comm_local_handle / wb_comm_connect on every rank first");
  WB_REQUIRE(!use_generic(p), "the fused exchange needs the default networks and kernel variant 0 or 1");
  if (int32_t rc = comm_healthy(p)) return rc;
  MlpParams m;
  fill_mlp_common(p, m, n, kModeGrad);
  m.states = states_dev;
  m.actions = actions_dev;
  m.old_logp = old_logp_dev;
  m.advantages = advantages_dev;
  m.returns = returns_dev;
  m.partials = p->d_partials;
  const int grid = grid_of(p, n);
  WB_CUDA(run_mlp(p, m));
  p->comm_epoch++;
  WB_CUDA(launch_reduce_exchange(p->d_partials, grid, p->d_grads, p->peers, p->comm_rank, p->comm_world, p->comm_epoch, p->d_comm_status,
                                 p->d_comm_dead, nullptr, p->stream));
  p->launches += 2;
  return WB_OK;
}

// DenseLayer.Adam bookkeeping: every dense layer's step counter advances (DenseLayer.cs:127) and its bias corrections are
// (float)(1 - Math.Pow(beta, t)) (:142-145)
static void next_corrections(wb_policy* p, float* corr1, float* corr2) {
  const int n_dense = p->actor.n_dense + p->critic.n_dense;
  for (int l = 0; l < n_dense; l++) {
    p->iterations[l] += 1;
    corr1[l] = (float)(1.0 - pow((double)p->hp.beta1, (double)p->iterations[l]));
    corr2[l] = (float)(1.0 - pow((double)p->hp.beta2, (double)p->iterations[l]));
  }
}
static void next_adam_params(wb_policy* p, AdamParams& a) {  // default networks: 3 + 2 dense layers
  a = AdamParams{};
  a.params = p->d_params;
  a.grads = p->d_grads;
  a.m = p->d_m;
  a.v = p->d_v;
  a.alpha = p->hp.alpha;
  a.beta1 = p->hp.beta1;
  a.beta2 = p->hp.beta2;
  a.eps = p->hp.adam_epsilon;
  next_corrections(p, a.corr1, a.corr2);
}
static cudaError_t adam_any(wb_policy* p) {
  if (p->default_topology) {
    AdamParams a;
    next_adam_params(p, a);
    return launch_adam(a, p->stream);
  }
  GenAdamParams g{};
  g.params = p->d_params;
  g.grads = p->d_grads;
  g.m = p->d_m;
  g.v = p->d_v;
  g.n_params = p->n_total;
  g.n_dense = generic_layer_ends(p->actor, p->critic, g.layer_end);
  g.alpha = p->hp.alpha;
  g.beta1 = p->hp.beta1;
  g.beta2 = p->hp.beta2;
  g.eps = p->hp.adam_epsilon;
  next_corrections(p, g.corr1, g.corr2);
  return launch_adam_generic(g, p->stream);
}

// the five device inputs of a gradient call + an optional row index (PPOAgent.CreateBatches fused into the kernel's prefetch)
struct TrainInputs {
  const float *states, *actions, *old_logp, *advantages, *returns;
  const int32_t* index;
};

static int32_t train_on_device(wb_policy* p, int32_t n, TrainInputs in) {
  WB_REQUIRE(n > 0, "n must be positive");
  WB_REQUIRE(p->hp.batch_size > 0, "batch_size must be positive");
  if (int32_t rc = comm_healthy(p)) return rc;
  const int world = p->comm_world >= 2 ? p->comm_world : 1;
  const int grid = grid_of(p, n);
  const bool one_launch = !use_generic(p) && p->variant == 0 && grid <= p->sm_count;
  if (in.index && !one_launch) {
    // the other kernels read contiguous minibatches: gather the rows first (PPOAgent.CreateBatches as its own launch)
    if (p->actor.input != kIn || p->actor.output != kAct)
      return fail(WB_ERR_UNSUPPORTED, "the minibatch gather is laid out for 12 observations and 4 actions");
    const size_t N = (size_t)n;
    if (int32_t rc = ensure_stage(p, N * (kIn + kAct + kAct + 2))) return rc;
    float* g_states = p->d_stage;
    float* g_actions = g_states + N * kIn;
    float* g_logp = g_actions + N * kAct;
    float* g_adv = g_logp + N * kAct;
    float* g_ret = g_adv + N;
    WB_CUDA(launch_gather_minibatch(in.index, n, in.states, in.actions, in.old_logp, in.advantages, in.returns, g_states, g_actions, g_logp,
                                    g_adv, g_ret, p->stream));
    p->launches++;
    in = TrainInputs{g_states, g_actions, g_logp, g_adv, g_ret, nullptr};
  }
  MlpParams m;
  fill_mlp_common(p, m, n, kModeGrad);
  m.states = in.states;
  m.actions = in.actions;
  m.old_logp = in.old_logp;
  m.advantages = in.advantages;
  m.returns = in.returns;
  m.index = in.index;
  m.partials = p->d_partials;
  if (use_generic(p)) {  // any topology: reduction and Adam as separate launches (single rank; data-parallel callers use the NCCL path)
    WB_REQUIRE(p->comm_world < 2, "a connected policy needs the default networks and kernel variant 0 or 1");
    WB_CUDA(run_mlp(p, m));
    WB_CUDA(reduce_grads(p, grid));
    WB_CUDA(adam_any(p));
    p->launches += 3;
    return WB_OK;
  }
  AdamParams a;
  next_adam_params(p, a);
  if (one_launch) {
    // ONE launch: the tensor-core gradient kernel reduces its own partials behind a grid barrier (the grid is persistent, one CTA
    // per SM, so every CTA is resident), exchanges its slices with the peers over NVLink when connected, and applies Adam
    FusedTail t{};
    t.enabled = 1;
    t.counter = p->d_grid_sync;
    p->grid_sync_target += (uint32_t)grid;
    t.target = p->grid_sync_target;
    t.grads = p->d_grads;
    t.adam = a;
    t.world = world;
    if (world > 1) {
      t.peers = p->peers;
      t.rank = p->comm_rank;
      t.epoch = ++p->comm_epoch;
      t.status = p->d_comm_status;
      t.dead = p->d_comm_dead;
    }
    WB_CUDA(launch_mlp_tc(m, grid, p->stream, &t));
    p->launches += 1;
    return WB_OK;
  }
  WB_CUDA(run_mlp(p, m));
  if (world > 1) p->comm_epoch++;
  WB_CUDA(launch_reduce_exchange(p->d_partials, grid, p->d_grads, p->peers, world > 1 ? p->comm_rank : 0, world, p->comm_epoch,
                                 p->d_comm_status, p->d_comm_dead, &a, p->stream));
  p->launches += 2;
  return WB_OK;
}

int32_t wb_ppo_train_dev(wb_policy* p, int32_t n, const float* states_dev, const float* actions_dev, const float* old_logp_dev,
                         const float* advantages_dev, const float* returns_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && old_logp_dev && advantages_dev && returns_dev, "null argument");
  return train_on_device(p, n, TrainInputs{states_dev, actions_dev, old_logp_dev, advantages_dev, returns_dev, nullptr});
}

int32_t wb_ppo_train_indexed_dev(wb_policy* p, int32_t n, const int32_t* index_dev, const float* states_pool, const float* actions_pool,
                                 const float* logp_pool, const float* advantages_pool, const float* returns_pool) {
  WB_REQUIRE(p && index_dev && states_pool && actions_pool && logp_pool && advantages_pool && returns_pool, "null argument");
  return train_on_device(p, n, TrainInputs{states_pool, actions_pool, logp_pool, advantages_pool, returns_pool, index_dev});
}

// device view of a host minibatch: the buffers' own device aliases when all five are page-locked (the kernel then reads them over
// PCIe while it computes: no staging copy), else a staged copy
static int32_t minibatch_on_device(wb_policy* p, int32_t n, const float* states_host, const float* actions_host, const float* old_logp_host,
                                   const float* advantages_host, const float* returns_host, TrainInputs* out) {
  const size_t IN = (size_t)p->actor.input, ACT = (size_t)p->actor.output;
  const size_t N = (size_t)n;
  static const bool zero_copy_enabled = getenv("WB_NO_ZERO_COPY") == nullptr;
  // (only the tensor-core kernel streams every input exactly once through a prefetch that hides the PCIe latency)
  if (zero_copy_enabled && !use_generic(p) && p->variant == 0) {
    const float* s = static_cast<const float*>(device_alias_of_pinned(states_host, sizeof(float) * N * IN));
    const float* a = static_cast<const float*>(device_alias_of_pinned(actions_host, sizeof(float) * N * ACT));
    const float* l = static_cast<const float*>(device_alias_of_pinned(old_logp_host, sizeof(float) * N * ACT));
    const float* ad = static_cast<const float*>(device_alias_of_pinned(advantages_host, sizeof(float) * N));
    const float* r = static_cast<const float*>(device_alias_of_pinned(returns_host, sizeof(float) * N));
    const uintptr_t all = reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(l) |
                          reinterpret_cast<uintptr_t>(ad) | reinterpret_cast<uintptr_t>(r);
    if (s && a && l && ad && r && (all & 15) == 0) {  // (the kernels use vector loads)
      *out = TrainInputs{s, a, l, ad, r, nullptr};
      return WB_OK;
    }
  }
  if (int32_t rc = ensure_stage(p, N * (IN + ACT + ACT + 2))) return rc;
  float* d_states = p->d_stage;
  float* d_actions = d_states + N * IN;
  float* d_logp = d_actions + N * ACT;
  float* d_adv = d_logp + N * ACT;
  float* d_ret = d_adv + N;
  WB_CUDA(cudaMemcpyAsync(d_states, states_host, sizeof(float) * N * IN, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_actions, actions_host, sizeof(float) * N * ACT, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_logp, old_logp_host, sizeof(float) * N * ACT, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_adv, advantages_host, sizeof(float) * N, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_ret, returns_host, sizeof(float) * N, cudaMemcpyHostToDevice, p->stream));
  *out = TrainInputs{d_states, d_actions, d_logp, d_adv, d_ret, nullptr};
  return WB_OK;
}

static int32_t read_losses(wb_policy* p, float* losses_host, int32_t* skipped_host) {
  float tail[3] = {0.f, 0.f, 0.f};
  WB_CUDA(cudaMemcpyAsync(tail, p->d_grads + p->n_total, sizeof(tail), cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  if (losses_host) {
    losses_host[0] = tail[0];
    losses_host[1] = tail[1];
  }
  if (skipped_host) *skipped_host = (int32_t)tail[2];
  return WB_OK;
}

int32_t wb_ppo_grad(wb_policy* p, int32_t n, const float* states_host, const float* actions_host, const float* old_logp_host,
                    const float* advantages_host, const float* returns_host, float* losses_host, int32_t* skipped_host) {
  WB_REQUIRE(p && states_host && actions_host && old_logp_host && advantages_host && returns_host, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  TrainInputs in{};
  if (int32_t rc = minibatch_on_device(p, n, states_host, actions_host, old_logp_host, advantages_host, returns_host, &in)) return rc;
  if (int32_t rc = wb_ppo_grad_dev(p, n, in.states, in.actions, in.old_logp, in.advantages, in.returns)) return rc;
  return read_losses(p, losses_host, skipped_host);
}

int32_t wb_ppo_train(wb_policy* p, int32_t n, const float* states_host, const float* actions_host, const float* old_logp_host,
                     const float* advantages_host, const float* returns_host, float* losses_host, int32_t* skipped_host) {
  WB_REQUIRE(p && states_host && actions_host && old_logp_host && advantages_host && returns_host, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  TrainInputs in{};
  if (int32_t rc = minibatch_on_device(p, n, states_host, actions_host, old_logp_host, advantages_host, returns_host, &in)) return rc;
  if (int32_t rc = train_on_device(p, n, in)) return rc;
  return read_losses(p, losses_host, skipped_host);
}

int32_t wb_adam_step(wb_policy* p) {
  WB_REQUIRE(p, "policy is null");
  WB_CUDA(adam_any(p));
  p->launches++;
  return WB_OK;
}

int32_t wb_policy_grad_buffer(wb_policy* p, void** dev_ptr_out, int32_t* n_floats_out) {
  WB_REQUIRE(p && dev_ptr_out && n_floats_out, "null argument");
  *dev_ptr_out = p->d_grads;
  *n_floats_out = p->grad_floats;
  return WB_OK;
}

int32_t wb_policy_launch_count(const wb_policy* p, int64_t* count_out) {
  WB_REQUIRE(p && count_out, "null argument");
  *count_out = p->launches;
  return WB_OK;
}

int32_t wb_returns_advantages(wb_policy* p, int32_t n, const float* rewards_host, const float* values_host, float* returns_host,
                              float* advantages_host) {
  WB_REQUIRE(p && rewards_host && values_host && returns_host && advantages_host, "null argument");
  WB_REQUIRE(n > 0, "n must be positive");
  const size_t N = (size_t)n;
  if (int32_t rc = ensure_stage(p, N * 4)) return rc;
  float* d_r = p->d_stage;
  float* d_v = d_r + N;
  float* d_G = d_v + N;
  float* d_A = d_G + N;
  WB_CUDA(cudaMemcpyAsync(d_r, rewards_host, sizeof(float) * N, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_v, values_host, sizeof(float) * N, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(launch_returns(d_r, d_v, n, p->hp.gamma, p->hp.lambda, p->hp.use_gae, p->hp.normalize_advantages, p->hp.epsilon, d_G, d_A,
                         p->stream));
  p->launches++;
  WB_CUDA(cudaMemcpyAsync(returns_host, d_G, sizeof(float) * N, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaMemcpyAsync(advantages_host, d_A, sizeof(float) * N, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

// ---- PPOAgent.Train(Trajectory) for a list of trajectories
// offsets: non-decreasing, offsets[0] >= 0; counts the Adam steps (epochs x floor(T_e / B) per trajectory) and index entries
static int32_t check_trajectories(const wb_policy* p, int32_t n_traj, const int32_t* offsets_host, int32_t epochs, int64_t* steps,
                                  int64_t* n_index) {
  WB_REQUIRE(offsets_host, "offsets_host is null");
  WB_REQUIRE(n_traj >= 1, "n_traj must be at least 1");
  WB_REQUIRE(epochs >= 0, "epochs must be >= 0");
  WB_REQUIRE(p->hp.batch_size >= 1, "hp.batch_size must be positive");
  if (p->comm_world > 1)
    return fail(WB_ERR_UNSUPPORTED, "the per-episode schedule is single-process (PPOAgent.cs:147-172); this policy is connected for data-parallel exchange");
  WB_REQUIRE(offsets_host[0] >= 0, "offsets[0] must be >= 0");
  *steps = 0;
  *n_index = 0;
  for (int32_t e = 0; e < n_traj; e++) {
    if (offsets_host[e + 1] < offsets_host[e]) return fail(WB_ERR_INVALID, "offsets must be non-decreasing (offsets[%d] > offsets[%d])", e, e + 1);
    const int64_t nb = (int64_t)epochs * ((offsets_host[e + 1] - offsets_host[e]) / p->hp.batch_size);
    *steps += nb;
    *n_index += nb * p->hp.batch_size;
  }
  WB_REQUIRE(*n_index <= INT32_MAX, "too many mini-batch indices for one call");
  return WB_OK;
}

static int32_t grow(float** buf, size_t* have, size_t want) {
  if (want <= *have) return WB_OK;
  cudaFree(*buf);
  *buf = nullptr;
  *have = 0;
  WB_CUDA(cudaMalloc(buf, want * sizeof(float)));
  *have = want;
  return WB_OK;
}

int32_t wb_ppo_train_trajectories_dev(wb_policy* p, int32_t n_traj, const int32_t* offsets_host, int32_t epochs, const float* states_dev,
                                      const float* actions_dev, const float* old_logp_dev, const float* rewards_dev,
                                      const int32_t* batch_index_dev, float* values_dev, float* returns_dev, float* advantages_dev,
                                      float* losses_dev, int32_t* skipped_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && old_logp_dev && rewards_dev, "null argument");
  int64_t steps = 0, n_index = 0;
  if (int32_t rc = check_trajectories(p, n_traj, offsets_host, epochs, &steps, &n_index)) return rc;
  WB_REQUIRE(batch_index_dev || n_index == 0, "batch_index is null");
  const size_t rows = (size_t)offsets_host[n_traj];
  const int B = p->hp.batch_size;
  const size_t IN = (size_t)p->actor.input, ACT = (size_t)p->actor.output;
  // Trajectory.Values / Returns / Advantages the caller does not want, and the sequenced path's gathered mini-batch
  const size_t mb_floats = use_generic(p) ? (size_t)B * (IN + 2 * ACT + 2) : 0;
  const size_t scratch_rows = (values_dev ? 0 : rows) + (returns_dev ? 0 : rows) + (advantages_dev ? 0 : rows);
  if (int32_t rc = grow(&p->d_episode_scratch, &p->episode_scratch_floats, scratch_rows + mb_floats + 1)) return rc;
  float* scratch = p->d_episode_scratch;
  if (!values_dev) { values_dev = scratch; scratch += rows; }
  if (!returns_dev) { returns_dev = scratch; scratch += rows; }
  if (!advantages_dev) { advantages_dev = scratch; scratch += rows; }

  if (use_generic(p)) {
    // networks the one-launch kernel does not cover: the per-trajectory / per-mini-batch kernels, enqueued without a host sync
    float* g_states = scratch;
    float* g_actions = g_states + (size_t)B * IN;
    float* g_logp = g_actions + (size_t)B * ACT;
    float* g_adv = g_logp + (size_t)B * ACT;
    float* g_ret = g_adv + B;
    if (losses_dev) WB_CUDA(cudaMemsetAsync(losses_dev, 0, sizeof(float) * 2 * n_traj, p->stream));
    if (skipped_dev) WB_CUDA(cudaMemsetAsync(skipped_dev, 0, sizeof(int32_t) * n_traj, p->stream));
    const int32_t* index = batch_index_dev;
    for (int32_t e = 0; e < n_traj; e++) {
      const int r0 = offsets_host[e], T = offsets_host[e + 1] - r0;
      if (T == 0) continue;
      MlpParams f;
      fill_mlp_common(p, f, T, kModeForward);
      f.states = states_dev + (size_t)r0 * IN;
      f.value = values_dev + r0;
      WB_CUDA(run_mlp(p, f));
      WB_CUDA(launch_returns(rewards_dev + r0, values_dev + r0, T, p->hp.gamma, p->hp.lambda, p->hp.use_gae, p->hp.normalize_advantages,
                             p->hp.epsilon, returns_dev + r0, advantages_dev + r0, p->stream));
      p->launches += 2;
      const int nb = epochs * (T / B);
      for (int b = 0; b < nb; b++, index += B) {
        WB_CUDA(launch_gather_rows(index, B, r0, (int)IN, (int)ACT, states_dev, actions_dev, old_logp_dev, advantages_dev, returns_dev, g_states,
                                   g_actions, g_logp, g_adv, g_ret, p->stream));
        MlpParams m;
        fill_mlp_common(p, m, B, kModeGrad);
        m.states = g_states;
        m.actions = g_actions;
        m.old_logp = g_logp;
        m.advantages = g_adv;
        m.returns = g_ret;
        m.partials = p->d_partials;
        WB_CUDA(run_mlp(p, m));
        WB_CUDA(reduce_grads(p, grid_of(p, B)));
        WB_CUDA(adam_any(p));
        WB_CUDA(launch_episode_losses(p->d_grads + p->n_total, losses_dev ? losses_dev + 2 * e : nullptr, skipped_dev ? skipped_dev + e : nullptr,
                                      p->stream));
        p->launches += 5;
      }
    }
    return WB_OK;
  }

  // default networks: ONE launch.  Table = device offsets [n_traj + 1] then the Adam bias corrections [steps][10] (next_corrections,
  // the function every other Adam entry uses, so wb_policy_get_adam reports what the per-mini-batch path reports)
  const size_t off_bytes = ((sizeof(int32_t) * (n_traj + 1)) + 15) / 16 * 16;
  const size_t tab_bytes = off_bytes + sizeof(float) * 10 * (size_t)steps;
  if (!p->episode_tab_copied) WB_CUDA(cudaEventCreateWithFlags(&p->episode_tab_copied, cudaEventDisableTiming));
  WB_CUDA(cudaEventSynchronize(p->episode_tab_copied));  // (the previous call's upload has read the pinned copy)
  if (tab_bytes > p->episode_tab_bytes) {
    if (p->h_episode_tab) cudaFreeHost(p->h_episode_tab);
    cudaFree(p->d_episode_tab);
    p->h_episode_tab = nullptr;
    p->d_episode_tab = nullptr;
    p->episode_tab_bytes = 0;
    WB_CUDA(cudaHostAlloc(&p->h_episode_tab, tab_bytes, cudaHostAllocDefault));
    WB_CUDA(cudaMalloc(&p->d_episode_tab, tab_bytes));
    p->episode_tab_bytes = tab_bytes;
  }
  memcpy(p->h_episode_tab, offsets_host, sizeof(int32_t) * (n_traj + 1));
  float* corr = reinterpret_cast<float*>(p->h_episode_tab + off_bytes);
  for (int64_t st = 0; st < steps; st++) next_corrections(p, corr + 10 * st, corr + 10 * st + 5);
  WB_CUDA(cudaMemcpyAsync(p->d_episode_tab, p->h_episode_tab, tab_bytes, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaEventRecord(p->episode_tab_copied, p->stream));
  EpisodeParams e{};
  e.rewards = rewards_dev;
  e.values = values_dev;
  e.returns = returns_dev;
  e.advantages = advantages_dev;
  e.offsets = reinterpret_cast<const int32_t*>(p->d_episode_tab);
  e.batch_index = batch_index_dev;
  e.corr = reinterpret_cast<const float*>(p->d_episode_tab + off_bytes);
  e.grads = p->d_grads;
  e.losses = losses_dev;
  e.skipped = skipped_dev;
  e.adam.params = p->d_params;
  e.adam.grads = p->d_grads;
  e.adam.m = p->d_m;
  e.adam.v = p->d_v;
  e.adam.alpha = p->hp.alpha;
  e.adam.beta1 = p->hp.beta1;
  e.adam.beta2 = p->hp.beta2;
  e.adam.eps = p->hp.adam_epsilon;
  e.n_traj = n_traj;
  e.epochs = epochs;
  e.batch = B;
  e.use_gae = p->hp.use_gae;
  e.normalize = p->hp.normalize_advantages;
  e.gamma = p->hp.gamma;
  e.lambda = p->hp.lambda;
  e.norm_eps = p->hp.epsilon;
  MlpParams m;
  fill_mlp_common(p, m, (int)rows, kModeGrad);
  m.states = states_dev;
  m.actions = actions_dev;
  m.old_logp = old_logp_dev;
  m.advantages = advantages_dev;
  m.returns = returns_dev;
  WB_CUDA(launch_episodes(e, m, p->stream));
  p->launches++;
  return WB_OK;
}

int32_t wb_ppo_train_trajectories(wb_policy* p, int32_t n_traj, const int32_t* offsets_host, int32_t epochs, const float* states_host,
                                  const float* actions_host, const float* old_logp_host, const float* rewards_host,
                                  const int32_t* batch_index_host, float* values_host, float* returns_host, float* advantages_host,
                                  float* losses_host, int32_t* skipped_host) {
  WB_REQUIRE(p && states_host && actions_host && old_logp_host && rewards_host, "null argument");
  int64_t steps = 0, n_index = 0;
  if (int32_t rc = check_trajectories(p, n_traj, offsets_host, epochs, &steps, &n_index)) return rc;
  WB_REQUIRE(batch_index_host || n_index == 0, "batch_index is null");
  // every index must be a local row of its trajectory: checked before anything on the device changes
  {
    const int B = p->hp.batch_size;
    const int32_t* ix = batch_index_host;
    for (int32_t e = 0; e < n_traj; e++) {
      const int T = offsets_host[e + 1] - offsets_host[e];
      const int64_t cnt = (int64_t)epochs * (T / B) * B;
      for (int64_t i = 0; i < cnt; i++, ix++)
        if (*ix < 0 || *ix >= T) return fail(WB_ERR_INVALID, "batch_index of trajectory %d holds %d, outside its %d rows", e, *ix, T);
    }
  }
  const size_t rows = (size_t)offsets_host[n_traj];
  const size_t IN = (size_t)p->actor.input, ACT = (size_t)p->actor.output, N = (size_t)n_traj;
  const size_t floats = rows * (IN + 2 * ACT + 4) + (size_t)n_index + 3 * N + 8;
  if (int32_t rc = ensure_stage(p, floats)) return rc;
  float* d_states = p->d_stage;
  float* d_actions = d_states + rows * IN;
  float* d_logp = d_actions + rows * ACT;
  float* d_rewards = d_logp + rows * ACT;
  float* d_values = d_rewards + rows;
  float* d_returns = d_values + rows;
  float* d_adv = d_returns + rows;
  float* d_losses = d_adv + rows;
  int32_t* d_skipped = reinterpret_cast<int32_t*>(d_losses + 2 * N);
  int32_t* d_index = d_skipped + N;
  if (rows) {
    WB_CUDA(cudaMemcpyAsync(d_states, states_host, sizeof(float) * rows * IN, cudaMemcpyHostToDevice, p->stream));
    WB_CUDA(cudaMemcpyAsync(d_actions, actions_host, sizeof(float) * rows * ACT, cudaMemcpyHostToDevice, p->stream));
    WB_CUDA(cudaMemcpyAsync(d_logp, old_logp_host, sizeof(float) * rows * ACT, cudaMemcpyHostToDevice, p->stream));
    WB_CUDA(cudaMemcpyAsync(d_rewards, rewards_host, sizeof(float) * rows, cudaMemcpyHostToDevice, p->stream));
  }
  if (n_index) WB_CUDA(cudaMemcpyAsync(d_index, batch_index_host, sizeof(int32_t) * n_index, cudaMemcpyHostToDevice, p->stream));
  if (int32_t rc = wb_ppo_train_trajectories_dev(p, n_traj, offsets_host, epochs, d_states, d_actions, d_logp, d_rewards, d_index, d_values,
                                                 d_returns, d_adv, d_losses, d_skipped))
    return rc;
  if (rows) {
    if (values_host) WB_CUDA(cudaMemcpyAsync(values_host, d_values, sizeof(float) * rows, cudaMemcpyDeviceToHost, p->stream));
    if (returns_host) WB_CUDA(cudaMemcpyAsync(returns_host, d_returns, sizeof(float) * rows, cudaMemcpyDeviceToHost, p->stream));
    if (advantages_host) WB_CUDA(cudaMemcpyAsync(advantages_host, d_adv, sizeof(float) * rows, cudaMemcpyDeviceToHost, p->stream));
  }
  if (losses_host) WB_CUDA(cudaMemcpyAsync(losses_host, d_losses, sizeof(float) * 2 * N, cudaMemcpyDeviceToHost, p->stream));
  if (skipped_host) WB_CUDA(cudaMemcpyAsync(skipped_host, d_skipped, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

int32_t wb_debug_tc_gemm(int32_t M, int32_t N, int32_t K, int32_t a_mn_major, int32_t b_mn_major, int32_t passes, const float* A_host,
                         const float* B_host, float* D_host) {
  WB_REQUIRE(A_host && B_host && D_host, "null argument");
  WB_REQUIRE((M == 64 || M == 128) && N >= 8 && N <= 128 && N % 8 == 0 && K >= 8 && K % 8 == 0, "unsupported test shape");
  WB_REQUIRE(sizeof(float) * 2 * ((size_t)M * K + (size_t)N * K) <= 200 * 1024, "test shape exceeds shared memory");
  if (int32_t rc = require_device()) return rc;
  float *dA = nullptr, *dB = nullptr, *dD = nullptr;
  WB_CUDA(cudaMalloc(&dA, sizeof(float) * M * K));
  WB_CUDA(cudaMalloc(&dB, sizeof(float) * N * K));
  WB_CUDA(cudaMalloc(&dD, sizeof(float) * M * N));
  cudaError_t e = cudaMemcpy(dA, A_host, sizeof(float) * M * K, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dB, B_host, sizeof(float) * N * K, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(dD, 0, sizeof(float) * M * N);
  if (e == cudaSuccess) e = launch_tc_gemm_test(dA, dB, dD, M, N, K, a_mn_major, b_mn_major, passes, nullptr);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(D_host, dD, sizeof(float) * M * N, cudaMemcpyDeviceToHost);
  cudaFree(dA);
  cudaFree(dB);
  cudaFree(dD);
  if (e != cudaSuccess) return fail(WB_ERR_CUDA, "wb_debug_tc_gemm: %s", cudaGetErrorString(e));
  return WB_OK;
}

}  // extern "C"

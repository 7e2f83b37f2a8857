// mlp.cuh -- declarations shared by the PPO kernels (mlp.cu) and the policy C ABI (api_policy.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/walker_b200.h"

namespace wb {

// The reference's default topologies (Hyperparameters.cs:91-92): the fused kernels are specialised for them.
//   actor : 12 -> 64 LeakyReLU -> 64 LeakyReLU -> 4 TanH        (5 252 parameters)
//   critic: 12 -> 64 LeakyReLU -> 1                             (  897 parameters)
constexpr int kIn = 12, kHid = 64, kAct = 4;
// flat parameter layout (DenseLayer.Save order: W[out][in] row-major then b[out], layer after layer)
constexpr int kOffW1 = 0;                       // [64][12]
constexpr int kOffB1 = kOffW1 + kHid * kIn;     // 768
constexpr int kOffW2 = kOffB1 + kHid;           // 832   [64][64]
constexpr int kOffB2 = kOffW2 + kHid * kHid;    // 4928
constexpr int kOffW3 = kOffB2 + kHid;           // 4992  [4][64]
constexpr int kOffB3 = kOffW3 + kAct * kHid;    // 5248
constexpr int kActorParams = kOffB3 + kAct;     // 5252
constexpr int kOffWc1 = kActorParams;           // [64][12]
constexpr int kOffBc1 = kOffWc1 + kHid * kIn;   // +768
constexpr int kOffWc2 = kOffBc1 + kHid;         // [1][64]
constexpr int kOffBc2 = kOffWc2 + kHid;
constexpr int kTotalParams = kOffBc2 + 1;       // 6149
constexpr int kCriticParams = kTotalParams - kActorParams;  // 897
// gradient buffer: [6149 grads | sum g_V | sum mean_k g_mu | skipped samples] padded to a float4 multiple
constexpr int kGradLossV = kTotalParams;
constexpr int kGradLossA = kTotalParams + 1;
constexpr int kGradSkipped = kTotalParams + 2;
constexpr int kGradFloats = 6152;

constexpr int kTile = 64;        // samples per CTA iteration
constexpr int kMlpThreads = 256;

enum : int { kModeForward = 0, kModeSample = 1, kModeSamplePhilox = 2, kModeGrad = 3 };

struct MlpParams {
  const float* params;  // [6149] actor | critic
  int32_t n;
  int32_t mode;
  // inputs
  const float* states;     // [n][12]
  const float* actions;    // [n][4]   (grad)
  const float* old_logp;   // [n][4]   (grad)
  const float* advantages; // [n]      (grad)
  const float* returns;    // [n]      (grad)
  const float* uniforms;   // [n][4][2] (sample)
  // (grad, tensor-core kernel only) sample s of the call is row index[s] of the five input arrays -- PPOAgent.CreateBatches fused
  // into the gradient kernel's input prefetch; nullptr = row s
  const int32_t* index;
  uint64_t seed, step;     // (sample, philox)
  // outputs
  float* mean;         // [n][4] or null
  float* value;        // [n] or null
  float* out_actions;  // [n][4] (sample)
  float* out_logp;     // [n][4] (sample)
  float* partials;     // [grid][kGradFloats] (grad)
  // hyper-parameters
  float log_std, epsilon, batch_size;
};

struct AdamParams {
  float* params;
  const float* grads;
  float* m;
  float* v;
  float alpha, beta1, beta2, eps;
  // bias corrections (float)(1 - Math.Pow(beta, t)) per dense layer: actor L1,L2,L3, critic L1,L2
  float corr1[5], corr2[5];
};

#ifdef __CUDACC__
// DenseLayer.Adam for one parameter (DenseLayer.cs:125-159; every product and sum individually rounded, as the Matrix operators do)
__device__ __forceinline__ void adam_update(const AdamParams& a, int i, float g) {
  const int layer = (i < kOffW2) ? 0 : (i < kOffW3) ? 1 : (i < kActorParams) ? 2 : (i < kOffWc2) ? 3 : 4;
  const float m = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, a.beta1), g), __fmul_rn(a.beta1, a.m[i]));
  const float v = __fadd_rn(__fmul_rn(a.beta2, a.v[i]), __fmul_rn(__fsub_rn(1.0f, a.beta2), __fmul_rn(g, g)));
  a.m[i] = m;
  a.v[i] = v;
  const float mhat = __fdiv_rn(m, a.corr1[layer]);
  const float vhat = __fdiv_rn(v, a.corr2[layer]);
  const float denom = __fadd_rn(__fsqrt_rn(vhat), a.eps);
  a.params[i] = __fsub_rn(a.params[i], __fmul_rn(a.alpha, __fdiv_rn(mhat, denom)));
}
#endif

// PPOAgent.Train(Trajectory) over a list of trajectories in one launch (ppo_episodes_kernel, default networks).  The row arrays
// (states / actions / old_logp of the MlpParams, rewards, values, returns, advantages) hold the trajectories back to back.
struct EpisodeParams {
  const float* rewards;
  float* values;
  float* returns;
  float* advantages;
  const int32_t* offsets;      // [n_traj + 1] (device copy of the host's offsets)
  const int32_t* batch_index;  // per mini-batch B local row numbers, in call order
  const float* corr;           // [Adam steps][10]: corr1 of the 5 dense layers, then corr2
  float* grads;                // the gradient buffer (last mini-batch's gradient, loss sums, skipped)
  float* losses;               // [n_traj][2] or null
  int32_t* skipped;            // [n_traj] or null
  AdamParams adam;             // params / m / v and the hyper-parameters (the corrections come from the table)
  int32_t n_traj, epochs, batch;
  int32_t use_gae, normalize;
  float gamma, lambda, norm_eps;
};
cudaError_t launch_episodes(const EpisodeParams& e, const MlpParams& p, cudaStream_t stream);
cudaError_t launch_gather_rows(const int32_t* index, int B, int row_base, int sdim, int adim, const float* states, const float* actions,
                               const float* logp, const float* adv, const float* ret, float* o_states, float* o_actions, float* o_logp,
                               float* o_adv, float* o_ret, cudaStream_t stream);
// losses[2] <- grads_tail[0..1], *skipped += grads_tail[2] (either may be null)
cudaError_t launch_episode_losses(const float* grads_tail, float* losses, int32_t* skipped, cudaStream_t stream);

// ---- populations: P independent agents of the default networks (population_act_kernel / population_episodes_kernel, mlp.cu)
// Every agent's parameters, Adam moments and gradient buffer sit at agent * kAgentStride floats (16-byte aligned rows).
constexpr int kAgentStride = kGradFloats;  // 6152 >= kTotalParams + 3
constexpr int kPopMaxLen = 1024;           // longest episode a population trains (the reference caps one at MaxTimesteps + 1 = 1 001)
constexpr int kActWarps = 4;               // walkers (one warp each) per CTA of population_act_kernel
// per-agent constants, built on the host from the agent's wb_hyperparams (population_agent_consts)
struct PopAgent {
  float stdv, neg_log_std, log_sqrt_2pi, upper, lower, variance;  // GradConsts
  float alpha, beta1, beta2, adam_eps;
  float gamma, lambda, norm_eps, batch_size_f;
  int32_t batch, use_gae, normalize;
  float log_std, clip_eps;  // the raw values: the any-topology kernels derive sigma and the clip range on the device, as ppo_generic_kernel
  int32_t pad[3];
};
void population_agent_consts(const wb_hyperparams& hp, PopAgent* out);
struct PopActParams {
  const float* params;     // [P][kAgentStride]
  const PopAgent* agents;  // [P]
  int32_t n, mode;         // walker w acts with agent w; mode kModeSample (uniforms) or kModeSamplePhilox
  const float* states;     // [n][12]
  const float* uniforms;   // [n][4][2] (kModeSample)
  uint64_t seed, step;     // (kModeSamplePhilox)
  float* actions;          // [n][4]
  float* logp;             // [n][4]
  float* mean;             // [n][4] or null
  float* value;            // [n] or null
};
cudaError_t launch_population_act(const PopActParams& a, cudaStream_t stream);
// one item = one finished episode: rows ((t0 + i) mod ring_rows) * columns + column, i < length
struct PopItem {
  int32_t out;        // position of the item in the caller's list (losses / skipped)
  int32_t column, t0, length;
  int32_t index_off;  // first of its caller-drawn mini-batch indices (unused for device draws)
  int32_t corr_off;   // first of its Adam steps in the correction table
  int32_t episode;    // episodes of this agent trained before this one (device draws)
  int32_t pad;
};
struct PopCta {
  int32_t agent, first, count, pad;  // items [first, first + count) of the table, in list order
};
struct PopTrainParams {
  const float* states;      // ring [R][C][12]
  const float* actions;     // ring [R][C][4]
  const float* old_logp;    // ring [R][C][4]
  const float* rewards;     // ring [R][C]
  float* values;            // ring [R][C]
  float* returns;           // ring [R][C]
  float* advantages;        // ring [R][C]
  const int32_t* batch_index;  // caller-drawn local rows, or null: drawn on the device
  const PopCta* ctas;
  const PopItem* items;
  const float* corr;        // [Adam steps][10]
  const PopAgent* agents;
  float* params;            // [P][kAgentStride]
  float* m;
  float* v;
  float* grads;
  float* losses;            // [n_items][2] or null
  int32_t* skipped;         // [n_items] or null
  int32_t ring_rows, columns, epochs;
  uint64_t seed;
};
cudaError_t launch_population_episodes(const PopTrainParams& t, int n_ctas, cudaStream_t stream);

int mlp_grid_for(int n, int sm_count);
cudaError_t launch_mlp(const MlpParams& p, int grid, cudaStream_t stream);
cudaError_t launch_reduce_partials(const float* partials, int nparts, float* grads, cudaStream_t stream);
cudaError_t launch_adam(const AdamParams& p, cudaStream_t stream);
cudaError_t launch_returns(const float* rewards, const float* values, int n, float gamma, float lambda, int use_gae, int normalize,
                           float norm_eps, float* returns, float* advantages, cudaStream_t stream);

// ---- exchange buffer of the fused reduce + all-reduce (one allocation per rank, shared with the peers through CUDA IPC)
constexpr int kExchMaxWorld = 8;
constexpr int kExchThreads = 256;
constexpr int kExchLanes = 16;   // threads per float4 of the gradient buffer: each sums every 16th per-CTA partial
constexpr int kExchCtas = (kGradFloats / 4 + kExchThreads / kExchLanes - 1) / (kExchThreads / kExchLanes);  // 97 slices of 16 float4
// flags per (parity, rank): one per CTA of whichever kernel runs the exchange -- reduce_exchange_kernel (97 CTAs) or the tail of the
// tensor-core gradient kernel (one CTA per SM)
constexpr int kExchFlagSlots = 192;
struct ExchPeers {
  float* base[kExchMaxWorld];  // every rank's exchange buffer as seen from this process
};
// layout (floats): slots [2 parities][kExchMaxWorld ranks][kGradFloats], then flags (uint32) [2][kExchMaxWorld][kExchFlagSlots]
constexpr size_t kExchSlotFloats = (size_t)2 * kExchMaxWorld * kGradFloats;
constexpr size_t kExchBytes = kExchSlotFloats * sizeof(float) + (size_t)2 * kExchMaxWorld * kExchFlagSlots * sizeof(uint32_t);
__host__ __device__ inline size_t exch_slot_offset(int parity, int rank) { return ((size_t)parity * kExchMaxWorld + rank) * kGradFloats; }
__host__ __device__ inline uint32_t* exch_flag(float* base, int parity, int rank, int cta) {
  return reinterpret_cast<uint32_t*>(base + kExchSlotFloats) + ((size_t)parity * kExchMaxWorld + rank) * kExchFlagSlots + cta;
}
#ifdef __CUDACC__
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
#endif

// Tail of the tensor-core gradient kernel: PPOAgent.Train(Batch) in ONE launch.  After a grid-wide barrier (every CTA of the
// persistent grid is resident: one per SM) each CTA reduces its slice of the per-CTA partials in a fixed order; with world > 1 it
// then pushes the slice into slot [rank] of every peer's exchange buffer over NVLink, publishes / awaits the epoch flags of ITS
// slice (the protocol of reduce_exchange_kernel, mlp.cu) and adds the world's slots in rank order; finally it applies
// DenseLayer.Adam to the slice.  Every rank must launch the same grid (same n), so that the slices agree.
struct FusedTail {
  int32_t enabled;
  uint32_t* counter;   // monotonically increasing arrival counter of the grid barrier
  uint32_t target;     // value the counter reaches when every CTA of THIS launch has arrived
  float* grads;        // [kGradFloats] reduced gradient (+ loss sums, skipped)
  AdamParams adam;
  // exchange (world > 1)
  ExchPeers peers;
  int32_t rank, world;
  uint32_t epoch;
  uint32_t* status;    // mapped host word: set on a time-out (the host reads it without a copy)
  uint32_t* dead;      // its device copy: what every later launch checks (a host-memory read per CTA would serialise over PCIe)
};

// adam != nullptr: DenseLayer.Adam is applied to the reduced gradient inside the same kernel
cudaError_t launch_reduce_exchange(const float* partials, int nparts, float* grads, const ExchPeers& peers, int rank, int world,
                                   uint32_t epoch, uint32_t* status, uint32_t* dead, const AdamParams* adam, cudaStream_t stream);

// last_values: V(s_T) per environment (bootstrap of a segment that ends mid-episode) or nullptr (truncate like a trajectory end)
cudaError_t launch_segment_returns(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, int n_envs,
                                   int T, float gamma, float lambda, int use_gae, float* returns, float* advantages, cudaStream_t stream);
// PPOAgent.Normalize over a pool, three stages (0: sum, 1: squared deviations, 2: apply); stats = double[2 * kNormCtas]
constexpr int kNormCtas = 128;
constexpr int kNormThreads = 256;
cudaError_t launch_normalize_stage(float* x, long n_local, double count_global, int stage, float epsilon, double* stats, cudaStream_t stream);
cudaError_t launch_gather_minibatch(const int32_t* index, int B, const float* states, const float* actions, const float* logp,
                                    const float* adv, const float* ret, float* o_states, float* o_actions, float* o_logp, float* o_adv,
                                    float* o_ret, cudaStream_t stream);

// ---- any topology the reference's DSL can describe (mlp_generic.cu)
constexpr int kGenMaxLayers = 16;   // layers (dense + activation) per network
constexpr int kGenMaxWidth = 128;   // widest layer / state size
constexpr int kGenMaxDense = 32;    // dense layers of both networks together (Adam bias corrections)
constexpr int kGenThreads = 256;
struct GenLayer {
  int32_t kind, in, out;       // WB_DENSE: in -> out; activation: in == out
  int32_t w_off, b_off;        // dense: offsets inside THIS network's flat parameter vector (W[out][in] row-major, then b[out])
  int32_t cache_off;           // offset of this layer's INPUT inside a sample's cache row (NeuralNetwork._cache)
};
struct GenNet {
  int32_t n_layers, input, output, n_params, n_dense, cache_floats;  // cache_floats: sum of the layers' input widths
  GenLayer L[kGenMaxLayers];
};
struct GenParams {
  GenNet actor, critic;
  const float* params;  // actor | critic
  int32_t n, mode, ts, grad_floats;
  const float* states;
  const float* actions;
  const float* old_logp;
  const float* advantages;
  const float* returns;
  const float* uniforms;
  uint64_t seed, step;
  float* mean;
  float* value;
  float* out_actions;
  float* out_logp;
  float* partials;      // [grid][grad_floats]
  float log_std, epsilon, batch_size;
};
struct GenAdamParams {
  float* params;
  const float* grads;
  float* m;
  float* v;
  int32_t n_params, n_dense;
  int32_t layer_end[kGenMaxDense];  // one past the last parameter of every dense layer (actor layers, then critic layers)
  float corr1[kGenMaxDense], corr2[kGenMaxDense];
  float alpha, beta1, beta2, eps;
};
size_t generic_smem_bytes(const GenNet& actor, const GenNet& critic, int ts);
int generic_tile_samples(const GenNet& actor, const GenNet& critic);  // 0: the caches do not fit shared memory even for one sample
int generic_grid_for(int n, int ts, int sm_count);
cudaError_t launch_mlp_generic(const GenParams& p, int grid, cudaStream_t stream);
cudaError_t launch_reduce_partials_n(const float* partials, int nparts, float* grads, int n_floats, cudaStream_t stream);
cudaError_t launch_adam_generic(const GenAdamParams& a, cudaStream_t stream);

// the two networks of a wb_policy / wb_population, validated (wb_policy_create's limits and statuses; a failure records the message)
struct Networks {
  GenNet actor, critic;
  int gen_ts;             // generic_tile_samples
  bool default_topology;  // the reference's default networks: the specialised kernels apply
};
int32_t build_networks(int32_t state_size, int32_t action_size, const int32_t* actor_kinds, const int32_t* actor_sizes, int32_t actor_layers,
                       const int32_t* critic_kinds, const int32_t* critic_sizes, int32_t critic_layers, Networks* out);
// one past the last parameter of every dense layer (actor layers, then critic layers at + actor.n_params); returns their number
int generic_layer_ends(const GenNet& actor, const GenNet& critic, int32_t* layer_end);

// ---- populations of any topology (population_generic_act_kernel / population_generic_episodes_kernel, mlp_generic.cu)
constexpr int kGenActWarps = 2;  // walkers (one warp each) per CTA of population_generic_act_kernel
constexpr size_t kPopGenMaxSmem = 227 * 1024;  // shared memory a CTA may hold on sm_100
struct PopGenActParams {
  GenNet actor, critic;
  int32_t stride;        // floats per agent row
  int32_t chunk_floats;  // generic_act_chunk_floats
  PopActParams a;        // states [n][state], uniforms [n][act][2], actions / logp / mean [n][act], value [n]
};
struct PopGenTrainParams {
  GenNet actor, critic;
  int32_t stride, ts, grad_floats, n_dense;
  int32_t layer_end[kGenMaxDense];
  PopTrainParams t;  // corr: [Adam steps][2 * n_dense]
};
int generic_act_chunk_floats(const GenNet& actor, const GenNet& critic);
size_t generic_episodes_smem_bytes(const GenNet& actor, const GenNet& critic, int ts);
cudaError_t launch_population_generic_act(const PopGenActParams& g, cudaStream_t stream);
cudaError_t launch_population_generic_episodes(const PopGenTrainParams& g, int n_ctas, cudaStream_t stream);

int tc_grid_for(int n, int sm_count);
cudaError_t launch_mlp_tc(const MlpParams& p, int grid, cudaStream_t stream, const FusedTail* tail = nullptr);
cudaError_t launch_tc_gemm_test(const float* A, const float* B, float* D, int M, int N, int K, int a_mn, int b_mn, int passes,
                                cudaStream_t stream);

}  // namespace wb

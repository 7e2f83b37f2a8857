// ppo_device.cuh -- device helpers shared by the default-network kernels (mlp.cu) and the any-topology kernels (mlp_generic.cu):
// the Philox stream, the per-trajectory returns / advantages and the device draw of an episode's mini-batch permutation.  One
// definition, so that both translation units compute the same bits.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace wb {

// Philox-4x32-10 (counter-based; extension -- the reference's System.Random is unseedable)
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// PPOAgent.MonteCarloReturn/MonteCarloAdvantages (:475-498), GeneralizedAdvantageEstimate (:414-444, whose nextGae is
// never updated in the reference), Normalize (:461-472).  One trajectory: an inherently sequential fp32 recurrence.
__device__ __forceinline__ void trajectory_returns(const float* __restrict__ rewards, const float* __restrict__ values, int n, float gamma,
                                                   float lambda, int use_gae, int normalize, float norm_eps, float* __restrict__ returns,
                                                   float* __restrict__ advantages) {
  if (use_gae) {
    const float next_gae = 0.0f;
    float next_value = 0.0f;
    for (int i = n - 1; i >= 0; i--) {
      const float cur = values[i];
      const float delta = __fsub_rn(__fadd_rn(rewards[i], __fmul_rn(gamma, next_value)), cur);
      next_value = cur;
      const float gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gamma, lambda), next_gae));
      advantages[i] = gae;
      returns[i] = __fadd_rn(gae, values[i]);
    }
  } else {
    float g = 0.0f;
    for (int i = n - 1; i >= 0; i--) {
      g = __fadd_rn(rewards[i], __fmul_rn(g, gamma));
      returns[i] = g;
    }
    for (int i = 0; i < n; i++) advantages[i] = __fsub_rn(returns[i], values[i]);
  }
  if (normalize && n > 0) {
    double acc = 0.0;
    for (int i = 0; i < n; i++) acc += (double)advantages[i];
    const float mean = (float)(acc / (double)n);
    double ss = 0.0;
    for (int i = 0; i < n; i++) {
      const double d = (double)__fsub_rn(advantages[i], mean);
      ss += d * d;
    }
    const float sd = (float)sqrt(ss / (double)n);
    const float div = __fadd_rn(sd, norm_eps);
    for (int i = 0; i < n; i++) advantages[i] = __fdiv_rn(__fsub_rn(advantages[i], mean), div);
  }
}

// PPOAgent.CreateBatches (PPOAgent.cs:501-540: sampling without replacement) drawn on the device by a CTA of kThreads threads:
// local row i of the episode gets key(i) = Philox-4x32-10(counter (i, epoch, episode, agent), key (seed lo, seed hi)).x, where
// `episode` counts the agent's episodes trained before this one; perm = the rows ordered by (key, row).  Each row's rank is
// counted over the <= 1 024 keys.  key / perm: shared-memory arrays of at least L entries.
template <int kThreads>
__device__ __forceinline__ void draw_permutation(uint32_t* key, int32_t* perm, int L, int epoch, int episode, int agent, uint64_t seed,
                                                 int tid) {
  for (int i = tid; i < L; i += kThreads)
    key[i] = philox4x32(make_uint4((uint32_t)i, (uint32_t)epoch, (uint32_t)episode, (uint32_t)agent),
                        make_uint2((uint32_t)seed, (uint32_t)(seed >> 32))).x;
  __syncthreads();
  for (int j = tid; j < L; j += kThreads) {
    const uint32_t kj = key[j];
    int rank = 0;
    for (int i = 0; i < L; i++) {
      const uint32_t ki = key[i];
      rank += (ki < kj || (ki == kj && i < j)) ? 1 : 0;
    }
    perm[rank] = j;
  }
  __syncthreads();
}

}  // namespace wb

// mlp.cu -- PPO policy/value MLP kernels for sm_100a (fp32 CUDA-core version of the fused pipeline).
//
// Replaces the reference's per-sample Matrix-library pipeline (Walker/PPO/Matrix.cs, Network/DenseLayer.cs,
// Network/ActivationLayer.cs, PPOAgent.cs:218-346,381-398, NormalDistribution.cs) with batched kernels:
//
//   ppo_fused_kernel  persistent CTAs; each iteration stages a tile of 64 samples in shared memory and runs
//                     actor + critic forward, the per-sample clipped-surrogate gradient (Appendix B of
//                     SURVEY.md), and the full backward pass as tile GEMMs; weight-gradient tiles are held in
//                     registers across all tiles of the CTA and written once as a per-CTA partial.
//   reduce_partials   deterministic fixed-order sum of the per-CTA partials (no atomics) -> gradient buffer.
//   adam_kernel       DenseLayer.Adam (DenseLayer.cs:125-159) with the reference's operation order.
//   returns_kernel    Monte-Carlo return / the reference's GAE variant / Normalize (PPOAgent.cs:414-498).
//
// Dot products accumulate in the reference's left-to-right order (Matrix.Multiply, Matrix.cs:604-616) with
// fused multiply-add; the cross-sample sum of dW is tiled (per CTA, then across CTAs) instead of the
// reference's strictly sequential per-sample accumulation -- covered by the 1e-4 relative tolerance.
#include "mlp.cuh"
#include "ppo_device.cuh"

#include <cfloat>

namespace wb {

constexpr int kPad = 68;  // row stride (floats) of [*][64] tiles in shared memory: float4-aligned, bank-staggered

struct __align__(16) MlpSmem {
  float W1[kHid * kIn];
  float W2[kHid * kPad];
  float W3[kAct * kPad];
  float Wc1[kHid * kIn];
  float Wc2[kHid];
  float b1[kHid], b2[kHid], bc1[kHid];
  float b3[kAct], bc2[4];
  float X[kTile * kIn];
  float A1[kTile * kPad], A2[kTile * kPad], C1[kTile * kPad];   // post-activation hidden layers
  float G2[kTile * kPad], G1[kTile * kPad], Gc1[kTile * kPad];  // dL/dz of the hidden layers
  float MU[kTile * kAct], G3[kTile * kAct], V[kTile], GV[kTile];
  float red[kMlpThreads];
};

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// ActivationLayer.cs:46-59
__device__ __forceinline__ float leaky(float v) { return fmaxf(0.2f * v, v); }
__device__ __forceinline__ float leaky_grad_from_output(float a) { return a < 0.0f ? 0.2f : 1.0f; }  // sign(a) == sign(z)

// out[s][o] = act(sum_i in[s][i] * W[o][i] + b[o]) for a 64-sample x 64-output tile; thread = 4 samples x 4 outputs
template <int K, int LDIN, int LDW>
__device__ __forceinline__ void dense64_forward(const float* in, const float* W, const float* b, float* out) {
  const int ts = threadIdx.x >> 4, to = threadIdx.x & 15;
  float acc[4][4];
#pragma unroll
  for (int k = 0; k < 4; k++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[k][j] = 0.0f;
#pragma unroll 4
  for (int i = 0; i < K; i += 4) {
    float4 a[4], w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) a[k] = ld4(in + (ts * 4 + k) * LDIN + i);
#pragma unroll
    for (int j = 0; j < 4; j++) w[j] = ld4(W + (to + 16 * j) * LDW + i);
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
      for (int j = 0; j < 4; j++) {
        acc[k][j] = fmaf(a[k].x, w[j].x, acc[k][j]);
        acc[k][j] = fmaf(a[k].y, w[j].y, acc[k][j]);
        acc[k][j] = fmaf(a[k].z, w[j].z, acc[k][j]);
        acc[k][j] = fmaf(a[k].w, w[j].w, acc[k][j]);
      }
  }
#pragma unroll
  for (int k = 0; k < 4; k++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int o = to + 16 * j;
      out[(ts * 4 + k) * kPad + o] = leaky(acc[k][j] + b[o]);
    }
}

// NormalDistribution.LogProbabilityDensity, NormalDistribution.cs:24-32 (-ln(std) and ln(sqrt(2pi)) precomputed on the host)
__device__ __forceinline__ float log_prob(float mean, float stdv, float action, float neg_log_std, float log_sqrt_2pi) {
  float fraction = (action - mean) / stdv;
  fraction *= fraction;
  fraction /= 2.0f;
  return neg_log_std - log_sqrt_2pi - fraction;
}

struct GradConsts {
  float stdv, neg_log_std, log_sqrt_2pi, upper, lower, variance;
};

// The sampling of ppo_fused_kernel's forward modes, restated for population_act_kernel (the same expressions in the same
// translation unit and flags: the same arithmetic; ppo_fused_kernel keeps its own copy so that its SASS stays as it is).
// The two uniforms of action dimension k of sample gs: injected (kModeSample) or from the Philox stream (gs, k, step) under seed
__device__ __forceinline__ void sample_uniforms(int mode, const float* uniforms, uint64_t seed, uint64_t step, int gs, int k, float& u1,
                                                float& u2) {
  if (mode == kModeSample) {
    u1 = uniforms[((size_t)gs * kAct + k) * 2];
    u2 = uniforms[((size_t)gs * kAct + k) * 2 + 1];
  } else {
    const uint4 r = philox4x32(make_uint4((uint32_t)gs, (uint32_t)k, (uint32_t)step, (uint32_t)(step >> 32)),
                               make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    u1 = (float)(r.x >> 8) * (1.0f / 16777216.0f);  // [0,1) like (float)Random.NextDouble()
    u2 = (float)(r.y >> 8) * (1.0f / 16777216.0f);
  }
}

// NormalDistribution.BoxMullerTransform (NormalDistribution.cs:12-19) around mu, and the action's log-probability
__device__ __forceinline__ void sample_action(float mu, float stdv, float neg_log_std, float log_sqrt_2pi, float u1, float u2, float& a,
                                              float& lp) {
  if (u1 == 0.0f) u1 = 1.0f;
  const float z = sqrtf(-2.0f * logf(u1)) * sinf(2.0f * 3.14159274f * u2);
  a = mu + (stdv * z);
  lp = log_prob(mu, stdv, a, neg_log_std, log_sqrt_2pi);
}

// ---- the 64-sample tile pipeline of PPOAgent.Train(Batch), shared by ppo_fused_kernel and ppo_episodes_kernel (one CTA of
// kMlpThreads threads over MlpSmem; the callers stage the tile's states in S.X and own the weight-gradient accumulators and loss
// sums, which stay in registers across every tile the CTA processes)

// weights p.params -> shared memory (padded rows)
__device__ __forceinline__ void stage_weights(MlpSmem& S, const MlpParams& p, int tid) {
  for (int i = tid; i < kHid * kIn; i += kMlpThreads) {
    S.W1[i] = p.params[kOffW1 + i];
    S.Wc1[i] = p.params[kOffWc1 + i];
  }
  for (int i = tid; i < kHid * kHid; i += kMlpThreads) S.W2[(i >> 6) * kPad + (i & 63)] = p.params[kOffW2 + i];
  for (int i = tid; i < kAct * kHid; i += kMlpThreads) S.W3[(i >> 6) * kPad + (i & 63)] = p.params[kOffW3 + i];
  if (tid < kHid) {
    S.b1[tid] = p.params[kOffB1 + tid];
    S.b2[tid] = p.params[kOffB2 + tid];
    S.bc1[tid] = p.params[kOffBc1 + tid];
    S.Wc2[tid] = p.params[kOffWc2 + tid];
  }
  if (tid < kAct) S.b3[tid] = p.params[kOffB3 + tid];
  if (tid == 0) S.bc2[0] = p.params[kOffBc2];
}

// S.X -> S.A1, S.C1, S.A2, S.MU, S.V; ends with a barrier
__device__ __forceinline__ void tile_forward(MlpSmem& S, int tid) {
  // ---- forward: actor L1, critic L1, actor L2 (NeuralNetwork.FeedForward, DenseLayer.FeedForward)
  dense64_forward<kIn, kIn, kIn>(S.X, S.W1, S.b1, S.A1);
  dense64_forward<kIn, kIn, kIn>(S.X, S.Wc1, S.bc1, S.C1);
  __syncthreads();
  dense64_forward<kHid, kPad, kPad>(S.A1, S.W2, S.b2, S.A2);
  __syncthreads();
  {  // actor L3 + TanH: thread = (sample, action dim); critic L2: threads 0..63
    const int s = tid >> 2, k = tid & 3;
    int i = 0;
    float sum = 0.0f;
#pragma unroll 4
    for (; i < kHid; i += 4) {
      const float4 a = ld4(S.A2 + s * kPad + i), w = ld4(S.W3 + k * kPad + i);
      sum = fmaf(a.x, w.x, sum);
      sum = fmaf(a.y, w.y, sum);
      sum = fmaf(a.z, w.z, sum);
      sum = fmaf(a.w, w.w, sum);
    }
    S.MU[s * kAct + k] = tanhf(sum + S.b3[k]);
    if (tid < kTile) {
      float v = 0.0f;
#pragma unroll 4
      for (int i = 0; i < kHid; i += 4) {
        const float4 a = ld4(S.C1 + tid * kPad + i), w = ld4(S.Wc2 + i);
        v = fmaf(a.x, w.x, v);
        v = fmaf(a.y, w.y, v);
        v = fmaf(a.z, w.z, v);
        v = fmaf(a.w, w.w, v);
      }
      S.V[tid] = v + S.bc2[0];
    }
  }
  __syncthreads();
}

// row_of(s): the row of p's actions / old_logp / advantages / returns that sample s < nvalid of the tile is;
// S.G3 / S.GV <- dL/dmu * tanh', dL/dV; ends with a barrier
template <class RowOf>
__device__ __forceinline__ void tile_surrogate(MlpSmem& S, const MlpParams p, const GradConsts gc, int nvalid, RowOf row_of, float& lossV,
                                               float& lossA, float& skipped, int tid) {
  // ---- per-sample clipped-surrogate gradient, PPOAgent.cs:232-326 (thread = sample)
  if (tid < kTile) {
    const int s = tid, gs = row_of(s);
    float g[kAct] = {0.f, 0.f, 0.f, 0.f};
    float gv = 0.0f;
    if (s < nvalid) {
      const float adv = p.advantages[gs];
      bool skip = false;
#pragma unroll
      for (int k = 0; k < kAct; k++) {
        const float mu = S.MU[s * kAct + k];
        const float a = p.actions[(size_t)gs * kAct + k];
        const float lp_old = p.old_logp[(size_t)gs * kAct + k];
        const float lp = log_prob(mu, gc.stdv, a, gc.neg_log_std, gc.log_sqrt_2pi);
        const float ratio = expf(lp - lp_old);
        const float clipped = ratio >= gc.upper ? gc.upper : (ratio <= gc.lower ? gc.lower : ratio);  // Matrix.Clip
        const float cra = clipped * adv, ra = ratio * adv;
        const float partA = (ra <= cra ? 1.0f : 0.0f) * adv;                              // Matrix.LessThan
        const float partB = (cra < ra ? 1.0f : 0.0f) * adv;                               // Matrix.LessThanNotEquals
        const float partC = (ratio >= gc.lower && ratio <= gc.upper) ? 1.0f : 0.0f;       // Matrix.InRange
        float dclip = (partA + partB * partC) * -1.0f;
        const float pold = expf(lp_old);
        if (pold == 0.0f) skip = true;  // HadamardDivision throws -> the sample is skipped (PPOAgent.cs:286-290)
        dclip = dclip / pold;
        const float prob = expf(lp);
        const float dmean = prob * ((a - mu) / gc.variance);
        g[k] = (dmean * dclip) / p.batch_size;
      }
      gv = (2.0f * (S.V[s] - p.returns[gs])) / p.batch_size;
      if (skip) {
#pragma unroll
        for (int k = 0; k < kAct; k++) g[k] = 0.0f;
        gv = 0.0f;
        skipped += 1.0f;
      } else {
        lossV += gv;
        lossA += (((g[0] + g[1]) + g[2]) + g[3]) / (float)kAct;  // Matrix.Average
      }
    }
    // TanhLayer.FeedBack: g * (1 - tanh(z)^2), ActivationLayer.cs:18-21,69-72
#pragma unroll
    for (int k = 0; k < kAct; k++) {
      const float mu = S.MU[s * kAct + k];
      S.G3[s * kAct + k] = g[k] * (1.0f - (mu * mu));
    }
    S.GV[s] = gv;
  }
  __syncthreads();
}

// backward pass of the tile into the accumulators; ends WITHOUT a barrier (the next tile's staging starts with one)
__device__ __forceinline__ void tile_backward(MlpSmem& S, float (&accW2)[4][4], float (&accW1)[3], float (&accWc1)[3], float& accW3, float& accS,
                                              float& accT, int tid) {
  // ---- dL/dz2 = (W3^T g3) * leaky'(z2); dL/dzc1 = (Wc2^T gv) * leaky'(zc1)
  {
    const int s = tid >> 2, i0 = (tid & 3) * 16;
    const float4 g3 = ld4(S.G3 + s * kAct);
    const float gv = S.GV[s];
#pragma unroll
    for (int i = i0; i < i0 + 16; i++) {
      float sum = 0.0f;
      sum = fmaf(S.W3[0 * kPad + i], g3.x, sum);
      sum = fmaf(S.W3[1 * kPad + i], g3.y, sum);
      sum = fmaf(S.W3[2 * kPad + i], g3.z, sum);
      sum = fmaf(S.W3[3 * kPad + i], g3.w, sum);
      S.G2[s * kPad + i] = sum * leaky_grad_from_output(S.A2[s * kPad + i]);
      S.Gc1[s * kPad + i] = (0.0f + S.Wc2[i] * gv) * leaky_grad_from_output(S.C1[s * kPad + i]);
    }
  }
  __syncthreads();

  // ---- dW3 += g3^T A2 ; dW2 += G2^T A1 ; dL/dz1 = (W2^T G2) * leaky'(z1)
  {
    const int k = tid >> 6, i = tid & 63;
#pragma unroll 8
    for (int s = 0; s < kTile; s++) accW3 = fmaf(S.G3[s * kAct + k], S.A2[s * kPad + i], accW3);
  }
  {
    const int og = tid >> 4, ig = tid & 15;
#pragma unroll 4
    for (int s = 0; s < kTile; s++) {
      const float4 g4 = ld4(S.G2 + s * kPad + og * 4);
      const float4 a4 = ld4(S.A1 + s * kPad + ig * 4);
      const float gg[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
      for (int j = 0; j < 4; j++) {
        accW2[j][0] = fmaf(gg[j], a4.x, accW2[j][0]);
        accW2[j][1] = fmaf(gg[j], a4.y, accW2[j][1]);
        accW2[j][2] = fmaf(gg[j], a4.z, accW2[j][2]);
        accW2[j][3] = fmaf(gg[j], a4.w, accW2[j][3]);
      }
    }
  }
  {
    const int ts = tid >> 4, ig = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
      for (int l = 0; l < 4; l++) acc[k][l] = 0.0f;
#pragma unroll 2
    for (int o = 0; o < kHid; o += 4) {
      float4 g4[4], w4[4];
#pragma unroll
      for (int k = 0; k < 4; k++) g4[k] = ld4(S.G2 + (ts * 4 + k) * kPad + o);
#pragma unroll
      for (int q = 0; q < 4; q++) w4[q] = ld4(S.W2 + (o + q) * kPad + ig * 4);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const float gq[4] = {g4[k].x, g4[k].y, g4[k].z, g4[k].w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
          acc[k][0] = fmaf(w4[q].x, gq[q], acc[k][0]);
          acc[k][1] = fmaf(w4[q].y, gq[q], acc[k][1]);
          acc[k][2] = fmaf(w4[q].z, gq[q], acc[k][2]);
          acc[k][3] = fmaf(w4[q].w, gq[q], acc[k][3]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int s = ts * 4 + k;
      const float4 a = ld4(S.A1 + s * kPad + ig * 4);
      float4 r;
      r.x = acc[k][0] * leaky_grad_from_output(a.x);
      r.y = acc[k][1] * leaky_grad_from_output(a.y);
      r.z = acc[k][2] * leaky_grad_from_output(a.z);
      r.w = acc[k][3] * leaky_grad_from_output(a.w);
      *reinterpret_cast<float4*>(S.G1 + s * kPad + ig * 4) = r;
    }
  }
  __syncthreads();

  // ---- dW1 += G1^T X ; dWc1 += Gc1^T X ; biases and the critic head
  {
    const int o = tid >> 2, ib = (tid & 3) * 3;
#pragma unroll 4
    for (int s = 0; s < kTile; s++) {
      const float ga = S.G1[s * kPad + o], gcr = S.Gc1[s * kPad + o];
      const float x0 = S.X[s * kIn + ib], x1 = S.X[s * kIn + ib + 1], x2 = S.X[s * kIn + ib + 2];
      accW1[0] = fmaf(ga, x0, accW1[0]);
      accW1[1] = fmaf(ga, x1, accW1[1]);
      accW1[2] = fmaf(ga, x2, accW1[2]);
      accWc1[0] = fmaf(gcr, x0, accWc1[0]);
      accWc1[1] = fmaf(gcr, x1, accWc1[1]);
      accWc1[2] = fmaf(gcr, x2, accWc1[2]);
    }
  }
  {
    const int q = tid >> 6, o = tid & 63;  // q: 0 db1, 1 db2, 2 dbc1, 3 dWc2
    const float* src = (q == 0) ? S.G1 : (q == 1) ? S.G2 : (q == 2) ? S.Gc1 : S.C1;
#pragma unroll 8
    for (int s = 0; s < kTile; s++) {
      const float v = src[s * kPad + o];
      accS = (q == 3) ? fmaf(S.GV[s], v, accS) : accS + v;
    }
    if (tid < kAct + 1) {
#pragma unroll 8
      for (int s = 0; s < kTile; s++) accT += (tid < kAct) ? S.G3[s * kAct + tid] : S.GV[s];
    }
  }
}

// the CTA's gradient (flat parameter layout) + loss sums -> out[0 .. kTotalParams + 3); ends with a barrier
__device__ __forceinline__ void write_grad(MlpSmem& S, const float (&accW2)[4][4], const float (&accW1)[3], const float (&accWc1)[3], float accW3,
                                           float accS, float accT, float lossV, float lossA, float skipped, float* out, int tid) {
  {
    const int og = tid >> 4, ig = tid & 15;
#pragma unroll
    for (int j = 0; j < 4; j++)
      *reinterpret_cast<float4*>(out + kOffW2 + (og * 4 + j) * kHid + ig * 4) =
          make_float4(accW2[j][0], accW2[j][1], accW2[j][2], accW2[j][3]);
  }
  {
    const int o = tid >> 2, ib = (tid & 3) * 3;
#pragma unroll
    for (int l = 0; l < 3; l++) {
      out[kOffW1 + o * kIn + ib + l] = accW1[l];
      out[kOffWc1 + o * kIn + ib + l] = accWc1[l];
    }
  }
  out[kOffW3 + (tid >> 6) * kHid + (tid & 63)] = accW3;
  {
    const int q = tid >> 6, o = tid & 63;
    const int off = (q == 0) ? kOffB1 : (q == 1) ? kOffB2 : (q == 2) ? kOffBc1 : kOffWc2;
    out[off + o] = accS;
  }
  if (tid < kAct) out[kOffB3 + tid] = accT;
  if (tid == kAct) out[kOffBc2] = accT;
  // loss sums: only threads < 64 hold non-zero values; fixed-order tree reduction
  __syncthreads();
  float* red = S.red;
  for (int pass = 0; pass < 3; pass++) {
    red[tid] = (pass == 0) ? lossV : (pass == 1) ? lossA : skipped;
    __syncthreads();
    for (int w = kMlpThreads / 2; w > 0; w >>= 1) {
      if (tid < w) red[tid] += red[tid + w];
      __syncthreads();
    }
    if (tid == 0) out[kTotalParams + pass] = red[0];
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kMlpThreads, 1) ppo_fused_kernel(const MlpParams p, const GradConsts gc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  const int tid = threadIdx.x;

  stage_weights(S, p, tid);
  const bool grad = p.mode == kModeGrad;
  // weight-gradient accumulators, resident in registers across every tile this CTA processes
  float accW2[4][4];
#pragma unroll
  for (int j = 0; j < 4; j++)
#pragma unroll
    for (int l = 0; l < 4; l++) accW2[j][l] = 0.0f;
  float accW1[3] = {0.f, 0.f, 0.f}, accWc1[3] = {0.f, 0.f, 0.f};
  float accW3 = 0.0f, accS = 0.0f, accT = 0.0f;
  float lossV = 0.0f, lossA = 0.0f, skipped = 0.0f;

  const int ntiles = (p.n + kTile - 1) / kTile;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int s0 = tile * kTile;
    const int nvalid = min(kTile, p.n - s0);
    __syncthreads();  // previous tile fully consumed (also orders the weight staging on the first pass)
    for (int i = tid; i < kTile * kIn; i += kMlpThreads) S.X[i] = (i < nvalid * kIn) ? p.states[(size_t)s0 * kIn + i] : 0.0f;
    __syncthreads();
    tile_forward(S, tid);
    if (!grad) {
      const int s = tid >> 2, k = tid & 3;
      const int gs = s0 + s;
      if (s < nvalid) {
        const float mu = S.MU[s * kAct + k];
        if (p.mean) p.mean[(size_t)gs * kAct + k] = mu;
        if (p.value && k == 0) p.value[gs] = S.V[s];
        if (p.mode == kModeSample || p.mode == kModeSamplePhilox) {
          float u1, u2;
          if (p.mode == kModeSample) {
            u1 = p.uniforms[((size_t)gs * kAct + k) * 2];
            u2 = p.uniforms[((size_t)gs * kAct + k) * 2 + 1];
          } else {
            const uint4 r = philox4x32(make_uint4((uint32_t)gs, (uint32_t)k, (uint32_t)p.step, (uint32_t)(p.step >> 32)),
                                       make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32)));
            u1 = (float)(r.x >> 8) * (1.0f / 16777216.0f);  // [0,1) like (float)Random.NextDouble()
            u2 = (float)(r.y >> 8) * (1.0f / 16777216.0f);
          }
          // NormalDistribution.BoxMullerTransform, NormalDistribution.cs:12-19
          if (u1 == 0.0f) u1 = 1.0f;
          const float z = sqrtf(-2.0f * logf(u1)) * sinf(2.0f * 3.14159274f * u2);
          const float a = mu + (gc.stdv * z);
          p.out_actions[(size_t)gs * kAct + k] = a;
          p.out_logp[(size_t)gs * kAct + k] = log_prob(mu, gc.stdv, a, gc.neg_log_std, gc.log_sqrt_2pi);
        }
      }
      continue;
    }

    tile_surrogate(S, p, gc, nvalid, [&](int s) { return s0 + s; }, lossV, lossA, skipped, tid);
    tile_backward(S, accW2, accW1, accWc1, accW3, accS, accT, tid);
  }

  if (!grad) return;
  // per-CTA partial gradient + loss sums
  write_grad(S, accW2, accW1, accWc1, accW3, accS, accT, lossV, lossA, skipped, p.partials + (size_t)blockIdx.x * kGradFloats, tid);
}

// grads[i] = sum over CTAs (fixed order) -- this is also NeuralNetwork.Zero(): the buffer is overwritten
__global__ void reduce_partials_kernel(const float* __restrict__ partials, int nparts, float* __restrict__ grads) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kGradFloats) return;
  float sum = 0.0f;
  for (int c = 0; c < nparts; c++) sum += partials[(size_t)c * kGradFloats + i];
  grads[i] = sum;
}

__global__ void adam_kernel(const AdamParams a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kTotalParams) return;
  adam_update(a, i, a.grads[i]);
}

__global__ void returns_kernel(const float* rewards, const float* values, int n, float gamma, float lambda, int use_gae,
                               int normalize, float norm_eps, float* returns, float* advantages) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  trajectory_returns(rewards, values, n, gamma, lambda, use_gae, normalize, norm_eps, returns, advantages);
}

// PPOAgent.Train(Trajectory) (PPOAgent.cs:147-172) for a list of trajectories, in list order, as ONE persistent CTA: the Adam
// steps form a serial chain (each mini-batch is trained with the weights the previous one left), so one SM without host round
// trips is the shape of the work.  Per trajectory: critic forward over its rows (tile_forward, as the forward mode of
// ppo_fused_kernel), returns / advantages (trajectory_returns, as returns_kernel), then epochs x floor(T / B) mini-batches:
// the indexed rows are gathered into the tile, ceil(B / 64) tiles accumulate in registers (the tile pipeline of
// ppo_fused_kernel), the gradient goes to the gradient buffer, and DenseLayer.Adam runs over every parameter with that step's
// bias corrections from the host's table before the shared-memory weights are refreshed.
struct __align__(16) EpisodeSmem {
  MlpSmem m;
  int32_t rows[kTile];  // pool row of every sample of the current mini-batch tile
};

__global__ void __launch_bounds__(kMlpThreads, 1) ppo_episodes_kernel(const EpisodeParams e, const MlpParams p, const GradConsts gc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EpisodeSmem& E = *reinterpret_cast<EpisodeSmem*>(smem_raw);
  MlpSmem& S = E.m;
  const int tid = threadIdx.x;
  const int B = e.batch;
  stage_weights(S, p, tid);
  int step = 0;
  const int32_t* index = e.batch_index;
  for (int t = 0; t < e.n_traj; t++) {
    const int r0 = e.offsets[t], T = e.offsets[t + 1] - r0;
    // ---- CalculateValues (PPOAgent.cs:175-189): the critic over the trajectory's rows with the current weights
    for (int s0 = 0; s0 < T; s0 += kTile) {
      const int nvalid = min(kTile, T - s0);
      __syncthreads();
      for (int i = tid; i < kTile * kIn; i += kMlpThreads) S.X[i] = (i < nvalid * kIn) ? p.states[(size_t)(r0 + s0) * kIn + i] : 0.0f;
      __syncthreads();
      tile_forward(S, tid);
      if (tid < nvalid) e.values[r0 + s0 + tid] = S.V[tid];
    }
    __syncthreads();
    if (tid == 0 && T > 0)
      trajectory_returns(e.rewards + r0, e.values + r0, T, e.gamma, e.lambda, e.use_gae, e.normalize, e.norm_eps, e.returns + r0,
                         e.advantages + r0);
    __syncthreads();
    // ---- epochs x floor(T / B) mini-batches, each Train(Batch) + NeuralNetwork.Optimise
    const int nb = e.epochs * (T / B);
    float skipped_total = 0.0f;
    for (int b = 0; b < nb; b++, step++, index += B) {
      float accW2[4][4];
#pragma unroll
      for (int j = 0; j < 4; j++)
#pragma unroll
        for (int l = 0; l < 4; l++) accW2[j][l] = 0.0f;
      float accW1[3] = {0.f, 0.f, 0.f}, accWc1[3] = {0.f, 0.f, 0.f};
      float accW3 = 0.0f, accS = 0.0f, accT = 0.0f;
      float lossV = 0.0f, lossA = 0.0f, skipped = 0.0f;
      for (int b0 = 0; b0 < B; b0 += kTile) {
        const int nvalid = min(kTile, B - b0);
        __syncthreads();
        if (tid < kTile) E.rows[tid] = r0 + (tid < nvalid ? index[b0 + tid] : 0);
        __syncthreads();
        for (int i = tid; i < kTile * kIn; i += kMlpThreads) {
          const int s = i / kIn;
          S.X[i] = (s < nvalid) ? p.states[(size_t)E.rows[s] * kIn + (i - s * kIn)] : 0.0f;
        }
        __syncthreads();
        tile_forward(S, tid);
        tile_surrogate(S, p, gc, nvalid, [&](int s) { return E.rows[s]; }, lossV, lossA, skipped, tid);
        tile_backward(S, accW2, accW1, accWc1, accW3, accS, accT, tid);
      }
      __syncthreads();
      write_grad(S, accW2, accW1, accWc1, accW3, accS, accT, lossV, lossA, skipped, e.grads, tid);
      // the per-mini-batch path reduces ONE partial (0 + partial + 0 ...): the same values, with -0 stored as +0
      AdamParams a = e.adam;
#pragma unroll
      for (int l = 0; l < 5; l++) {
        a.corr1[l] = e.corr[step * 10 + l];
        a.corr2[l] = e.corr[step * 10 + 5 + l];
      }
      for (int i = tid; i < kTotalParams + 3; i += kMlpThreads) {
        const float g = __fadd_rn(e.grads[i], 0.0f);
        e.grads[i] = g;
        if (i < kTotalParams) adam_update(a, i, g);
      }
      __syncthreads();
      if (tid == 0) skipped_total += e.grads[kGradSkipped];
      stage_weights(S, p, tid);  // (ordered before the next use by the next tile's first barrier)
    }
    if (tid == 0) {
      if (e.losses) {
        e.losses[2 * t] = nb > 0 ? e.grads[kGradLossV] : 0.0f;
        e.losses[2 * t + 1] = nb > 0 ? e.grads[kGradLossA] : 0.0f;
      }
      if (e.skipped) e.skipped[t] = (int32_t)skipped_total;
    }
  }
}

// ---- populations: P independent agents of the default networks, agent a at a * kAgentStride of the parameter / Adam / gradient
// arrays (new Walker() builds its own PPOAgent(12, 4), Walker.cs:25-34; N walkers of the reference are N independent learners)

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// population_act_kernel: PPOAgent.SampleActions (PPOAgent.cs:381-398) for N walkers, walker w with agent w.  One warp per walker:
// its 5 252 actor parameters (21 KB, every env-step) are copied into the warp's shared memory with cp.async, W2 into rows padded
// to kPad floats so that the lanes' float4 row reads are conflict-free.  Lane o computes hidden units o and o + 32, lanes 0..3
// the four means and the sampling, lane 4 the optional critic value.  Every dot product is the chain of dense64_forward /
// tile_forward (a left-to-right fmaf chain from 0, then + b, then leaky or tanhf) and the sampling is ppo_fused_kernel's, so
// each row equals wb_policy_act_dev / wb_policy_sample of that agent on kernel variant 1 bit for bit.  Bandwidth-bound.
constexpr int kActHead = kHid * kIn + kHid;          // W1, b1
constexpr int kActTail = kHid + kAct * kHid + kAct;  // b2, W3, b3
struct __align__(16) ActWarpSmem {
  float head[kActHead];
  float W2[kHid * kPad];
  float tail[kActTail];
  float x[16];
  float a1[kHid], a2[kHid], c1[kHid];
};

__global__ void __launch_bounds__(kActWarps * 32) population_act_kernel(const PopActParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * kActWarps + warp;
  if (w >= P.n) return;  // (warp-uniform; the kernel has no CTA-wide barrier)
  ActWarpSmem& S = reinterpret_cast<ActWarpSmem*>(smem_raw)[warp];
  const float* prm = P.params + (size_t)w * kAgentStride;
  for (int c = lane; c < kActHead / 4; c += 32) cp_async16(S.head + 4 * c, prm + 4 * c);
  for (int c = lane; c < kHid * kHid / 4; c += 32) cp_async16(S.W2 + (c >> 4) * kPad + (c & 15) * 4, prm + kOffW2 + 4 * c);
  for (int c = lane; c < kActTail / 4; c += 32) cp_async16(S.tail + 4 * c, prm + kOffB2 + 4 * c);
  if (lane < kIn) S.x[lane] = P.states[(size_t)w * kIn + lane];
  cp_async_wait_all();
  __syncwarp();
  const float *W1 = S.head, *b1 = S.head + kHid * kIn, *b2 = S.tail, *W3 = S.tail + kHid, *b3 = W3 + kAct * kHid;
#pragma unroll
  for (int h = 0; h < 2; h++) {  // actor L1
    const int o = lane + 32 * h;
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < kIn; i += 4) {
      const float4 a = ld4(S.x + i), wv = ld4(W1 + o * kIn + i);
      acc = fmaf(a.x, wv.x, acc);
      acc = fmaf(a.y, wv.y, acc);
      acc = fmaf(a.z, wv.z, acc);
      acc = fmaf(a.w, wv.w, acc);
    }
    S.a1[o] = leaky(acc + b1[o]);
  }
  if (P.value) {  // critic L1, straight from global memory (read only when the value is asked for)
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int o = lane + 32 * h;
      float acc = 0.0f;
#pragma unroll
      for (int i = 0; i < kIn; i += 4) {
        const float4 a = ld4(S.x + i), wv = __ldg(reinterpret_cast<const float4*>(prm + kOffWc1 + o * kIn + i));
        acc = fmaf(a.x, wv.x, acc);
        acc = fmaf(a.y, wv.y, acc);
        acc = fmaf(a.z, wv.z, acc);
        acc = fmaf(a.w, wv.w, acc);
      }
      S.c1[o] = leaky(acc + __ldg(prm + kOffBc1 + o));
    }
  }
  __syncwarp();
  {  // actor L2
    float acc0 = 0.0f, acc1 = 0.0f;
#pragma unroll 4
    for (int i = 0; i < kHid; i += 4) {
      const float4 a = ld4(S.a1 + i), w0 = ld4(S.W2 + lane * kPad + i), w1 = ld4(S.W2 + (lane + 32) * kPad + i);
      acc0 = fmaf(a.x, w0.x, acc0);
      acc0 = fmaf(a.y, w0.y, acc0);
      acc0 = fmaf(a.z, w0.z, acc0);
      acc0 = fmaf(a.w, w0.w, acc0);
      acc1 = fmaf(a.x, w1.x, acc1);
      acc1 = fmaf(a.y, w1.y, acc1);
      acc1 = fmaf(a.z, w1.z, acc1);
      acc1 = fmaf(a.w, w1.w, acc1);
    }
    S.a2[lane] = leaky(acc0 + b2[lane]);
    S.a2[lane + 32] = leaky(acc1 + b2[lane + 32]);
  }
  __syncwarp();
  if (lane < kAct) {  // actor L3 + TanH, then Box-Muller and log_prob
    const int k = lane;
    float sum = 0.0f;
#pragma unroll 4
    for (int i = 0; i < kHid; i += 4) {
      const float4 a = ld4(S.a2 + i), wv = ld4(W3 + k * kHid + i);
      sum = fmaf(a.x, wv.x, sum);
      sum = fmaf(a.y, wv.y, sum);
      sum = fmaf(a.z, wv.z, sum);
      sum = fmaf(a.w, wv.w, sum);
    }
    const float mu = tanhf(sum + b3[k]);
    const PopAgent& ag = P.agents[w];
    float u1, u2, a, lp;
    sample_uniforms(P.mode, P.uniforms, P.seed, P.step, w, k, u1, u2);
    sample_action(mu, ag.stdv, ag.neg_log_std, ag.log_sqrt_2pi, u1, u2, a, lp);
    P.actions[(size_t)w * kAct + k] = a;
    P.logp[(size_t)w * kAct + k] = lp;
    if (P.mean) P.mean[(size_t)w * kAct + k] = mu;
  } else if (lane == kAct && P.value) {  // critic L2
    float v = 0.0f;
#pragma unroll 4
    for (int i = 0; i < kHid; i += 4) {
      const float4 a = ld4(S.c1 + i), wv = __ldg(reinterpret_cast<const float4*>(prm + kOffWc2 + i));
      v = fmaf(a.x, wv.x, v);
      v = fmaf(a.y, wv.y, v);
      v = fmaf(a.z, wv.z, v);
      v = fmaf(a.w, wv.w, v);
    }
    P.value[w] = v + __ldg(prm + kOffBc2);
  }
}

// population_episodes_kernel: ppo_episodes_kernel over many agents -- one CTA per agent with work in the call, training that agent's
// items (finished episodes) in list order with the agent's own parameters, Adam moments, gradient buffer, constants and slice of
// the host's Adam correction table.  Independent networks, so the CTAs need no exchange (one SM per agent).  An item's rows live
// in a time-major ring [R][C]: row i = ((t0 + i) mod R) * C + column.  Its rewards and values are gathered into shared memory for
// trajectory_returns and the returns / advantages scattered back.  Mini-batch indices come from the caller or, with a null index
// pointer, from draw_permutation (ppo_device.cuh).
struct __align__(16) PopSmem {
  MlpSmem m;
  int32_t rows[kTile];
  float rew[kPopMaxLen], val[kPopMaxLen], ret[kPopMaxLen], adv[kPopMaxLen];
  uint32_t key[kPopMaxLen];
  int32_t perm[kPopMaxLen];
};

__global__ void __launch_bounds__(kMlpThreads, 1) population_episodes_kernel(const PopTrainParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PopSmem& E = *reinterpret_cast<PopSmem*>(smem_raw);
  MlpSmem& S = E.m;
  const int tid = threadIdx.x;
  const PopCta cta = P.ctas[blockIdx.x];
  const PopAgent ag = P.agents[cta.agent];
  const size_t base = (size_t)cta.agent * kAgentStride;
  MlpParams p{};
  p.params = P.params + base;
  p.states = P.states;
  p.actions = P.actions;
  p.old_logp = P.old_logp;
  p.advantages = P.advantages;
  p.returns = P.returns;
  p.batch_size = ag.batch_size_f;
  const GradConsts gc{ag.stdv, ag.neg_log_std, ag.log_sqrt_2pi, ag.upper, ag.lower, ag.variance};
  float* grads = P.grads + base;
  AdamParams adam{};
  adam.params = P.params + base;
  adam.grads = grads;
  adam.m = P.m + base;
  adam.v = P.v + base;
  adam.alpha = ag.alpha;
  adam.beta1 = ag.beta1;
  adam.beta2 = ag.beta2;
  adam.eps = ag.adam_eps;
  const int B = ag.batch, R = P.ring_rows, C = P.columns;
  stage_weights(S, p, tid);
  for (int it = 0; it < cta.count; it++) {
    const PopItem item = P.items[cta.first + it];
    const int L = item.length;
    auto row_of = [&](int i) {
      const int t = item.t0 + i;
      return (t >= R ? t - R : t) * C + item.column;
    };
    // ---- CalculateValues (PPOAgent.cs:175-189)
    for (int s0 = 0; s0 < L; s0 += kTile) {
      const int nvalid = min(kTile, L - s0);
      __syncthreads();
      for (int i = tid; i < kTile * kIn; i += kMlpThreads) {
        const int s = i / kIn;
        S.X[i] = (s < nvalid) ? p.states[(size_t)row_of(s0 + s) * kIn + (i - s * kIn)] : 0.0f;
      }
      __syncthreads();
      tile_forward(S, tid);
      if (tid < nvalid) E.val[s0 + tid] = S.V[tid];
    }
    for (int i = tid; i < L; i += kMlpThreads) E.rew[i] = P.rewards[row_of(i)];
    __syncthreads();
    if (tid == 0 && L > 0)
      trajectory_returns(E.rew, E.val, L, ag.gamma, ag.lambda, ag.use_gae, ag.normalize, ag.norm_eps, E.ret, E.adv);
    __syncthreads();
    for (int i = tid; i < L; i += kMlpThreads) {
      const int r = row_of(i);
      P.values[r] = E.val[i];
      P.returns[r] = E.ret[i];
      P.advantages[r] = E.adv[i];
    }
    __syncthreads();  // (the surrogate reads the returns / advantages back from global memory)
    // ---- epochs x floor(L / B) mini-batches, each Train(Batch) + NeuralNetwork.Optimise
    const int per_epoch = L / B;
    int step = 0;
    float skipped_total = 0.0f;
    for (int epoch = 0; epoch < P.epochs && per_epoch > 0; epoch++) {
      const int32_t* index = E.perm;
      if (P.batch_index) index = P.batch_index + item.index_off + (size_t)epoch * per_epoch * B;
      else draw_permutation<kMlpThreads>(E.key, E.perm, L, epoch, item.episode, cta.agent, P.seed, tid);
      for (int b = 0; b < per_epoch; b++, step++, index += B) {
        float accW2[4][4];
#pragma unroll
        for (int j = 0; j < 4; j++)
#pragma unroll
          for (int l = 0; l < 4; l++) accW2[j][l] = 0.0f;
        float accW1[3] = {0.f, 0.f, 0.f}, accWc1[3] = {0.f, 0.f, 0.f};
        float accW3 = 0.0f, accS = 0.0f, accT = 0.0f;
        float lossV = 0.0f, lossA = 0.0f, skipped = 0.0f;
        for (int b0 = 0; b0 < B; b0 += kTile) {
          const int nvalid = min(kTile, B - b0);
          __syncthreads();
          if (tid < kTile) E.rows[tid] = row_of(tid < nvalid ? index[b0 + tid] : 0);
          __syncthreads();
          for (int i = tid; i < kTile * kIn; i += kMlpThreads) {
            const int s = i / kIn;
            S.X[i] = (s < nvalid) ? p.states[(size_t)E.rows[s] * kIn + (i - s * kIn)] : 0.0f;
          }
          __syncthreads();
          tile_forward(S, tid);
          tile_surrogate(S, p, gc, nvalid, [&](int s) { return E.rows[s]; }, lossV, lossA, skipped, tid);
          tile_backward(S, accW2, accW1, accWc1, accW3, accS, accT, tid);
        }
        __syncthreads();
        write_grad(S, accW2, accW1, accWc1, accW3, accS, accT, lossV, lossA, skipped, grads, tid);
        AdamParams a = adam;
        const float* corr = P.corr + (size_t)(item.corr_off + step) * 10;
#pragma unroll
        for (int l = 0; l < 5; l++) {
          a.corr1[l] = corr[l];
          a.corr2[l] = corr[5 + l];
        }
        for (int i = tid; i < kTotalParams + 3; i += kMlpThreads) {
          const float g = __fadd_rn(grads[i], 0.0f);  // (as ppo_episodes_kernel: what the one-partial reduction stores)
          grads[i] = g;
          if (i < kTotalParams) adam_update(a, i, g);
        }
        __syncthreads();
        if (tid == 0) skipped_total += grads[kGradSkipped];
        stage_weights(S, p, tid);  // (ordered before the next use by the next tile's first barrier)
      }
    }
    if (tid == 0) {
      const bool trained = P.epochs > 0 && per_epoch > 0;
      if (P.losses) {
        P.losses[2 * item.out] = trained ? grads[kGradLossV] : 0.0f;
        P.losses[2 * item.out + 1] = trained ? grads[kGradLossA] : 0.0f;
      }
      if (P.skipped) P.skipped[item.out] = (int32_t)skipped_total;
    }
  }
}

// The same recurrences over a time-major rollout buffer [T][N] of N lockstep environments (the reference trains on one
// episode of one environment, PPOAgent.cs:147; here every environment contributes the fragments of its episodes that fall
// inside the T-step segment).  One thread per environment, reverse scan; a step with done != 0 is the LAST step of its
// episode, so the recurrence restarts there exactly like at the end of a trajectory (next return / next value = 0).
// The segment end: an episode that is still running when the segment ends is NOT over, so its tail must not be scored as if
// the return stopped there.  With `last_values` (the critic's estimate V(s_T) of the observation AFTER the last step) the scan
// starts from it -- next return = next value = V(s_T) unless dones[T-1] is set -- which is the standard bootstrap for a
// fixed-horizon rollout; the reference never needs it because it only trains on complete episodes.  last_values == nullptr
// keeps the reference's trajectory-end semantics at the segment end (truncation: the form the oracle comparison uses).
__global__ void segment_returns_kernel(const float* __restrict__ rewards, const float* __restrict__ values, const uint8_t* __restrict__ dones,
                                       const float* __restrict__ last_values, int n_envs, int T, float gamma, float lambda, int use_gae,
                                       float* __restrict__ returns, float* __restrict__ advantages) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_envs) return;
  const float boot = last_values != nullptr ? last_values[e] : 0.0f;
  if (use_gae) {
    const float next_gae = 0.0f;  // never updated in the reference (PPOAgent.cs:414-444)
    float next_value = boot;
    for (int t = T - 1; t >= 0; t--) {
      const size_t i = (size_t)t * n_envs + e;
      if (dones[i]) next_value = 0.0f;
      const float cur = values[i];
      const float delta = __fsub_rn(__fadd_rn(rewards[i], __fmul_rn(gamma, next_value)), cur);
      next_value = cur;
      const float gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gamma, lambda), next_gae));
      advantages[i] = gae;
      returns[i] = __fadd_rn(gae, cur);
    }
  } else {
    float g = boot;
    for (int t = T - 1; t >= 0; t--) {
      const size_t i = (size_t)t * n_envs + e;
      if (dones[i]) g = 0.0f;
      g = __fadd_rn(rewards[i], __fmul_rn(g, gamma));
      returns[i] = g;
      advantages[i] = __fsub_rn(g, values[i]);
    }
  }
}

// PPOAgent.Normalize (PPOAgent.cs:461-472) over a pool of advantages, in three launches so that a data-parallel caller can
// all-reduce the two double sums in between (stats[0] = sum x, stats[1] = sum ((double)(x - mean))^2, both accumulated in
// double like List<float>.Average() / Sum(Math.Pow(value - mean, 2)); the summation order is a fixed tree instead of the
// reference's left-to-right loop, a difference of ~1e-16 relative in the double sums before they are rounded to float).
//   stage 0: partial sums of x                         -> stats[0 .. kNormCtas)
//   stage 1: mean = (float)(sum / count); partial sums of ((double)(x - mean))^2 -> stats[kNormCtas .. 2 kNormCtas)
//   stage 2: std = (float)sqrt(sum2 / count); x = (x - mean) / (std + epsilon)
// Every consumer adds the kNormCtas partials in index order, so the totals are identical wherever they are formed (a
// data-parallel caller all-reduces the partial arrays element by element between the stages).
__device__ __forceinline__ double norm_total(const double* stats, int stage, double* s_bcast) {
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int g = 0; g < kNormCtas; g++) t += stats[stage * kNormCtas + g];
    *s_bcast = t;
  }
  __syncthreads();
  return *s_bcast;
}
__global__ void __launch_bounds__(kNormThreads) normalize_sums_kernel(const float* __restrict__ x, long n, double count, int stage, double* stats) {
  __shared__ double red[kNormThreads];
  __shared__ double s_sum;
  float mean = 0.0f;
  if (stage == 1) mean = (float)(norm_total(stats, 0, &s_sum) / count);
  double acc = 0.0;
  for (long i = (long)blockIdx.x * kNormThreads + threadIdx.x; i < n; i += (long)kNormCtas * kNormThreads) {
    if (stage == 0) {
      acc += (double)x[i];
    } else {
      const double d = (double)__fsub_rn(x[i], mean);
      acc += d * d;
    }
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int w = kNormThreads / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) stats[stage * kNormCtas + blockIdx.x] = red[0];
}
__global__ void __launch_bounds__(256) normalize_apply_kernel(float* __restrict__ x, long n, double count, float epsilon, const double* __restrict__ stats) {
  __shared__ double s_sum, s_sum2;
  const float mean = (float)(norm_total(stats, 0, &s_sum) / count);
  const float sd = (float)sqrt(norm_total(stats, 1, &s_sum2) / count);
  const float div = __fadd_rn(sd, epsilon);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) x[i] = __fdiv_rn(__fsub_rn(x[i], mean), div);
}

// PPOAgent.CreateBatches (PPOAgent.cs:501-540) on the device: rows index[b] of the rollout pool -> a contiguous minibatch.
// 22 floats per sample: state 12, action 4, log-probability 4, advantage, return; one thread per (sample, float).
__global__ void gather_minibatch_kernel(const int32_t* __restrict__ index, int B, const float* __restrict__ states,
                                        const float* __restrict__ actions, const float* __restrict__ logp, const float* __restrict__ adv,
                                        const float* __restrict__ ret, float* __restrict__ o_states, float* __restrict__ o_actions,
                                        float* __restrict__ o_logp, float* __restrict__ o_adv, float* __restrict__ o_ret) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = gid / 22, f = gid % 22;
  if (b >= B) return;
  const size_t src = (size_t)index[b];
  if (f < 12) o_states[(size_t)b * 12 + f] = states[src * 12 + f];
  else if (f < 16) o_actions[(size_t)b * 4 + (f - 12)] = actions[src * 4 + (f - 12)];
  else if (f < 20) o_logp[(size_t)b * 4 + (f - 16)] = logp[src * 4 + (f - 16)];
  else if (f == 20) o_adv[b] = adv[src];
  else o_ret[b] = ret[src];
}

// ---------------------------------------------------------------- host side
static GradConsts grad_consts(float log_std, float epsilon) {
  GradConsts gc;
  gc.stdv = expf(log_std);                         // PPOAgent.GetStandardDeviations, PPOAgent.cs:367-378
  gc.neg_log_std = -logf(gc.stdv);                 // NormalDistribution.cs:31
  gc.log_sqrt_2pi = logf(sqrtf(2.0f * 3.14159274f));
  gc.upper = 1.0f + epsilon;
  gc.lower = 1.0f - epsilon;
  gc.variance = gc.stdv * gc.stdv;
  return gc;
}

void population_agent_consts(const wb_hyperparams& hp, PopAgent* o) {
  const GradConsts gc = grad_consts(hp.log_std, hp.epsilon);
  *o = PopAgent{};
  o->stdv = gc.stdv;
  o->neg_log_std = gc.neg_log_std;
  o->log_sqrt_2pi = gc.log_sqrt_2pi;
  o->upper = gc.upper;
  o->lower = gc.lower;
  o->variance = gc.variance;
  o->alpha = hp.alpha;
  o->beta1 = hp.beta1;
  o->beta2 = hp.beta2;
  o->adam_eps = hp.adam_epsilon;
  o->gamma = hp.gamma;
  o->lambda = hp.lambda;
  o->norm_eps = hp.epsilon;  // PPOAgent.Normalize divides by std + the PPO clip epsilon, as trajectory_returns' callers pass it
  o->batch_size_f = (float)hp.batch_size;
  o->batch = hp.batch_size;
  o->use_gae = hp.use_gae;
  o->normalize = hp.normalize_advantages;
  o->log_std = hp.log_std;
  o->clip_eps = hp.epsilon;
}

cudaError_t launch_population_act(const PopActParams& a, cudaStream_t stream) {
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  const int smem = (int)(kActWarps * sizeof(ActWarpSmem));
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t err = cudaFuncSetAttribute(population_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  population_act_kernel<<<(a.n + kActWarps - 1) / kActWarps, kActWarps * 32, smem, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_population_episodes(const PopTrainParams& t, int n_ctas, cudaStream_t stream) {
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t err = cudaFuncSetAttribute(population_episodes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PopSmem));
    if (err != cudaSuccess) return err;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  population_episodes_kernel<<<n_ctas, kMlpThreads, sizeof(PopSmem), stream>>>(t);
  return cudaGetLastError();
}

cudaError_t launch_segment_returns(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, int n_envs,
                                   int T, float gamma, float lambda, int use_gae, float* returns, float* advantages, cudaStream_t stream) {
  segment_returns_kernel<<<(n_envs + 127) / 128, 128, 0, stream>>>(rewards, values, dones, last_values, n_envs, T, gamma, lambda, use_gae,
                                                                   returns, advantages);
  return cudaGetLastError();
}

cudaError_t launch_normalize_stage(float* x, long n_local, double count_global, int stage, float epsilon, double* stats, cudaStream_t stream) {
  if (stage == 0 || stage == 1)
    normalize_sums_kernel<<<kNormCtas, kNormThreads, 0, stream>>>(x, n_local, count_global, stage, stats);
  else
    normalize_apply_kernel<<<296, 256, 0, stream>>>(x, n_local, count_global, epsilon, stats);
  return cudaGetLastError();
}

cudaError_t launch_gather_minibatch(const int32_t* index, int B, const float* states, const float* actions, const float* logp,
                                    const float* adv, const float* ret, float* o_states, float* o_actions, float* o_logp, float* o_adv,
                                    float* o_ret, cudaStream_t stream) {
  const long total = (long)B * 22;
  gather_minibatch_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(index, B, states, actions, logp, adv, ret, o_states,
                                                                               o_actions, o_logp, o_adv, o_ret);
  return cudaGetLastError();
}

int mlp_grid_for(int n, int sm_count) {
  const int ntiles = (n + kTile - 1) / kTile;
  return ntiles < sm_count ? (ntiles > 0 ? ntiles : 1) : sm_count;
}

cudaError_t launch_mlp(const MlpParams& p, int grid, cudaStream_t stream) {
  // opt in to > 48 KB of dynamic shared memory: a per-DEVICE function attribute (a process may drive several GPUs)
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(ppo_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MlpSmem));
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  ppo_fused_kernel<<<grid, kMlpThreads, sizeof(MlpSmem), stream>>>(p, grad_consts(p.log_std, p.epsilon));
  return cudaGetLastError();
}

// ---------------------------------------------------------------- fused gradient reduction + all-reduce over NVLink peer memory
// The data-parallel update needs sum over ranks of (sum over this rank's CTAs of the partial gradients): a 24.6 KB message,
// latency bound.  Instead of reduce_partials_kernel followed by an NCCL all-reduce, ONE kernel does both: CTA c owns float4
// slice c of the gradient buffer; it sums the rank's per-CTA partials for its slice in fixed order, PUSHES the slice into slot
// [rank] of every peer's exchange buffer with plain stores over NVLink (peer pointers opened through CUDA IPC), publishes an
// epoch flag per (peer, rank, slice) with a system-scope release, waits for the world's flags in its OWN buffer (acquire) and
// adds the world's slots in rank order -- every rank performs the same additions in the same order, so the reduced gradient
// (and therefore Adam and the weights) is bit-identical everywhere.  Slices are independent (no grid-wide barrier) and the
// slots are double buffered by epoch parity: a rank can run at most one exchange ahead of the slowest peer.
// (st_release_sys / ld_acquire_sys: mlp.cuh)

__global__ void __launch_bounds__(kExchThreads) reduce_exchange_kernel(const float* __restrict__ partials, int nparts, float* __restrict__ grads,
                                                                       ExchPeers peers, int rank, int world, uint32_t epoch, uint32_t* status, uint32_t* dead,
                                                                       AdamParams adam, int do_adam) {
  // kExchLanes threads per float4 of the slice: each sums every kExchLanes-th per-CTA partial (<= 10 independent loads in flight
  // per thread, 97 CTAs: the 3.6 MB of partials are read at memory speed instead of as 13 CTAs' dependent chains), then the
  // partial sums are combined pairwise by shuffles -- a fixed order, so the result is deterministic
  const int part = threadIdx.x & (kExchLanes - 1);
  const int i4 = blockIdx.x * (kExchThreads / kExchLanes) + (threadIdx.x / kExchLanes);  // float4 index inside the gradient buffer
  const bool in = i4 < kGradFloats / 4;
  const int par = (int)(epoch & 1u);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (in) {
    const float4* p4 = reinterpret_cast<const float4*>(partials) + i4;
#pragma unroll 10
    for (int q = part; q < nparts; q += kExchLanes) {
      const float4 v = p4[(size_t)q * (kGradFloats / 4)];
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
  }
#pragma unroll
  for (int m = 1; m < kExchLanes; m <<= 1) {
    acc.x += __shfl_xor_sync(0xFFFFFFFFu, acc.x, m);
    acc.y += __shfl_xor_sync(0xFFFFFFFFu, acc.y, m);
    acc.z += __shfl_xor_sync(0xFFFFFFFFu, acc.z, m);
    acc.w += __shfl_xor_sync(0xFFFFFFFFu, acc.w, m);
  }
  float4 s = acc;
  bool ok = true;
  if (world > 1) {  // (world is a kernel argument: uniform)
    // a previous exchange of this handle timed out: the ranks' weights can no longer be assumed identical -- every later launch
    // is a no-op (no store, no Adam) until the host has seen the status word (wb_comm_status / wb_ppo_train_dev refuse)
    // (`dead` is the DEVICE copy of the status word: reading the mapped host word from every CTA costs one PCIe round trip per
    //  CTA, and those serialise -- ~1 us each, 100 us per exchange with 97 CTAs)
    if (__syncthreads_or(threadIdx.x == 0 && *reinterpret_cast<volatile uint32_t*>(dead) != 0u)) return;  // (CTA-uniform)
    if (in) {
      // push my slice into slot [par][rank] of every rank (NVLink stores; r == rank is local); the lanes of an element share the peers
      for (int r = part; r < world; r += kExchLanes) reinterpret_cast<float4*>(peers.base[r] + exch_slot_offset(par, rank))[i4] = acc;
    }
    // the CTA's pushes are ordered before the flags by the barrier + ONE system-scope release per flag (release is cumulative over
    // what the barrier made visible to the flag's thread).  A __threadfence_system() in every thread of every CTA -- 25 000
    // MEMBAR.SYS per exchange -- cost ~100 us on its own.
    __syncthreads();
    if ((int)threadIdx.x < world) {
      __threadfence_system();
      st_release_sys(exch_flag(peers.base[threadIdx.x], par, rank, blockIdx.x), epoch);
    }
    bool timed_out = false;
    if ((int)threadIdx.x < world) {  // wait for rank threadIdx.x's slice in MY buffer
      const uint32_t* f = exch_flag(peers.base[rank], par, threadIdx.x, blockIdx.x);
      long spins = 0;
      while (ld_acquire_sys(f) != epoch) {
        if (++spins > (1L << 31)) {  // a peer never arrived (crashed?): give up loudly instead of hanging the GPU
          *reinterpret_cast<volatile uint32_t*>(status) = 1u;  // (mapped host memory: the host sees it without a copy)
          *reinterpret_cast<volatile uint32_t*>(dead) = 1u;    // (device copy: what later launches check)
          __threadfence_system();
          timed_out = true;
          break;
        }
      }
    }
    // a slice whose peers did not all arrive holds stale slot data: it must neither be stored nor reach Adam
    ok = __syncthreads_or(timed_out) == 0;
    if (ok && in && part == 0) {
      s = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int r = 0; r < world; r++) {  // rank order on every rank: bit-identical sums
        const float4 v = __ldcg(reinterpret_cast<const float4*>(peers.base[rank] + exch_slot_offset(par, r)) + i4);
        s.x += v.x;
        s.y += v.y;
        s.z += v.z;
        s.w += v.w;
      }
    }
  }
  if (ok && in && part == 0) {
    reinterpret_cast<float4*>(grads)[i4] = s;
    if (do_adam) {  // NeuralNetwork.Optimise fused behind the reduction: the gradient never makes another round trip
      const float g[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
      for (int c = 0; c < 4; c++)
        if (i4 * 4 + c < kTotalParams) adam_update(adam, i4 * 4 + c, g[c]);
    }
  }
}

cudaError_t launch_reduce_exchange(const float* partials, int nparts, float* grads, const ExchPeers& peers, int rank, int world,
                                   uint32_t epoch, uint32_t* status, uint32_t* dead, const AdamParams* adam, cudaStream_t stream) {
  AdamParams a{};
  if (adam) a = *adam;
  reduce_exchange_kernel<<<kExchCtas, kExchThreads, 0, stream>>>(partials, nparts, grads, peers, rank, world, epoch, status, dead, a, adam != nullptr);
  return cudaGetLastError();
}

cudaError_t launch_reduce_partials(const float* partials, int nparts, float* grads, cudaStream_t stream) {
  reduce_partials_kernel<<<(kGradFloats + 127) / 128, 128, 0, stream>>>(partials, nparts, grads);
  return cudaGetLastError();
}

cudaError_t launch_adam(const AdamParams& p, cudaStream_t stream) {
  adam_kernel<<<(kTotalParams + 127) / 128, 128, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_episodes(const EpisodeParams& e, const MlpParams& p, cudaStream_t stream) {
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t err = cudaFuncSetAttribute(ppo_episodes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EpisodeSmem));
    if (err != cudaSuccess) return err;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  ppo_episodes_kernel<<<1, kMlpThreads, sizeof(EpisodeSmem), stream>>>(e, p, grad_consts(p.log_std, p.epsilon));
  return cudaGetLastError();
}

// rows row_base + index[b] of the row arrays -> a contiguous mini-batch, any state / action width (one thread per (sample, float))
__global__ void gather_rows_kernel(const int32_t* __restrict__ index, int B, int row_base, int sdim, int adim, const float* __restrict__ states,
                                   const float* __restrict__ actions, const float* __restrict__ logp, const float* __restrict__ adv,
                                   const float* __restrict__ ret, float* __restrict__ o_states, float* __restrict__ o_actions,
                                   float* __restrict__ o_logp, float* __restrict__ o_adv, float* __restrict__ o_ret) {
  const int per = sdim + 2 * adim + 2;
  const long gid = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(gid / per), f = (int)(gid % per);
  if (b >= B) return;
  const size_t src = (size_t)row_base + index[b];
  if (f < sdim) o_states[(size_t)b * sdim + f] = states[src * sdim + f];
  else if (f < sdim + adim) o_actions[(size_t)b * adim + (f - sdim)] = actions[src * adim + (f - sdim)];
  else if (f < sdim + 2 * adim) o_logp[(size_t)b * adim + (f - sdim - adim)] = logp[src * adim + (f - sdim - adim)];
  else if (f == sdim + 2 * adim) o_adv[b] = adv[src];
  else o_ret[b] = ret[src];
}

// losses[2] <- the gradient buffer's loss sums, skipped += its skipped count (one trajectory's mini-batches, in order)
__global__ void episode_losses_kernel(const float* __restrict__ tail, float* losses, int32_t* skipped) {
  if (threadIdx.x != 0) return;
  if (losses) {
    losses[0] = tail[0];
    losses[1] = tail[1];
  }
  if (skipped) *skipped += (int32_t)tail[2];
}

cudaError_t launch_gather_rows(const int32_t* index, int B, int row_base, int sdim, int adim, const float* states, const float* actions,
                               const float* logp, const float* adv, const float* ret, float* o_states, float* o_actions, float* o_logp,
                               float* o_adv, float* o_ret, cudaStream_t stream) {
  const long total = (long)B * (sdim + 2 * adim + 2);
  gather_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(index, B, row_base, sdim, adim, states, actions, logp, adv, ret,
                                                                          o_states, o_actions, o_logp, o_adv, o_ret);
  return cudaGetLastError();
}

cudaError_t launch_episode_losses(const float* grads_tail, float* losses, int32_t* skipped, cudaStream_t stream) {
  episode_losses_kernel<<<1, 32, 0, stream>>>(grads_tail, losses, skipped);
  return cudaGetLastError();
}

cudaError_t launch_returns(const float* rewards, const float* values, int n, float gamma, float lambda, int use_gae, int normalize,
                           float norm_eps, float* returns, float* advantages, cudaStream_t stream) {
  returns_kernel<<<1, 32, 0, stream>>>(rewards, values, n, gamma, lambda, use_gae, normalize, norm_eps, returns, advantages);
  return cudaGetLastError();
}

}  // namespace wb

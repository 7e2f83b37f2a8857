// mlp_generic.cu -- the PPO pipeline for ANY network the reference's DSL can describe (PPOAgent.ParseLayers, PPOAgent.cs:96-143):
// any sequence of dense layers (widths 1..128) and ReLU / LeakyReLU / TanH activations (ActivationLayer.cs:32-73), any state and
// action size.  The tensor-core kernel (mlp_tc.cu) and the register-blocked fp32 kernel (mlp.cu) are specialised for the
// reference's default topologies; a user-edited Hyperparameters.ActorNeuralNetwork / CriticNeuralNetwork lands here instead of
// falling off the GPU path.  General, not tuned: one CTA per tile of TS samples, the layer inputs the reference caches
// (NeuralNetwork._cache: the INPUT of every layer, NeuralNetwork.cs:52-64) live in shared memory, every dot product runs left to
// right like Matrix.Multiply (Matrix.cs:604-616) with the product and the sum rounded separately (no FMA: a pre-activation that
// lands within rounding distance of an activation's kink takes the same side as in the C# loop), the cross-sample sums of
// dW / db are formed per CTA in sample order and added to a per-CTA partial that the same thread always owns (deterministic),
// then reduced by reduce_partials_n.
//
//   forward    NeuralNetwork.FeedForward / DenseLayer.FeedForward (DenseLayer.cs:82-98)
//   sample     PPOAgent.SampleActions (PPOAgent.cs:381-398), Box-Muller sin branch (NormalDistribution.cs:12-19)
//   gradient   PPOAgent.Train(Batch) (PPOAgent.cs:218-342): per-dimension ratio / clip, HadamardDivision zero divisor => sample
//              skipped, losses; NeuralNetwork.FeedBack / DenseLayer.FeedBack (DenseLayer.cs:103-120) / ActivationLayer.FeedBack
//
// The population kernels below (population_generic_act_kernel, population_generic_episodes_kernel) run P independent agents of
// such networks and share the forward, backward, surrogate and sampling code with ppo_generic_kernel, so that agent a computes
// the bits of one wb_policy on this kernel.
#include "common.h"
#include "mlp.cuh"
#include "ppo_device.cuh"

namespace wb {

namespace {

__device__ __forceinline__ float gen_activate(int kind, float v) {
  if (kind == WB_RELU) return fmaxf(0.0f, v);             // MathF.Max(0, value)
  if (kind == WB_LEAKYRELU) return fmaxf(0.2f * v, v);    // MathF.Max(Alpha * value, value)
  return tanhf(v);                                        // MathF.Tanh
}
__device__ __forceinline__ float gen_derivative(int kind, float v) {
  if (kind == WB_RELU) return v < 0.0f ? 0.0f : 1.0f;
  if (kind == WB_LEAKYRELU) return v < 0.0f ? 0.2f : 1.0f;
  const float t = tanhf(v);
  return 1.0f - (t * t);
}

__device__ __forceinline__ float gen_log_prob(float mean, float stdv, float action, float neg_log_std, float log_sqrt_2pi) {
  float fraction = (action - mean) / stdv;  // NormalDistribution.LogProbabilityDensity, NormalDistribution.cs:24-32
  fraction *= fraction;
  fraction /= 2.0f;
  return neg_log_std - log_sqrt_2pi - fraction;
}

// Weight loads: kLdg = true reads through the read-only data cache (ppo_generic_kernel: the weights do not change during the
// launch); kLdg = false is a plain coherent load, for a kernel that rewrites the weights with Adam inside the same launch
template <bool kLdg>
__device__ __forceinline__ float ld_weight(const float* p) {
  if (kLdg) return __ldg(p);
  return *p;
}

// NeuralNetwork.FeedForward over a tile: cache row of sample s = cache + s * stride; layer l reads its input at L[l].cache_off and
// writes the next layer's input (the last layer writes at net.cache_floats: the network output)
template <bool kLdg>
__device__ void gen_forward(const GenNet& net, const float* params, float* cache, int stride, int ts) {
  for (int l = 0; l < net.n_layers; l++) {
    const GenLayer& L = net.L[l];
    const int out_off = (l + 1 < net.n_layers) ? net.L[l + 1].cache_off : net.cache_floats;
    if (L.kind == WB_DENSE) {
      const float* W = params + L.w_off;
      const float* b = params + L.b_off;
      for (int idx = threadIdx.x; idx < ts * L.out; idx += blockDim.x) {
        const int s = idx / L.out, o = idx - s * L.out;
        const float* x = cache + (size_t)s * stride + L.cache_off;
        const float* w = W + (size_t)o * L.in;
        float acc = 0.0f;
        for (int i = 0; i < L.in; i++) acc = __fadd_rn(acc, __fmul_rn(x[i], ld_weight<kLdg>(w + i)));  // product and sum individually rounded, like the C# loop
        cache[(size_t)s * stride + out_off + o] = acc + ld_weight<kLdg>(b + o);
      }
    } else {
      for (int idx = threadIdx.x; idx < ts * L.in; idx += blockDim.x) {
        const int s = idx / L.in, j = idx - s * L.in;
        cache[(size_t)s * stride + out_off + j] = gen_activate(L.kind, cache[(size_t)s * stride + L.cache_off + j]);
      }
    }
    __syncthreads();
  }
}

// NeuralNetwork.FeedBack over a tile: g0 holds dL/d(output) [ts][kGenMaxWidth]; g1 is the ping-pong partner.  The per-CTA partial
// sums of dW / db are added to `partial` (flat parameter layout of this network); every element is always added by the same thread.
template <bool kLdg>
__device__ void gen_backward(const GenNet& net, const float* params, const float* cache, int stride, int ts, float* g0, float* g1,
                             float* partial) {
  float* g = g0;
  float* gn = g1;
  for (int l = net.n_layers - 1; l >= 0; l--) {
    const GenLayer& L = net.L[l];
    if (L.kind == WB_DENSE) {
      const float* W = params + L.w_off;
      // db += g ; dW += g x^T  (DenseLayer.FeedBack, DenseLayer.cs:103-120); element (o, i), i == in: the bias
      for (int idx = threadIdx.x; idx < L.out * (L.in + 1); idx += blockDim.x) {
        const int o = idx / (L.in + 1), i = idx - o * (L.in + 1);
        float acc = 0.0f;
        for (int s = 0; s < ts; s++) {
          const float gs = g[s * kGenMaxWidth + o];
          acc = __fadd_rn(acc, (i < L.in) ? __fmul_rn(gs, cache[(size_t)s * stride + L.cache_off + i]) : gs);
        }
        float* dst = partial + (i < L.in ? L.w_off + o * L.in + i : L.b_off + o);
        *dst += acc;
      }
      // g <- W^T g (sum over the outputs from 0, Matrix.Multiply order); the reference also does this for the first layer, where
      // nothing reads the result
      if (l > 0) {
        for (int idx = threadIdx.x; idx < ts * L.in; idx += blockDim.x) {
          const int s = idx / L.in, i = idx - s * L.in;
          float acc = 0.0f;
          for (int o = 0; o < L.out; o++) acc = __fadd_rn(acc, __fmul_rn(ld_weight<kLdg>(W + (size_t)o * L.in + i), g[s * kGenMaxWidth + o]));
          gn[s * kGenMaxWidth + i] = acc;
        }
        __syncthreads();
        float* t = g;
        g = gn;
        gn = t;
      } else {
        __syncthreads();
      }
    } else {
      for (int idx = threadIdx.x; idx < ts * L.in; idx += blockDim.x) {
        const int s = idx / L.in, j = idx - s * L.in;
        g[s * kGenMaxWidth + j] *= gen_derivative(L.kind, cache[(size_t)s * stride + L.cache_off + j]);
      }
      __syncthreads();
    }
  }
}

// PPOAgent.GetStandardDeviations (PPOAgent.cs:367-378), NormalDistribution.cs:31 and the clip range, on the device
struct GenConsts {
  float stdv, neg_log_std, log_sqrt_2pi, upper, lower, variance;
};
__device__ __forceinline__ GenConsts gen_consts(float log_std, float epsilon) {
  GenConsts c;
  c.stdv = expf(log_std);
  c.neg_log_std = -logf(c.stdv);
  c.log_sqrt_2pi = logf(sqrtf(2.0f * 3.14159274f));
  c.upper = 1.0f + epsilon;
  c.lower = 1.0f - epsilon;
  c.variance = c.stdv * c.stdv;
  return c;
}

// PPOAgent.SampleActions for action dimension k of sample gs: the two uniforms injected (kModeSample, uniforms [n][act][2]) or from
// the Philox stream (gs, k, step) under seed, then NormalDistribution.BoxMullerTransform (NormalDistribution.cs:12-19) around mu
__device__ __forceinline__ void gen_sample(int mode, const float* uniforms, uint64_t seed, uint64_t step, size_t gs, int k, int act, float mu,
                                           const GenConsts& c, float& a, float& lp) {
  float u1, u2;
  if (mode == kModeSample) {
    u1 = uniforms[(gs * act + k) * 2];
    u2 = uniforms[(gs * act + k) * 2 + 1];
  } else {
    const uint4 r = philox4x32(make_uint4((uint32_t)gs, (uint32_t)k, (uint32_t)step, (uint32_t)(step >> 32)),
                               make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    u1 = (float)(r.x >> 8) * (1.0f / 16777216.0f);
    u2 = (float)(r.y >> 8) * (1.0f / 16777216.0f);
  }
  if (u1 == 0.0f) u1 = 1.0f;
  const float z = sqrtf(-2.0f * logf(u1)) * sinf(2.0f * 3.14159274f * u2);
  a = mu + (c.stdv * z);
  lp = gen_log_prob(mu, c.stdv, a, c.neg_log_std, c.log_sqrt_2pi);
}

// The clipped-surrogate gradient of one sample (PPOAgent.cs:232-326), action dimensions in order: dL/dmu into g0_row[0..act),
// dL/dV into *gv, and for the loss sums g1_row[0] = skipped (0 / 1), g1_row[1] = the sample's actor loss term.  mu / a / lp_old:
// the sample's means, actions and old log-probabilities.
__device__ __forceinline__ void gen_surrogate(const float* mu_row, const float* a_row, const float* lp_row, float adv, float value, float ret,
                                              int act, float batch_size, const GenConsts& c, float* g0_row, float* g1_row, float* gv) {
  float gvs = (2.0f * (value - ret)) / batch_size;
  bool skip = false;
  float sum = 0.0f;
  for (int k = 0; k < act; k++) {
    const float mu = mu_row[k];
    const float a = a_row[k];
    const float lp_old = lp_row[k];
    const float lp = gen_log_prob(mu, c.stdv, a, c.neg_log_std, c.log_sqrt_2pi);
    const float ratio = expf(lp - lp_old);
    const float clipped = ratio >= c.upper ? c.upper : (ratio <= c.lower ? c.lower : ratio);  // Matrix.Clip, Matrix.cs:377-405
    const float cra = clipped * adv, ra = ratio * adv;
    const float partA = (ra <= cra ? 1.0f : 0.0f) * adv;                                    // Matrix.LessThan (<=)
    const float partB = (cra < ra ? 1.0f : 0.0f) * adv;                                     // Matrix.LessThanNotEquals
    const float partC = (ratio >= c.lower && ratio <= c.upper) ? 1.0f : 0.0f;               // Matrix.InRange
    float dclip = (partA + partB * partC) * -1.0f;
    const float pold = expf(lp_old);
    if (pold == 0.0f) skip = true;                                                          // HadamardDivision throws (Matrix.cs:348-374)
    dclip = dclip / pold;
    const float dmean = expf(lp) * ((a - mu) / c.variance);
    const float gk = (dmean * dclip) / batch_size;
    g0_row[k] = gk;
    sum += gk;
  }
  if (skip) {  // the reference `continue`s: no feedback for this sample, no loss contribution
    for (int k = 0; k < act; k++) g0_row[k] = 0.0f;
    gvs = 0.0f;
  }
  *gv = gvs;
  g1_row[0] = skip ? 1.0f : 0.0f;
  g1_row[1] = skip ? 0.0f : sum / (float)act;  // Matrix.Average, PPOAgent.cs:332
}

// thread 0: the tile's loss V, loss A and skipped count added to sums[0..2] in sample order
__device__ __forceinline__ void gen_add_loss_sums(const float* gv, const float* g1, int ts, float* sums) {
  for (int s = 0; s < ts; s++) {
    sums[0] += gv[s];
    sums[1] += g1[s * kGenMaxWidth + 1];
    sums[2] += g1[s * kGenMaxWidth];
  }
}

__global__ void __launch_bounds__(kGenThreads) ppo_generic_kernel(const GenParams p) {
  extern __shared__ __align__(16) float gsm[];
  const int ts_max = p.ts;
  const int strideA = p.actor.cache_floats + p.actor.output, strideC = p.critic.cache_floats + p.critic.output;
  float* cacheA = gsm;
  float* cacheC = cacheA + (size_t)ts_max * strideA;
  float* g0 = cacheC + (size_t)ts_max * strideC;
  float* g1 = g0 + (size_t)ts_max * kGenMaxWidth;
  float* gv = g1 + (size_t)ts_max * kGenMaxWidth;       // [ts] dL/dV per sample
  float* sums = gv + ts_max;                            // [4]: loss V, loss A, skipped
  const int tid = threadIdx.x;
  const int act = p.actor.output, sdim = p.actor.input;
  const float* paramsA = p.params;
  const float* paramsC = p.params + p.actor.n_params;
  const bool grad = p.mode == kModeGrad;
  float* partial = grad ? p.partials + (size_t)blockIdx.x * p.grad_floats : nullptr;
  if (grad) {
    for (int i = tid; i < p.grad_floats; i += blockDim.x) partial[i] = 0.0f;
    if (tid < 4) sums[tid] = 0.0f;
    __syncthreads();
  }
  const GenConsts c = gen_consts(p.log_std, p.epsilon);

  const int ntiles = (p.n + ts_max - 1) / ts_max;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int s0 = tile * ts_max;
    const int ts = min(ts_max, p.n - s0);
    for (int idx = tid; idx < ts * sdim; idx += blockDim.x) {
      const int s = idx / sdim, i = idx - s * sdim;
      const float v = p.states[(size_t)(s0 + s) * sdim + i];
      cacheA[(size_t)s * strideA + p.actor.L[0].cache_off + i] = v;
      cacheC[(size_t)s * strideC + p.critic.L[0].cache_off + i] = v;
    }
    __syncthreads();
    gen_forward<true>(p.actor, paramsA, cacheA, strideA, ts);
    gen_forward<true>(p.critic, paramsC, cacheC, strideC, ts);
    const float* mu_of = cacheA + p.actor.cache_floats;   // + s * strideA
    const float* v_of = cacheC + p.critic.cache_floats;   // + s * strideC

    if (!grad) {
      for (int idx = tid; idx < ts * act; idx += blockDim.x) {
        const int s = idx / act, k = idx - s * act;
        const size_t gs = (size_t)(s0 + s);
        const float mu = mu_of[(size_t)s * strideA + k];
        if (p.mean) p.mean[gs * act + k] = mu;
        if (p.mode == kModeSample || p.mode == kModeSamplePhilox) {
          float a, lp;
          gen_sample(p.mode, p.uniforms, p.seed, p.step, gs, k, act, mu, c, a, lp);
          p.out_actions[gs * act + k] = a;
          p.out_logp[gs * act + k] = lp;
        }
      }
      if (p.value)
        for (int s = tid; s < ts; s += blockDim.x) p.value[s0 + s] = v_of[(size_t)s * strideC];
      __syncthreads();
      continue;
    }

    // ---- per-sample clipped-surrogate gradient: one thread per sample
    for (int s = tid; s < ts; s += blockDim.x) {
      const size_t gs = (size_t)(s0 + s);
      gen_surrogate(mu_of + (size_t)s * strideA, p.actions + gs * act, p.old_logp + gs * act, p.advantages[gs], v_of[(size_t)s * strideC],
                    p.returns[gs], act, p.batch_size, c, g0 + s * kGenMaxWidth, g1 + s * kGenMaxWidth, gv + s);
    }
    __syncthreads();
    if (tid == 0) gen_add_loss_sums(gv, g1, ts, sums);  // (losses and the skipped count in sample order)
    __syncthreads();
    // actor: g0 holds dL/dmu
    gen_backward<true>(p.actor, paramsA, cacheA, strideA, ts, g0, g1, partial);
    // critic: dL/dV into column 0 of g0
    for (int s = tid; s < ts; s += blockDim.x) g0[s * kGenMaxWidth] = gv[s];
    __syncthreads();
    gen_backward<true>(p.critic, paramsC, cacheC, strideC, ts, g0, g1, partial + p.actor.n_params);
  }
  if (grad) {
    __syncthreads();
    const int total = p.actor.n_params + p.critic.n_params;
    if (tid < 3) partial[total + tid] = sums[tid];
  }
}

__global__ void reduce_partials_n_kernel(const float* __restrict__ partials, int nparts, float* __restrict__ grads, int n_floats) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_floats) return;
  float sum = 0.0f;
  for (int c = 0; c < nparts; c++) sum += partials[(size_t)c * n_floats + i];
  grads[i] = sum;
}

// DenseLayer.Adam for one parameter of any topology (DenseLayer.cs:125-159): same operation order as adam_update in mlp.cu
__global__ void adam_generic_kernel(const GenAdamParams a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n_params) return;
  int layer = 0;
  while (layer + 1 < a.n_dense && i >= a.layer_end[layer]) layer++;
  const float g = a.grads[i];
  const float m = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, a.beta1), g), __fmul_rn(a.beta1, a.m[i]));
  const float v = __fadd_rn(__fmul_rn(a.beta2, a.v[i]), __fmul_rn(__fsub_rn(1.0f, a.beta2), __fmul_rn(g, g)));
  a.m[i] = m;
  a.v[i] = v;
  const float mhat = __fdiv_rn(m, a.corr1[layer]);
  const float vhat = __fdiv_rn(v, a.corr2[layer]);
  const float denom = __fadd_rn(__fsqrt_rn(vhat), a.eps);
  a.params[i] = __fsub_rn(a.params[i], __fmul_rn(a.alpha, __fdiv_rn(mhat, denom)));
}

// ---- populations of any topology: agent a's parameters, Adam moments and gradient buffer at a * stride floats (actor | critic)

__device__ __forceinline__ void cp_async4(float* smem, const float* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_prev() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// Rows [row0, row0 + 32) of dense layer L into a warp's chunk buffer: row r at r * (L.in | 1) floats (an odd pitch: lane r reading
// column i of its row hits bank (r + i) mod 32, conflict-free), the 32 biases after the rows.  Coalesced 4-byte copies: the
// layer's rows are contiguous in global memory, but a layer's offset and width need not be multiples of four floats.
__device__ __forceinline__ void stage_chunk(const GenLayer& L, const float* params, int row0, float* buf, int lane) {
  const int rows = min(32, L.out - row0), in = L.in, pitch = in | 1, n = rows * in;
  const float* W = params + L.w_off + (size_t)row0 * in;
  int r = lane / in, c = lane - r * in;
  for (int j = lane; j < n; j += 32) {
    cp_async4(buf + r * pitch + c, W + j);
    c += 32;
    while (c >= in) {
      c -= in;
      r++;
    }
  }
  if (lane < rows) cp_async4(buf + 32 * pitch + lane, params + L.b_off + row0 + lane);
}
// the next chunk of a network's dense layers after (l, row0); l == n_layers: none
__device__ __forceinline__ void next_chunk(const GenNet& net, int& l, int& row0) {
  row0 += 32;
  if (row0 < net.L[l].out) return;
  row0 = 0;
  do l++;
  while (l < net.n_layers && net.L[l].kind != WB_DENSE);
}

// NeuralNetwork.FeedForward of one sample by one warp: x holds the input, y is scratch (kGenMaxWidth floats each); returns the
// buffer that holds the output.  The dense layers stream through two chunk buffers of chunk_floats with cp.async: chunk k + 2 is
// copied while chunk k + 1 is in flight and chunk k is computed, across layer ends.  Lane o of a chunk computes output row0 + o
// with gen_forward's chain (a left-to-right __fadd_rn(acc, __fmul_rn(x[i], w[i])) from 0, then + b); activation layers are
// applied in place.
__device__ float* warp_forward(const GenNet& net, const float* params, float* x, float* y, float* bufs, int chunk_floats, int lane) {
  int pl = 0, pr = 0;  // the next chunk to copy: the first dense layer's first rows
  while (pl < net.n_layers && net.L[pl].kind != WB_DENSE) pl++;
  for (int k = 0; k < 2; k++) {
    if (pl < net.n_layers) {
      stage_chunk(net.L[pl], params, pr, bufs + k * chunk_floats, lane);
      next_chunk(net, pl, pr);
    }
    cp_async_commit();
  }
  int bi = 0;
  for (int l = 0; l < net.n_layers; l++) {
    const GenLayer& L = net.L[l];
    if (L.kind != WB_DENSE) {
      for (int j = lane; j < L.in; j += 32) x[j] = gen_activate(L.kind, x[j]);
      __syncwarp();
      continue;
    }
    const int pitch = L.in | 1;
    for (int row0 = 0; row0 < L.out; row0 += 32) {
      cp_async_wait_prev();
      __syncwarp();
      float* B = bufs + bi * chunk_floats;
      const int o = row0 + lane;
      if (o < L.out) {
        const float* w = B + lane * pitch;
        float acc = 0.0f;
        for (int i = 0; i < L.in; i++) acc = __fadd_rn(acc, __fmul_rn(x[i], w[i]));
        y[o] = acc + B[32 * pitch + lane];
      }
      __syncwarp();
      if (pl < net.n_layers) {
        stage_chunk(net.L[pl], params, pr, B, lane);
        next_chunk(net, pl, pr);
      }
      cp_async_commit();
      bi ^= 1;
    }
    float* t = x;
    x = y;
    y = t;
  }
  return x;
}

// population_generic_act_kernel: PPOAgent.SampleActions for N walkers, walker w with agent w, for networks the default kernel does
// not cover.  One warp per walker (warp_forward); lanes k < act sample action k as ppo_generic_kernel does (gen_sample, sigma
// from the agent's log_std on the device).  The critic runs only when the value is asked for.
__global__ void __launch_bounds__(kGenActWarps * 32) population_generic_act_kernel(const PopGenActParams G) {
  extern __shared__ __align__(16) float gsm[];
  const PopActParams& P = G.a;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * kGenActWarps + warp;
  if (w >= P.n) return;  // (warp-uniform; the kernel has no CTA-wide barrier)
  float* bufs = gsm + (size_t)warp * (2 * G.chunk_floats + 2 * kGenMaxWidth);
  float* x = bufs + 2 * G.chunk_floats;
  float* y = x + kGenMaxWidth;
  const float* prm = P.params + (size_t)w * G.stride;
  const int sdim = G.actor.input, act = G.actor.output;
  for (int j = lane; j < sdim; j += 32) x[j] = P.states[(size_t)w * sdim + j];
  __syncwarp();
  const float* mu = warp_forward(G.actor, prm, x, y, bufs, G.chunk_floats, lane);
  const PopAgent& ag = P.agents[w];
  const GenConsts c = gen_consts(ag.log_std, ag.clip_eps);
  for (int k = lane; k < act; k += 32) {
    float a, lp;
    gen_sample(P.mode, P.uniforms, P.seed, P.step, (size_t)w, k, act, mu[k], c, a, lp);
    P.actions[(size_t)w * act + k] = a;
    P.logp[(size_t)w * act + k] = lp;
    if (P.mean) P.mean[(size_t)w * act + k] = mu[k];
  }
  if (P.value) {
    __syncwarp();
    for (int j = lane; j < sdim; j += 32) x[j] = P.states[(size_t)w * sdim + j];
    __syncwarp();
    const float* v = warp_forward(G.critic, prm + G.actor.n_params, x, y, bufs, G.chunk_floats, lane);
    if (lane == 0) P.value[w] = v[0];
  }
}

// population_generic_episodes_kernel: population_episodes_kernel for networks the default kernel does not cover.  One CTA per
// agent with work, its items in list order, the same tables, ring addressing and device draws.  Per item: the critic forward over
// the episode in tiles, trajectory_returns on shared-memory copies, then epochs x floor(L / B) mini-batches, each followed by
// DenseLayer.Adam (adam_generic_kernel's operations) before the next reads the weights.
// Summation order: a wb_policy on ppo_generic_kernel forms a mini-batch's gradient on one CTA per tile of ts samples (B <= 1 024,
// so at most 128 tiles, fewer than the grid cap), each tile's sums in sample order in a zeroed partial, then reduce_partials_n
// adds the partials in tile order from 0.  Here the tiles run in order on one CTA and gen_backward adds each tile's sums to the
// zeroed gradient buffer: the same additions (0 + p never differs from p in a sum that starts at +0).  ts must be the policy's.
__global__ void __launch_bounds__(kGenThreads, 1) population_generic_episodes_kernel(const PopGenTrainParams G) {
  extern __shared__ __align__(16) float gsm[];
  const PopTrainParams& P = G.t;
  const int ts_max = G.ts;
  const GenNet& actor = G.actor;
  const GenNet& critic = G.critic;
  const int strideA = actor.cache_floats + actor.output, strideC = critic.cache_floats + critic.output;
  float* cacheA = gsm;
  float* cacheC = cacheA + (size_t)ts_max * strideA;
  float* g0 = cacheC + (size_t)ts_max * strideC;
  float* g1 = g0 + (size_t)ts_max * kGenMaxWidth;
  float* gv = g1 + (size_t)ts_max * kGenMaxWidth;
  float* sums = gv + ts_max;
  float* rew = sums + 4;  // generic_smem_bytes ends here; the episode arrays follow
  float* val = rew + kPopMaxLen;
  float* ret = val + kPopMaxLen;
  float* adv = ret + kPopMaxLen;
  uint32_t* key = reinterpret_cast<uint32_t*>(adv + kPopMaxLen);
  int32_t* perm = reinterpret_cast<int32_t*>(key + kPopMaxLen);
  int32_t* loc = perm + kPopMaxLen;  // [ts] local row of every sample of the current tile
  const int tid = threadIdx.x;
  const PopCta cta = P.ctas[blockIdx.x];
  const PopAgent ag = P.agents[cta.agent];
  const size_t base = (size_t)cta.agent * G.stride;
  float* params = P.params + base;
  float* grads = P.grads + base;
  float* m = P.m + base;
  float* v = P.v + base;
  const float* paramsA = params;
  const float* paramsC = params + actor.n_params;
  const int n_total = actor.n_params + critic.n_params, sdim = actor.input, act = actor.output;
  const GenConsts c = gen_consts(ag.log_std, ag.clip_eps);
  const int B = ag.batch, R = P.ring_rows, C = P.columns;
  for (int it = 0; it < cta.count; it++) {
    const PopItem item = P.items[cta.first + it];
    const int L = item.length;
    auto row_of = [&](int i) {
      const int t = item.t0 + i;
      return (t >= R ? t - R : t) * C + item.column;
    };
    // ---- CalculateValues (PPOAgent.cs:175-189)
    for (int s0 = 0; s0 < L; s0 += ts_max) {
      const int ts = min(ts_max, L - s0);
      __syncthreads();
      for (int idx = tid; idx < ts * sdim; idx += kGenThreads) {
        const int s = idx / sdim, i = idx - s * sdim;
        cacheC[(size_t)s * strideC + critic.L[0].cache_off + i] = P.states[(size_t)row_of(s0 + s) * sdim + i];
      }
      __syncthreads();
      gen_forward<false>(critic, paramsC, cacheC, strideC, ts);
      for (int s = tid; s < ts; s += kGenThreads) val[s0 + s] = cacheC[(size_t)s * strideC + critic.cache_floats];
    }
    for (int i = tid; i < L; i += kGenThreads) rew[i] = P.rewards[row_of(i)];
    __syncthreads();
    if (tid == 0 && L > 0) trajectory_returns(rew, val, L, ag.gamma, ag.lambda, ag.use_gae, ag.normalize, ag.norm_eps, ret, adv);
    __syncthreads();
    for (int i = tid; i < L; i += kGenThreads) {
      const int r = row_of(i);
      P.values[r] = val[i];
      P.returns[r] = ret[i];
      P.advantages[r] = adv[i];
    }
    // ---- epochs x floor(L / B) mini-batches, each Train(Batch) + NeuralNetwork.Optimise
    const int per_epoch = L / B;
    int step = 0;
    float skipped_total = 0.0f;
    for (int epoch = 0; epoch < P.epochs && per_epoch > 0; epoch++) {
      const int32_t* index = perm;
      if (P.batch_index) index = P.batch_index + item.index_off + (size_t)epoch * per_epoch * B;
      else draw_permutation<kGenThreads>(key, perm, L, epoch, item.episode, cta.agent, P.seed, tid);
      for (int b = 0; b < per_epoch; b++, step++, index += B) {
        for (int i = tid; i < G.grad_floats; i += kGenThreads) grads[i] = 0.0f;
        for (int s0 = 0; s0 < B; s0 += ts_max) {
          const int ts = min(ts_max, B - s0);
          __syncthreads();
          if (tid < ts) loc[tid] = index[s0 + tid];
          if (tid < 4) sums[tid] = 0.0f;
          __syncthreads();
          for (int idx = tid; idx < ts * sdim; idx += kGenThreads) {
            const int s = idx / sdim, i = idx - s * sdim;
            const float x = P.states[(size_t)row_of(loc[s]) * sdim + i];
            cacheA[(size_t)s * strideA + actor.L[0].cache_off + i] = x;
            cacheC[(size_t)s * strideC + critic.L[0].cache_off + i] = x;
          }
          __syncthreads();
          gen_forward<false>(actor, paramsA, cacheA, strideA, ts);
          gen_forward<false>(critic, paramsC, cacheC, strideC, ts);
          for (int s = tid; s < ts; s += kGenThreads) {
            const int li = loc[s];
            const size_t r = (size_t)row_of(li);
            gen_surrogate(cacheA + (size_t)s * strideA + actor.cache_floats, P.actions + r * act, P.old_logp + r * act, adv[li],
                          cacheC[(size_t)s * strideC + critic.cache_floats], ret[li], act, ag.batch_size_f, c, g0 + s * kGenMaxWidth,
                          g1 + s * kGenMaxWidth, gv + s);
          }
          __syncthreads();
          if (tid == 0) {
            gen_add_loss_sums(gv, g1, ts, sums);
            for (int k = 0; k < 3; k++) grads[n_total + k] += sums[k];
          }
          __syncthreads();
          gen_backward<false>(actor, paramsA, cacheA, strideA, ts, g0, g1, grads);
          for (int s = tid; s < ts; s += kGenThreads) g0[s * kGenMaxWidth] = gv[s];
          __syncthreads();
          gen_backward<false>(critic, paramsC, cacheC, strideC, ts, g0, g1, grads + actor.n_params);
        }
        __syncthreads();
        // (read before the barrier that ends this step: the next mini-batch zeroes the buffer from other warps)
        if (tid == 0) skipped_total += grads[n_total + 2];
        // DenseLayer.Adam with this step's bias corrections [2 * n_dense] from the host table (adam_generic_kernel, op for op)
        const float* corr = P.corr + (size_t)(item.corr_off + step) * 2 * G.n_dense;
        for (int i = tid; i < n_total; i += kGenThreads) {
          int layer = 0;
          while (layer + 1 < G.n_dense && i >= G.layer_end[layer]) layer++;
          const float g = grads[i];
          const float mi = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, ag.beta1), g), __fmul_rn(ag.beta1, m[i]));
          const float vi = __fadd_rn(__fmul_rn(ag.beta2, v[i]), __fmul_rn(__fsub_rn(1.0f, ag.beta2), __fmul_rn(g, g)));
          m[i] = mi;
          v[i] = vi;
          const float mhat = __fdiv_rn(mi, corr[layer]);
          const float vhat = __fdiv_rn(vi, corr[G.n_dense + layer]);
          const float denom = __fadd_rn(__fsqrt_rn(vhat), ag.adam_eps);
          params[i] = __fsub_rn(params[i], __fmul_rn(ag.alpha, __fdiv_rn(mhat, denom)));
        }
        __syncthreads();
      }
    }
    if (tid == 0) {
      const bool trained = P.epochs > 0 && per_epoch > 0;
      if (P.losses) {
        P.losses[2 * item.out] = trained ? grads[n_total] : 0.0f;
        P.losses[2 * item.out + 1] = trained ? grads[n_total + 1] : 0.0f;
      }
      if (P.skipped) P.skipped[item.out] = (int32_t)skipped_total;
    }
    __syncthreads();
  }
}

}  // namespace

size_t generic_smem_bytes(const GenNet& actor, const GenNet& critic, int ts) {
  const size_t strideA = (size_t)actor.cache_floats + actor.output, strideC = (size_t)critic.cache_floats + critic.output;
  return sizeof(float) * ((size_t)ts * (strideA + strideC + 2 * kGenMaxWidth + 1) + 4);
}

int generic_tile_samples(const GenNet& actor, const GenNet& critic) {
  for (int ts = 32; ts >= 1; ts >>= 1)
    if (generic_smem_bytes(actor, critic, ts) <= 200 * 1024) return ts;
  return 0;
}

int generic_grid_for(int n, int ts, int sm_count) {
  const int ntiles = (n + ts - 1) / ts;
  const int cap = sm_count * 2;
  return ntiles < cap ? (ntiles > 0 ? ntiles : 1) : cap;
}

cudaError_t launch_mlp_generic(const GenParams& p, int grid, cudaStream_t stream) {
  const size_t smem = generic_smem_bytes(p.actor, p.critic, p.ts);
  static size_t configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || configured[dev] < smem) {
    cudaError_t e = cudaFuncSetAttribute(ppo_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024));
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = 200 * 1024;
  }
  ppo_generic_kernel<<<grid, kGenThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_reduce_partials_n(const float* partials, int nparts, float* grads, int n_floats, cudaStream_t stream) {
  reduce_partials_n_kernel<<<(n_floats + 127) / 128, 128, 0, stream>>>(partials, nparts, grads, n_floats);
  return cudaGetLastError();
}

// PPOAgent.ParseLayers output (kinds / sizes) -> layer table; false when the DSL instance is outside what the kernels cover
static bool build_net(int32_t input, const int32_t* kinds, const int32_t* sizes, int32_t n_layers, GenNet* net, const char** why) {
  *net = GenNet{};
  if (n_layers < 1 || n_layers > kGenMaxLayers) { *why = "a network holds 1..16 layers"; return false; }
  if (input < 1 || input > kGenMaxWidth) { *why = "the state size must be 1..128"; return false; }
  net->n_layers = n_layers;
  net->input = input;
  int width = input, cache = 0, off = 0;
  for (int l = 0; l < n_layers; l++) {
    GenLayer& L = net->L[l];
    L.kind = kinds[l];
    L.in = width;
    L.cache_off = cache;
    cache += width;
    if (kinds[l] == WB_DENSE) {
      if (sizes[l] < 1 || sizes[l] > kGenMaxWidth) { *why = "dense layer widths must be 1..128"; return false; }
      L.out = sizes[l];
      L.w_off = off;
      off += L.out * L.in;
      L.b_off = off;
      off += L.out;
      width = L.out;
      net->n_dense++;
    } else if (kinds[l] == WB_RELU || kinds[l] == WB_LEAKYRELU || kinds[l] == WB_TANH) {
      L.out = width;
    } else {
      *why = "unknown layer kind";
      return false;
    }
  }
  if (net->n_dense < 1) { *why = "a network needs at least one dense layer"; return false; }
  net->output = width;
  net->n_params = off;
  net->cache_floats = cache;
  return true;
}

static bool is_default_topology(int32_t state_size, int32_t action_size, const int32_t* ak, const int32_t* as, int32_t al,
                                const int32_t* ck, const int32_t* cs, int32_t cl) {
  if (state_size != kIn || action_size != kAct || al != 6 || cl != 3) return false;
  const int32_t want_ak[6] = {WB_DENSE, WB_LEAKYRELU, WB_DENSE, WB_LEAKYRELU, WB_DENSE, WB_TANH};
  const int32_t want_as[6] = {kHid, 0, kHid, 0, kAct, 0};
  for (int i = 0; i < 6; i++) {
    if (ak[i] != want_ak[i]) return false;
    if (ak[i] == WB_DENSE && as[i] != want_as[i]) return false;
  }
  const int32_t want_ck[3] = {WB_DENSE, WB_LEAKYRELU, WB_DENSE};
  const int32_t want_cs[3] = {kHid, 0, 1};
  for (int i = 0; i < 3; i++) {
    if (ck[i] != want_ck[i]) return false;
    if (ck[i] == WB_DENSE && cs[i] != want_cs[i]) return false;
  }
  return true;
}

int32_t build_networks(int32_t state_size, int32_t action_size, const int32_t* actor_kinds, const int32_t* actor_sizes, int32_t actor_layers,
                       const int32_t* critic_kinds, const int32_t* critic_sizes, int32_t critic_layers, Networks* out) {
  if (!(actor_kinds && actor_sizes && critic_kinds && critic_sizes)) return fail(WB_ERR_INVALID, "%s", "null layer list");
  Networks& n = *out;
  const char* why = "";
  if (!build_net(state_size, actor_kinds, actor_sizes, actor_layers, &n.actor, &why)) return fail(WB_ERR_UNSUPPORTED, "actor network: %s", why);
  if (!build_net(state_size, critic_kinds, critic_sizes, critic_layers, &n.critic, &why)) return fail(WB_ERR_UNSUPPORTED, "critic network: %s", why);
  // PPOAgent.CreateNetworks checks the two output sizes (PPOAgent.cs:78-92); the host shim falls back to the defaults like the reference
  if (n.actor.output != action_size) return fail(WB_ERR_INVALID, "the actor's last dense layer must have action_size outputs (PPOAgent.cs:86)");
  if (n.critic.output != 1) return fail(WB_ERR_INVALID, "the critic's last dense layer must have one output (PPOAgent.cs:78)");
  if (action_size > 64) return fail(WB_ERR_UNSUPPORTED, "action_size must be 1..64");
  if (n.actor.n_dense + n.critic.n_dense > kGenMaxDense) return fail(WB_ERR_UNSUPPORTED, "at most 32 dense layers in both networks together");
  n.gen_ts = generic_tile_samples(n.actor, n.critic);
  if (n.gen_ts == 0) return fail(WB_ERR_UNSUPPORTED, "the layer caches of one sample exceed shared memory (sum of layer widths too large)");
  n.default_topology = is_default_topology(state_size, action_size, actor_kinds, actor_sizes, actor_layers, critic_kinds, critic_sizes, critic_layers);
  return WB_OK;
}

int generic_layer_ends(const GenNet& actor, const GenNet& critic, int32_t* layer_end) {
  int k = 0;
  for (int l = 0; l < actor.n_layers; l++)
    if (actor.L[l].kind == WB_DENSE) layer_end[k++] = actor.L[l].b_off + actor.L[l].out;
  for (int l = 0; l < critic.n_layers; l++)
    if (critic.L[l].kind == WB_DENSE) layer_end[k++] = actor.n_params + critic.L[l].b_off + critic.L[l].out;
  return k;
}

int generic_act_chunk_floats(const GenNet& actor, const GenNet& critic) {
  int most = 0;
  for (const GenNet* net : {&actor, &critic})
    for (int l = 0; l < net->n_layers; l++)
      if (net->L[l].kind == WB_DENSE) most = max(most, 32 * (net->L[l].in | 1) + 32);
  return (most + 3) / 4 * 4;
}

size_t generic_episodes_smem_bytes(const GenNet& actor, const GenNet& critic, int ts) {
  return generic_smem_bytes(actor, critic, ts) + sizeof(float) * 6 * (size_t)kPopMaxLen + sizeof(int32_t) * 32;
}

cudaError_t launch_population_generic_act(const PopGenActParams& g, cudaStream_t stream) {
  static bool configured[64] = {};
  const int smem_max = (int)(sizeof(float) * kGenActWarps * (2 * (32 * (kGenMaxWidth + 1) + 32) + 2 * kGenMaxWidth));
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(population_generic_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  const size_t smem = sizeof(float) * kGenActWarps * (2 * (size_t)g.chunk_floats + 2 * kGenMaxWidth);
  population_generic_act_kernel<<<(g.a.n + kGenActWarps - 1) / kGenActWarps, kGenActWarps * 32, smem, stream>>>(g);
  return cudaGetLastError();
}

cudaError_t launch_population_generic_episodes(const PopGenTrainParams& g, int n_ctas, cudaStream_t stream) {
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(population_generic_episodes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPopGenMaxSmem);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  population_generic_episodes_kernel<<<n_ctas, kGenThreads, generic_episodes_smem_bytes(g.actor, g.critic, g.ts), stream>>>(g);
  return cudaGetLastError();
}

cudaError_t launch_adam_generic(const GenAdamParams& a, cudaStream_t stream) {
  adam_generic_kernel<<<(a.n_params + 127) / 128, 128, 0, stream>>>(a);
  return cudaGetLastError();
}

}  // namespace wb

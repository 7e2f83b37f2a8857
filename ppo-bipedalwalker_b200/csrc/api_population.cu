// api_population.cu -- C ABI of a population of independent PPO agents (include/walker_b200.h, wb_population_*).  Compute is in
// mlp.cu (population_act_kernel, population_episodes_kernel: the reference's default networks) and mlp_generic.cu
// (population_generic_act_kernel, population_generic_episodes_kernel: any other network the DSL describes).
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "common.h"
#include "mlp.cuh"

using namespace wb;

struct wb_population {
  int device = 0;
  cudaStream_t stream = nullptr;
  int n = 0;
  int64_t launches = 0;
  Networks nets{};                  // default_topology: the default kernels; otherwise the any-topology ones
  int state = kIn, action = kAct;
  int n_total = kTotalParams;       // actor | critic parameters of one agent
  int stride = kAgentStride;        // floats per agent row: n_total + 3 (loss sums, skipped) rounded up to a float4 multiple
  int n_dense = 5;                  // dense layers of both networks (actor first)
  int32_t layer_end[kGenMaxDense] = {};
  std::vector<wb_hyperparams> hp;
  std::vector<int32_t> iterations;  // [n][n_dense] DenseLayer._iteration per dense layer
  std::vector<int32_t> episodes;    // [n] episodes trained so far (counter of the device-drawn mini-batches)
  float* d_params = nullptr;        // [n][stride] actor | critic
  float* d_m = nullptr;
  float* d_v = nullptr;
  float* d_grads = nullptr;
  PopAgent* d_agents = nullptr;     // [n]
  // staging of the host entries (grown on demand)
  float* d_stage = nullptr;
  size_t stage_bytes = 0;
  PinnedTable tab;                  // the table of a train call (items + Adam corrections) or a copy call (pairs + constants)
};

static int32_t grow_stage(wb_population* p, size_t bytes) {
  if (bytes <= p->stage_bytes) return WB_OK;
  cudaFree(p->d_stage);
  p->d_stage = nullptr;
  p->stage_bytes = 0;
  WB_CUDA(cudaMalloc(&p->d_stage, bytes));
  p->stage_bytes = bytes;
  return WB_OK;
}

// one train call, validated and enqueued: items [n_items][4] = (agent, column, t0, length) in list order
static int32_t enqueue_train(wb_population* p, int32_t n_items, const int32_t* items, int32_t ring_rows, int32_t columns, int32_t epochs,
                             uint64_t seed, const float* states, const float* actions, const float* logp, const float* rewards,
                             const int32_t* batch_index, float* values, float* returns, float* advantages, float* losses,
                             int32_t* skipped) {
  WB_REQUIRE(items, "items is null");
  WB_REQUIRE(states && actions && logp && rewards && values && returns && advantages, "null argument");
  WB_REQUIRE(n_items >= 1, "n_items must be at least 1");
  WB_REQUIRE(ring_rows >= 1 && columns >= 1, "ring_rows and columns must be positive");
  WB_REQUIRE((int64_t)ring_rows * columns <= INT32_MAX, "the ring holds more than 2^31 rows");
  WB_REQUIRE(epochs >= 0, "epochs must be >= 0");
  int64_t steps = 0;
  for (int32_t i = 0; i < n_items; i++) {
    const int32_t a = items[4 * i], c = items[4 * i + 1], t0 = items[4 * i + 2], L = items[4 * i + 3];
    if (a < 0 || a >= p->n) return fail(WB_ERR_INVALID, "item %d: agent %d outside 0..%d", i, a, p->n - 1);
    if (c < 0 || c >= columns) return fail(WB_ERR_INVALID, "item %d: column %d outside 0..%d", i, c, columns - 1);
    if (t0 < 0 || t0 >= ring_rows) return fail(WB_ERR_INVALID, "item %d: first step %d outside the ring's %d rows", i, t0, ring_rows);
    if (L < 0 || L > ring_rows) return fail(WB_ERR_INVALID, "item %d: length %d outside 0..%d (the ring's rows)", i, L, ring_rows);
    if (L > kPopMaxLen) return fail(WB_ERR_UNSUPPORTED, "item %d: an episode of %d steps (at most %d)", i, L, kPopMaxLen);
    steps += (int64_t)epochs * (L / p->hp[a].batch_size);
  }
  // (the correction table holds 2 * n_dense floats per Adam step)
  WB_REQUIRE(steps <= INT32_MAX / (2 * p->n_dense), "too many Adam steps for one call");
  // CTAs: the agents with work, in order of first appearance; each trains its items in list order
  std::vector<int32_t> first_cta(p->n, -1);
  std::vector<PopCta> ctas;
  for (int32_t i = 0; i < n_items; i++) {
    const int32_t a = items[4 * i];
    if (first_cta[a] < 0) {
      first_cta[a] = (int32_t)ctas.size();
      ctas.push_back(PopCta{a, 0, 0, 0});
    }
    ctas[first_cta[a]].count++;
  }
  for (size_t k = 1; k < ctas.size(); k++) ctas[k].first = ctas[k - 1].first + ctas[k - 1].count;
  const size_t cta_bytes = align16(sizeof(PopCta) * ctas.size());
  const size_t item_bytes = align16(sizeof(PopItem) * n_items);
  const int nd = p->n_dense;
  const size_t tab_bytes = cta_bytes + item_bytes + sizeof(float) * 2 * nd * (size_t)steps;
  if (int32_t rc = p->tab.reserve(tab_bytes)) return rc;
  // nothing fails below this line: the step counters and episode counters advance only for a call that is enqueued
  memcpy(p->tab.host, ctas.data(), sizeof(PopCta) * ctas.size());
  PopItem* tab_items = reinterpret_cast<PopItem*>(p->tab.host + cta_bytes);
  float* corr = reinterpret_cast<float*>(p->tab.host + cta_bytes + item_bytes);
  std::vector<int32_t> fill(ctas.size(), 0);
  int64_t index_off = 0, corr_off = 0;
  for (int32_t i = 0; i < n_items; i++) {
    const int32_t a = items[4 * i], L = items[4 * i + 3], B = p->hp[a].batch_size;
    const int32_t k = first_cta[a];
    const int64_t nb = (int64_t)epochs * (L / B);
    PopItem& it = tab_items[ctas[k].first + fill[k]++];
    it = PopItem{i, items[4 * i + 1], items[4 * i + 2], L, (int32_t)index_off, (int32_t)corr_off, p->episodes[a]++, 0};
    // DenseLayer.Adam bias corrections (float)(1 - Math.Pow(beta, t)) (DenseLayer.cs:127,142-145), as next_corrections computes them
    int32_t* iter = &p->iterations[(size_t)a * nd];
    for (int64_t s = 0; s < nb; s++) {
      float* c = corr + 2 * nd * (corr_off + s);
      for (int l = 0; l < nd; l++) {
        iter[l] += 1;
        c[l] = (float)(1.0 - pow((double)p->hp[a].beta1, (double)iter[l]));
        c[nd + l] = (float)(1.0 - pow((double)p->hp[a].beta2, (double)iter[l]));
      }
    }
    index_off += nb * B;
    corr_off += nb;
  }
  if (int32_t rc = p->tab.upload(tab_bytes, p->stream)) return rc;
  PopTrainParams t{};
  t.states = states;
  t.actions = actions;
  t.old_logp = logp;
  t.rewards = rewards;
  t.values = values;
  t.returns = returns;
  t.advantages = advantages;
  t.batch_index = batch_index;
  t.ctas = reinterpret_cast<const PopCta*>(p->tab.dev);
  t.items = reinterpret_cast<const PopItem*>(p->tab.dev + cta_bytes);
  t.corr = reinterpret_cast<const float*>(p->tab.dev + cta_bytes + item_bytes);
  t.agents = p->d_agents;
  t.params = p->d_params;
  t.m = p->d_m;
  t.v = p->d_v;
  t.grads = p->d_grads;
  t.losses = losses;
  t.skipped = skipped;
  t.ring_rows = ring_rows;
  t.columns = columns;
  t.epochs = epochs;
  t.seed = seed;
  if (p->nets.default_topology) {
    WB_CUDA(launch_population_episodes(t, (int)ctas.size(), p->stream));
  } else {
    PopGenTrainParams g{};
    g.actor = p->nets.actor;
    g.critic = p->nets.critic;
    g.stride = p->stride;
    g.ts = p->nets.gen_ts;
    g.grad_floats = p->stride;
    g.n_dense = nd;
    memcpy(g.layer_end, p->layer_end, sizeof(g.layer_end));
    g.t = t;
    WB_CUDA(launch_population_generic_episodes(g, (int)ctas.size(), p->stream));
  }
  p->launches++;
  return WB_OK;
}

static int32_t copy_agent(wb_population* p, int32_t agent, float* dev_base, const float* src_host, float* dst_host) {
  WB_REQUIRE(agent >= 0 && agent < p->n, "agent outside the population");
  float* d = dev_base + (size_t)agent * p->stride;
  if (src_host) WB_CUDA(cudaMemcpyAsync(d, src_host, sizeof(float) * p->n_total, cudaMemcpyHostToDevice, p->stream));
  if (dst_host) WB_CUDA(cudaMemcpyAsync(dst_host, d, sizeof(float) * p->n_total, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

static int32_t act(wb_population* p, int32_t n, int32_t mode, const float* states, const float* uniforms, uint64_t seed, uint64_t step,
                   float* actions, float* logp, float* mean, float* value) {
  WB_REQUIRE(n == p->n, "n must equal the population size (walker w acts with agent w)");
  PopActParams a{};
  a.params = p->d_params;
  a.agents = p->d_agents;
  a.n = n;
  a.mode = mode;
  a.states = states;
  a.uniforms = uniforms;
  a.seed = seed;
  a.step = step;
  a.actions = actions;
  a.logp = logp;
  a.mean = mean;
  a.value = value;
  if (p->nets.default_topology) {
    WB_CUDA(launch_population_act(a, p->stream));
  } else {
    PopGenActParams g{};
    g.actor = p->nets.actor;
    g.critic = p->nets.critic;
    g.stride = p->stride;
    g.chunk_floats = generic_act_chunk_floats(p->nets.actor, p->nets.critic);
    g.a = a;
    WB_CUDA(launch_population_generic_act(g, p->stream));
  }
  p->launches++;
  return WB_OK;
}

extern "C" {

int32_t wb_population_create_net(int32_t n_agents, int32_t state_size, int32_t action_size, const int32_t* actor_kinds,
                                 const int32_t* actor_sizes, int32_t actor_layers, const int32_t* critic_kinds, const int32_t* critic_sizes,
                                 int32_t critic_layers, const wb_hyperparams* hp, wb_population** out) {
  WB_REQUIRE(out, "out is null");
  *out = nullptr;
  Networks nets;
  if (int32_t rc = build_networks(state_size, action_size, actor_kinds, actor_sizes, actor_layers, critic_kinds, critic_sizes, critic_layers, &nets))
    return rc;
  if (!nets.default_topology && generic_episodes_smem_bytes(nets.actor, nets.critic, nets.gen_ts) > kPopGenMaxSmem)
    return fail(WB_ERR_UNSUPPORTED, "the layer caches and one episode's arrays exceed shared memory");
  WB_REQUIRE(n_agents >= 1, "n_agents must be at least 1");
  if (hp)
    for (int32_t a = 0; a < n_agents; a++)
      if (hp[a].batch_size < 1) return fail(WB_ERR_INVALID, "agent %d: batch_size must be positive", a);
  if (int32_t rc = require_device()) return rc;
  wb_population* p = new (std::nothrow) wb_population();
  WB_REQUIRE(p, "out of host memory");
  p->n = n_agents;
  p->nets = nets;
  p->state = state_size;
  p->action = action_size;
  p->n_total = nets.actor.n_params + nets.critic.n_params;
  p->stride = (p->n_total + 3 + 3) / 4 * 4;
  p->n_dense = generic_layer_ends(nets.actor, nets.critic, p->layer_end);
  cudaGetDevice(&p->device);
  try {
    p->hp.resize(n_agents);
    p->iterations.assign((size_t)n_agents * p->n_dense, 0);
    p->episodes.assign(n_agents, 0);
  } catch (const std::bad_alloc&) {
    delete p;
    return fail(WB_ERR_INVALID, "out of host memory");
  }
  std::vector<PopAgent> consts(n_agents);
  for (int32_t a = 0; a < n_agents; a++) {
    if (hp) p->hp[a] = hp[a]; else wb_hyperparams_default(&p->hp[a]);
    population_agent_consts(p->hp[a], &consts[a]);
  }
  const size_t bytes = sizeof(float) * p->stride * (size_t)n_agents;
  cudaError_t e = cudaMalloc(&p->d_params, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_m, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_v, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_grads, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&p->d_agents, sizeof(PopAgent) * n_agents);
  if (e == cudaSuccess) e = cudaMemset(p->d_params, 0, bytes);
  if (e == cudaSuccess) e = cudaMemset(p->d_m, 0, bytes);
  if (e == cudaSuccess) e = cudaMemset(p->d_v, 0, bytes);
  if (e == cudaSuccess) e = cudaMemset(p->d_grads, 0, bytes);
  if (e == cudaSuccess) e = cudaMemcpy(p->d_agents, consts.data(), sizeof(PopAgent) * n_agents, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    wb_population_destroy(p);
    return fail(WB_ERR_CUDA, "wb_population_create: %s", cudaGetErrorString(e));
  }
  *out = p;
  return WB_OK;
}

int32_t wb_population_create(int32_t n_agents, const wb_hyperparams* hp, wb_population** out) {
  const int32_t ak[6] = {WB_DENSE, WB_LEAKYRELU, WB_DENSE, WB_LEAKYRELU, WB_DENSE, WB_TANH}, as[6] = {kHid, 0, kHid, 0, kAct, 0};
  const int32_t ck[3] = {WB_DENSE, WB_LEAKYRELU, WB_DENSE}, cs[3] = {kHid, 0, 1};
  return wb_population_create_net(n_agents, kIn, kAct, ak, as, 6, ck, cs, 3, hp, out);
}

int32_t wb_population_destroy(wb_population* p) {
  if (!p) return WB_OK;
  cudaFree(p->d_params);
  cudaFree(p->d_m);
  cudaFree(p->d_v);
  cudaFree(p->d_grads);
  cudaFree(p->d_agents);
  cudaFree(p->d_stage);
  delete p;
  return WB_OK;
}

int32_t wb_population_set_stream(wb_population* p, void* cuda_stream) {
  WB_REQUIRE(p, "population is null");
  p->stream = (cudaStream_t)cuda_stream;
  return WB_OK;
}

int32_t wb_population_sync(wb_population* p) {
  WB_REQUIRE(p, "population is null");
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

int32_t wb_population_launch_count(const wb_population* p, int64_t* count_out) {
  WB_REQUIRE(p && count_out, "null argument");
  *count_out = p->launches;
  return WB_OK;
}

int32_t wb_population_set_weights(wb_population* p, int32_t agent, const float* flat_host) {
  WB_REQUIRE(p && flat_host, "null argument");
  return copy_agent(p, agent, p->d_params, flat_host, nullptr);
}

int32_t wb_population_get_weights(wb_population* p, int32_t agent, float* flat_host) {
  WB_REQUIRE(p && flat_host, "null argument");
  return copy_agent(p, agent, p->d_params, nullptr, flat_host);
}

int32_t wb_population_get_grads(wb_population* p, int32_t agent, float* flat_host) {
  WB_REQUIRE(p && flat_host, "null argument");
  return copy_agent(p, agent, p->d_grads, nullptr, flat_host);
}

int32_t wb_population_get_adam(wb_population* p, int32_t agent, float* m_host, float* v_host, int32_t* steps_host) {
  WB_REQUIRE(p && m_host && v_host && steps_host, "null argument");
  if (int32_t rc = copy_agent(p, agent, p->d_m, nullptr, m_host)) return rc;
  if (int32_t rc = copy_agent(p, agent, p->d_v, nullptr, v_host)) return rc;
  memcpy(steps_host, &p->iterations[(size_t)agent * p->n_dense], sizeof(int32_t) * p->n_dense);
  return WB_OK;
}

int32_t wb_population_set_adam(wb_population* p, int32_t agent, const float* m_host, const float* v_host, const int32_t* steps_host) {
  WB_REQUIRE(p && m_host && v_host && steps_host, "null argument");
  if (int32_t rc = copy_agent(p, agent, p->d_m, m_host, nullptr)) return rc;
  if (int32_t rc = copy_agent(p, agent, p->d_v, v_host, nullptr)) return rc;
  memcpy(&p->iterations[(size_t)agent * p->n_dense], steps_host, sizeof(int32_t) * p->n_dense);
  return WB_OK;
}

int32_t wb_population_set_hyperparams(wb_population* p, int32_t agent, const wb_hyperparams* hp) {
  WB_REQUIRE(p && hp, "null argument");
  WB_REQUIRE(agent >= 0 && agent < p->n, "agent outside the population");
  WB_REQUIRE(hp->batch_size >= 1, "batch_size must be positive");
  PopAgent c;
  population_agent_consts(*hp, &c);
  WB_CUDA(cudaMemcpyAsync(p->d_agents + agent, &c, sizeof(PopAgent), cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  p->hp[agent] = *hp;
  return WB_OK;
}

int32_t wb_population_get_hyperparams(const wb_population* p, int32_t agent, wb_hyperparams* hp_out) {
  WB_REQUIRE(p && hp_out, "null argument");
  WB_REQUIRE(agent >= 0 && agent < p->n, "agent outside the population");
  *hp_out = p->hp[agent];
  return WB_OK;
}

int32_t wb_population_copy_agents(wb_population* p, int32_t n_pairs, const int32_t* dst_host, const int32_t* src_host,
                                  const wb_hyperparams* hp_host) {
  WB_REQUIRE(p && dst_host && src_host, "null argument");
  WB_REQUIRE(n_pairs >= 1, "n_pairs must be at least 1");
  // every dst distinct and never a src: the pairs are independent copies, in any order
  enum : uint8_t { kNone, kDst, kSrc };
  std::vector<uint8_t> role(p->n, kNone);
  for (int32_t i = 0; i < n_pairs; i++) {
    const int32_t d = dst_host[i], s = src_host[i];
    if (d < 0 || d >= p->n) return fail(WB_ERR_INVALID, "pair %d: dst %d outside 0..%d", i, d, p->n - 1);
    if (s < 0 || s >= p->n) return fail(WB_ERR_INVALID, "pair %d: src %d outside 0..%d", i, s, p->n - 1);
    if (d == s) return fail(WB_ERR_INVALID, "pair %d: agent %d copies itself", i, d);
    if (role[d] == kDst) return fail(WB_ERR_INVALID, "pair %d: dst %d is listed twice", i, d);
    role[d] = kDst;
    if (hp_host && hp_host[i].batch_size < 1) return fail(WB_ERR_INVALID, "pair %d: batch_size must be positive", i);
  }
  for (int32_t i = 0; i < n_pairs; i++)
    if (role[src_host[i]] == kDst) return fail(WB_ERR_INVALID, "pair %d: agent %d is both a src and a dst", i, src_host[i]);
  const size_t pair_bytes = align16(sizeof(int32_t) * 2 * n_pairs);
  const size_t tab_bytes = pair_bytes + sizeof(PopAgent) * n_pairs;
  if (int32_t rc = p->tab.reserve(tab_bytes)) return rc;
  int32_t* tab_pairs = reinterpret_cast<int32_t*>(p->tab.host);
  PopAgent* tab_consts = reinterpret_cast<PopAgent*>(p->tab.host + pair_bytes);
  std::vector<wb_hyperparams> hp(n_pairs);
  for (int32_t i = 0; i < n_pairs; i++) {
    tab_pairs[2 * i] = dst_host[i];
    tab_pairs[2 * i + 1] = src_host[i];
    hp[i] = hp_host ? hp_host[i] : p->hp[src_host[i]];
    population_agent_consts(hp[i], &tab_consts[i]);
  }
  if (int32_t rc = p->tab.upload(tab_bytes, p->stream)) return rc;
  PopCopyParams c{};
  c.params = p->d_params;
  c.m = p->d_m;
  c.v = p->d_v;
  c.agents = p->d_agents;
  c.pairs = reinterpret_cast<const int32_t*>(p->tab.dev);
  c.consts = reinterpret_cast<const PopAgent*>(p->tab.dev + pair_bytes);
  c.n_pairs = n_pairs;
  c.stride = p->stride;
  WB_CUDA(launch_population_copy(c, p->stream));
  p->launches++;
  // the host half: dst's hyper-parameters and Adam step counters (the bias corrections); its episode counter stays its own
  const int nd = p->n_dense;
  for (int32_t i = 0; i < n_pairs; i++) {
    p->hp[dst_host[i]] = hp[i];
    memcpy(&p->iterations[(size_t)dst_host[i] * nd], &p->iterations[(size_t)src_host[i] * nd], sizeof(int32_t) * nd);
  }
  return WB_OK;
}

int32_t wb_population_num_params(const wb_population* p, int32_t which, int32_t* n_out) {
  WB_REQUIRE(p && n_out, "null argument");
  if (which == 0) *n_out = p->nets.actor.n_params;
  else if (which == 1) *n_out = p->nets.critic.n_params;
  else return fail(WB_ERR_INVALID, "which must be 0 (actor) or 1 (critic)");
  return WB_OK;
}

int32_t wb_population_act_dev(wb_population* p, int32_t n, const float* states_dev, uint64_t seed, uint64_t step, float* actions_dev,
                              float* logp_dev, float* mean_dev, float* value_dev) {
  WB_REQUIRE(p && states_dev && actions_dev && logp_dev, "null argument");
  return act(p, n, kModeSamplePhilox, states_dev, nullptr, seed, step, actions_dev, logp_dev, mean_dev, value_dev);
}

int32_t wb_population_sample(wb_population* p, int32_t n, const float* states_host, const float* uniforms_host, float* actions_host,
                             float* logp_host, float* mean_host) {
  WB_REQUIRE(p && states_host && uniforms_host && actions_host && logp_host, "null argument");
  WB_REQUIRE(n == p->n, "n must equal the population size (walker w acts with agent w)");
  const size_t N = (size_t)n, IN = (size_t)p->state, ACT = (size_t)p->action;
  if (int32_t rc = grow_stage(p, sizeof(float) * N * (IN + 2 * ACT + 3 * ACT))) return rc;
  float* d_states = p->d_stage;
  float* d_uni = d_states + N * IN;
  float* d_act = d_uni + N * ACT * 2;
  float* d_logp = d_act + N * ACT;
  float* d_mean = d_logp + N * ACT;
  WB_CUDA(cudaMemcpyAsync(d_states, states_host, sizeof(float) * N * IN, cudaMemcpyHostToDevice, p->stream));
  WB_CUDA(cudaMemcpyAsync(d_uni, uniforms_host, sizeof(float) * N * ACT * 2, cudaMemcpyHostToDevice, p->stream));
  if (int32_t rc = act(p, n, kModeSample, d_states, d_uni, 0, 0, d_act, d_logp, d_mean, nullptr)) return rc;
  WB_CUDA(cudaMemcpyAsync(actions_host, d_act, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaMemcpyAsync(logp_host, d_logp, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  if (mean_host) WB_CUDA(cudaMemcpyAsync(mean_host, d_mean, sizeof(float) * N * ACT, cudaMemcpyDeviceToHost, p->stream));
  WB_CUDA(cudaStreamSynchronize(p->stream));
  return WB_OK;
}

int32_t wb_population_train_dev(wb_population* p, int32_t n_items, const int32_t* items_host, int32_t ring_rows, int32_t columns,
                                int32_t epochs, uint64_t seed, const float* states_dev, const float* actions_dev, const float* logp_dev,
                                const float* rewards_dev, const int32_t* batch_index_dev, float* values_dev, float* returns_dev,
                                float* advantages_dev, float* losses_dev, int32_t* skipped_dev) {
  WB_REQUIRE(p, "population is null");
  return enqueue_train(p, n_items, items_host, ring_rows, columns, epochs, seed, states_dev, actions_dev, logp_dev, rewards_dev,
                       batch_index_dev, values_dev, returns_dev, advantages_dev, losses_dev, skipped_dev);
}

int32_t wb_population_train_trajectories(wb_population* p, int32_t n_traj, const int32_t* agent_host, const int32_t* offsets_host,
                                         int32_t epochs, const float* states_host, const float* actions_host, const float* logp_host,
                                         const float* rewards_host, const int32_t* batch_index_host, float* values_host,
                                         float* returns_host, float* advantages_host, float* losses_host, int32_t* skipped_host) {
  WB_REQUIRE(p && agent_host && offsets_host && states_host && actions_host && logp_host && rewards_host, "null argument");
  WB_REQUIRE(n_traj >= 1, "n_traj must be at least 1");
  WB_REQUIRE(epochs >= 0, "epochs must be >= 0");
  WB_REQUIRE(offsets_host[0] >= 0, "offsets[0] must be >= 0");
  // a packed list is a ring of one column whose rows are the trajectories back to back: item e = (agent, 0, offsets[e], T_e)
  std::vector<int32_t> items((size_t)4 * n_traj);
  int64_t n_index = 0;
  for (int32_t e = 0; e < n_traj; e++) {
    const int32_t a = agent_host[e], T = offsets_host[e + 1] - offsets_host[e];
    if (T < 0) return fail(WB_ERR_INVALID, "offsets must be non-decreasing (offsets[%d] > offsets[%d])", e, e + 1);
    if (a < 0 || a >= p->n) return fail(WB_ERR_INVALID, "trajectory %d: agent %d outside 0..%d", e, a, p->n - 1);
    const int32_t B = p->hp[a].batch_size;
    const int64_t cnt = (int64_t)epochs * (T / B) * B;
    WB_REQUIRE(batch_index_host || cnt == 0, "batch_index is null");
    for (int64_t i = 0; i < cnt; i++) {
      const int32_t ix = batch_index_host[n_index + i];
      if (ix < 0 || ix >= T) return fail(WB_ERR_INVALID, "batch_index of trajectory %d holds %d, outside its %d rows", e, ix, T);
    }
    n_index += cnt;
    items[4 * e] = a;
    items[4 * e + 1] = 0;
    items[4 * e + 2] = T > 0 ? offsets_host[e] : 0;
    items[4 * e + 3] = T;
  }
  WB_REQUIRE(n_index <= INT32_MAX, "too many mini-batch indices for one call");
  const size_t rows = (size_t)offsets_host[n_traj], R = rows > 0 ? rows : 1, N = (size_t)n_traj;
  WB_REQUIRE(rows <= (size_t)INT32_MAX, "too many rows");
  const size_t IN = (size_t)p->state, ACT = (size_t)p->action;
  const size_t floats = R * (IN + 2 * ACT + 4) + 2 * N;
  if (int32_t rc = grow_stage(p, sizeof(float) * floats + sizeof(int32_t) * (N + (size_t)n_index) + 16)) return rc;
  float* d_states = p->d_stage;
  float* d_actions = d_states + R * IN;
  float* d_logp = d_actions + R * ACT;
  float* d_rewards = d_logp + R * ACT;
  float* d_values = d_rewards + R;
  float* d_returns = d_values + R;
  float* d_adv = d_returns + R;
  float* d_losses = d_adv + R;
  int32_t* d_skipped = reinterpret_cast<int32_t*>(d_losses + 2 * N);
  int32_t* d_index = d_skipped + N;
  if (rows) {
    WB_CUDA(cudaMemcpyAsync(d_states, states_host, sizeof(float) * rows * IN, cudaMemcpyHostToDevice, p->stream));
    WB_CUDA(cudaMemcpyAsync(d_actions, actions_host, sizeof(float) * rows * ACT, cudaMemcpyHostToDevice, p->stream));
    WB_CUDA(cudaMemcpyAsync(d_logp, logp_host, sizeof(float) * rows * ACT, cudaMemcpyHostToDevice, p->stream));
    WB_CUDA(cudaMemcpyAsync(d_rewards, rewards_host, sizeof(float) * rows, cudaMemcpyHostToDevice, p->stream));
  }
  if (n_index) WB_CUDA(cudaMemcpyAsync(d_index, batch_index_host, sizeof(int32_t) * n_index, cudaMemcpyHostToDevice, p->stream));
  if (int32_t rc = enqueue_train(p, n_traj, items.data(), (int32_t)R, 1, epochs, 0, d_states, d_actions, d_logp, d_rewards, d_index,
                                 d_values, d_returns, d_adv, d_losses, d_skipped))
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

}  // extern "C"

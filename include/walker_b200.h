/*
 * walker_b200.h -- C ABI of libwalker_b200.so: the B200-native (sm_100a) hot path of
 * De-Rosa/PPO-BipedalWalker -- the lockstep rigid-body physics step over N independent walkers and the
 * PPO policy/value MLP forward / clipped-surrogate gradient / backward / Adam.
 *
 * The reference (C#/MonoGame) has no FFI boundary; its "operator API" for this path is the public method
 * surface of Environment / Walker / Joint / RigidBody / IObject / IMaterial / PPOAgent / NeuralNetwork.
 * Each export below names the reference method(s) it replaces (file:line relative to the reference root);
 * INTEGRATION.md shows the P/Invoke stubs a maintainer adds on the C# side.
 *
 * Conventions
 *   - every call returns int32 status (WB_OK == 0); wb_last_error() gives the message of the last failure
 *     on the calling thread; nothing throws across the boundary.  The reference logs-and-continues
 *     (RigidBody.cs:91-94, PPOAgent.cs:238-341); the host shim maps status != 0 to ErrorLogger.LogError.
 *   - plain pointers + sizes only.  "host" pointers are ordinary (or pinned) CPU memory, copied inside
 *     the call on the handle's stream and synchronised before returning.  "_dev" variants take DEVICE
 *     pointers, enqueue on the handle's stream and return without synchronising.
 *   - handles own all device state; a handle is bound to the device current at creation; not thread-safe
 *     per handle, safe across handles.
 *   - there is no CPU fallback: every compute entry fails with WB_ERR_NO_DEVICE without a CUDA device.
 *
 * State record ("identical start state" contract, SURVEY.md section 8b): per environment 92 floats + 2 int32,
 *   f[ 0..57] vertices   LLL(6) LLU(6) Body(5) RLL(6) RLU(6), x/y interleaved   (Skeleton._vectors)
 *   f[58..67] centroids  x/y per body (cached, never recomputed after Rotate: Skeleton.cs:89-97)
 *   f[68..77] linear velocity x/y per body                                       (RigidBody.cs:30)
 *   f[78..82] angular velocity, f[83..87] tracked angle                          (RigidBody.cs:31,33)
 *   f[88..91] Joint._currentTorque                                               (Joint.cs:18)
 *   i[0] flags: bit0-4 Collided(LLL,LLU,Body,RLL,RLU) bit5 Walker.Terminal bit6 floor-first list order
 *   i[1] Environment._steps
 * wb_env_{get,set}_state exchange the records as structure-of-arrays blobs on the host side ([92][N] floats, [2][N] ints).
 * On the device the state is also a structure of arrays over walkers, with the x and y of a point adjacent (float2 rows for
 * vertices / centroids / velocities, float rows for the rest; csrc/physics.cuh) -- the library converts.
 */
#ifndef WALKER_B200_H
#define WALKER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WB_OK 0
#define WB_ERR_INVALID 1    /* bad argument                                   */
#define WB_ERR_NO_DEVICE 2  /* no CUDA device / wrong architecture            */
#define WB_ERR_CUDA 3       /* CUDA runtime error (message in wb_last_error)  */
#define WB_ERR_UNSUPPORTED 4
#define WB_ERR_COMM 5       /* a data-parallel gradient exchange timed out    */

#define WB_STATE_FLOATS 92
#define WB_STATE_INTS 2
#define WB_OBS 12
#define WB_ACT 4
#define WB_PAIR_SLOTS 9

#define WB_FLAG_TERMINAL (1 << 5)
#define WB_FLAG_FLOOR_FIRST (1 << 6)

/* built-in materials, Materials/{Ice,Wood,Paper,Titanium,Carpet,Rubber,Metal,SuperRubber}.cs:7-9 */
enum { WB_ICE = 0, WB_WOOD, WB_PAPER, WB_TITANIUM, WB_CARPET, WB_RUBBER, WB_METAL, WB_SUPERRUBBER, WB_NUM_BUILTIN_MATERIALS };
#define WB_MAX_MATERIALS 64

typedef struct wb_env_batch wb_env_batch;
typedef struct wb_policy wb_policy;

/* Hyperparameters.cs:83-121 (only the fields the hot path reads). */
typedef struct {
  int32_t iterations;    /* :86  physics substeps per env-step (50)      */
  int32_t max_timesteps; /* :87  (1000)                                  */
  int32_t batch_size;    /* :111 divisor of the per-sample gradients (64)*/
  int32_t use_gae;       /* :112                                         */
  int32_t normalize_advantages; /* :113                                  */
  float alpha, beta1, beta2, adam_epsilon; /* :104-107                   */
  float gamma, lambda;   /* :116-117                                     */
  float epsilon;         /* :120 PPO clip                                */
  float log_std;         /* :121                                         */
} wb_hyperparams;

/* per ordered candidate pair per substep; slot = LLL:{0,1} LLU:{2,3} Body:{4} RLL:{5,6} RLU:{7,8},
 * second index = position of the candidate in Environment._rigidBodies order (RigidBody.cs:66-96). */
typedef struct {
  int32_t other, aabb, sat, axis;
  float nx, ny, depth;
  int32_t ncontacts;
  float c0x, c0y, c1x, c1y;
} wb_pair_trace;

typedef struct {
  int32_t active;
  float depth;
} wb_joint_trace;

/* ---- library ---- */
const char* wb_version(void);
int32_t wb_last_error(char* buf, size_t buf_len);
/* selects the device (cudaSetDevice) and checks it is sm_100 */
int32_t wb_init(int32_t device);
int32_t wb_hyperparams_default(wb_hyperparams* hp); /* Hyperparameters.cs:83-121 defaults */
/* new IMaterial implementation (Materials/IMaterial.cs:6-11) -> id usable in wb_env_create */
int32_t wb_material_register(float inverse_mass, float restitution, float friction, int32_t* id_out);
int32_t wb_material_get(int32_t id, float* inverse_mass, float* restitution, float* friction);

/* ---- environments: Environment.cs / Walker/Walker.cs / Bodies / Objects ---- */
/* new Environment(...) x N (Environment.cs:39-51: Walker ctor + CreateCreature + CreateFloor + InitialState).
 * floor_material_ids / walker_material_ids: host arrays [n] or NULL (Metal floor Environment.cs:223, Carpet walker Walker.cs:30). */
int32_t wb_env_create(int32_t n_envs, const uint8_t* floor_material_ids, const uint8_t* walker_material_ids,
                      const wb_hyperparams* hp, wb_env_batch** out);
int32_t wb_env_destroy(wb_env_batch* env);
int32_t wb_env_count(const wb_env_batch* env, int32_t* n_out);
/* bind all work of this handle to a caller-owned cudaStream_t (NULL = default stream) */
int32_t wb_env_set_stream(wb_env_batch* env, void* cuda_stream);
int32_t wb_env_sync(wb_env_batch* env);

/* Environment.Reset + Walker.Reset + InitialState (Environment.cs:167-180, Walker.cs:212-236) for envs whose
 * mask byte != 0 (mask == NULL: all).  first_episode != 0 restores the constructor's list order instead. */
int32_t wb_env_reset(wb_env_batch* env, const uint8_t* mask_host, int32_t first_episode);
/* SoA blobs: state_f [92][N], state_i [2][N] (flags row, steps row) */
int32_t wb_env_set_state(wb_env_batch* env, const float* state_f_host, const int32_t* state_i_host);
int32_t wb_env_get_state(wb_env_batch* env, float* state_f_host, int32_t* state_i_host);

/* Matrix.Clip(action,1,-1) + Walker.TakeActions + Joint.SetTorque (Environment.cs:78, Walker.cs:66-75, Joint.cs:56-61); actions [N][4] */
int32_t wb_env_take_actions(wb_env_batch* env, const float* actions_host);
/* Environment.StepObjects(deltaTime) (Environment.cs:126-143): deltaTime /= iterations; iterations x (4 Joint.Step + every IObject.Update) */
int32_t wb_env_step_objects(wb_env_batch* env, float delta_time);
/* same, recording every candidate pair / joint: pair_trace [N][iterations][9], joint_trace [N][iterations][4] (host) */
int32_t wb_env_debug_contacts(wb_env_batch* env, float delta_time, wb_pair_trace* pair_trace_host,
                              wb_joint_trace* joint_trace_host);
/* tail of Environment.Step (Environment.cs:101-121): Walker.Update, CalculateReward (:148-154), terminal logic, Walker.GetState (Walker.cs:132-152).
 * obs [N][12], reward [N], done [N] */
int32_t wb_env_observe(wb_env_batch* env, float* obs_host, float* reward_host, uint8_t* done_host);
/* Walker.GetState only */
int32_t wb_env_get_obs(wb_env_batch* env, float* obs_host);

/* Environment.Update minus the policy (Environment.cs:64-92): _steps++, TakeActions(Clip(a)), Step, and when
 * auto_reset != 0 the Reset + InitialState that follows a terminal step (the returned obs is then the
 * initial observation).  One fused kernel launch; host buffers.  When every buffer of the call is page-locked
 * (cudaHostAlloc / cudaHostRegister / wb_host_pin) the kernel reads the actions and writes obs / reward / done directly
 * through the device-side aliases of the caller's buffers (zero-copy: no staging copies, one synchronisation); pageable
 * buffers take H2D copy + launch + D2H copies.  The results are identical. */
int32_t wb_env_step(wb_env_batch* env, const float* actions_host, float delta_time, int32_t auto_reset, float* obs_host,
                    float* reward_host, uint8_t* done_host);
/* device-pointer variant: enqueue only (no copies, no sync) */
int32_t wb_env_step_dev(wb_env_batch* env, const float* actions_dev, float delta_time, int32_t auto_reset, float* obs_dev,
                        float* reward_dev, uint8_t* done_dev);
/* Page-lock / release a host buffer the caller owns (e.g. a pinned GCHandle of a C# array: the reference keeps its
 * observation / action Matrix objects on the managed heap, Environment.cs:64-92) so that wb_env_step takes the zero-copy
 * path.  The buffer must stay allocated and un-moved until wb_host_unpin. */
int32_t wb_host_pin(void* host_ptr, size_t bytes);
int32_t wb_host_unpin(void* host_ptr);
/* number of kernel launches this handle has issued (bench.py "gpu_launches") */
int32_t wb_env_launch_count(const wb_env_batch* env, int64_t* count_out);
/* physics kernel variant: 2, 4, 8 or 16 lanes per walker (the lanes split the two legs, the SAT axes and the vertices: latency,
 * small batches), 1 (one thread per walker) or 1001 (one thread per walker + CTA-level work compaction: throughput, GPU full);
 * 104/108/116 = lanes without the leg split (kept for comparison); 0 = chosen from the batch size (the default) */
int32_t wb_env_set_variant(wb_env_batch* env, int32_t lanes_per_env);
int32_t wb_env_get_variant(const wb_env_batch* env, int32_t* lanes_per_env_out);

/* test hook: the rotation coefficients (float)Math.Cos((double)r), (float)Math.Sin((double)r) of Matrix.CreateRotationZ as used by
 * Skeleton.Rotate (Skeleton.cs:93). mode 0: production path, 1: forced double-double path, 2: forced device sincos path */
int32_t wb_debug_rotz(int32_t n, const float* radians_host, int32_t mode, float* cos_host, float* sin_host);

/* test hook: the kernels evaluate Vector2.Normalize's factor 1f / sqrt(s) (two correctly rounded steps, MonoGame Vector2.Normalize as
 * used by SATCollision.cs:46, ContactPoints.cs:27,84,86, Joint.cs:36) with a branch-free sequence; this compares it with the
 * two-intrinsic form for every float bit pattern in [first_bits, first_bits + count) and returns the number of mismatches */
int32_t wb_debug_rcp_sqrt_check(uint32_t first_bits, uint64_t count, uint64_t* mismatches_out, uint32_t* first_bad_bits_out);

/* ---- general scenes: the IObject plugin surface (Objects/IObject.cs:7-10) ----
 * N lockstep copies of an arbitrary list of convex polygons (Square / Triangle / Hexagon / Pole / Hull ..., 3..16 vertices,
 * Objects/RigidBodies/{Square,Triangle,Hexagon,Pole,Hull}.cs) with any IMaterial, static / floor flags, association ("no collide") lists (RigidBody.cs:143-152) and
 * joints (Joint.cs), stepped by Environment.StepObjects (Environment.cs:126-143).  List order = index order.  The walker-specialised
 * wb_env_* path covers the reference's default scene much faster; this path covers everything else the engine can be asked to do. */
typedef struct wb_scene wb_scene;
typedef struct {
  int32_t n_vertices;        /* Skeleton.AddVectors: 3..16 */
  int32_t is_static;         /* RigidBody ctor isStatic (RigidBody.cs:36-50) */
  int32_t is_floor;          /* isFloor: an AABB overlap with it latches the other body's Collided (RigidBody.cs:75-76) */
  int32_t material;          /* built-in id or wb_material_register */
  uint32_t associated_mask;  /* bit j: body j is associated (never tested against) */
  float accel_x, accel_y;    /* RigidBody.AddAcceleration (Walker.cs:191-198 adds (0, 980)) */
  float inverse_inertia;     /* < 0: 0.001f * inverse mass (RigidBody.cs:49); >= 0: override (Walker.cs:168) */
} wb_body_desc;
typedef struct {
  int32_t body_a, vertex_a, body_b, vertex_b; /* new Joint(bodyA, bodyB, indexA, indexB), Joint.cs:20-28 */
} wb_joint_desc;
/* vertices_xy: all polygons' vertices concatenated in body order, (x, y) interleaved */
int32_t wb_scene_create(int32_t n_envs, const wb_body_desc* bodies, int32_t n_bodies, const float* vertices_xy, const wb_joint_desc* joints,
                        int32_t n_joints, int32_t iterations, wb_scene** out);
int32_t wb_scene_destroy(wb_scene* scene);
int32_t wb_scene_set_stream(wb_scene* scene, void* cuda_stream);
/* per-copy record: 2*V vertex floats (body by body), 2B cached centroids, 2B linear velocities, B angular velocities, B tracked
 * angles, J Joint._currentTorque; host blobs are SoA [floats][N]; collided [N] has one bit per body */
int32_t wb_scene_state_floats(const wb_scene* scene, int32_t* per_copy_out);
int32_t wb_scene_set_state(wb_scene* scene, const float* state_host, const int32_t* collided_host);
int32_t wb_scene_get_state(wb_scene* scene, float* state_host, int32_t* collided_host);
/* Joint.SetTorque for every joint (Joint.cs:56-61); torques [N][J] */
int32_t wb_scene_set_torques(wb_scene* scene, const float* torques_host);
/* Environment.StepObjects(deltaTime) */
int32_t wb_scene_step_objects(wb_scene* scene, float delta_time);

/* ---- the walker on arbitrary terrain: Environment.Update with any IObject list in place of Environment.CreateFloor ----
 * Hyperparameters.RoughFloor (Hyperparameters.cs:88) -> Environment.CreateRoughFloor (Environment.cs:230-261), or any 1..11 bodies
 * (static floor hulls, obstacles, loose dynamic bodies).  Scene per copy: the walker's bodies [LLL, LLU, Body, RLL, RLU] and joints
 * exactly as Walker.CreateCreature builds them (Walker.cs:40-46,155-209), then the terrain bodies; the association masks of the
 * terrain descriptions index the terrain list.  List order: walker first as constructed (Environment.cs:46-48), terrain first
 * after a Reset, which re-creates the walker and appends it (Environment.cs:167-173).  Same phases and results contract as
 * wb_env_step: Terminal latches when Body, LLU or RLU touches any is_floor body (Walker.cs:49-54).  A Reset re-creates the
 * walker only: terrain bodies keep their state.  Static terrain bodies are never written by an impulse, like the wb_env_* floor:
 * finite impulses leave them unchanged anyway, and a NaN one (NaN actions) cannot corrupt terrain that outlives the walker's
 * resets.  More than 11 terrain bodies: WB_ERR_UNSUPPORTED. */
typedef struct wb_terrain_env wb_terrain_env;
/* new Environment(...) x N (Environment.cs:39-51) over the terrain: vertices_xy = all terrain vertices, body by body, (x, y) */
int32_t wb_terrain_env_create(int32_t n_envs, const wb_body_desc* terrain, int32_t n_terrain, const float* vertices_xy,
                              int32_t walker_material, const wb_hyperparams* hp, wb_terrain_env** out);
int32_t wb_terrain_env_destroy(wb_terrain_env* env);
int32_t wb_terrain_env_set_stream(wb_terrain_env* env, void* cuda_stream);
int32_t wb_terrain_env_state_floats(const wb_terrain_env* env, int32_t* per_copy_out);
/* per-copy terrain: vertices [N][2 * terrain vertices] (same vertex counts as at create); cached centroids recomputed like
 * Skeleton.FindCentroid (Skeleton.cs:100-113); terrain velocities / omega / angle and Collided cleared; the walker is not touched */
int32_t wb_terrain_env_set_terrain(wb_terrain_env* env, const float* vertices_host);
/* Environment.Reset + Walker.Reset + InitialState (Environment.cs:167-180, Walker.cs:212-236) for copies whose mask byte != 0
 * (NULL: all); first_episode != 0 restores the constructor's list order (walker first) */
int32_t wb_terrain_env_reset(wb_terrain_env* env, const uint8_t* mask_host, int32_t first_episode);
/* floats [rows][N]: the wb_scene_* record, bodies in INDEX order [LLL, LLU, Body, RLL, RLU, terrain...], then the 4 joint torques;
 * ints [3][N]: Collided bit per body index, flags (WB_FLAG_TERMINAL, WB_FLAG_FLOOR_FIRST = terrain before walker), Environment._steps */
int32_t wb_terrain_env_get_state(wb_terrain_env* env, float* state_f_host, int32_t* state_i_host);
int32_t wb_terrain_env_set_state(wb_terrain_env* env, const float* state_f_host, const int32_t* state_i_host);
/* Walker.GetState (Walker.cs:132-152): obs [N][12] */
int32_t wb_terrain_env_get_obs(wb_terrain_env* env, float* obs_host);
/* Environment.Update minus the policy (Environment.cs:64-92), one launch: as wb_env_step; host buffers are staged (copy, launch,
 * copy back, sync) */
int32_t wb_terrain_env_step(wb_terrain_env* env, const float* actions_host, float delta_time, int32_t auto_reset, float* obs_host,
                            float* reward_host, uint8_t* done_host);
/* device-pointer variant: enqueue only (no copies, no sync) */
int32_t wb_terrain_env_step_dev(wb_terrain_env* env, const float* actions_dev, float delta_time, int32_t auto_reset, float* obs_dev,
                                float* reward_dev, uint8_t* done_dev);
/* number of kernel launches this handle has issued */
int32_t wb_terrain_env_launch_count(const wb_terrain_env* env, int64_t* count_out);

/* ---- policy: Walker/PPO/PPOAgent.cs, Network/, Matrix.cs ---- */
/* layer kinds of the network DSL (PPOAgent.ParseLayers, PPOAgent.cs:96-143) */
enum { WB_DENSE = 0, WB_RELU = 1, WB_LEAKYRELU = 2, WB_TANH = 3 };

/* new PPOAgent(stateSize, actionSize) (PPOAgent.cs:23-37) with already-parsed layer lists (kinds[i] / sizes[i]; size is read
 * for WB_DENSE only).  Any network the DSL describes is accepted within: 1..16 layers per network, state size and dense widths
 * 1..128, action size 1..64, actor output == action_size, critic output == 1 (PPOAgent.cs:78-92), at most 32 dense layers in
 * total; anything else fails with WB_ERR_UNSUPPORTED / WB_ERR_INVALID -- never a fallback.  The reference's default networks
 * (Hyperparameters.cs:91-92) run on the tensor-core kernel, every other network on the any-topology kernel.
 * Weights start at zero: load them with wb_policy_set_weights (Xavier init is host-side, Matrix.cs:59-80). */
int32_t wb_policy_create(int32_t state_size, int32_t action_size, const int32_t* actor_kinds, const int32_t* actor_sizes,
                         int32_t actor_layers, const int32_t* critic_kinds, const int32_t* critic_sizes, int32_t critic_layers,
                         const wb_hyperparams* hp, wb_policy** out);
int32_t wb_policy_destroy(wb_policy* p);
int32_t wb_policy_set_stream(wb_policy* p, void* cuda_stream);
int32_t wb_policy_sync(wb_policy* p);
/* kernel variant of the MLP path: 0 = tcgen05 tensor-core kernel with 3xTF32 operands (default networks; the default),
 * 1 = fp32 CUDA-core kernel (default networks), 2 = the any-topology kernel (what non-default networks always use) */
int32_t wb_policy_set_variant(wb_policy* p, int32_t variant);
int32_t wb_policy_set_hyperparams(wb_policy* p, const wb_hyperparams* hp);
/* flat parameter vectors, per dense layer W[out][in] row-major then b[out] (DenseLayer.Save, DenseLayer.cs:73-79). which: 0 actor, 1 critic */
int32_t wb_policy_num_params(const wb_policy* p, int32_t which, int32_t* n_out);
int32_t wb_policy_set_weights(wb_policy* p, int32_t which, const float* flat_host);
int32_t wb_policy_get_weights(wb_policy* p, int32_t which, float* flat_host);
int32_t wb_policy_get_grads(wb_policy* p, int32_t which, float* flat_host);
/* Adam moments + per-dense-layer step counters (DenseLayer.cs:15-20) */
int32_t wb_policy_get_adam(wb_policy* p, int32_t which, float* m_host, float* v_host, int32_t* iterations_host);
int32_t wb_policy_set_adam(wb_policy* p, int32_t which, const float* m_host, const float* v_host, const int32_t* iterations_host);

/* NeuralNetwork.FeedForward for n states (NeuralNetwork.cs:52-64): mean [n][act] (actor), value [n] (critic); either may be NULL */
int32_t wb_policy_forward(wb_policy* p, int32_t n, const float* states_host, float* mean_host, float* value_host);
int32_t wb_policy_forward_dev(wb_policy* p, int32_t n, const float* states_dev, float* mean_dev, float* value_dev);
/* PPOAgent.SampleActions (PPOAgent.cs:381-398) with the two uniforms of each Box-Muller draw injected:
 * uniforms [n][act][2] -> actions [n][act], logp [n][act] (NormalDistribution.cs:12-32) */
int32_t wb_policy_sample(wb_policy* p, int32_t n, const float* states_host, const float* uniforms_host, float* actions_host,
                         float* logp_host, float* mean_host);
int32_t wb_policy_sample_dev(wb_policy* p, int32_t n, const float* states_dev, const float* uniforms_dev, float* actions_dev,
                             float* logp_dev, float* mean_dev);
/* same, uniforms from an on-device Philox-4x32-10 counter stream (seed, step): extension, the reference RNG is unseedable */
int32_t wb_policy_sample_philox_dev(wb_policy* p, int32_t n, const float* states_dev, uint64_t seed, uint64_t step,
                                    float* actions_dev, float* logp_dev, float* mean_dev);

/* one policy step of a lockstep rollout, all on the device: SampleActions (Philox stream (seed, step)) and the critic's value
 * estimate (PPOAgent.GetValueEstimate, PPOAgent.cs:350-364) in ONE launch; mean_dev / value_dev may be NULL */
int32_t wb_policy_act_dev(wb_policy* p, int32_t n, const float* states_dev, uint64_t seed, uint64_t step, float* actions_dev,
                          float* logp_dev, float* mean_dev, float* value_dev);
/* rollout -> update glue for N lockstep environments (PPOAgent.cs:414-498 applied per episode fragment): time-major buffers
 * [horizon][n_envs]; done != 0 marks the last step of an episode (the recurrences restart there like at a trajectory end).
 * Segment end: last_values_dev [n_envs] = the critic's estimate of the observation AFTER the last step; an episode still
 * running at the segment end continues the recurrence from it (next return = next value = V(s_T)).  This is a DEVIATION the
 * lockstep form needs -- the reference only ever trains on complete episodes (PPOAgent.cs:147) -- and is skipped where
 * dones[horizon-1] is set.  last_values_dev == NULL truncates instead (the segment end is scored like a trajectory end).
 * With hp.normalize_advantages the whole [horizon x n_envs] pool is normalised (wb_normalize_advantages_dev, stage -1). */
int32_t wb_segment_returns_dev(wb_policy* p, int32_t n_envs, int32_t horizon, const float* rewards_dev, const float* values_dev,
                               const uint8_t* dones_dev, const float* last_values_dev, float* returns_dev, float* advantages_dev);
/* PPOAgent.Normalize (PPOAgent.cs:461-472) over a pool of advantages: mean = (float)(sum / count) and
 * std = (float)sqrt(sum (x - mean)^2 / count) accumulated in double, x = (x - mean) / (std + hp.epsilon) (the reference
 * uses the PPO clip epsilon here).  stage -1 runs everything for a single process.  A data-parallel caller runs stage 0,
 * all-reduces (sum) the stats buffer, runs stage 1, all-reduces it again, runs stage 2; n_global = pool size over all ranks. */
int32_t wb_normalize_advantages_dev(wb_policy* p, int32_t stage, int64_t n_local, int64_t n_global, float* advantages_dev);
/* device address + length (in doubles) of the partial-sum buffer the stages above exchange through */
int32_t wb_normalize_stats_buffer(wb_policy* p, void** dev_ptr_out, int32_t* n_doubles_out);
/* PPOAgent.CreateBatches (PPOAgent.cs:501-540): gather rows index_dev[0..batch) of the rollout pool into a contiguous minibatch */
int32_t wb_gather_minibatch_dev(wb_policy* p, int32_t batch, const int32_t* index_dev, const float* states_pool, const float* actions_pool,
                                const float* logp_pool, const float* advantages_pool, const float* returns_pool, float* states_out,
                                float* actions_out, float* logp_out, float* advantages_out, float* returns_out);

/* PPOAgent.Train(Batch) gradient part (PPOAgent.cs:218-342): Zero(), then for every sample the
 * clipped-surrogate dL/dmu and 2(V-G)/B, back-propagated and accumulated; gradients stay on the device
 * (wb_policy_get_grads).  n = samples in this call (this rank's shard); hp.batch_size is the divisor B.
 * losses_host[2] = {sum g_V, sum mean_k g_mu} (the reference's "losses", PPOAgent.cs:331-332); skipped_host = samples skipped (:286-290). */
int32_t wb_ppo_grad(wb_policy* p, int32_t n, const float* states_host, const float* actions_host, const float* old_logp_host,
                    const float* advantages_host, const float* returns_host, float* losses_host, int32_t* skipped_host);
int32_t wb_ppo_grad_dev(wb_policy* p, int32_t n, const float* states_dev, const float* actions_dev, const float* old_logp_dev,
                        const float* advantages_dev, const float* returns_dev);
/* Data-parallel variant for one process per GPU on one NVLink/NVSwitch box (no reference equivalent: the reference is one process):
 * the per-CTA partial gradients are reduced AND summed over all ranks by ONE kernel that pushes slices into the peers' exchange
 * buffers over NVLink (CUDA IPC peer memory) -- no NCCL call, bit-identical result on every rank.  Setup: every rank calls
 * wb_comm_local_handle, the 64-byte handles are all-gathered by the host (any transport), every rank calls wb_comm_connect with
 * the gathered array [world][64].  Every rank must then issue the same sequence of wb_ppo_grad_allreduce_dev calls. */
int32_t wb_comm_local_handle(wb_policy* p, void* handle64_out);
int32_t wb_comm_connect(wb_policy* p, int32_t rank, int32_t world, const void* all_handles64);
/* failed_out != 0: an exchange gave up waiting for a peer (bounded spin).  The slices that timed out were neither stored nor
 * passed to Adam, every later exchange of the handle is a no-op on the device, and wb_ppo_train_dev / wb_ppo_grad_allreduce_dev
 * return WB_ERR_COMM from then on (the status word is mapped host memory: the check costs nothing and needs no sync) */
int32_t wb_comm_status(wb_policy* p, int32_t* connected_world_out, int32_t* failed_out);
int32_t wb_ppo_grad_allreduce_dev(wb_policy* p, int32_t n, const float* states_dev, const float* actions_dev, const float* old_logp_dev,
                                  const float* advantages_dev, const float* returns_dev);
/* PPOAgent.Train(Batch) complete (PPOAgent.cs:218-345): gradient, reduction of the per-CTA partials, all-reduce over NVLink when
 * the policy is connected (wb_comm_connect; a single rank otherwise) and DenseLayer.Adam on both networks; the reduced gradient is
 * also left in the gradient buffer (losses / skipped included).  With the default networks and the tensor-core kernel this is ONE
 * launch: the gradient kernel reduces, exchanges and applies Adam in its own tail behind a grid barrier (every rank must then pass
 * the same n, so that the ranks' slices agree); otherwise the gradient kernel is followed by one reduce / exchange / Adam kernel. */
int32_t wb_ppo_train_dev(wb_policy* p, int32_t n, const float* states_dev, const float* actions_dev, const float* old_logp_dev,
                         const float* advantages_dev, const float* returns_dev);
/* The same on rows index_dev[0..n) of a rollout pool: PPOAgent.CreateBatches (PPOAgent.cs:501-540) fused into the gradient kernel's
 * input prefetch (no gathered copy of the minibatch is written; kernels without that path gather first, as wb_gather_minibatch_dev).
 * Every index must be a valid row of the pool arrays: the kernel does not range-check device indices. */
int32_t wb_ppo_train_indexed_dev(wb_policy* p, int32_t n, const int32_t* index_dev, const float* states_pool, const float* actions_pool,
                                 const float* logp_pool, const float* advantages_pool, const float* returns_pool);
/* PPOAgent.Train(Batch) from host buffers: wb_ppo_grad + wb_adam_step as one call (one launch on the default path).  When all five
 * buffers are page-locked (cudaHostAlloc / cudaHostRegister / wb_host_pin) and 16-byte aligned the tensor-core kernel reads them in
 * place over PCIe while it computes (no staging copy); wb_ppo_grad takes the same zero-copy path; the other kernel variants and
 * pageable buffers are staged.  losses / skipped as wb_ppo_grad. */
int32_t wb_ppo_train(wb_policy* p, int32_t n, const float* states_host, const float* actions_host, const float* old_logp_host,
                     const float* advantages_host, const float* returns_host, float* losses_host, int32_t* skipped_host);
/* PPOAgent.Train(Trajectory) (PPOAgent.cs:147-172) for n_traj complete episodes, in list order: trajectory e is trained with the
 * weights trajectory e-1 left, exactly as n_traj calls of Train.  offsets_host[n_traj+1] (HOST, in both entries; non-decreasing,
 * offsets[0] >= 0) delimits trajectory e = rows [offsets[e], offsets[e+1]) of states [.][state], actions / old_logp [.][act]
 * (UNclipped, Environment.cs:87-88) and rewards [.].  Per trajectory: CalculateValues (critic forward), MC return or GAE and the
 * optional Normalize (PPOAgent.cs:175-189,414-498), then epochs x floor(T_e / B) mini-batches of B = hp.batch_size samples, each
 * Train(Batch) + Adam.  batch_index: per trajectory, epochs x floor(T_e / B) x B LOCAL row numbers (PPOAgent.CreateBatches,
 * :501-540; the caller draws them, like the injected Box-Muller uniforms), blocks concatenated in trajectory order.
 * values / returns / advantages [.] (Trajectory.Values / Returns / Advantages) may be NULL.  losses [n_traj][2] = the last
 * mini-batch's {sum g_V, sum mean_k g_mu} (0 if T_e < B), skipped [n_traj] = skipped samples over all of the trajectory's
 * mini-batches; either may be NULL.  A trajectory with T_e < B gets its values / returns / advantages but trains nothing and
 * consumes no Adam step.  The Adam bias corrections are computed on the host exactly as for wb_adam_step; the gradient buffer
 * then holds the last trained mini-batch's gradient, losses and skipped count, as after wb_ppo_train.  The default networks
 * (kernel variants 0 and 1) train in ONE launch: one persistent CTA runs the whole chain of Adam steps without a host round
 * trip; other networks and variant 2 enqueue the per-trajectory and per-mini-batch kernels with no host sync.  The host entry
 * range-checks every index and refuses bad offsets, epochs < 0, n_traj < 1 and hp.batch_size < 1 with WB_ERR_INVALID before
 * anything on the device changes.  A policy connected for data-parallel exchange (world > 1) gets WB_ERR_UNSUPPORTED. */
int32_t wb_ppo_train_trajectories(wb_policy* p, int32_t n_traj, const int32_t* offsets_host, int32_t epochs, const float* states_host,
                                  const float* actions_host, const float* old_logp_host, const float* rewards_host,
                                  const int32_t* batch_index_host, float* values_host, float* returns_host, float* advantages_host,
                                  float* losses_host, int32_t* skipped_host);
/* The same with every pointer except offsets_host on the device; enqueue only.  Every index must be a valid local row of its
 * trajectory: the kernels do not range-check device indices. */
int32_t wb_ppo_train_trajectories_dev(wb_policy* p, int32_t n_traj, const int32_t* offsets_host, int32_t epochs, const float* states_dev,
                                      const float* actions_dev, const float* old_logp_dev, const float* rewards_dev,
                                      const int32_t* batch_index_dev, float* values_dev, float* returns_dev, float* advantages_dev,
                                      float* losses_dev, int32_t* skipped_dev);
/* NeuralNetwork.Optimise -> DenseLayer.Adam on both networks (NeuralNetwork.cs:85-91, DenseLayer.cs:125-159) */
int32_t wb_adam_step(wb_policy* p);
/* device address + length of the contiguous gradient buffer [actor | critic | 2 loss sums | skipped] for the
 * caller's all-reduce (one NCCL all-reduce(sum) over NVLink per minibatch, issued by the host process) */
int32_t wb_policy_grad_buffer(wb_policy* p, void** dev_ptr_out, int32_t* n_floats_out);
int32_t wb_policy_launch_count(const wb_policy* p, int64_t* count_out);

/* ---- populations: one PPO brain per walker ----
 * In the reference every walker owns its agent (new Walker() builds its own PPOAgent(12, 4), Walker.cs:25-34) and trains it on each
 * of its own episodes as soon as the episode ends (Environment.cs:91,157-164 -> PPOAgent.Train(Trajectory), PPOAgent.cs:147-172).
 * A population holds P such agents, all with the same two networks: the reference's defaults (Hyperparameters.cs:91-92; 6 149
 * parameters, wb_population_create) or any pair the DSL describes (wb_population_create_net).  Each agent has its own weights,
 * Adam m / v, per-dense-layer step counters and wb_hyperparams (alpha, beta1, beta2, Adam epsilon, gamma, lambda, clip epsilon,
 * log_std, use_gae, normalize_advantages, batch_size).  Agent a behaves exactly as one wb_policy with the same networks, weights
 * and hyper-parameters -- on kernel variant 1 for the default networks, on the any-topology kernel (variant 2) otherwise: acting
 * and training give the same bits.  Agents that a call does not name are not touched.  Weights start at zero (load them with
 * wb_population_set_weights).  The longest episode trained is 1 024 steps (WB_ERR_UNSUPPORTED beyond).  Below, n_actor /
 * n_critic / n_dense are the population's parameter and dense-layer counts (wb_population_num_params; 5 252 / 897 / 3 + 2 for the
 * defaults), state / act its state and action sizes (12 / 4). */
typedef struct wb_population wb_population;
/* new PPOAgent(12, 4) x n_agents (PPOAgent.cs:23-37); hp = [n_agents] hyper-parameters or NULL (the defaults for every agent).
 * n_agents < 1 or a batch_size < 1: WB_ERR_INVALID */
int32_t wb_population_create(int32_t n_agents, const wb_hyperparams* hp, wb_population** out);
/* new PPOAgent(state_size, action_size) x n_agents with the networks of the layer lists (as wb_policy_create: the same checks and
 * statuses for a network outside the limits).  The default lists give the population of wb_population_create; other networks run
 * the any-topology population kernels.  A network whose layer caches and one episode's arrays exceed a CTA's shared memory:
 * WB_ERR_UNSUPPORTED. */
int32_t wb_population_create_net(int32_t n_agents, int32_t state_size, int32_t action_size, const int32_t* actor_kinds,
                                 const int32_t* actor_sizes, int32_t actor_layers, const int32_t* critic_kinds, const int32_t* critic_sizes,
                                 int32_t critic_layers, const wb_hyperparams* hp, wb_population** out);
/* parameters of each agent's actor (which = 0) or critic (which = 1) */
int32_t wb_population_num_params(const wb_population* pop, int32_t which, int32_t* n_out);
int32_t wb_population_destroy(wb_population* pop);
int32_t wb_population_set_stream(wb_population* pop, void* cuda_stream);
int32_t wb_population_sync(wb_population* pop);
/* number of kernel launches this handle has issued */
int32_t wb_population_launch_count(const wb_population* pop, int64_t* count_out);
/* agent a's flat parameters [n_actor + n_critic] = actor | critic, each in the DenseLayer.Save order (DenseLayer.cs:73-79) */
int32_t wb_population_set_weights(wb_population* pop, int32_t agent, const float* flat_host);
int32_t wb_population_get_weights(wb_population* pop, int32_t agent, float* flat_host);
/* agent a's gradient buffer [n_actor + n_critic] (the last mini-batch it trained, as wb_policy_get_grads) */
int32_t wb_population_get_grads(wb_population* pop, int32_t agent, float* flat_host);
/* agent a's Adam moments m / v [n_actor + n_critic] and the step counters [n_dense] of its dense layers (actor layers, then critic
 * layers; DenseLayer.cs:15-20) */
int32_t wb_population_get_adam(wb_population* pop, int32_t agent, float* m_host, float* v_host, int32_t* steps_host);
/* the mirror of wb_population_get_adam (and of wb_policy_set_adam): agent a's m / v [n_actor + n_critic] and step counters
 * [n_dense] (DenseLayer.cs:15-20) */
int32_t wb_population_set_adam(wb_population* pop, int32_t agent, const float* m_host, const float* v_host, const int32_t* steps_host);
/* agent a's wb_hyperparams (Hyperparameters.cs:83-121; set mirrors wb_policy_set_hyperparams).  The next call that acts or trains
 * with the agent uses them.  batch_size < 1: WB_ERR_INVALID, nothing changes. */
int32_t wb_population_set_hyperparams(wb_population* pop, int32_t agent, const wb_hyperparams* hp);
int32_t wb_population_get_hyperparams(const wb_population* pop, int32_t agent, wb_hyperparams* hp_out);
/* Population-based training's exploit step, an extension with no reference counterpart (the reference's agents are independent):
 * for i < n_pairs, agent dst_host[i] becomes a copy of agent src_host[i] -- its weights, Adam m / v and step counters, bit for
 * bit -- with the hyper-parameters hp_host[i] (hp_host NULL: src's).  dst keeps its own gradient buffer (scratch of its last
 * mini-batch) and its own count of trained episodes (which keys its device-drawn mini-batches).  Enqueue only: one launch on the
 * population's stream, after whatever is already enqueued there.  Refused with WB_ERR_INVALID before anything changes:
 * n_pairs < 1, an agent out of range, dst == src, a dst listed twice, an agent that is both a src and a dst, a batch_size < 1. */
int32_t wb_population_copy_agents(wb_population* pop, int32_t n_pairs, const int32_t* dst_host, const int32_t* src_host,
                                  const wb_hyperparams* hp_host);
/* PPOAgent.SampleActions (PPOAgent.cs:381-398) for n == P walkers, walker w with agent w, with the two System.Random uniforms of
 * each Box-Muller draw injected (NormalDistribution.cs:12-32): states [n][state], uniforms [n][act][2] -> actions, logp [n][act],
 * mean [n][act] or NULL.  Row w equals wb_policy_sample of agent w. */
int32_t wb_population_sample(wb_population* pop, int32_t n, const float* states_host, const float* uniforms_host, float* actions_host,
                             float* logp_host, float* mean_host);
/* the same from the Philox stream (seed, step) of wb_policy_act_dev (counter (walker, action dim, step)), enqueue only; mean_dev
 * and the critic's value estimate value_dev [n] (PPOAgent.GetValueEstimate, PPOAgent.cs:350-364) may be NULL.  One launch. */
int32_t wb_population_act_dev(wb_population* pop, int32_t n, const float* states_dev, uint64_t seed, uint64_t step, float* actions_dev,
                              float* logp_dev, float* mean_dev, float* value_dev);
/* PPOAgent.Train(Trajectory) (PPOAgent.cs:147-172) for n_traj finished episodes of several agents in ONE launch: trajectory e
 * belongs to agent agent_host[e] and is rows [offsets[e], offsets[e+1]) of the packed arrays, as in wb_ppo_train_trajectories.
 * Every agent trains its own trajectories in list order, so its final state equals wb_ppo_train_trajectories of its sub-list.
 * batch_index: per trajectory, in list order, epochs x floor(T_e / B_a) x B_a local row numbers (PPOAgent.CreateBatches,
 * :501-540, drawn by the caller), B_a = that agent's batch_size.  values / returns / advantages [rows], losses [n_traj][2] and
 * skipped [n_traj] as in wb_ppo_train_trajectories; each may be NULL.  Bad offsets, an agent out of range, epochs < 0,
 * n_traj < 1 or an index outside its trajectory: WB_ERR_INVALID before anything on the device changes. */
int32_t wb_population_train_trajectories(wb_population* pop, int32_t n_traj, const int32_t* agent_host, const int32_t* offsets_host,
                                         int32_t epochs, const float* states_host, const float* actions_host, const float* logp_host,
                                         const float* rewards_host, const int32_t* batch_index_host, float* values_host,
                                         float* returns_host, float* advantages_host, float* losses_host, int32_t* skipped_host);
/* The device form for lockstep walkers (Environment.Update -> TrainNetworks -> Reset, Environment.cs:64-92,157-173): the
 * rollout arrays are a time-major ring of ring_rows rows x columns (states [R][C][state], actions / logp [R][C][act], rewards /
 * values / returns / advantages [R][C]).  items_host [n_items][4] = (agent, column, t0, length): the episode's step i is row
 * ((t0 + i) mod ring_rows) * columns + column.  Every agent trains its items in list order, one CTA per agent with work.
 * batch_index_dev: caller-drawn indices in the layout of wb_population_train_trajectories, or NULL: the kernel draws them --
 * epoch k of an episode orders the local rows i < length by (key, i) with key = Philox-4x32-10(counter (i, k, episode, agent),
 * key (seed & 0xffffffff, seed >> 32)).x, where `episode` is the number of this agent's episodes (items, in both train entries)
 * trained before this one, and takes floor(length / B) blocks of B (the remainder is dropped).  The episode's values, returns and
 * advantages are written to its rows of values_dev / returns_dev / advantages_dev (required); losses_dev [n_items][2] and
 * skipped_dev [n_items] may be NULL.  Host arguments are checked before anything changes (WB_ERR_INVALID): n_items < 1, an
 * agent or column out of range, length < 0 or > ring_rows, t0 outside the ring, epochs < 0.  Device indices are not
 * range-checked.  Enqueue only: one launch. */
int32_t wb_population_train_dev(wb_population* pop, int32_t n_items, const int32_t* items_host, int32_t ring_rows, int32_t columns,
                                int32_t epochs, uint64_t seed, const float* states_dev, const float* actions_dev, const float* logp_dev,
                                const float* rewards_dev, const int32_t* batch_index_dev, float* values_dev, float* returns_dev,
                                float* advantages_dev, float* losses_dev, int32_t* skipped_dev);

/* test hook for the tcgen05 building block: one CTA computes D[M x N] = A[M x K] * B[N x K]^T on the tensor cores
 * (kind::tf32; passes = 1 plain TF32, 3 = 3xTF32 split).  a/b_mn_major choose how the operand tile is read (K-major / MN-major). */
int32_t wb_debug_tc_gemm(int32_t M, int32_t N, int32_t K, int32_t a_mn_major, int32_t b_mn_major, int32_t passes, const float* A_host,
                         const float* B_host, float* D_host);

/* rollout -> update glue (PPOAgent.cs:414-498), one trajectory of length n on the device */
int32_t wb_returns_advantages(wb_policy* p, int32_t n, const float* rewards_host, const float* values_host, float* returns_host,
                              float* advantages_host);

#ifdef __cplusplus
}
#endif
#endif /* WALKER_B200_H */

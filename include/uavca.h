/*
 * uavca.h — C-ABI of the B200-native batched UAV collision-avoidance environment step.
 *
 * The reference (dazchi/gym-uav-collision-avoidance) has no FFI: its boundary is the Python gym API of
 * two classes.  Every entry point below names the reference interface it replaces (file:line relative to
 * the reference checkout):
 *
 *   uavca_step_multi   <- MultiUAVWorld2D.step            gym_uav_collision_avoidance/envs/multi_uav_world_2d.py:177-241
 *                         UAVAgent.step/finish/uavs_in_range  gym_uav_collision_avoidance/envs/uav_agent.py:23-64
 *   uavca_step_f64     <- either step() fed NumPy float64 actions   uav_agent.py:26, uav_world_2d.py:142
 *   uavca_step_single  <- UAVWorld2D.step                 gym_uav_collision_avoidance/envs/uav_world_2d.py:137-173
 *   uavca_reset        <- MultiUAVWorld2D.reset :116-175 / UAVWorld2D.reset uav_world_2d.py:119-135
 *   uavca_observe      <- MultiUAVWorld2D._get_obs :60-109 / UAVWorld2D._get_obs uav_world_2d.py:77-112
 *   uavca_map_action   <- caller-side action mapping      test_sac_multi.py:77-80, test_pytorch_multi.py:80
 *   uavca_rollout      <- the random-action driver loops    run.py:10-16, run_multi.py:10-16 (K x env.step per call)
 *   uavca_step_multi_replay <- env.step + the N memory.push calls of a training step   test_sac_multi.py:99-103
 *   uavca_replay_push(_dev) / uavca_replay_sample <- ReplayMemory.push / .sample   pytorch_sac_temp/replay_memory.py:15-24
 *   uavca_stats        <- env.steps / target_reach_count / collision_count  multi_uav_world_2d.py:166-168,209,221,238
 *   uavca_config       <- constructor kwargs              multi_uav_world_2d.py:13-28, uav_world_2d.py:14-26
 *
 * Conventions: plain C, int return codes (0 = ok, negative = error, text via uavca_last_error()); no
 * exceptions cross the boundary.  Unless a parameter is documented as HOST memory, every pointer is a
 * DEVICE pointer borrowed for the duration of the call (the caller — PyTorch — owns all memory).  Every
 * call takes a cudaStream_t (passed as void*) and is asynchronous on it.  A handle is bound to one device,
 * is not thread-safe; distinct handles are independent.  There is no CPU fallback: without a usable CUDA
 * device uavca_create fails.
 */
#ifndef UAVCA_H_
#define UAVCA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UAVCA_VERSION 203

/* world kinds */
#define UAVCA_KIND_MULTI 0  /* MultiUAVWorld2D: N UAVs per env, 10-feature observation */
#define UAVCA_KIND_SINGLE 1 /* UAVWorld2D: one UAV per env, 4-feature observation */

/* action modes (what the `action` tensor holds) */
#define UAVCA_ACTION_CARTESIAN 0 /* env action [vx, vy] in m/s — what env.step() takes */
#define UAVCA_ACTION_POLAR 1     /* policy output in [-1,1]^2: v=(a0/2+0.5)*scale, th=a1*pi (test_sac_multi.py:77-80) */
#define UAVCA_ACTION_SCALED 2    /* policy output in [-1,1]^2: a*action_space.high (test_pytorch_multi.py:80) */

/* auto-reset trigger bits (0 = never reset inside step) */
#define UAVCA_RESET_ON_DONE0 1    /* training protocol: dones[0] (test_sac_multi.py:111-113) */
#define UAVCA_RESET_ON_ALL_DONE 2 /* evaluation protocol: all(dones) (test_sac_multi.py:115-117) */
#define UAVCA_RESET_ON_ANY_DONE 4 /* any UAV done (single-UAV world: its done flag, run.py:14-15) */

/* where an auto-reset or uavca_reset takes the new episode from */
#define UAVCA_SOURCE_PHILOX 0 /* counter-based Philox4x32-10 keyed by (seed, global env index, episode) */
#define UAVCA_SOURCE_POOL 1   /* host-supplied reset states (parity runs): uavca_set_reset_pool */

/* per-UAV flag bits in the state (`flags` array) */
#define UAVCA_FLAG_PARKED 1   /* UAVAgent.done latch (uav_agent.py:19,39) */
#define UAVCA_FLAG_COLLIDED 2 /* UAVAgent.collided latch (uav_agent.py:20; multi_uav_world_2d.py:210) */

#define UAVCA_OBS_DIM_MULTI 10
#define UAVCA_OBS_DIM_SINGLE 4
#define UAVCA_MAX_AGENTS 1024 /* up to 32 UAVs an env lives in one warp (the fast kernels); larger envs and the float64
                                 world of circular episodes run on the general one-thread-per-env kernel */

typedef struct uavca_config {
  int32_t kind;                 /* UAVCA_KIND_* */
  int32_t num_envs;             /* B, environments held by THIS handle (this GPU's shard) */
  int32_t num_agents;           /* N, UAVs per env (1..UAVCA_MAX_AGENTS); must be 1 for UAVCA_KIND_SINGLE */
  int32_t reset_mode;           /* UAVCA_RESET_* bits */
  int32_t max_episode_steps;    /* also reset when env steps >= this; 0 = no limit */
  int32_t reset_source;         /* UAVCA_SOURCE_* */
  int32_t circular;             /* multi reset: deterministic ring layout, reset(circular=True) (multi_uav_world_2d.py:157-163).
                                   The reference holds float64 locations from there on, so this mode is the FLOAT64 WORLD:
                                   positions, targets, distances in float64 (state fields pos64 / tgt64 / init64 / prev64;
                                   pos / tgt / init / prev keep float32 mirrors) */
  int32_t single_f32_first_step;/* single world: replicate the float32 first-step quotient the reference
                                   produces when handed float32 actions (uav_world_2d.py:122,142) */
  int64_t env_index_base;       /* global index of env 0 of this shard (Philox streams are shard-invariant) */
  uint64_t seed;                /* Philox key */
  double x_size, y_size;        /* box, centred on the origin */
  double max_speed;             /* per-component speed bound */
  double max_acceleration;      /* per-component acceleration bound */
  double tau;                   /* seconds per step (0.02 in the reference) */
  double collider_radius;       /* soft collision when d <= 2*collider_radius */
  double hard_collision_radius; /* HARD_COLLISION_RADIUS (multi_uav_world_2d.py:8) */
  double d_sense;               /* neighbour sensing range (strict <) */
  double reach_distance;        /* 0.5  (multi_uav_world_2d.py:218, uav_world_2d.py:159) */
  double reach_speed;           /* 0.2  (multi_uav_world_2d.py:218) */
  double polar_scale;           /* action scale of UAVCA_ACTION_POLAR: ||action_space.high|| (multi) or high[0] (single) */
  int32_t track_scores;         /* accumulate the per-episode scores the training loops keep on the host
                                   (test_sac_multi.py:105,152-156): score[b][0] += rewards[0],
                                   score[b][1] += sum_i rewards[i] * (1 - dones[i]); folded into stats at reset */
  int32_t reserved0;
} uavca_config;

/* Byte offsets of the structure-of-arrays fields inside one state blob (all 256-byte aligned).
 * M = num_envs * num_agents.  The blob is allocated by the caller (uavca_state_layout gives its size). */
typedef struct uavca_layout {
  size_t total_bytes;
  size_t stats;   /* 8 x 8 bytes over FINISHED episodes: uint64 episodes, reach, collisions, steps; double sum of
                     score[.][0], double sum of score[.][1] (track_scores); uint64 non-finite UAV-steps seen; 1 spare */
  size_t pos;     /* float  [M][2]  UAV location          (float32 in the reference after reset) */
  size_t vel;     /* double [M][2]  UAV velocity          (float64 in the reference) */
  size_t tgt;     /* float  [M][2]  target location */
  size_t init;    /* float  [M]     init_distance */
  size_t prev;    /* float  [M]     prev_distance */
  size_t flags;   /* uint8  [M]     UAVCA_FLAG_* */
  size_t steps;   /* int32  [B]     env.steps */
  size_t reach;   /* int32  [B]     env.target_reach_count */
  size_t coll;    /* int32  [B]     env.collision_count */
  size_t episode; /* uint32 [B]     episodes started by this env (Philox counter word) */
  size_t score;   /* double [B][2]  running scores of the episode in flight (track_scores) */
  size_t pos64;   /* double [M][2]  float64 world only (config.circular; zero-sized otherwise): location */
  size_t tgt64;   /* double [M][2]  target_location */
  size_t init64;  /* double [M]     init_distance */
  size_t prev64;  /* double [M]     prev_distance */
} uavca_layout;

typedef struct uavca_handle uavca_handle;

const char* uavca_last_error(void);
int uavca_version(void);

/* Fill *cfg with the reference defaults of the given world kind (ctor defaults cited above). */
int uavca_default_config(int kind, uavca_config* cfg);

int uavca_create(const uavca_config* cfg, int device, uavca_handle** out);
int uavca_destroy(uavca_handle* h);
int uavca_get_config(const uavca_handle* h, uavca_config* out);
int uavca_state_layout(const uavca_handle* h, uavca_layout* out);

/* Host-supplied reset states: `pool_state` is a state blob laid out for `pool_envs` environments (same N).
 * With reset_source = UAVCA_SOURCE_POOL env b starting its e-th episode copies pool env
 * (env_index_base + b + e) % pool_envs.  The pool is borrowed until replaced or the handle is destroyed. */
int uavca_set_reset_pool(uavca_handle* h, const void* pool_state, int32_t pool_envs);
/* Layout of a pool blob holding `pool_envs` environments. */
int uavca_pool_layout(const uavca_handle* h, int32_t pool_envs, uavca_layout* out);

/* Start a new episode in every env (mask == NULL) or in envs with mask[b] != 0, and write their
 * observations (rows of other envs are left untouched).  obs: float [B][N][obs_dim]. */
int uavca_reset(uavca_handle* h, void* state, const uint8_t* mask, float* obs, void* stream);

/* Recompute the observation of the current state (after the caller edited the state). */
int uavca_observe(uavca_handle* h, const void* state, float* obs, void* stream);

/* action: float [B][N][2]; obs: float [B][N][10]; reward: float [B][N]; done: uint8 [B][N].
 * obs is the observation the policy acts on next (post-reset for envs that auto-reset this step).
 * final_obs (nullable): the step's own next-observation before any reset (what the replay buffer stores).
 * reset_mask (nullable): uint8 [B], 1 where the env auto-reset this step. */
int uavca_step_multi(uavca_handle* h, void* state, const float* action, int action_mode, int evaluate,
                     float* obs, float* reward, uint8_t* done, float* final_obs, uint8_t* reset_mask,
                     void* stream);

/* action: float [B][2]; obs: float [B][4]; reward: float [B]; done: uint8 [B];
 * distance (nullable): float [B] = info["distance"]. */
int uavca_step_single(uavca_handle* h, void* state, const float* action, int action_mode, float* obs,
                      float* reward, uint8_t* done, float* distance, float* final_obs, uint8_t* reset_mask,
                      void* stream);

/* env.step() fed FLOAT64 cartesian actions — what the reference's own loops hand it: NumPy float64 arrays built on the
 * host (test_sac_multi.py:77-80, run.py:13), which `UAVAgent.step` consumes in float64 (uav_agent.py:26; uav_world_2d.py:142).
 * action: double [B][N][2] ([B][2] for the single world).  Serves both kinds (distance: single world only, nullable;
 * evaluate: multi world only).  Bit-exact for actions that float32 cannot hold.  Same kernels as the float32 entry points
 * (the warp kernel up to 32 UAVs per env, the general kernel beyond and in the float64 world); no action mapping: the
 * policy-space modes exist for float32 device policies. */
int uavca_step_f64(uavca_handle* h, void* state, const double* action, int evaluate, float* obs, float* reward, uint8_t* done,
                   float* distance, float* final_obs, uint8_t* reset_mask, void* stream);

/* The gym call as the reference makes it — `obs, reward, done, info = env.step(action)` returns values (multi_uav_world_2d.py:241,
 * uav_world_2d.py:173): one of the three steps above (action: float [B][N][2], or double when action_is_f64) followed by a
 * wait for `stream`, in ONE call.  With obs / reward / done / distance in mapped pinned host memory the results are readable
 * when it returns; this is what the B=1 drop-in classes call once per step (compat.py). */
int uavca_step_sync(uavca_handle* h, void* state, const void* action, int action_is_f64, int action_mode, int evaluate, float* obs,
                    float* reward, uint8_t* done, float* distance, float* final_obs, uint8_t* reset_mask, void* stream);

/* The caller-side action mapping on its own: in/out float [B][N][2]. */
int uavca_map_action(uavca_handle* h, const float* in, int action_mode, float* out, void* stream);

/* out8 (device int64[8]): episodes finished, reach, collisions, steps over finished episodes; then the
 * same three counters summed over the episodes in flight (reach, collisions, steps) and B.  The score sums and the
 * non-finite counter are read from the `stats` field of the state blob directly (see uavca_layout). */
int uavca_stats(uavca_handle* h, const void* state, int64_t* out8, void* stream);

/* End-to-end form with HOST buffers; ordered after the work already queued on `stream`, returns when the
 * outputs are in host memory.  `state` stays on the device.  Pinned (page-locked) buffers take the zero-copy
 * path: one launch on `stream` whose loads/stores go through PCIe directly (mapped host memory); outputs of
 * 256 MB and more leave by DMA instead (chunked pipeline).  Pageable buffers are staged: H2D actions, step,
 * D2H obs/reward/done, pipelined in chunks over internal streams forked from `stream`.  Works for both kinds
 * (obs_dim from the config). */
int uavca_step_host(uavca_handle* h, void* state, const float* host_action, int action_mode, int evaluate,
                    float* host_obs, float* host_reward, uint8_t* host_done, void* stream);

/* K consecutive steps in ONE launch (the loops of run.py:10-16 / run_multi.py:10-16).  The state stays in
 * registers for the K steps; per-step outputs are [K][...] blocks:
 *   obs float [K][B][N][obs_dim]; reward float [K][B][N]; done uint8 [K][B][N];
 *   final_obs (nullable) like obs; reset_mask (nullable) uint8 [K][B]; distance (nullable, single world) float [K][B].
 * Actions: action_block float [K][B][N][2] in `action_mode`, or NULL — then every UAV draws uniform policy-space
 * actions in [-1,1)^2 from Philox4x32-10 keyed by (action_seed, global env index, UAV, step0 + k) and mapped by
 * `action_mode` (UAVCA_ACTION_CARTESIAN then means a * max_speed: action_space.sample()); action_out (nullable)
 * float [K][B][N][2] receives the draws.  Results are bit-identical to K calls of uavca_step_* fed the same actions
 * (uavca_sample_actions reproduces the draws of one step).  K > 1 needs B*N*obs_dim*4 to be a multiple of 16.  The float64
 * world and envs of more than 32 UAVs run on the general kernel, which has no K loop: same call, same results, K launches. */
int uavca_rollout(uavca_handle* h, void* state, int32_t K, const float* action_block, int action_mode, int evaluate,
                  uint64_t action_seed, uint64_t step0, float* obs, float* reward, uint8_t* done, float* action_out,
                  float* final_obs, uint8_t* reset_mask, float* distance, void* stream);

/* out float [B][N][2]: the policy-space actions uavca_rollout draws at global step `step`. */
int uavca_sample_actions(uavca_handle* h, uint64_t action_seed, uint64_t step, float* out, void* stream);

/* Device-resident replay ring, the hand-off to the learner side ("next" row; replaces ReplayMemory.push,
 * pytorch_sac_temp/replay_memory.py:15-19, and ReplayBuffer.append, pytorch_ddpg/buffer_tensor.py:40-59).
 * Appends M transitions at ring slot `head`, wrapping at `capacity`, in one launch:
 *   obs, next_obs float [M][obs_dim]; action float [M][act_dim]; reward float [M]; done uint8 [M]
 *   ring_* float [capacity][...]; ring_mask[slot] = 1 - done  (mask = float(not done), test_sac_multi.py:101-103)
 * No handle: the ring belongs to the caller.  M <= capacity. */
int uavca_replay_push(const float* obs, const float* action, const float* reward, const float* next_obs,
                      const uint8_t* done, int64_t M, int32_t obs_dim, int32_t act_dim, float* ring_obs,
                      float* ring_action, float* ring_reward, float* ring_next_obs, float* ring_mask,
                      int64_t capacity, int64_t head, void* stream);

/* The same append with the ring head kept ON THE DEVICE: ring_meta int64[4] (device, zero-initialised by the caller)
 * holds [0] the slot the next append starts at, [1] scratch, [2] the number of transitions held (<= capacity), [3] the
 * number of appends so far (a per-step device counter, e.g. the `counter_dev` of uavca_policy_act).  The
 * call reads the head from ring_meta and advances it itself, so a CUDA-graph replay of an acting step appends where
 * the previous replay stopped. */
int uavca_replay_push_dev(const float* obs, const float* action, const float* reward, const float* next_obs,
                          const uint8_t* done, int64_t M, int32_t obs_dim, int32_t act_dim, float* ring_obs,
                          float* ring_action, float* ring_reward, float* ring_next_obs, float* ring_mask,
                          int64_t capacity, int64_t* ring_meta, void* stream);

/* Draw `batch` transitions from the ring and gather the five arrays in ONE launch ("next" row; replaces ReplayMemory.sample,
 * pytorch_sac_temp/replay_memory.py:21-24, and ReplayBuffer.get_batch, pytorch_ddpg/buffer_tensor.py:65-90).  Head and fill
 * level are read from ring_meta on the device; the slots come from word 0 (x) of the Philox4x32-10 block with key seed and
 * counter (j, ctr, 5 << 16 | j >> 32, ctr >> 32) for sample j and ctr = draw + appends so far (ring_meta[3]), uniformly over
 * the filled slots with replacement ((x * size) >> 32) or, with recency_weighted != 0, with probability rising linearly
 * with recency (the `unbalance_p` scheme of buffer_tensor.py:78-87: age = floor(sqrt((x + 0.5) / 2^32) * size), at most
 * size - 1, counted from the oldest slot).  The tag 5 in counter word 2 keeps the stream apart from every other Philox
 * stream of the library (env resets 0..2, rollout actions 3, policy noise 4) whatever the seeds.  No host synchronisation: safe inside a
 * CUDA graph of a learner step.  out_*: float [batch][obs_dim] / [batch][act_dim] / [batch]; out_index (nullable) int64
 * [batch] receives the slots.  An empty ring yields slot 0. */
int uavca_replay_sample(const float* ring_obs, const float* ring_action, const float* ring_reward, const float* ring_next_obs,
                        const float* ring_mask, int64_t capacity, int32_t obs_dim, int32_t act_dim, const int64_t* ring_meta,
                        int64_t batch, uint64_t seed, uint64_t draw, int recency_weighted, float* out_obs, float* out_action,
                        float* out_reward, float* out_next_obs, float* out_mask, int64_t* out_index, void* stream);

/* uavca_step_multi with the replay append folded into the SAME launch ("next" row; MultiUAVWorld2D.step followed by the N
 * memory.push calls of test_sac_multi.py:99-103).  Besides everything uavca_step_multi writes, UAV m's transition goes to
 * ring slot (head + m) mod capacity:
 *   ring_obs[slot]      = prev_obs[m]   (prev_obs float [B][N][10]: the observation `action` was taken on; not `obs`)
 *   ring_action[slot]   = action[m]     (as handed in, i.e. the policy-space action when action_mode maps it)
 *   ring_reward[slot]   = reward[m];  ring_next_obs[slot] = the step's own next observation (before any auto-reset);
 *   ring_mask[slot]     = 1 - done[m]
 * with the head in ring_meta (device int64[4], exactly as uavca_replay_push_dev keeps it: the two calls can be mixed on
 * one ring).  Result identical to uavca_step_multi + uavca_replay_push_dev; one pass over the transitions less.
 * Warp kernels only: num_agents <= 32 and not the float64 world (-2 otherwise: use the two calls); capacity * 10 < 2^31. */
int uavca_step_multi_replay(uavca_handle* h, void* state, const float* action, int action_mode, int evaluate,
                            const float* prev_obs, float* obs, float* reward, uint8_t* done, float* final_obs,
                            uint8_t* reset_mask, float* ring_obs, float* ring_action, float* ring_reward, float* ring_next_obs,
                            float* ring_mask, int64_t capacity, int64_t* ring_meta, void* stream);

/* Fused acting path of the shared SAC policy ("next" row; replaces the per-UAV SAC.select_action round trips,
 * pytorch_sac_temp/sac.py:38-44, with GaussianPolicy.forward/sample, pytorch_sac_temp/model.py:74-101, for all
 * M = B*N observations in one tcgen05 kernel).  Fixed architecture 10 -> 256 -> 256 -> (2 + 2); all weight
 * operands fp16, K-major, biases carried as an extra input column:
 *   obs float [M][10];
 *   w1  fp16 [256][16]  : linear1.weight in columns 0..9, linear1.bias in column 10, zeros elsewhere;
 *   w2  fp16 [256][256] : linear2.weight;            w2b fp16 [256][16] : linear2.bias in column 0, zeros;
 *   w3  fp16 [16][256]  : rows 0,1 mean_linear.weight, rows 2,3 log_std_linear.weight, zeros;
 *   w3b fp16 [16][16]   : mean_linear.bias, log_std_linear.bias in column 0 of rows 0..3, zeros;
 *   noise float [M][2] standard-normal draws or NULL: then Box-Muller on the Philox4x32-10 block with key seed and
 *   counter (row, ctr, 4 << 16 | row >> 32, ctr >> 32), ctr = counter + *counter_dev (tag 4: no other Philox stream of
 *   the library can produce that counter); counter_dev is a nullable DEVICE uint64 the caller advances between calls,
 *   which keeps a CUDA-graph replay of the call from repeating its noise;
 *   action float [M][2] = tanh(mean + exp(clamp(log_std, -20, 2)) * noise);  head (nullable) float [M][4] = mean, log_std.
 * No handle: weights and buffers belong to the caller. */
int uavca_policy_act(const float* obs, int64_t M, const void* w1, const void* w2, const void* w2b, const void* w3,
                     const void* w3b, const float* noise, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                     float* action, float* head, void* stream);

/* Launch bookkeeping: number of kernels this handle has launched so far. */
int64_t uavca_launch_count(const uavca_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* UAVCA_H_ */

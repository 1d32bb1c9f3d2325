// uavca_host.h — host-side declarations shared by the kernel translation unit and the C-ABI.
#pragma once

#include <cuda_runtime.h>

#include "uavca_device.cuh"

namespace uavca {

// One kernel per call when B > 0.  cta_pack: envs of 11 and 17..25 UAVs run on the CTA-packed kernel (uavca_cta.cuh);
// false keeps them on the one-env-per-warp kernel.
cudaError_t launch_step_multi(const KernelArgs& a, cudaStream_t st, bool cta_pack);
cudaError_t launch_step_multi_ring(const KernelArgs& a, const RingSink& g, cudaStream_t st);
cudaError_t launch_rollout_multi(const KernelArgs& a, const RolloutArgs& r, cudaStream_t st);
cudaError_t launch_rollout_single(const KernelArgs& a, const RolloutArgs& r, cudaStream_t st);
cudaError_t launch_sample_actions(const Consts& c, float* out, int B, int N, unsigned long long seed, unsigned long long t,
                                  cudaStream_t st);
cudaError_t launch_reset_multi(const KernelArgs& a, const uint8_t* mask, cudaStream_t st);
cudaError_t launch_observe_multi(const KernelArgs& a, cudaStream_t st);
cudaError_t launch_step_single(const KernelArgs& a, cudaStream_t st);
cudaError_t launch_reset_single(const KernelArgs& a, const uint8_t* mask, cudaStream_t st);
cudaError_t launch_observe_single(const KernelArgs& a, cudaStream_t st);
cudaError_t launch_map_action(const Consts& c, const float* in, float* out, long long M, int mode, cudaStream_t st);
cudaError_t launch_stats(const StateView& s, int B, long long* out8, cudaStream_t st);
cudaError_t launch_replay_push(const float* obs, const float* action, const float* reward, const float* next_obs,
                               const uint8_t* done, long long M, int obs_dim, int act_dim, float* r_obs, float* r_act,
                               float* r_rew, float* r_next, float* r_mask, long long capacity, long long head,
                               long long* meta, cudaStream_t st);

cudaError_t launch_replay_sample(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                                 const float* r_mask, long long capacity, int obs_dim, int act_dim, const long long* meta,
                                 long long batch, unsigned long long seed, unsigned long long draw, int recency, float* o_obs,
                                 float* o_act, float* o_rew, float* o_nxt, float* o_mask, long long* o_idx, cudaStream_t st);
// n-step returns (uavca_nstep.cuh): the slots of launch_replay_sample / launch_per_sample, then the n-step gather
cudaError_t launch_replay_sample_nstep(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                                       const float* r_mask, long long capacity, int obs_dim, int act_dim, const long long* meta,
                                       long long batch, unsigned long long seed, unsigned long long draw, int recency,
                                       long long stride, int n, double gamma, float* o_obs, float* o_act, float* o_rew,
                                       float* o_nxt, float* o_disc, long long* o_idx, cudaStream_t st);

// Prioritized replay (uavca_per.cu): the sum-tree over the ring's slots.
cudaError_t launch_per_sync(double* tree, long long L, long long* per_meta, const long long* ring_meta, long long capacity,
                            cudaStream_t st);
cudaError_t launch_per_update(double* tree, long long L, long long capacity, long long* per_meta, const long long* index,
                              const double* priority, long long n, cudaStream_t st);
cudaError_t launch_per_sample(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                              const float* r_mask, int obs_dim, int act_dim, const long long* ring_meta, double* tree,
                              long long L, long long batch, double beta, unsigned long long seed, unsigned long long draw,
                              float* o_obs, float* o_act, float* o_rew, float* o_nxt, float* o_mask, long long* o_idx,
                              float* o_w, cudaStream_t st);
cudaError_t launch_per_sample_nstep(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                                    const float* r_mask, long long capacity, int obs_dim, int act_dim,
                                    const long long* ring_meta, double* tree, long long L, long long batch, double beta,
                                    long long stride, int n, double gamma, unsigned long long seed, unsigned long long draw,
                                    float* o_obs, float* o_act, float* o_rew, float* o_nxt, float* o_disc, long long* o_idx,
                                    float* o_w, cudaStream_t st);

cudaError_t launch_policy_act(const float* obs, long long M, const void* w1, const void* w2, const void* w2b, const void* w3,
                              const void* w3b, const float* noise, unsigned long long seed, unsigned long long counter,
                              const unsigned long long* counter_dev, float* action, float* head, cudaStream_t st);

// Shift a view to the sub-range of envs starting at env0 (stats stay shared).
inline StateView offset_view(const StateView& v, long long env0, int N) {
  StateView o = v;
  const long long m0 = env0 * N;
  o.pos += m0; o.vel += m0; o.tgt += m0; o.init += m0; o.prev += m0; o.flags += m0;
  o.steps += env0; o.reach += env0; o.coll += env0; o.episode += env0; o.score += env0;
  if (o.pos64) { o.pos64 += m0; o.tgt64 += m0; o.init64 += m0; o.prev64 += m0; }
  return o;
}

}  // namespace uavca

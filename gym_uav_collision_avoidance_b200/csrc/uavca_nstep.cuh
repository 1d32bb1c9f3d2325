// uavca_nstep.cuh — the n-step gather shared by the uniform / recency sampler (replay_sample_nstep_kernel,
// uavca_kernels.cu) and the prioritized one (per_sample_kernel<true>, uavca_per.cu).  The rule is the contract of
// uavca_replay_sample_nstep in include/uavca.h; this is its one device statement.
#pragma once

#include "uavca_device.cuh"

namespace uavca {

constexpr int kNstepLanes = 16;  // lanes per sample in both samplers: lane i checks link i, so n <= 16

// The 16 lanes of sample j (lane g of the group, `mask` the group's shuffle mask) hold the drawn slot s = s_0.  Writes
// state = obs[s], action = act[s], reward = R, next_state = nxt[s_{k-1}] and discount, as the contract defines them.
//   age(s) = (head - 1 - s) mod cap; s_i = (s + i * stride) mod cap, with i * stride <= age(s) < cap for every successor
//   read, so one subtraction of cap wraps it.  Link i (1 <= i < n): mask[s_{i-1}] != 0, i * stride <= age(s), and
//   obs[s_i] equals nxt[s_{i-1}] bit for bit.  k = 1 + the links that hold consecutively from i = 1 (a 16-lane ballot).
__device__ __forceinline__ void nstep_gather(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                                             const float* r_mask, int od, int ad, long long cap, long long head,
                                             long long stride, int n, double gamma, long long slot, long long j, int g,
                                             unsigned mask, float* o_obs, float* o_act, float* o_rew, float* o_nxt,
                                             float* o_disc) {
  long long age = head - 1 - slot;
  age += age < 0 ? cap : 0;
  const long long step = (long long)g * stride;
  const bool present = g < n && step <= age;  // lane 0 always: age >= 0
  long long si = slot + step;
  si -= si >= cap ? cap : 0;
  float m = 0.0f, r = 0.0f;
  if (present) {
    m = r_mask[si];
    r = r_rew[si];
  }
  const float mprev = __shfl_up_sync(mask, m, 1, kNstepLanes);
  bool link = false;
  if (g > 0 && present && mprev != 0.0f) {
    long long sp = si - stride;
    sp += sp < 0 ? cap : 0;
    const float* a = r_obs + si * od;
    const float* b = r_nxt + sp * od;
    link = true;
    for (int k = 0; k < od; ++k) link &= __float_as_uint(a[k]) == __float_as_uint(b[k]);  // bits: -0.0 != 0.0
  }
  const unsigned bits = (__ballot_sync(mask, link) >> (threadIdx.x & 16)) & 0xFFFFu;
  const int kk = __ffs(~(bits >> 1));  // 1 + the links that hold consecutively from link 1
  // R = sum_{i<k} gamma^i r_i in float64, sequential and unfused; every lane folds the same shuffled rewards
  double R = 0.0, gg = 1.0;
  for (int i = 0; i < kk; ++i) {
    const float ri = __shfl_sync(mask, r, i, kNstepLanes);
    R = __dadd_rn(R, __dmul_rn(gg, (double)ri));
    gg = __dmul_rn(gg, gamma);
  }
  const float mlast = __shfl_sync(mask, m, kk - 1, kNstepLanes);
  const long long slast = __shfl_sync(mask, si, kk - 1, kNstepLanes);
  for (int k = g; k < od; k += kNstepLanes) {
    o_obs[j * od + k] = r_obs[slot * od + k];
    o_nxt[j * od + k] = r_nxt[slast * od + k];
  }
  for (int k = g; k < ad; k += kNstepLanes) o_act[j * ad + k] = r_act[slot * ad + k];
  if (g == 0) {
    o_rew[j] = __double2float_rn(R);
    o_disc[j] = mlast != 0.0f ? __double2float_rn(gg) : 0.0f;
  }
}

}  // namespace uavca

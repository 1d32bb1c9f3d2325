// uavca_device.cuh — device-side building blocks of the batched env step (sm_100a).
//
// Numerics contract (DESIGN.md §3): everything that feeds a comparison in the reference — velocity (float64),
// position (float32, one rounding of a float64 sum), float32 distances formed as sqrt(x*x + y*y) without
// fusion — is reproduced with explicit round-to-nearest intrinsics so that nvcc's FMA contraction cannot
// change a bit.  Quantities that are outputs only (reward, observation features) are computed to well inside
// the 1e-5 relative tolerance with cheaper single-precision transcendental code.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/uavca.h"

namespace uavca {

#ifndef UAVCA_WPB
#define UAVCA_WPB 4
#endif
#ifndef UAVCA_MINB
#define UAVCA_MINB 8
#endif
constexpr int kWarpsPerBlock = UAVCA_WPB;
constexpr int kThreads = kWarpsPerBlock * 32;
constexpr int kMinBlocksPerSM = UAVCA_MINB;  // step kernel: caps registers per thread (8 warps x 4 blocks -> 64 regs, 32 warps/SM)
constexpr unsigned kFull = 0xffffffffu;
constexpr unsigned kMaxResetAttempts = 4096u;  // the reference would loop forever in an over-crowded box

// Philox4x32-10 streams.  Every key is a seed the caller picks, so the streams are kept apart by their counters alone:
// each consumer puts its own tag in the upper half of counter word 2 (philox4x32_10 / philox_indexed below).
//   reset    (env, episode, stream << 16 | uav, attempt)         stream 0..2, uav < 2^16
//   actions  (env, t >> 1, 3 << 16 | uav, t >> 33)                uav < 2^16
//   policy   (row, ctr, 4 << 16 | row >> 32, ctr >> 32)          row < 2^48     (uavca_policy.cu)
//   sampler  (sample, ctr, 5 << 16 | sample >> 32, ctr >> 32)    sample < 2^48  (replay_sample_kernel)
//   per      (sample, ctr, 6 << 16 | sample >> 32, ctr >> 32)    sample < 2^48  (per_sample_kernel, uavca_per.cu)
// The n-step samplers (replay_sample_nstep_kernel, per_sample_kernel<true>) draw on the streams 5 and 6 of their one-step
// siblings through the same draw code, so the same (seed, draw, appends) gives the same slots: no stream of their own.
enum : int { kStreamPos = 0, kStreamTgt = 1, kStreamVel = 2, kStreamAct = 3, kStreamPolicy = 4, kStreamSample = 5,
             kStreamPerSample = 6 };

// Constants derived once on the host from uavca_config (capi.cu: derive_consts).
struct Consts {
  // float64 kinematics (uav_agent.py:26-29)
  double tau, inv_tau, amax, vmax;
  double clip_x;        // least x >= 0 with fl(x / tau) >= amax: beyond it the acceleration clip decides
  double vm2, inv_vm2;  // ||(vmax, vmax)|| as np.linalg.norm computes it, and its reciprocal
  double lox, hix, loy, hiy;  // box (float64 compare, multi_uav_world_2d.py:213,224)
  double reach_speed_sq;      // least s with sqrt(s) >= reach_speed: ||v|| < reach_speed  <=>  s < this
  double two_r_d, two_h_d, dsense_d, reach_dist_d, inv_diag_d;  // float64 world (uavca_seq.cuh): thresholds as python floats
  // float32 thresholds (python scalars are weak against float32 norms under NumPy 2)
  float two_r, two_h, dsense, reach_dist;
  // the same thresholds in squared-distance space (sqrt is monotone, so the flags stay bit-exact without a sqrt):
  //   d <= 2r  <=>  s <= s_two_r_le ;  d <= 2h  <=>  s <= s_two_h_le ;  d < d_sense  <=>  s < s_dsense_lt
  float s_two_r_le, s_two_h_le, s_dsense_lt;
  // soft / hard collision of the nearest neighbour, sensing range folded in: d < d_sense and d <= 2r  <=>  s <= s_coll_le
  float s_coll_le, s_hard_le;
  float s_reach_lt;  // dist < reach_distance  <=>  s < s_reach_lt
  // box as float32 bounds with identical compare results: float64(p) >= lo  <=>  p >= lox_f, ...
  float lox_f, hix_f, loy_f, hiy_f;
  float vm2_floor_f;  // greatest float32 <= vm2: float64(init) <= vm2  <=>  init <= vm2_floor_f
  float vm2_f, inv_dsense;
  float inv_diag, inv_vm2_f, inv_vmax_f, inv_pi;
  float polar_scale, vmax_f, tau_f;
  // episode control
  int reset_mode, max_steps, reset_source, circular, single_f32_first_step, track_scores;
  unsigned rs_any_mask, rs_all_off;  // reset_mode as masks over an env's done bits (step_core)
  int steps_limit;                   // max_steps, or INT_MAX when there is no limit
  int key_mask;                      // ~31: distance-bits mask of the neighbour keys (pair_scan)
  int near_key;                      // greatest key of a neighbour that may be within collision reach of pass A (neighbours())
  unsigned seed_lo, seed_hi;
  long long env_base;
};

// Structure-of-arrays state of one shard (pointers into the caller's blob).
struct StateView {
  float2* pos;
  double2* vel;
  float2* tgt;
  float* init;
  float* prev;
  uint8_t* flags;
  int* steps;
  int* reach;
  int* coll;
  unsigned* episode;
  double2* score;  // per env: (sum of rewards[0], sum_i rewards[i] * (1 - dones[i])) of the episode in flight
  double2 *pos64, *tgt64;  // float64 world (config.circular): the reference keeps float64 locations after reset(circular=True)
  double *init64, *prev64;
  unsigned long long* stats;
};

struct StepIO {
  const float2* action;
  const double2* action64;  // nullable: float64 cartesian actions (uavca_step_f64) instead of `action`
  float* obs;
  float* reward;
  uint8_t* done;
  float* final_obs;     // nullable
  uint8_t* reset_mask;  // nullable
  float* distance;      // nullable (single world)
  int action_mode;
  int evaluate;
};

struct KernelArgs {
  Consts c;
  StateView s;
  StateView pool;  // reset pool (pos == nullptr when absent)
  int pool_envs;
  const double4* ring64;  // reset(circular=True): per UAV (pos.x, pos.y, tgt.x, tgt.y), float64, computed with the host libm
  StepIO io;
  int B, N;
};

// K steps in one launch (uavca_rollout): per-step outputs are [K][...] blocks, actions come from a [K][M][2] block or
// from the counter-based Philox stream (run.py:10-16 / run_multi.py:10-16: env.step(env.action_space.sample())).
struct RolloutArgs {
  int K;
  const float2* action_block;  // [K][M] or nullptr: Philox actions
  float2* action_out;          // nullable [K][M]: the actions taken (policy space, before the action mapping)
  unsigned seed_lo, seed_hi;   // Philox key of the action stream
  unsigned long long step0;    // global index of step k = 0 (Philox counter word; the caller advances it by K)
  long long M;                 // B * N of this launch (stride of one step in the blocks)
  int B;
  unsigned KM;                 // K * M: end of the plain instances' 32-bit step offsets (set by launch_rollout_multi)
};

// Device replay ring fed straight from the step kernel (uavca_step_multi_replay): the step that produced a transition
// also appends it — (observation acted on, policy-space action, reward, the step's own next observation, 1 - done) as
// the training loop stores it (test_sac_multi.py:101-103).  Row indices are 32-bit: capacity * 10 < 2^31 is checked on
// the host.  meta (device int64[4]): ring head, block ticket, transitions held, appends so far (as uavca_replay_push_dev).
struct RingSink {
  const float2* prev_obs;  // [M][5]: the observation the action was taken on
  float2* obs;             // [capacity][5]
  float2* act;             // [capacity]
  float* rew;              // [capacity]
  float2* nxt;             // [capacity][5]
  float* mask;             // [capacity]
  long long* meta;
  int cap;
  int M;
};

// ---- exact float32 / float64 primitives ------------------------------------------------------------------

// squared float32 norm the way np.linalg.norm forms it: products and sum rounded separately (never fused)
__device__ __forceinline__ float sq32(float dx, float dy) {
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}
__device__ __forceinline__ float n32(float dx, float dy) { return __fsqrt_rn(sq32(dx, dy)); }

// squared float64 norm as the ddot kernel forms it: second product fused
__device__ __forceinline__ double sq64(double x, double y) { return fma(y, y, __dmul_rn(x, x)); }

__device__ __forceinline__ double clipd(double v, double lo, double hi) {
  // np.clip: NaN propagates (both comparisons are false)
  v = (v < lo) ? lo : v;
  v = (v > hi) ? hi : v;
  return v;
}

// Correctly rounded x / tau from the reciprocal and two FMA residual corrections (Markstein): after the first
// correction the quotient is faithful, after the second it is the round-to-nearest quotient.  Bit-identical
// to IEEE division for every finite x in the unclipped range; 5 DP instructions instead of ~25.
__device__ __forceinline__ double div_tau(double x, const Consts& c) {
  double q0 = __dmul_rn(x, c.inv_tau);
  double r0 = fma(-q0, c.tau, x);
  double q1 = fma(r0, c.inv_tau, q0);
  double r1 = fma(-q1, c.tau, x);
  return fma(r1, c.inv_tau, q1);
}

// dv = clip((a - v) / tau, -amax, amax)            (uav_agent.py:26)
__device__ __forceinline__ double accel(double a, double v, const Consts& c) {
  double x = __dsub_rn(a, v);
  double q = div_tau(x, c);
  // |x| >= clip_x  <=>  |fl(x/tau)| >= amax: the clip decides and the quotient (possibly inf/NaN for huge x) is unused
  q = (x >= c.clip_x) ? c.amax : q;
  q = (x <= -c.clip_x) ? -c.amax : q;
  return q;
}

// One UAV kinematic update: v = clip(v + dv*tau, +-vmax); p = float32(float64(p) + v*tau)   (uav_agent.py:27-29)
__device__ __forceinline__ void integrate(double ax, double ay, double& vx, double& vy, float& px, float& py,
                                          const Consts& c) {
  double dvx = accel(ax, vx, c), dvy = accel(ay, vy, c);
  vx = clipd(__dadd_rn(vx, __dmul_rn(dvx, c.tau)), -c.vmax, c.vmax);
  vy = clipd(__dadd_rn(vy, __dmul_rn(dvy, c.tau)), -c.vmax, c.vmax);
  px = __double2float_rn(__dadd_rn((double)px, __dmul_rn(vx, c.tau)));
  py = __double2float_rn(__dadd_rn((double)py, __dmul_rn(vy, c.tau)));
}

// atan2 for finite inputs whose larger magnitude is 0 or >= ~1e-30, branch-free: octant reduction, one approximate division and a degree-8 minimax
// polynomial in t^2 (fit in this repo; max relative error 1.2e-7 evaluated in float32, ~4e-7 with the division).
// Relative accuracy holds down to tiny angles (P(0) = 1 exactly).  atan2(0, 0) = 0 as in libm.
__device__ __forceinline__ float fast_atan2(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  const float t = __fdividef(mn, mx + 1e-37f);  // the tiny bias makes atan2(0, 0) = 0 without a select
  const float s = t * t;
  float p = 0.0029206890612840652f;
  p = fmaf(p, s, -0.016367916017770767f);
  p = fmaf(p, s, 0.04321184381842613f);
  p = fmaf(p, s, -0.07552213221788406f);
  p = fmaf(p, s, 0.10666003823280334f);
  p = fmaf(p, s, -0.14211055636405945f);
  p = fmaf(p, s, 0.19993773102760315f);
  p = fmaf(p, s, -0.33333152532577515f);
  p = fmaf(p, s, 1.0f);
  float r = t * p;
  r = (ay > ax) ? (1.57079637050628662f - r) : r;
  r = (x < 0.0f) ? (3.14159274101257324f - r) : r;
  return copysignf(r, y);
}

// Two atan2 at once: the polynomial runs on Blackwell's packed FP32 pipe (FMUL2/FFMA2, two lanes per instruction);
// octant reduction and fix-up stay scalar.  Same arithmetic per element as fast_atan2.  The coefficients are literals:
// FFMA2 takes a 32-bit immediate for both lanes, where a __constant__ table costs an LDC per coefficient and call.
__device__ __forceinline__ float2 fast_atan2_pair(float y0, float x0, float y1, float x1) {
  const float ax0 = fabsf(x0), ay0 = fabsf(y0), ax1 = fabsf(x1), ay1 = fabsf(y1);
  const float mx0 = fmaxf(ax0, ay0), mn0 = fminf(ax0, ay0), mx1 = fmaxf(ax1, ay1), mn1 = fminf(ax1, ay1);
  const float2 t = make_float2(__fdividef(mn0, mx0 + 1e-37f), __fdividef(mn1, mx1 + 1e-37f));
  const float2 s = __fmul2_rn(t, t);
  auto both = [](float v) { return make_float2(v, v); };
  float2 p = both(0.0029206890612840652f);
  p = __ffma2_rn(p, s, both(-0.016367916017770767f));
  p = __ffma2_rn(p, s, both(0.04321184381842613f));
  p = __ffma2_rn(p, s, both(-0.07552213221788406f));
  p = __ffma2_rn(p, s, both(0.10666003823280334f));
  p = __ffma2_rn(p, s, both(-0.14211055636405945f));
  p = __ffma2_rn(p, s, both(0.19993773102760315f));
  p = __ffma2_rn(p, s, both(-0.33333152532577515f));
  p = __ffma2_rn(p, s, both(1.0f));
  float2 r = __fmul2_rn(t, p);
  r.x = (ay0 > ax0) ? (1.57079637050628662f - r.x) : r.x;
  r.y = (ay1 > ax1) ? (1.57079637050628662f - r.y) : r.y;
  r.x = (x0 < 0.0f) ? (3.14159274101257324f - r.x) : r.x;
  r.y = (x1 < 0.0f) ? (3.14159274101257324f - r.y) : r.y;
  return make_float2(copysignf(r.x, y0), copysignf(r.y, y1));
}

// difference of two angles given in units of pi, wrapped to [-1, 1]
__device__ __forceinline__ float wrap_units(float d) {
  // d - 2*rint(d/2) with rint done by the 1.5*2^23 magic constant: three FMA-pipe instructions, no compare/select
  const float k = __fadd_rn(__fmaf_rn(d, 0.5f, 12582912.0f), -12582912.0f);
  return __fmaf_rn(k, -2.0f, d);
}
__device__ __forceinline__ float2 wrap_units2(float2 d) {
  const float2 m = make_float2(12582912.0f, 12582912.0f);
  const float2 k = __fadd2_rn(__ffma2_rn(d, make_float2(0.5f, 0.5f), m), make_float2(-12582912.0f, -12582912.0f));
  return __ffma2_rn(k, make_float2(-2.0f, -2.0f), d);
}

// Output-only square root / reciprocal (observation features, reward): flush-to-zero MUFU forms, no denormal fix-up.
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// sin and cos of |x| <= ~1e4 (here |x| <= pi): Cody-Waite reduction by pi/2 in three FMA steps and the usual
// minimax polynomials on [-pi/4, pi/4]; ~1.5 ulp.  Unlike sincosf() there is no huge-argument path, hence no
// local-memory frame in the kernels that inline it.
__device__ __forceinline__ void sincos_bounded(float x, float& sn, float& cs) {
  const float k = rintf(x * 0.636619747f);
  float r = fmaf(k, -1.57079601e+00f, x);
  r = fmaf(k, -3.13916473e-07f, r);
  r = fmaf(k, -5.39030253e-15f, r);
  const int q = (int)k;
  const float s = r * r;
  float ps = fmaf(-1.95152959e-4f, s, 8.33307933e-3f);
  ps = fmaf(ps, s, -1.66666597e-1f);
  ps = fmaf(ps * s, r, r);
  float pc = fmaf(2.44331571e-5f, s, -1.38873036e-3f);
  pc = fmaf(pc, s, 4.16666418e-2f);
  pc = fmaf(pc, s, -0.5f);
  pc = fmaf(pc, s, 1.0f);
  const bool swap = (q & 1) != 0;
  float a = swap ? pc : ps, b = swap ? ps : pc;
  sn = (q & 2) ? -a : a;
  cs = ((q + 1) & 2) ? -b : b;
}

// wrap(atan2(dy,dx) - atan2(hy,hx)) as ONE atan2 of the float64 cross/dot products of the two directions
// (relative error ~4e-7 even for tiny angles).  Callers deal with zero / denormal-tiny vectors.
__device__ __forceinline__ float rel_angle(double dx, double dy, double hx, double hy) {
  double cr = fma(hx, dy, -(hy * dx));
  double dt = fma(hx, dx, hy * dy);
  return fast_atan2((float)cr, (float)dt);
}

// libm-grade fallback for the rare degenerate inputs (velocity components below ~1e-30 but not both zero, or a
// UAV sitting exactly on its target): same formulas as the reference, in double.
static __device__ __noinline__ float2 angles_slow(double tdx, double tdy, double vx, double vy) {
  const double th = atan2(vy, vx);
  const double d = atan2(tdy, tdx) - th;
  return make_float2((float)(th * 0.3183098861837907), (float)(atan2(sin(d), cos(d)) * 0.3183098861837907));
}

// Caller-side action mapping (test_sac_multi.py:77-80; test_pytorch_multi.py:80).
__device__ __forceinline__ float2 map_action(float2 a, int mode, const Consts& c) {
  if (mode == UAVCA_ACTION_POLAR) {
    float v = __fmul_rn(__fadd_rn(__fmul_rn(a.x, 0.5f), 0.5f), c.polar_scale);
    float th = __fmul_rn(a.y, 3.14159274101257324f);
    float sn, cs;
    sincos_bounded(th, sn, cs);
    return make_float2(__fmul_rn(v, cs), __fmul_rn(v, sn));
  }
  if (mode == UAVCA_ACTION_SCALED) return make_float2(__fmul_rn(a.x, c.vmax_f), __fmul_rn(a.y, c.vmax_f));
  return a;
}

// ---- Philox4x32-10 -------------------------------------------------------------------------------------------

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
// The block of stream `tag` (kStreamPolicy, kStreamSample) for a 48-bit index and a 64-bit counter.
__device__ __forceinline__ uint4 philox_indexed(int tag, unsigned long long index, unsigned long long ctr, uint32_t k0,
                                                uint32_t k1) {
  return philox4x32_10((uint32_t)index, (uint32_t)ctr, ((uint32_t)tag << 16) | (uint32_t)(index >> 32), (uint32_t)(ctr >> 32),
                       k0, k1);
}

__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return __dmul_rn(__dadd_rn(__dmul_rn((double)(a >> 5), 67108864.0), (double)(b >> 6)), 1.0 / 9007199254740992.0);
}

// float32(np.random.uniform(lo, hi)) per component: lo + (hi-lo)*u, two roundings, then the float32 cast
__device__ __forceinline__ float2 draw_pair(const Consts& c, long long env_global, uint32_t episode, int stream,
                                            int uav, uint32_t attempt, double lox, double hix, double loy,
                                            double hiy) {
  uint4 r = philox4x32_10((uint32_t)env_global, episode, ((uint32_t)stream << 16) | (uint32_t)uav, attempt, c.seed_lo,
                          c.seed_hi);
  double ux = u53(r.x, r.y), uy = u53(r.z, r.w);
  float x = __double2float_rn(__dadd_rn(lox, __dmul_rn(__dsub_rn(hix, lox), ux)));
  float y = __double2float_rn(__dadd_rn(loy, __dmul_rn(__dsub_rn(hiy, loy), uy)));
  return make_float2(x, y);
}

// Uniform random action in [-1, 1)^2 for (global env, UAV, global step t): one Philox call serves steps 2q and 2q+1.
__device__ __forceinline__ uint4 action_words(unsigned seed_lo, unsigned seed_hi, long long env_global, int uav,
                                              unsigned long long t) {
  return philox4x32_10((uint32_t)env_global, (uint32_t)(t >> 1), ((uint32_t)kStreamAct << 16) | (uint32_t)uav,
                       (uint32_t)(t >> 33), seed_lo, seed_hi);
}
__device__ __forceinline__ float2 action_from_words(const uint4& w, unsigned long long t) {
  const uint32_t a = (t & 1ull) ? w.z : w.x, b = (t & 1ull) ? w.w : w.y;
  // 24-bit uniforms in [0, 1): exact in float32, then one FMA to [-1, 1)
  return make_float2(__fmaf_rn((float)(a >> 8), 2.0f / 16777216.0f, -1.0f), __fmaf_rn((float)(b >> 8), 2.0f / 16777216.0f, -1.0f));
}

// ---- streaming loads / stores ----------------------------------------------------------------------------------
// State and I/O are touched exactly once per step: keep them out of L1 (no reuse) but let L2 write-back merge.

template <typename T>
__device__ __forceinline__ T ld_stream(const T* p) {
  return __ldcs(p);
}
template <typename T>
__device__ __forceinline__ void st_stream(T* p, T v) {
  __stcs(p, v);
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(kFull, v, src); }

}  // namespace uavca

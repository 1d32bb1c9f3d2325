// uavca_kernels.cu — sm_100a kernels of the batched UAV collision-avoidance env step and their launchers.
//
//   step_multi_kernel   MultiUAVWorld2D.step      (multi_uav_world_2d.py:177-241, uav_agent.py:23-64), fused with
//                       observation build (:60-109), counters, done logic and in-place auto-reset (:116-175)
//   step_single_kernel  UAVWorld2D.step/reset     (uav_world_2d.py:137-173, 119-135)
//   reset_*/observe_*   standalone reset() and _get_obs()
//
// One pass over HBM per step: every state field and every output is read/written exactly once with coalesced,
// streaming accesses; neighbour interaction stays on chip (per-warp shared-memory ring, uavca_multi.cuh).  No tensor
// cores: there is no dense contraction anywhere in the step.  (The fused policy kernel, which is GEMM-shaped, lives
// in uavca_policy.cu.)
#include <atomic>
#include <cmath>
#include <cstdlib>

#include "uavca_host.h"
#include "uavca_multi.cuh"
#include "uavca_seq.cuh"
#include "uavca_cta.cuh"
#include "uavca_tma.cuh"

namespace uavca {

// ================================================================================================================
// Multi-UAV world
// ================================================================================================================

// I/O policy of step_core for per-lane streaming global accesses (ragged tails, unaligned tensors, any N).
struct GlobalIO {
  const KernelArgs& a;
  const Lane& L;
  float* stage;  // per-warp staging of the observation rows
  __device__ __forceinline__ Uav load_uav() const { return uavca::load_uav(a.s, L); }
  __device__ __forceinline__ float2 load_action() const {
    return L.valid ? ld_stream(a.io.action + L.m) : make_float2(0.f, 0.f);
  }
  __device__ __forceinline__ int load_steps() const { return L.valid ? a.s.steps[L.env] : 0; }
  // Programmatic dependent launch: every input is in registers, the next kernel of the stream may start launching
  __device__ __forceinline__ void loads_done() const { cudaTriggerProgrammaticLaunchCompletion(); }
  __device__ __forceinline__ void store_reward_done(float r, bool done) const {
    if (L.valid) {
      st_stream(a.io.reward + L.m, r);
      st_stream(a.io.done + L.m, (uint8_t)done);
    }
  }
  __device__ __forceinline__ bool wants_final() const { return a.io.final_obs != nullptr; }
  __device__ __forceinline__ void put_own(float2 o01, float2 o23) const { stage_own(stage, L.lane, o01, o23); }
  __device__ __forceinline__ void put_neighbours(const ObsTail& n) const { stage_neighbours(stage, L.lane, n); }
  __device__ __forceinline__ void commit(float* g) const {
    __syncwarp();
    flush_rows(stage, g, L);
    __syncwarp();
  }
  __device__ __forceinline__ void commit_obs() const { commit(a.io.obs); }
  __device__ __forceinline__ void commit_final() const { commit(a.io.final_obs); }
  __device__ __forceinline__ void store_state(const Uav& u) const { store_uav(a.s, L, u, false); }
  __device__ __forceinline__ void store_target(const Uav& u) const {
    st_stream(a.s.tgt + L.m, make_float2(u.tx, u.ty));
    st_stream(a.s.init + L.m, u.init);
  }
  __device__ __forceinline__ void store_steps(int v, bool leader) const {
    if (leader) a.s.steps[L.env] = v;
  }
  __device__ __forceinline__ void store_reset(bool rs) const {
    if (a.io.reset_mask) a.io.reset_mask[L.env] = (uint8_t)rs;
  }
};

// The same I/O with FLOAT64 cartesian actions (uavca_step_f64): what the reference's own loops hand env.step().
struct GlobalIO64 : GlobalIO {
  static constexpr bool kAction64 = true;
  __device__ __forceinline__ GlobalIO64(const KernelArgs& a_, const Lane& L_, float* stage_) : GlobalIO{a_, L_, stage_} {}
  __device__ __forceinline__ double2 load_action64() const {
    return L.valid ? ld_stream(a.io.action64 + L.m) : make_double2(0.0, 0.0);
  }
};

template <int NT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSM) step_multi_f64_kernel(const __grid_constant__ KernelArgs a) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  const WarpScratch ws = warp_scratch(smem);
  const int warp_global = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  cudaGridDependencySynchronize();
  const Lane L = make_lane<NT, false>(a.B, a.N, warp_global);
  GlobalIO64 io(a, L, ws.stage);
  step_core<NT>(a, ws, L, io);
}

template <int NT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSM) step_multi_kernel(const __grid_constant__ KernelArgs a) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  const WarpScratch ws = warp_scratch(smem);
  const int warp_global = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int N = NT > 0 ? NT : a.N;
  const bool full = uavs_left(a.B, N, warp_global) >= (32 / N) * N;  // warp-uniform
  // Programmatic dependent launch: this grid may have been scheduled while the previous kernel of the stream was
  // still draining; everything above overlapped with it, nothing below may (it reads memory that kernel wrote).
  cudaGridDependencySynchronize();
  if (full) {  // all warps but the last of a shard: no validity predicates
    const Lane L = make_lane<NT, true>(a.B, a.N, warp_global);
    GlobalIO io{a, L, ws.stage};
    step_core<NT>(a, ws, L, io);
  } else {
    const Lane L = make_lane<NT, false>(a.B, a.N, warp_global);
    GlobalIO io{a, L, ws.stage};
    step_core<NT>(a, ws, L, io);
  }
}


__device__ __forceinline__ void cp_async(void* smem_dst, const void* gsrc, int bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  if (bytes == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
  else if (bytes == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- step + replay append in one launch (uavca_step_multi_replay) ------------------------------------------------
// I/O policy of step_core that, besides GlobalIO's outputs, appends each UAV's transition to a device replay ring:
// the launch that computes (reward, next observation, done) is the one that stores them, so the acting step loses a
// whole pass over the transitions (163,840 x 96 bytes read again and written again) and a launch.  The ring slot of
// UAV m is (head + m) mod capacity with the head read once per thread from ring_meta; the last CTA to finish advances
// it (every CTA read the head before it took its ticket), so a CUDA-graph replay appends where the previous one stopped.
struct RingIO {
  const KernelArgs& a;
  const RingSink& g;
  const Lane& L;
  float* stage;
  float2* prev_stage;  // per warp [160]: the rows of prev_obs, in flight (cp.async) while the step is computed
  int head;
  __device__ __forceinline__ void fetch_prev() const {
    const int n2 = L.valid_lanes * 5;
    const float2* p2 = g.prev_obs + (size_t)L.warp_m0 * 5;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const int k = L.lane + 32 * r;
      if (k < n2) cp_async(prev_stage + k, p2 + k, 8);
    }
  }
  __device__ __forceinline__ int slot() const {
    const int s = head + L.m;
    return s >= g.cap ? s - g.cap : s;
  }
  __device__ __forceinline__ Uav load_uav() const {
    fetch_prev();
    return uavca::load_uav(a.s, L);
  }
  __device__ __forceinline__ float2 load_action() const {
    if (!L.valid) return make_float2(0.f, 0.f);
    const float2 act = ld_stream(a.io.action + L.m);
    st_stream(g.act + slot(), act);  // the policy-space action, before the action mapping (what memory.push receives)
    return act;
  }
  __device__ __forceinline__ int load_steps() const { return L.valid ? a.s.steps[L.env] : 0; }
  __device__ __forceinline__ void loads_done() const { cudaTriggerProgrammaticLaunchCompletion(); }
  __device__ __forceinline__ void store_reward_done(float r, bool done) const {
    if (L.valid) {
      st_stream(a.io.reward + L.m, r);
      st_stream(a.io.done + L.m, (uint8_t)done);
      const int s = slot();
      st_stream(g.rew + s, r);
      st_stream(g.mask + s, done ? 0.0f : 1.0f);  // mask = float(not done)
    }
  }
  __device__ __forceinline__ bool wants_final() const { return true; }
  __device__ __forceinline__ void put_own(float2 o01, float2 o23) const { stage_own(stage, L.lane, o01, o23); }
  __device__ __forceinline__ void put_neighbours(const ObsTail& n) const { stage_neighbours(stage, L.lane, n); }
  __device__ __forceinline__ void commit_obs() const {
    __syncwarp();
    flush_rows(stage, a.io.obs, L);
    __syncwarp();
  }
  // the step's own next observation (before any auto-reset) goes to the ring, and with it the row of the observation
  // the action was taken on: both are runs of valid_lanes * 5 float2 that may wrap at the end of the ring
  __device__ __forceinline__ void commit_final() const {
    __syncwarp();
    const int n2 = L.valid_lanes * 5, cap2 = g.cap * 5;
    const int d0 = (head + L.warp_m0 >= g.cap ? head + L.warp_m0 - g.cap : head + L.warp_m0) * 5;
    const float2* s2 = reinterpret_cast<const float2*>(stage);
    cp_async_wait_all();  // each lane reads back exactly the elements it fetched
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const int k = L.lane + 32 * r;
      if (k < n2) {
        int d = d0 + k;
        d = d >= cap2 ? d - cap2 : d;
        st_stream(g.nxt + d, s2[k]);
        st_stream(g.obs + d, prev_stage[k]);
      }
    }
    if (a.io.final_obs != nullptr) flush_rows(stage, a.io.final_obs, L);
    __syncwarp();
  }
  __device__ __forceinline__ void store_state(const Uav& u) const { store_uav(a.s, L, u, false); }
  __device__ __forceinline__ void store_target(const Uav& u) const {
    st_stream(a.s.tgt + L.m, make_float2(u.tx, u.ty));
    st_stream(a.s.init + L.m, u.init);
  }
  __device__ __forceinline__ void store_steps(int v, bool leader) const {
    if (leader) a.s.steps[L.env] = v;
  }
  __device__ __forceinline__ void store_reset(bool rs) const {
    if (a.io.reset_mask) a.io.reset_mask[L.env] = (uint8_t)rs;
  }
};

template <int NT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSM) step_multi_ring_kernel(const __grid_constant__ KernelArgs a,
                                                                                    const __grid_constant__ RingSink g) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  const WarpScratch ws = warp_scratch(smem);
  const int warp_global = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int N = NT > 0 ? NT : a.N;
  const bool full = uavs_left(a.B, N, warp_global) >= (32 / N) * N;  // warp-uniform
  cudaGridDependencySynchronize();
  __shared__ __align__(16) float2 prev_smem[kWarpsPerBlock * 160];
  float2* const prev_stage = prev_smem + (threadIdx.x >> 5) * 160;
  int head;  // < capacity < 2^31 / 10: the low word of meta[0]
  asm volatile("ld.global.ca.s32 %0, [%1];" : "=r"(head) : "l"(g.meta) : "memory");  // one load per thread, L1 serves most
  if (full) {
    const Lane L = make_lane<NT, true>(a.B, a.N, warp_global);
    RingIO io{a, g, L, ws.stage, prev_stage, head};
    step_core<NT>(a, ws, L, io);
  } else {
    const Lane L = make_lane<NT, false>(a.B, a.N, warp_global);
    RingIO io{a, g, L, ws.stage, prev_stage, head};
    step_core<NT>(a, ws, L, io);
  }
  // every warp of this CTA holds the head (its stores used it): take the CTA's ticket; the last one advances the ring
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(g.meta + 1), 1ull);
    if (t == (unsigned long long)gridDim.x - 1ull) {
      const long long nh = g.meta[0] + g.M;  // unchanged since every thread read it: only this branch writes it
      g.meta[0] = nh >= g.cap ? nh - g.cap : nh;
      const long long held = g.meta[2] + g.M;
      g.meta[2] = held > g.cap ? g.cap : held;
      g.meta[3] += 1;
      g.meta[1] = 0;
    }
  }
}



// ---- K steps per launch -------------------------------------------------------------------------------------------
// I/O policy of step_core for uavca_rollout: the state of the warp's UAVs stays in REGISTERS for all K steps (loaded
// once, stored once), only the per-step outputs stream out, as [K][...] blocks.  Removes the launch, ramp-up and tail
// of K-1 dependent launches and 66 of the 107 algorithmic bytes per UAV-step (the state round trip and, with Philox
// actions, the action read).  Runs the very same step_core as the one-step kernel, so the results are bit-identical
// to K single steps.
//
// The general instance tests the action source and every option of uavca_rollout (final_obs, reset_mask, action_out,
// score tracking, any action mode) at run time.
struct RolloutIO {
  const KernelArgs& a;
  const RolloutArgs& r;
  const Lane& L;
  float* stage;
  Uav cur;
  float2 act;
  int steps;
  int k;          // step of the launch: outputs go to slot k of the [K][...] blocks
  long long km;   // k * M
  __device__ __forceinline__ Uav load_uav() const { return cur; }
  __device__ __forceinline__ float2 load_action() const { return act; }
  __device__ __forceinline__ int load_steps() const { return steps; }
  __device__ __forceinline__ void loads_done() const {}
  __device__ __forceinline__ void store_reward_done(float rw, bool done) const {
    if (L.valid) {
      st_stream((a.io.reward + km) + (unsigned)L.m, rw);
      st_stream((a.io.done + km) + (unsigned)L.m, (uint8_t)done);
    }
  }
  __device__ __forceinline__ bool wants_final() const { return a.io.final_obs != nullptr; }
  __device__ __forceinline__ void put_own(float2 o01, float2 o23) const { stage_own(stage, L.lane, o01, o23); }
  __device__ __forceinline__ void put_neighbours(const ObsTail& n) const { stage_neighbours(stage, L.lane, n); }
  __device__ __forceinline__ void commit(float* g) const {
    __syncwarp();
    flush_warp_rows(stage, (g + km * UAVCA_OBS_DIM_MULTI) + (unsigned)L.warp_m0 * (size_t)UAVCA_OBS_DIM_MULTI, L);
    __syncwarp();
  }
  __device__ __forceinline__ void commit_obs() const { commit(a.io.obs); }
  __device__ __forceinline__ void commit_final() const { commit(a.io.final_obs); }
  __device__ __forceinline__ void store_state(const Uav& u) { cur = u; }
  __device__ __forceinline__ void store_target(const Uav&) const {}  // store_state carried the new target already
  __device__ __forceinline__ void store_steps(int v, bool) { steps = v; }
  __device__ __forceinline__ void store_reset(bool rs) const {
    if (a.io.reset_mask) a.io.reset_mask[(size_t)k * r.B + L.env] = (uint8_t)rs;
  }
};

// PLAIN: the launch of an open-loop driver loop (bench.py, run_multi.py): cartesian actions (block actions as given,
// Philox actions scaled to the action box before step_core sees them), no final_obs, reset_mask, action_out or score
// tracking.  Those options then cost nothing per step.
// Every per-step address is the lane's element offset off = k * M + m, one 32-bit register advanced by M per step: an
// address is the parameter base plus off * sizeof (a LEA pair), with no step counter and no 64-bit index arithmetic in
// the loop.  The launcher runs this instance only where K * M * 10 < 2^31, so the observation offset off * 10 fits too.
// The observation stage is written and read through its shared-memory address, computed once before the loop.
struct PlainRolloutIO {
  static constexpr bool kPlain = true;
  const KernelArgs& a;
  const Lane& L;
  unsigned stage;  // shared-memory address of the warp's observation stage
  Uav cur;
  float2 act;
  int steps;
  unsigned off;  // k * M + m
  __device__ __forceinline__ Uav load_uav() const { return cur; }
  __device__ __forceinline__ float2 load_action() const { return act; }
  __device__ __forceinline__ int load_steps() const { return steps; }
  __device__ __forceinline__ void loads_done() const {}
  __device__ __forceinline__ void store_reward_done(float rw, bool done) const {
    if (L.valid) {
      st_stream(a.io.reward + off, rw);
      st_stream(a.io.done + off, (uint8_t)done);
    }
  }
  __device__ __forceinline__ bool wants_final() const { return false; }
  __device__ __forceinline__ void put_own(float2 o01, float2 o23) const { stage_own(stage, L.lane, o01, o23); }
  __device__ __forceinline__ void put_neighbours(const ObsTail& n) const { stage_neighbours(stage, L.lane, n); }
  __device__ __forceinline__ void commit_obs() const {
    __syncwarp();
    flush_warp_rows(stage, a.io.obs + (off - (unsigned)L.lane) * (unsigned)UAVCA_OBS_DIM_MULTI, L);  // (k * M + warp_m0) * 10
    __syncwarp();
  }
  __device__ __forceinline__ void commit_final() const {}
  __device__ __forceinline__ void store_state(const Uav& u) { cur = u; }
  __device__ __forceinline__ void store_target(const Uav&) const {}  // store_state carried the new target already
  __device__ __forceinline__ void store_steps(int v, bool) { steps = v; }
  __device__ __forceinline__ void store_reset(bool) const {}
};

// the action slots by their shared-memory address: one 32-bit register per lane, no generic-address conversion per step
__device__ __forceinline__ void cp_async8(unsigned smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}

// Instances of the rollout kernel: the plain launch (PlainRolloutIO) with an action block and with Philox actions, each
// with its action source fixed at compile time, and one general instance (RolloutIO) that tests the action source and
// every option at run time.
enum RolloutKind : int { kRolloutGeneral = 0, kRolloutPlainBlock = 1, kRolloutPlainPhilox = 2 };

// Everything that does not change from step to step (the lane geometry, the lane's action slot, the warp's row offset)
// is computed once, before the K loop.
// Action block: the action of step k+1 travels while step k is computed — by cp.async into a per-lane shared-memory
// slot (two slots, alternating), not into registers: at 64 registers ptxas sinks a register prefetch down to its use,
// and ncu showed 15 % of the warp-time waiting on that load (profiles/r2_full_rollout_n32.md).  The two slots of a lane
// lie 256 bytes apart in the warp's 512-byte aligned block: the other slot is slot ^ 256.
template <int NT, bool FULL, int KIND>
__device__ __forceinline__ void rollout_multi_body(const KernelArgs& a, const RolloutArgs& r, const WarpScratch& ws,
                                                   float2* act_smem, int warp_global) {
  const Lane L = make_lane<NT, FULL>(a.B, a.N, warp_global);
  unsigned slot = (unsigned)__cvta_generic_to_shared(act_smem + L.lane);
  const long long env_global = a.c.env_base + L.env;  // Philox actions
  if constexpr (KIND != kRolloutGeneral) {
    PlainRolloutIO io{a, L, (unsigned)__cvta_generic_to_shared(ws.stage), load_uav(a.s, L), make_float2(0.f, 0.f),
                      L.valid ? a.s.steps[L.env] : 0, (unsigned)L.m};
    cudaTriggerProgrammaticLaunchCompletion();
    const unsigned M = (unsigned)r.M;
    if constexpr (KIND == kRolloutPlainBlock) {
      const unsigned end = r.KM + (unsigned)L.m;  // end - off is the same in every lane: the loop is warp-uniform
      if (L.valid) cp_async8(slot, r.action_block + io.off);
      do {
        cp_async_wait_all();
        io.act = L.valid ? lds_float2(slot) : make_float2(0.f, 0.f);
        const unsigned next = io.off + M;
        if (next < end && L.valid) cp_async8(slot ^ 256u, r.action_block + next);
        step_core<NT>(a, ws, L, io);
        io.off = next;
        slot ^= 256u;
      } while (io.off < end);
    } else {
      // the Philox counter needs the step index itself: k stays, the addresses still come from the offset alone
      uint4 words = make_uint4(0u, 0u, 0u, 0u);
      for (int k = 0; k < r.K; ++k) {
        const unsigned long long t = r.step0 + (unsigned long long)k;
        if (k == 0 || (t & 1ull) == 0ull) words = action_words(r.seed_lo, r.seed_hi, env_global, L.i, t);
        io.act = map_action(action_from_words(words, t), UAVCA_ACTION_SCALED, a.c);  // what step_core would do with the launch's mode
        step_core<NT>(a, ws, L, io);
        io.off += M;
      }
    }
    store_uav(a.s, L, io.cur, true);
    if (L.valid & (L.i == 0)) a.s.steps[L.env] = io.steps;
  } else {
    const bool block = r.action_block != nullptr;  // warp-uniform
    RolloutIO io{a, r, L, ws.stage, load_uav(a.s, L), make_float2(0.f, 0.f), L.valid ? a.s.steps[L.env] : 0, 0, 0};
    cudaTriggerProgrammaticLaunchCompletion();
    if (block && L.valid) cp_async8(slot, r.action_block + L.m);
    uint4 words = make_uint4(0u, 0u, 0u, 0u);
    for (int k = 0; k < r.K; ++k) {
      io.k = k;
      io.km = (long long)k * r.M;
      if (block) {
        cp_async_wait_all();
        io.act = L.valid ? lds_float2(slot + (k & 1) * 256) : make_float2(0.f, 0.f);
        if (k + 1 < r.K && L.valid) cp_async8(slot + ((k + 1) & 1) * 256, (r.action_block + (io.km + r.M)) + (unsigned)L.m);
      } else {
        const unsigned long long t = r.step0 + (unsigned long long)k;
        if (k == 0 || (t & 1ull) == 0ull) words = action_words(r.seed_lo, r.seed_hi, env_global, L.i, t);
        io.act = action_from_words(words, t);
        if (r.action_out != nullptr && L.valid) st_stream((r.action_out + io.km) + L.m, io.act);
      }
      step_core<NT>(a, ws, L, io);
    }
    store_uav(a.s, L, io.cur, true);
    if (L.valid & (L.i == 0)) a.s.steps[L.env] = io.steps;
  }
}

// Resident CTAs per SM of the rollout kernel (measured on B200, profiles/r2_rollout_minb.md: 8 CTAs x 64 registers beats
// 6 x 80 and 5 x 96 at N = 16 / 32 and with action blocks, and ties at N = 8 with Philox actions).
#ifndef UAVCA_ROLLOUT_MINB
#define UAVCA_ROLLOUT_MINB 8
#endif
template <int NT, int KIND>
__global__ void __launch_bounds__(kThreads, UAVCA_ROLLOUT_MINB) rollout_multi_kernel(const __grid_constant__ KernelArgs a,
                                                                                  const __grid_constant__ RolloutArgs r) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  __shared__ __align__(512) float2 act_smem[kWarpsPerBlock * 64];  // per warp: two slots of 32 float2 actions
  const WarpScratch ws = warp_scratch(smem);
  const int warp_global = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int N = NT > 0 ? NT : a.N;
  const bool full = uavs_left(a.B, N, warp_global) >= (32 / N) * N;  // warp-uniform
  cudaGridDependencySynchronize();
  float2* const my_act = act_smem + (threadIdx.x >> 5) * 64;
  if (full) rollout_multi_body<NT, true, KIND>(a, r, ws, my_act, warp_global);
  else rollout_multi_body<NT, false, KIND>(a, r, ws, my_act, warp_global);
}

// The action stream of uavca_rollout on its own, one step: out[m] = the policy-space action of global step t.
__global__ void __launch_bounds__(kThreads) sample_actions_kernel(const __grid_constant__ Consts c, float2* out, int B, int N,
                                                                  unsigned seed_lo, unsigned seed_hi, unsigned long long t) {
  const long long m = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (m >= (long long)B * N) return;
  const long long env = m / N;
  const int i = (int)(m - env * N);
  out[m] = action_from_words(action_words(seed_lo, seed_hi, c.env_base + env, i, t), t);
}

// ---- persistent variant with cp.async input prefetch (large batches) ----------------------------------------------------
// ncu on step_multi_kernel<32> (profiles/r2_full_c4_step_multi_n32.md): a fifth of the warp-time is spent waiting for
// the warp's own state to arrive (long scoreboard on the first use of the loads).  Here every warp walks warp-tiles
// w, w + G, w + 2G, ...; while it computes one tile, the next tile's state and actions are already on their way INTO
// SHARED MEMORY (cp.async / LDGSTS: no registers held, unlike a register prefetch).  Same step_core, same outputs.
// MEASURED (profiles/r2_prefetch_variant.md): the long-scoreboard stall disappears (2.05 -> 0.16 warps per issue cycle)
// but issue utilisation does not rise (76.5 % -> 72.5 %): the idle issue slots come from the dependent integer min/max
// chains and ALU-pipe contention, not from load latency, and the hardware CTA scheduler already overlaps one CTA's loads
// with its neighbours' compute.  151.6 vs 132.3 us at N=32, B=131,072 — slower everywhere, hence opt-in only
// (UAVCA_STEP_PATH=prefetch), parity-tested.
constexpr int kPfStageBytes = 32 * (16 + 8 + 8 + 8 + 4 + 4);  // vel, pos, tgt, action, init, prev of one warp-tile


struct PfStage {
  double2* vel;
  float2 *pos, *tgt, *act;
  float *init, *prev;
};
__device__ __forceinline__ PfStage pf_stage(unsigned char* base) {
  PfStage st;
  st.vel = reinterpret_cast<double2*>(base);
  st.pos = reinterpret_cast<float2*>(base + 32 * 16);
  st.tgt = st.pos + 32;
  st.act = st.tgt + 32;
  st.init = reinterpret_cast<float*>(st.act + 32);
  st.prev = st.init + 32;
  return st;
}

struct PfIO : GlobalIO {
  Uav pre;
  float2 act;
  int steps;
  __device__ __forceinline__ Uav load_uav() const { return pre; }
  __device__ __forceinline__ float2 load_action() const { return act; }
  __device__ __forceinline__ int load_steps() const { return steps; }
  __device__ __forceinline__ void loads_done() const {}
};

template <int NT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSM) step_multi_pf_kernel(const __grid_constant__ KernelArgs a,
                                                                                  const int num_tiles) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  __shared__ __align__(16) unsigned char stage_mem[kWarpsPerBlock * kPfStageBytes];
  const WarpScratch ws = warp_scratch(smem);
  const PfStage st = pf_stage(stage_mem + (threadIdx.x >> 5) * kPfStageBytes);
  const int lane = threadIdx.x & 31;
  const int stride = gridDim.x * kWarpsPerBlock;
  int wt = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  cudaGridDependencySynchronize();
  if (wt >= num_tiles) return;
  // every tile of this kernel is a FULL warp-tile (the launcher hands the ragged rest to the per-lane kernel)
  unsigned nflags = 0u;
  int nsteps = 0;
  auto prefetch = [&](int tile) {
    const Lane P = make_lane<NT, true>(a.B, a.N, tile);
    if (P.valid) {
      cp_async(st.vel + lane, a.s.vel + P.m, 16);
      cp_async(st.pos + lane, a.s.pos + P.m, 8);
      cp_async(st.tgt + lane, a.s.tgt + P.m, 8);
      cp_async(st.act + lane, a.io.action + P.m, 8);
      cp_async(st.init + lane, a.s.init + P.m, 4);
      cp_async(st.prev + lane, a.s.prev + P.m, 4);
      nflags = ld_stream(a.s.flags + P.m);  // one register each: consumed only at the top of the next tile
      nsteps = a.s.steps[P.env];
    }
  };
  prefetch(wt);
  cudaTriggerProgrammaticLaunchCompletion();
  while (true) {
    const Lane L = make_lane<NT, true>(a.B, a.N, wt);
    cp_async_wait_all();
    __syncwarp();
    PfIO io{{a, L, ws.stage}, Uav{}, make_float2(0.f, 0.f), 0};
    if (L.valid) {
      const double2 v = st.vel[lane];
      const float2 p = st.pos[lane], t = st.tgt[lane];
      io.pre.px = p.x; io.pre.py = p.y; io.pre.tx = t.x; io.pre.ty = t.y; io.pre.vx = v.x; io.pre.vy = v.y;
      io.pre.init = st.init[lane]; io.pre.prev = st.prev[lane]; io.pre.flags = nflags;
      io.act = st.act[lane];
      io.steps = nsteps;
    } else {  // idle lanes (32 is not a multiple of N): a harmless UAV in ordinary flight, as in load_uav()
      io.pre.px = io.pre.py = io.pre.ty = 0.f; io.pre.tx = 8.f; io.pre.init = io.pre.prev = 8.f;
      io.pre.vx = 1.0; io.pre.vy = 0.0; io.pre.flags = 0u;
    }
    __syncwarp();  // the stage has been read out: refill it for the next tile while this one is computed
    const int next = wt + stride;
    if (next < num_tiles) prefetch(next);
    step_core<NT>(a, ws, L, io);
    if (next >= num_tiles) break;
    wt = next;
  }
}

template <int NT>
__global__ void __launch_bounds__(kThreads) reset_multi_kernel(const __grid_constant__ KernelArgs a, const uint8_t* mask) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  const WarpScratch ws = warp_scratch(smem);
  const Lane L = make_lane<NT>(a.B, a.N);
  Uav u = load_uav(a.s, L);
  const bool rs = L.valid && (mask == nullptr || mask[L.env] != 0);
  const bool leader = L.valid & (L.i == 0);
  unsigned episode = 0;
  if (leader) episode = a.s.episode[L.env];
  episode = __shfl_sync(kFull, episode, L.base);
  if (leader && rs) {
    if (episode > 0u) {
      atomicAdd(a.s.stats + 0, 1ull);
      atomicAdd(a.s.stats + 1, (unsigned long long)a.s.reach[L.env]);
      atomicAdd(a.s.stats + 2, (unsigned long long)a.s.coll[L.env]);
      atomicAdd(a.s.stats + 3, (unsigned long long)a.s.steps[L.env]);
      if (a.c.track_scores) fold_scores(a.s, L.env);
    }
    a.s.steps[L.env] = 0; a.s.reach[L.env] = 0; a.s.coll[L.env] = 0;
    a.s.episode[L.env] = episode + 1u;
  }
  reset_multi(a, L, rs, episode, u);
  const ObsRow o = observe_state<NT>(a.c, ws, L, u);
  if (a.io.obs) {
    if (mask == nullptr) {
      store_obs_rows(ws.stage, a.io.obs, L, o);
    } else if (rs) {  // rows of other envs stay untouched
      float2* row = reinterpret_cast<float2*>(a.io.obs + (size_t)L.m * 10);
      row[0] = o.o01; row[1] = o.o23; row[2] = o.n.a; row[3] = o.n.b; row[4] = o.n.c;
    }
  }
  if (rs) store_uav(a.s, L, u, true);
}

template <int NT>
__global__ void __launch_bounds__(kThreads) observe_multi_kernel(const __grid_constant__ KernelArgs a) {
  __shared__ __align__(16) float smem[kWarpsPerBlock * kScratchFloats];
  const WarpScratch ws = warp_scratch(smem);
  const Lane L = make_lane<NT>(a.B, a.N);
  const Uav u = load_uav(a.s, L);
  store_obs_rows(ws.stage, a.io.obs, L, observe_state<NT>(a.c, ws, L, u));
}

// ================================================================================================================
// Single-UAV world: one thread per env
// ================================================================================================================

struct SingleEnv {
  float px, py, tx, ty, init, prev;
  double vx, vy;
  int steps;
};

__device__ __forceinline__ void obs_single(const Consts& c, const SingleEnv& e, bool vel_is_f32, float o[4]) {
  // UAVWorld2D._get_obs (uav_world_2d.py:88-97)
  const float speed = vel_is_f32 ? n32((float)e.vx, (float)e.vy) : sqrt_approx((float)sq64(e.vx, e.vy));
  o[0] = speed * c.inv_vmax_f;
  o[1] = fast_atan2((float)e.vy, (float)e.vx) * c.inv_pi;
  const float tdx = __fsub_rn(e.tx, e.px), tdy = __fsub_rn(e.ty, e.py);
  o[2] = n32(tdx, tdy) * c.inv_diag;
  o[3] = rel_angle((double)tdx, (double)tdy, e.vx, e.vy) * c.inv_pi;
}

__device__ __forceinline__ void reset_single(const KernelArgs& a, long long b, unsigned episode, SingleEnv& e) {
  // UAVWorld2D.reset (uav_world_2d.py:121-131)
  const Consts& c = a.c;
  const long long env_global = c.env_base + b;
  if (c.reset_source == UAVCA_SOURCE_POOL && a.pool.pos != nullptr) {
    const long long p = (env_global + (long long)episode) % a.pool_envs;
    float2 pp = a.pool.pos[p], pt = a.pool.tgt[p];
    double2 pv = a.pool.vel[p];
    e.px = pp.x; e.py = pp.y; e.tx = pt.x; e.ty = pt.y; e.vx = pv.x; e.vy = pv.y;
    e.init = a.pool.init[p]; e.prev = a.pool.prev[p];
  } else {
    float2 p = draw_pair(c, env_global, episode, kStreamPos, 0, 0u, c.lox, c.hix, c.loy, c.hiy);
    float2 v = draw_pair(c, env_global, episode, kStreamVel, 0, 0u, -c.vmax, c.vmax, -c.vmax, c.vmax);
    float2 t = draw_pair(c, env_global, episode, kStreamTgt, 0, 0u, c.lox, c.hix, c.loy, c.hiy);
    e.px = p.x; e.py = p.y; e.vx = (double)v.x; e.vy = (double)v.y; e.tx = t.x; e.ty = t.y;
    e.init = n32(__fsub_rn(e.tx, e.px), __fsub_rn(e.ty, e.py));
    e.prev = e.init;
  }
  e.steps = 0;
}

__device__ __forceinline__ SingleEnv load_single(const StateView& s, long long b) {
  SingleEnv e;
  float2 p = ld_stream(s.pos + b), t = ld_stream(s.tgt + b);
  double2 v = ld_stream(s.vel + b);
  e.px = p.x; e.py = p.y; e.tx = t.x; e.ty = t.y; e.vx = v.x; e.vy = v.y;
  e.init = ld_stream(s.init + b); e.prev = ld_stream(s.prev + b); e.steps = ld_stream(s.steps + b);
  return e;
}

__device__ __forceinline__ void store_single(const StateView& s, long long b, const SingleEnv& e, bool with_target) {
  st_stream(s.pos + b, make_float2(e.px, e.py));
  st_stream(s.vel + b, make_double2(e.vx, e.vy));
  st_stream(s.prev + b, e.prev);
  st_stream(s.steps + b, e.steps);
  if (with_target) {
    st_stream(s.tgt + b, make_float2(e.tx, e.ty));
    st_stream(s.init + b, e.init);
  }
}

__device__ __forceinline__ void fold_single(const KernelArgs& a, long long b, unsigned episode, int steps) {
  if (episode > 0u) {
    atomicAdd(a.s.stats + 0, 1ull);
    atomicAdd(a.s.stats + 1, (unsigned long long)a.s.reach[b]);
    atomicAdd(a.s.stats + 3, (unsigned long long)steps);
    if (a.c.track_scores) fold_scores(a.s, (int)b);
  }
  a.s.reach[b] = 0; a.s.coll[b] = 0;
  a.s.episode[b] = episode + 1u;
}

// One UAVWorld2D.step of env b held in registers (uav_world_2d.py:137-173); outputs go to row `o` of the output
// tensors (o = b for one step per launch, k * B + b inside a rollout).  Returns true when the env auto-reset.
__device__ __forceinline__ bool step_single_core(const KernelArgs& a, long long b, long long o, SingleEnv& e, float2 act_raw,
                                                 const double2* act64 = nullptr) {
  const Consts& c = a.c;
  const float2 act = map_action(act_raw, a.io.action_mode, c);

  // UAVWorld2D.step (uav_world_2d.py:142-147)
  if (act64 != nullptr) {  // a float64 action: float64 arithmetic from the first step on
    integrate(act64->x, act64->y, e.vx, e.vy, e.px, e.py, c);
  } else if (c.single_f32_first_step && e.steps == 0) {
    // float32 action against the float32 reset speed: the quotient is formed in float32 (:122,:142)
    const double qx = (double)__fdiv_rn(__fsub_rn(act.x, (float)e.vx), c.tau_f);
    const double qy = (double)__fdiv_rn(__fsub_rn(act.y, (float)e.vy), c.tau_f);
    const double dvx = clipd(qx, -c.amax, c.amax), dvy = clipd(qy, -c.amax, c.amax);
    e.vx = clipd(__dadd_rn(e.vx, __dmul_rn(dvx, c.tau)), -c.vmax, c.vmax);
    e.vy = clipd(__dadd_rn(e.vy, __dmul_rn(dvy, c.tau)), -c.vmax, c.vmax);
    e.px = __double2float_rn(__dadd_rn((double)e.px, __dmul_rn(e.vx, c.tau)));
    e.py = __double2float_rn(__dadd_rn((double)e.py, __dmul_rn(e.vy, c.tau)));
  } else {
    integrate((double)act.x, (double)act.y, e.vx, e.vy, e.px, e.py, c);
  }
  const float tdx = __fsub_rn(e.tx, e.px), tdy = __fsub_rn(e.ty, e.py);
  const float dist = n32(tdx, tdy);                                               // :150
  const float dth = rel_angle((double)tdx, (double)tdy, e.vx, e.vy);              // :155-156
  // reward (:152-157): float32 under NumPy 2, the angle term is a python float rounded to float32 first
  float r = __fsub_rn(0.0f, __fdiv_rn(1.0f, e.init));
  r = __fadd_rn(r, __fmul_rn(10.0f, __fsub_rn(e.prev, dist)));
  r = __fsub_rn(r, (float)(0.1 * (double)fabsf(dth)));
  const bool inside = (e.px >= c.lox_f) & (e.px <= c.hix_f) & (e.py >= c.loy_f) & (e.py <= c.hiy_f);
  const bool reached = dist < c.reach_dist;                                       // :159
  if (reached) r = __fadd_rn(r, 1000.0f);                                         // :161
  const bool done = reached | !inside;                                            // :159-166
  e.steps += 1;                                                                   // :170
  e.prev = dist;                                                                  // :172
  if (reached) a.s.reach[b] += 1;
  if (c.track_scores) {  // test_sac.py-style score: sum of rewards; and rewards * (1 - done)
    double2 sc = a.s.score[b];
    sc.x += (double)r;
    sc.y += done ? 0.0 : (double)r;
    a.s.score[b] = sc;
  }
  if (!(fabsf(r) <= 3.4e38f) | !(fabsf(e.px) + fabsf(e.py) <= 3.4e38f)) atomicAdd(a.s.stats + 6, 1ull);

  float ob[4];
  obs_single(c, e, false, ob);
  st_stream(a.io.reward + o, r);
  st_stream(a.io.done + o, (uint8_t)done);
  if (a.io.distance) st_stream(a.io.distance + o, dist);                          // info["distance"] :169
  if (a.io.final_obs) st_stream(reinterpret_cast<float4*>(a.io.final_obs) + o, make_float4(ob[0], ob[1], ob[2], ob[3]));

  bool rs = false;
  if (c.reset_mode & (UAVCA_RESET_ON_DONE0 | UAVCA_RESET_ON_ALL_DONE | UAVCA_RESET_ON_ANY_DONE)) rs |= done;
  if (c.max_steps > 0) rs |= e.steps >= c.max_steps;
  if (a.io.reset_mask) a.io.reset_mask[o] = (uint8_t)rs;
  if (rs) {
    const unsigned episode = a.s.episode[b];
    fold_single(a, b, episode, e.steps);
    reset_single(a, b, episode, e);
    obs_single(c, e, true, ob);
  }
  st_stream(reinterpret_cast<float4*>(a.io.obs) + o, make_float4(ob[0], ob[1], ob[2], ob[3]));
  return rs;
}

__global__ void __launch_bounds__(kThreads) step_single_kernel(const __grid_constant__ KernelArgs a) {
  const long long b = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (b >= a.B) return;
  SingleEnv e = load_single(a.s, b);
  double2 q = make_double2(0.0, 0.0);
  float2 af = make_float2(0.f, 0.f);
  const bool f64 = a.io.action64 != nullptr;  // uavca_step_f64 (kernel-uniform)
  if (f64) q = a.io.action64[b];
  else af = ld_stream(a.io.action + b);
  const bool rs = step_single_core(a, b, b, e, af, f64 ? &q : nullptr);
  store_single(a.s, b, e, rs);
}

// K steps of UAVWorld2D per launch, the env in registers throughout (see RolloutIO above).
__global__ void __launch_bounds__(kThreads) rollout_single_kernel(const __grid_constant__ KernelArgs a,
                                                                  const __grid_constant__ RolloutArgs r) {
  __shared__ __align__(16) float2 act_smem[2 * kThreads];  // per thread two alternating slots: the next step's action by cp.async
  const long long b = (long long)blockIdx.x * kThreads + threadIdx.x;
  cudaGridDependencySynchronize();
  if (b >= a.B) return;
  SingleEnv e = load_single(a.s, b);
  cudaTriggerProgrammaticLaunchCompletion();
  uint4 words = make_uint4(0u, 0u, 0u, 0u);
  float2* slot = act_smem + threadIdx.x;
  if (r.action_block != nullptr) cp_async(slot, r.action_block + b, 8);
  for (int k = 0; k < r.K; ++k) {
    float2 act;
    if (r.action_block != nullptr) {
      cp_async_wait_all();
      act = slot[(k & 1) * kThreads];
      if (k + 1 < r.K) cp_async(slot + ((k + 1) & 1) * kThreads, r.action_block + (size_t)(k + 1) * r.M + b, 8);
    } else {
      const unsigned long long t = r.step0 + (unsigned long long)k;
      if (k == 0 || (t & 1ull) == 0ull) words = action_words(r.seed_lo, r.seed_hi, a.c.env_base + b, 0, t);
      act = action_from_words(words, t);
      if (r.action_out != nullptr) st_stream(r.action_out + (size_t)k * r.M + b, act);
    }
    step_single_core(a, b, (long long)k * r.M + b, e, act);
  }
  store_single(a.s, b, e, true);
}

__global__ void __launch_bounds__(kThreads) reset_single_kernel(const __grid_constant__ KernelArgs a, const uint8_t* mask) {
  const long long b = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (b >= a.B) return;
  if (mask != nullptr && mask[b] == 0) return;
  SingleEnv e = load_single(a.s, b);
  const unsigned episode = a.s.episode[b];
  fold_single(a, b, episode, e.steps);
  reset_single(a, b, episode, e);
  a.s.flags[b] = 0;
  float o[4];
  obs_single(a.c, e, true, o);
  if (a.io.obs) st_stream(reinterpret_cast<float4*>(a.io.obs) + b, make_float4(o[0], o[1], o[2], o[3]));
  store_single(a.s, b, e, true);
}

__global__ void __launch_bounds__(kThreads) observe_single_kernel(const __grid_constant__ KernelArgs a) {
  const long long b = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (b >= a.B) return;
  const SingleEnv e = load_single(a.s, b);
  float o[4];
  obs_single(a.c, e, e.steps == 0, o);
  st_stream(reinterpret_cast<float4*>(a.io.obs) + b, make_float4(o[0], o[1], o[2], o[3]));
}

// ================================================================================================================
// Small utility kernels
// ================================================================================================================

__global__ void __launch_bounds__(kThreads) map_action_kernel(const __grid_constant__ Consts c, const float2* in,
                                                              float2* out, long long M, int mode) {
  const long long m = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (m < M) out[m] = map_action(in[m], mode, c);
}

// out8: finished-episode totals (episodes, reach, collisions, steps), in-flight sums (reach, collisions, steps), B
__global__ void __launch_bounds__(kThreads) stats_kernel(StateView s, int B, long long* out8) {
  long long reach = 0, coll = 0, steps = 0;
  for (long long b = (long long)blockIdx.x * kThreads + threadIdx.x; b < B; b += (long long)gridDim.x * kThreads) {
    reach += s.reach[b]; coll += s.coll[b]; steps += s.steps[b];
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    reach += __shfl_xor_sync(kFull, reach, d);
    coll += __shfl_xor_sync(kFull, coll, d);
    steps += __shfl_xor_sync(kFull, steps, d);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(reinterpret_cast<unsigned long long*>(out8 + 4), (unsigned long long)reach);
    atomicAdd(reinterpret_cast<unsigned long long*>(out8 + 5), (unsigned long long)coll);
    atomicAdd(reinterpret_cast<unsigned long long*>(out8 + 6), (unsigned long long)steps);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    out8[0] = (long long)s.stats[0]; out8[1] = (long long)s.stats[1];
    out8[2] = (long long)s.stats[2]; out8[3] = (long long)s.stats[3];
    out8[7] = B;
  }
}

// Replay ring append: every array is a run of whole rows, so the ring write is a flat copy whose destination index
// wraps at capacity * row.  V = float2 when both row widths are even and the pointers 8-byte aligned, else float.
constexpr int kPushThreads = 1024;  // big blocks: one head ticket (a same-address atomic) per block
template <typename V>
__global__ void __launch_bounds__(kPushThreads) replay_push_kernel(const V* obs, const V* act, const float* rew, const V* nxt,
                                                               const uint8_t* done, long long M, long long od, long long ad,
                                                               V* r_obs, V* r_act, float* r_rew, V* r_nxt, float* r_mask,
                                                               long long cap, long long head, long long* meta) {
  // meta (nullable, device): [0] ring head, [1] block ticket, [2] transitions held, [3] appends so far.  With it the head
  // lives on the device, so a CUDA-graph replay of the push appends where the previous replay stopped.  Every thread
  // reads the head (an ordinary load: L1 serves all but the first warp of an SM — a volatile load from 25,000 warps made
  // the one L2 sector a hot spot, 28 us); once all threads of a block HOLD it (the barrier's predicate depends on the
  // loaded value) the block takes a ticket, and the last ticket holder — every block has read the head by then —
  // advances it.  Nothing waits for the data stores (the kernel boundary orders them for the consumers).
  if (meta != nullptr) {
    asm volatile("ld.global.ca.s64 %0, [%1];" : "=l"(head) : "l"(meta) : "memory");  // exactly one load, L1-cacheable
    if (__syncthreads_or(head < 0)) return;  // never taken
    if (threadIdx.x == 0) {
      const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(meta + 1), 1ull);
      if (t == (unsigned long long)gridDim.x - 1ull) {
        const long long nh = head + M;
        meta[0] = nh >= cap ? nh - cap : nh;
        const long long held = meta[2] + M;
        meta[2] = held > cap ? cap : held;
        meta[3] += 1;  // appends so far: a per-step device counter other kernels of an acting step can key their RNG on
        meta[1] = 0;
      }
    }
  }
  const long long j = (long long)blockIdx.x * kPushThreads + threadIdx.x;
  if (j < M * od) {
    long long d = head * od + j;
    if (d >= cap * od) d -= cap * od;
    r_obs[d] = ld_stream(obs + j);
    r_nxt[d] = ld_stream(nxt + j);
  }
  if (j < M * ad) {
    long long d = head * ad + j;
    if (d >= cap * ad) d -= cap * ad;
    r_act[d] = ld_stream(act + j);
  }
  if (j < M) {
    long long d = head + j;
    if (d >= cap) d -= cap;
    r_rew[d] = ld_stream(rew + j);
    r_mask[d] = done[j] ? 0.0f : 1.0f;
  }
}

// Replay sampling (ReplayMemory.sample, pytorch_sac_temp/replay_memory.py:21-24; ReplayBuffer.get_batch with its recency
// weighting, pytorch_ddpg/buffer_tensor.py:65-90): draw `batch` slots and gather the five arrays in ONE launch.  Ring head
// and fill level are read on the device (ring_meta), the draws come from the sampler's Philox4x32-10 stream keyed by (seed,
// sample, draw + appends so far) (uavca_device.cuh), so a learner step captured in a CUDA graph samples fresh transitions
// from the ring as it grows.  An empty ring yields slot 0.
// 16 threads per sample: they share the slot and copy the rows element-wise.
constexpr int kSampleLanes = 16;
__global__ void __launch_bounds__(kThreads) replay_sample_kernel(const float* r_obs, const float* r_act, const float* r_rew,
                                                                 const float* r_nxt, const float* r_mask, long long cap, int od,
                                                                 int ad, const long long* meta, long long batch, unsigned seed_lo,
                                                                 unsigned seed_hi, unsigned long long draw, int recency,
                                                                 float* o_obs, float* o_act, float* o_rew, float* o_nxt,
                                                                 float* o_mask, long long* o_idx) {
  const long long j = ((long long)blockIdx.x * kThreads + threadIdx.x) / kSampleLanes;
  const int l = threadIdx.x % kSampleLanes;
  if (j >= batch) return;
  const long long head = meta[0], size = meta[2];
  const unsigned long long ctr = draw + (unsigned long long)meta[3];
  const uint4 r = philox_indexed(kStreamSample, (unsigned long long)j, ctr, seed_lo, seed_hi);
  long long slot = 0;
  if (size > 0) {
    if (recency) {
      // probability rising linearly with recency: inverse CDF of p_i ~ i + 1/2 over insertion order (buffer_tensor.py:78-87)
      const double u = ((double)r.x + 0.5) * (1.0 / 4294967296.0);
      long long age = (long long)(sqrt(u) * (double)size);
      age = age >= size ? size - 1 : age;
      const long long oldest = size == cap ? head : 0;
      slot = oldest + age;
      slot -= slot >= cap ? cap : 0;
    } else {
      slot = (long long)(((unsigned long long)r.x * (unsigned long long)size) >> 32);  // uniform over the filled slots (size < 2^32)
    }
  }
  for (int k = l; k < od; k += kSampleLanes) {
    o_obs[j * od + k] = r_obs[slot * od + k];
    o_nxt[j * od + k] = r_nxt[slot * od + k];
  }
  for (int k = l; k < ad; k += kSampleLanes) o_act[j * ad + k] = r_act[slot * ad + k];
  if (l == 0) {
    o_rew[j] = r_rew[slot];
    o_mask[j] = r_mask[slot];
    if (o_idx) o_idx[j] = slot;
  }
}

// ================================================================================================================
// Launchers
// ================================================================================================================

static inline int flat_grid(long long n) { return (int)((n + kThreads - 1) / kThreads); }

static inline int multi_grid(int B, int N) {
  const int epw = 32 / N;
  const long long warps = ((long long)B + epw - 1) / epw;
  return (int)((warps + kWarpsPerBlock - 1) / kWarpsPerBlock);
}

#define UAVCA_DISPATCH_N(N, CALL)            \
  switch (N) {                               \
    case 2: { constexpr int NT = 2; CALL; } break;   \
    case 4: { constexpr int NT = 4; CALL; } break;   \
    case 5: { constexpr int NT = 5; CALL; } break;   \
    case 8: { constexpr int NT = 8; CALL; } break;   \
    case 10: { constexpr int NT = 10; CALL; } break; \
    case 16: { constexpr int NT = 16; CALL; } break; \
    case 32: { constexpr int NT = 32; CALL; } break; \
    default: { constexpr int NT = 0; CALL; } break;  \
  }

// The step kernel is launched with programmatic stream serialization (PDL): its blocks may become resident while
// the previous kernel in the stream drains, and wait in cudaGridDependencySynchronize() before touching memory.
template <int NT>
static cudaError_t launch_step_multi_n(const KernelArgs& a, int grid, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, step_multi_kernel<NT>, a);
}

// ---- bulk path (uavca_tma.cuh): persistent grid sized to the SM slots the kernel can hold --------------------------

template <typename Kernel>
static cudaError_t launch_pdl(Kernel kernel, int grid, int threads, size_t smem, cudaStream_t st, const KernelArgs& a,
                              int num_tiles) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, a, num_tiles);
}

template <int NT, bool FINAL>
static cudaError_t launch_step_tma_n(const KernelArgs& a, int num_tiles, cudaStream_t st) {
  using G = TmaGeom<NT, FINAL>;
  constexpr int kMaxDev = 64;
  static std::atomic<int> slots[kMaxDev];  // resident CTAs per device for this instantiation (0 = not configured yet)
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= kMaxDev) return cudaErrorInvalidDevice;
  auto kernel = step_multi_tma_kernel<NT, FINAL>;
  if (slots[dev] == 0) {
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    int per_sm = 0, sms = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, G::THREADS, G::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    slots[dev] = per_sm * sms;
  }
  const int n_slots = slots[dev];
  const int grid = num_tiles < n_slots ? num_tiles : n_slots;
  return launch_pdl(kernel, grid, G::THREADS, G::SMEM_BYTES, st, a, num_tiles);
}

// envs per tile of the bulk path for this N (0: no bulk path, the per-lane kernel takes everything)
static int tma_tile_envs(int N) {
  switch (N) {
    case 2: return TmaGeom<2, false>::E;
    case 4: return TmaGeom<4, false>::E;
    case 5: return TmaGeom<5, false>::E;
    case 8: return TmaGeom<8, false>::E;
    case 10: return TmaGeom<10, false>::E;
    case 16: return TmaGeom<16, false>::E;
    case 32: return TmaGeom<32, false>::E;
    default: return 0;
  }
}

#define UAVCA_DISPATCH_TMA(N, CALL)                  \
  switch (N) {                                       \
    case 2: { constexpr int NT = 2; CALL; } break;   \
    case 4: { constexpr int NT = 4; CALL; } break;   \
    case 5: { constexpr int NT = 5; CALL; } break;   \
    case 8: { constexpr int NT = 8; CALL; } break;   \
    case 10: { constexpr int NT = 10; CALL; } break; \
    case 16: { constexpr int NT = 16; CALL; } break; \
    case 32: { constexpr int NT = 32; CALL; } break; \
    default: break;                                  \
  }

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// persistent prefetching kernel: grid = resident CTA slots of the device
template <int NT>
static cudaError_t launch_step_pf_n(const KernelArgs& a, int num_tiles, cudaStream_t st) {
  constexpr int kMaxDev = 64;
  static std::atomic<int> slots[kMaxDev];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= kMaxDev) return cudaErrorInvalidDevice;
  auto kernel = step_multi_pf_kernel<NT>;
  if (slots[dev] == 0) {
    int per_sm = 0, sms = 0;
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, 0);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    slots[dev] = per_sm * sms;
  }
  const int ctas = (num_tiles + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const int n_slots = slots[dev];
  return launch_pdl(kernel, ctas < n_slots ? ctas : n_slots, kThreads, 0, st, a, num_tiles);
}


// the general one-thread-per-env kernels (uavca_seq.cuh) serve the float64 world and envs wider than a warp
static inline bool wants_seq(const KernelArgs& a) { return a.c.circular != 0 || a.N > 32; }

template <int NT>
static cudaError_t launch_step_multi_f64_n(const KernelArgs& a, int grid, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, step_multi_f64_kernel<NT>, a);
}

cudaError_t launch_step_multi(const KernelArgs& a, cudaStream_t st, int* launched, int path) {
  if (launched) *launched = 0;
  if (a.B <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  if (wants_seq(a)) {
    if (a.c.circular) step_multi_seq_kernel<double><<<flat_grid(a.B), kThreads, 0, st>>>(a);
    else step_multi_seq_kernel<float><<<flat_grid(a.B), kThreads, 0, st>>>(a);
    if (launched) *launched = 1;
    return cudaGetLastError();
  }
  if (a.io.action64 != nullptr) {  // float64 actions: the warp kernel fed by GlobalIO64
    UAVCA_DISPATCH_N(a.N, (e = launch_step_multi_f64_n<NT>(a, multi_grid(a.B, a.N), st)));
    if (e != cudaSuccess) return e;
    if (launched) *launched = 1;
    return cudaGetLastError();
  }
  if (cta_packs(a.N, false) && path != UAVCA_PATH_PLAIN && path != UAVCA_PATH_PREFETCH && path != UAVCA_PATH_AUTO) {
    // 17..25 UAVs per env: 5..7 envs packed across the 4 warps of a CTA instead of one env per warp (uavca_cta.cuh).
    // Measured (B*N = 2 Mi UAVs, one stream): N=17 98 vs 136 us, N=20 101 vs 122, N=24 107 vs 113; from N=26 a CTA
    // holds 4 envs like 4 warps do and the barriers only cost (N=28 119 vs 108 us), so those stay on the warp kernel.
    const int envs_per_cta = kThreads / a.N;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((a.B + envs_per_cta - 1) / envs_per_cta);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, step_multi_cta_kernel, a);
    if (e != cudaSuccess) return e;
    if (launched) *launched = 1;
    return cudaGetLastError();
  }
  if (path == UAVCA_PATH_PREFETCH) {
    // opt-in (UAVCA_STEP_PATH=prefetch; measured slower than the per-lane kernel at every size, DESIGN.md 6.3): whole
    // warp-tiles go through the persistent cp.async-prefetch kernel, the ragged rest through the per-lane kernel
    const int epw = 32 / a.N;
    const int full_tiles = a.B / epw;
    if (full_tiles > 0 && aligned16(a.s.vel) && aligned16(a.s.pos) && aligned16(a.s.tgt) && aligned16(a.io.action)) {
      UAVCA_DISPATCH_N(a.N, (e = launch_step_pf_n<NT>(a, full_tiles, st)));
      if (e != cudaSuccess) return e;
      if (launched) *launched += 1;
      const int done_envs = full_tiles * epw;
      if (done_envs < a.B) {
        KernelArgs r = a;
        const long long m0 = (long long)done_envs * a.N;
        r.s = offset_view(a.s, done_envs, a.N);
        r.c.env_base += done_envs;
        r.B = a.B - done_envs;
        r.io.action += m0;
        r.io.obs += m0 * UAVCA_OBS_DIM_MULTI;
        r.io.reward += m0;
        r.io.done += m0;
        if (r.io.final_obs) r.io.final_obs += m0 * UAVCA_OBS_DIM_MULTI;
        if (r.io.reset_mask) r.io.reset_mask += done_envs;
        UAVCA_DISPATCH_N(r.N, (e = launch_step_multi_n<NT>(r, multi_grid(r.B, r.N), st)));
        if (e != cudaSuccess) return e;
        if (launched) *launched += 1;
      }
      return cudaGetLastError();
    }
  }
  // whole tiles go through the bulk (TMA) kernel, the ragged rest through the per-lane kernel
  int tile_envs = path == UAVCA_PATH_AUTO ? tma_tile_envs(a.N) : 0;
  if (tile_envs && !(aligned16(a.io.action) && aligned16(a.io.obs) && aligned16(a.io.reward) && aligned16(a.io.done) &&
                     aligned16(a.io.final_obs) && aligned16(a.s.pos) && aligned16(a.s.vel) && aligned16(a.s.tgt) &&
                     aligned16(a.s.init) && aligned16(a.s.prev) && aligned16(a.s.flags) && aligned16(a.s.steps)))
    tile_envs = 0;
  const int tiles = tile_envs ? a.B / tile_envs : 0;
  const int bulk_envs = tiles * tile_envs;
  if (tiles > 0) {
    if (a.io.final_obs) {
      UAVCA_DISPATCH_TMA(a.N, (e = launch_step_tma_n<NT, true>(a, tiles, st)));
    } else {
      UAVCA_DISPATCH_TMA(a.N, (e = launch_step_tma_n<NT, false>(a, tiles, st)));
    }
    if (e != cudaSuccess) return e;
    if (launched) *launched += 1;
  }
  if (bulk_envs < a.B) {
    KernelArgs r = a;
    const long long m0 = (long long)bulk_envs * a.N;
    r.s = offset_view(a.s, bulk_envs, a.N);
    r.c.env_base += bulk_envs;
    r.B = a.B - bulk_envs;
    r.io.action += m0;
    r.io.obs += m0 * UAVCA_OBS_DIM_MULTI;
    r.io.reward += m0;
    r.io.done += m0;
    if (r.io.final_obs) r.io.final_obs += m0 * UAVCA_OBS_DIM_MULTI;
    if (r.io.reset_mask) r.io.reset_mask += bulk_envs;
    const int grid = multi_grid(r.B, r.N);
    UAVCA_DISPATCH_N(r.N, (e = launch_step_multi_n<NT>(r, grid, st)));
    if (e != cudaSuccess) return e;
    if (launched) *launched += 1;
  }
  return cudaGetLastError();
}

template <int NT>
static cudaError_t launch_step_multi_ring_n(const KernelArgs& a, const RingSink& g, int grid, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, step_multi_ring_kernel<NT>, a, g);
}

// step + replay append in one launch: the warp kernels only (N <= 32, float32 world)
cudaError_t launch_step_multi_ring(const KernelArgs& a, const RingSink& g, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  if (wants_seq(a)) return cudaErrorNotSupported;
  cudaError_t e = cudaSuccess;
  UAVCA_DISPATCH_N(a.N, (e = launch_step_multi_ring_n<NT>(a, g, multi_grid(a.B, a.N), st)));
  if (e != cudaSuccess) return e;
  return cudaGetLastError();
}

template <typename Kernel>
static cudaError_t launch_pdl2(Kernel kernel, int grid, cudaStream_t st, const KernelArgs& a, const RolloutArgs& r) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, a, r);
}

cudaError_t launch_rollout_multi(const KernelArgs& a, const RolloutArgs& r, cudaStream_t st) {
  if (a.B <= 0 || r.K <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  // 17..25 UAVs per env: the CTA-packed kernel (5..7 envs on the 128 threads of a CTA instead of one env per warp), as in
  // launch_step_multi; UAVCA_ROLLOUT_CTA=0 keeps the warp kernel (A/B measurements)
  static const bool cta_ok = [] { const char* v = getenv("UAVCA_ROLLOUT_CTA"); return !(v && v[0] == '0'); }();
  if (cta_ok && cta_packs(a.N, true)) {
    const int envs_per_cta = kThreads / a.N;
    e = launch_pdl2(rollout_multi_cta_kernel, (a.B + envs_per_cta - 1) / envs_per_cta, st, a, r);
    return e != cudaSuccess ? e : cudaGetLastError();
  }
  const int grid = multi_grid(a.B, a.N);
  const bool block = r.action_block != nullptr;
  // the plain instance (PlainRolloutIO): the action mode the plain call implies — cartesian block actions, Philox actions
  // scaled to the action box — and none of the optional outputs or accumulators.  Its step offsets are 32-bit: every
  // element offset of the launch's blocks, up to the observations' K * M * 10, must stay below 2^31.
  const bool plain = a.io.final_obs == nullptr && a.io.reset_mask == nullptr && !a.c.track_scores &&
                     (block ? a.io.action_mode == UAVCA_ACTION_CARTESIAN
                            : a.io.action_mode == UAVCA_ACTION_SCALED && r.action_out == nullptr) &&
                     (long long)r.K * r.M * UAVCA_OBS_DIM_MULTI < (1ll << 31);
  RolloutArgs rp = r;
  rp.KM = plain ? (unsigned)(r.K * r.M) : 0u;
  if (block && plain) {
    UAVCA_DISPATCH_N(a.N, (e = launch_pdl2(rollout_multi_kernel<NT, kRolloutPlainBlock>, grid, st, a, rp)));
  } else if (plain) {
    UAVCA_DISPATCH_N(a.N, (e = launch_pdl2(rollout_multi_kernel<NT, kRolloutPlainPhilox>, grid, st, a, rp)));
  } else {
    UAVCA_DISPATCH_N(a.N, (e = launch_pdl2(rollout_multi_kernel<NT, kRolloutGeneral>, grid, st, a, r)));
  }
  return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_rollout_single(const KernelArgs& a, const RolloutArgs& r, cudaStream_t st) {
  if (a.B <= 0 || r.K <= 0) return cudaSuccess;
  const cudaError_t e = launch_pdl2(rollout_single_kernel, flat_grid(a.B), st, a, r);
  return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_sample_actions(const Consts& c, float* out, int B, int N, unsigned long long seed, unsigned long long t,
                                  cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  sample_actions_kernel<<<flat_grid((long long)B * N), kThreads, 0, st>>>(c, reinterpret_cast<float2*>(out), B, N,
                                                                          (unsigned)(seed & 0xffffffffull),
                                                                          (unsigned)(seed >> 32), t);
  return cudaGetLastError();
}

cudaError_t launch_reset_multi(const KernelArgs& a, const uint8_t* mask, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  if (wants_seq(a)) {
    if (a.c.circular) reset_multi_seq_kernel<double><<<flat_grid(a.B), kThreads, 0, st>>>(a, mask);
    else reset_multi_seq_kernel<float><<<flat_grid(a.B), kThreads, 0, st>>>(a, mask);
    return cudaGetLastError();
  }
  const int grid = multi_grid(a.B, a.N);
  UAVCA_DISPATCH_N(a.N, (reset_multi_kernel<NT><<<grid, kThreads, 0, st>>>(a, mask)));
  return cudaGetLastError();
}

cudaError_t launch_observe_multi(const KernelArgs& a, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  if (wants_seq(a)) {
    if (a.c.circular) observe_multi_seq_kernel<double><<<flat_grid(a.B), kThreads, 0, st>>>(a);
    else observe_multi_seq_kernel<float><<<flat_grid(a.B), kThreads, 0, st>>>(a);
    return cudaGetLastError();
  }
  const int grid = multi_grid(a.B, a.N);
  UAVCA_DISPATCH_N(a.N, (observe_multi_kernel<NT><<<grid, kThreads, 0, st>>>(a)));
  return cudaGetLastError();
}

cudaError_t launch_step_single(const KernelArgs& a, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  step_single_kernel<<<flat_grid(a.B), kThreads, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_reset_single(const KernelArgs& a, const uint8_t* mask, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  reset_single_kernel<<<flat_grid(a.B), kThreads, 0, st>>>(a, mask);
  return cudaGetLastError();
}

cudaError_t launch_observe_single(const KernelArgs& a, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  observe_single_kernel<<<flat_grid(a.B), kThreads, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_map_action(const Consts& c, const float* in, float* out, long long M, int mode, cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  map_action_kernel<<<flat_grid(M), kThreads, 0, st>>>(c, reinterpret_cast<const float2*>(in),
                                                       reinterpret_cast<float2*>(out), M, mode);
  return cudaGetLastError();
}

cudaError_t launch_replay_sample(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                                 const float* r_mask, long long capacity, int obs_dim, int act_dim, const long long* meta,
                                 long long batch, unsigned long long seed, unsigned long long draw, int recency, float* o_obs,
                                 float* o_act, float* o_rew, float* o_nxt, float* o_mask, long long* o_idx, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  replay_sample_kernel<<<flat_grid(batch * kSampleLanes), kThreads, 0, st>>>(
      r_obs, r_act, r_rew, r_nxt, r_mask, capacity, obs_dim, act_dim, meta, batch, (unsigned)(seed & 0xffffffffull),
      (unsigned)(seed >> 32), draw, recency, o_obs, o_act, o_rew, o_nxt, o_mask, o_idx);
  return cudaGetLastError();
}

cudaError_t launch_replay_push(const float* obs, const float* action, const float* reward, const float* next_obs,
                               const uint8_t* done, long long M, int obs_dim, int act_dim, float* r_obs, float* r_act,
                               float* r_rew, float* r_next, float* r_mask, long long capacity, long long head,
                               long long* meta, cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  auto a8 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; };
  const bool wide = (obs_dim % 2 == 0) && (act_dim % 2 == 0) && a8(obs) && a8(action) && a8(next_obs) && a8(r_obs) &&
                    a8(r_act) && a8(r_next);
  const long long widest = (long long)(obs_dim > act_dim ? obs_dim : act_dim);
  if (wide) {
    const long long n = M * (widest / 2) > M ? M * (widest / 2) : M;
    replay_push_kernel<float2><<<(int)((n + kPushThreads - 1) / kPushThreads), kPushThreads, 0, st>>>(
        reinterpret_cast<const float2*>(obs), reinterpret_cast<const float2*>(action), reward,
        reinterpret_cast<const float2*>(next_obs), done, M, obs_dim / 2, act_dim / 2, reinterpret_cast<float2*>(r_obs),
        reinterpret_cast<float2*>(r_act), r_rew, reinterpret_cast<float2*>(r_next), r_mask, capacity, head, meta);
  } else {
    const long long n = M * (widest > 1 ? widest : 1);
    replay_push_kernel<float><<<(int)((n + kPushThreads - 1) / kPushThreads), kPushThreads, 0, st>>>(obs, action, reward, next_obs, done, M, obs_dim, act_dim,
                                                                  r_obs, r_act, r_rew, r_next, r_mask, capacity, head, meta);
  }
  return cudaGetLastError();
}

cudaError_t launch_stats(const StateView& s, int B, long long* out8, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(out8, 0, 8 * sizeof(long long), st);
  if (e != cudaSuccess) return e;
  int grid = flat_grid(B);
  if (grid > 148 * 4) grid = 148 * 4;
  if (grid < 1) grid = 1;
  stats_kernel<<<grid, kThreads, 0, st>>>(s, B, out8);
  return cudaGetLastError();
}

}  // namespace uavca

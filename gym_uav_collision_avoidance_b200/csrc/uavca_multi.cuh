// uavca_multi.cuh — warp-cooperative pieces of the multi-UAV world (MultiUAVWorld2D) shared by the step,
// reset and observe kernels.
//
// Thread mapping: one lane per UAV, the N lanes of an env are adjacent in one warp, floor(32/N) envs per warp.
// The flat UAV index of lane l in (global) warp w is  w * lanes_used + l, so every per-UAV array is read and
// written as one contiguous, coalesced run per warp.  Neighbour data never touches memory: lanes exchange
// positions and headings through a per-warp shared-memory scratch (broadcast loads).
#pragma once

#include "uavca_device.cuh"

namespace uavca {

struct Lane {
  int N;           // UAVs per env
  int lanes_used;  // floor(32/N) * N
  int lane;
  int i;            // UAV index inside its env
  int base;         // first lane of this lane's env
  int ring;         // float4 offset of this env's ring in WarpScratch::pairs
  unsigned envmask; // N low bits
  int env;          // env index inside the shard
  int m;            // flat UAV index env*N + i  (B*N < 2^31 is checked at uavca_create)
  int warp_m0;      // flat UAV index of lane 0 of this warp
  int valid_lanes;  // lanes of this warp that map to real UAVs (a prefix)
  bool valid;
};

// UAVs from warp `warp_global`'s first env to the end of the shard (>= lanes_used: the warp is full)
__device__ __forceinline__ int uavs_left(int B, int N, int warp_global) { return (B - warp_global * (32 / N)) * N; }

// FULL: the caller knows that every env slot of this warp maps to a real env (all warps but the last of a shard);
// the validity predicates then fold to compile-time constants.
template <int NT, bool FULL = false>
__device__ __forceinline__ Lane make_lane(int B, int Nrt, int warp_global) {
  Lane L;
  L.N = NT > 0 ? NT : Nrt;
  const int epw = 32 / L.N;
  L.lanes_used = epw * L.N;
  L.lane = threadIdx.x & 31;
  const int e_local = L.lane / L.N;
  L.i = L.lane - e_local * L.N;
  L.base = e_local * L.N;
  L.ring = e_local * (L.N + 1);
  L.envmask = L.N >= 32 ? 0xffffffffu : ((1u << L.N) - 1u);
  L.env = warp_global * epw + e_local;
  L.warp_m0 = warp_global * L.lanes_used;
  if (FULL) {
    L.valid_lanes = L.lanes_used;
  } else {
    const int left = uavs_left(B, L.N, warp_global);
    L.valid_lanes = left <= 0 ? 0 : (left < L.lanes_used ? left : L.lanes_used);
  }
  L.valid = L.lane < L.valid_lanes;
  L.m = L.warp_m0 + L.lane;
  if (!L.valid) { L.base = 0; L.ring = 0; L.i = 0; }  // idle lanes shadow UAV 0 of the warp's first env and never store
  return L;
}
template <int NT>
__device__ __forceinline__ Lane make_lane(int B, int Nrt) {
  return make_lane<NT, false>(B, Nrt, blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5));
}

struct Uav {
  float px, py, tx, ty, init, prev;
  double vx, vy;
  unsigned flags;
};

__device__ __forceinline__ Uav load_uav(const StateView& s, const Lane& L) {
  Uav u;
  if (L.valid) {
    float2 p = ld_stream(s.pos + L.m);
    double2 v = ld_stream(s.vel + L.m);
    float2 t = ld_stream(s.tgt + L.m);
    u.init = ld_stream(s.init + L.m);
    u.prev = ld_stream(s.prev + L.m);
    u.flags = ld_stream(s.flags + L.m);
    u.px = p.x; u.py = p.y; u.vx = v.x; u.vy = v.y; u.tx = t.x; u.ty = t.y;
  } else {
    // idle lanes (32 is not a multiple of N, or the ragged end of a shard) carry a harmless UAV in ordinary flight:
    // moving, 8 m from its target, inside the box.  A zero state would sit exactly on its target with zero velocity
    // and drag the whole warp through the rare paths (double-precision angles, finish()) on every step.
    u.px = u.py = u.ty = 0.f; u.tx = 8.f; u.init = u.prev = 8.f; u.vx = 1.0; u.vy = 0.0; u.flags = 0u;
  }
  return u;
}

__device__ __forceinline__ void store_uav(const StateView& s, const Lane& L, const Uav& u, bool with_target) {
  if (!L.valid) return;
  st_stream(s.pos + L.m, make_float2(u.px, u.py));
  st_stream(s.vel + L.m, make_double2(u.vx, u.vy));
  st_stream(s.prev + L.m, u.prev);
  st_stream(s.flags + L.m, (uint8_t)u.flags);
  if (with_target) {
    st_stream(s.tgt + L.m, make_float2(u.tx, u.ty));
    st_stream(s.init + L.m, u.init);
  }
}

// Per-warp shared-memory scratch.  Neighbour data never goes to global memory.
//   pairs  per env a DOUBLED ring of the NEW positions, two ring slots per float4: element q of an env's ring holds
//          (x[2q], x[2q+1], y[2q], y[2q+1]) with slot s < N = UAV s and slot N+s = UAV s again.  Lane i sweeps the slots
//          from its own even-aligned start, so one LDS.128 brings TWO neighbours laid out for packed FP32 (both
//          squared distances of the pair come out of 2 FADD2 + 2 FFMA2 with a +0 addend + 1 FADD2) and ring
//          neighbour i+k needs no index arithmetic, compare or select.
//   cand   per UAV (new.x, new.y, old.x, old.y): what the few selected neighbours are looked up in afterwards
//   th     per UAV heading / pi
struct WarpScratch {
  float4* pairs;  // [48]  env e_local at float4 offset e_local * (N + 1)
  float4* cand;   // [32]  by lane of the UAV
  float* th;      // [32]  by lane of the UAV
  float* stage;   // [320] observation rows of the warp
  // Small envs (SweepKind::kMixed) use the same memory as ONE doubled ring of (old, new) positions instead (see below):
  __device__ __forceinline__ float4* ring() const { return pairs; }                                    // [64]
  __device__ __forceinline__ float* ring_th() const { return reinterpret_cast<float*>(pairs) + 256; }  // [64]
};
// Up to this many UAVs per env the neighbour sweep computes BOTH distances of a neighbour (sequential pass and
// observation pass) in one packed instruction stream — 11.5 instructions per neighbour and nothing afterwards; above it
// the two-neighbours-per-load sweep of the new positions (8 per neighbour + ~30 once) wins.  Crossover at N ~ 12
// (ncu: N=8 executes 575 warp-instructions per step with the latter, ~550 with the former).
constexpr int kMixedMaxN = 10;
template <int NT>
struct SweepKind {
  static constexpr bool kMixed = NT > 0 && NT <= kMixedMaxN;
};
constexpr int kRingFloats = 48 * 4 + 32 * 4 + 32;
constexpr int kScratchFloats = kRingFloats + 32 * 10;

__device__ __forceinline__ WarpScratch warp_scratch(float* block_smem) {
  float* w = block_smem + (threadIdx.x >> 5) * kScratchFloats;
  return WarpScratch{reinterpret_cast<float4*>(w), reinterpret_cast<float4*>(w + 192), w + 320, w + kRingFloats};
}

__device__ __forceinline__ void publish(const WarpScratch& ws, const Lane& L, float nx, float ny, float ox, float oy, float th_u) {
  if (L.valid) {
    float* ring = reinterpret_cast<float*>(ws.pairs + L.ring);
    const int s0 = L.i, s1 = L.i + L.N;
    const int a0 = ((s0 >> 1) << 2) + (s0 & 1), a1 = ((s1 >> 1) << 2) + (s1 & 1);
    ring[a0] = nx; ring[a0 + 2] = ny;
    ring[a1] = nx; ring[a1 + 2] = ny;
    ws.cand[L.lane] = make_float4(nx, ny, ox, oy);
    ws.th[L.lane] = th_u;
  }
  __syncwarp();
}

// ---- neighbour search -----------------------------------------------------------------------------------------------
// The two nearest other UAVs of the env, ordered by (squared float32 distance, ring offset) — the order of
// `relative_distances.argsort()` (uav_agent.py:62) with the lowest ring offset first among exactly equal distances
// (the reference's own order of exact ties is undefined, SURVEY.md 7.3-4).  Results are ring offsets k (neighbour
// j = (i + k) mod N); 0 = none.

constexpr int kInfBits = 0x7f800000;

// Exact reference selection: branch-free insertion on the float32 squared distances themselves.  Out of line: it
// only runs for the rare lanes whose fast selection below is ambiguous.
static __device__ __noinline__ int nearest2_exact(const float4* cand, int i, int N, float px, float py) {
  const float inf = __int_as_float(kInfBits);
  float s1 = inf, s2 = inf;
  int j1 = 0, j2 = 0;
  for (int k = 1; k < N; ++k) {
    int j = i + k;
    j -= j >= N ? N : 0;
    const float4 q = cand[j];
    const float s = sq32(__fsub_rn(q.x, px), __fsub_rn(q.y, py));
    const bool p1 = s < s1, p2 = s < s2;
    j2 = p1 ? j1 : (p2 ? k : j2);
    s2 = p1 ? s1 : (p2 ? s : s2);
    j1 = p1 ? k : j1;
    s1 = p1 ? s : s1;
  }
  return j1 | (j2 << 8);
}

// Pass A of MultiUAVWorld2D.step in full (multi_uav_world_2d.py:198-210): the squared distance to the nearest other
// UAV with j < i at its NEW position and j > i at its OLD one (the reference moves and tests the UAVs one after the
// other).  Out of line: only lanes with three or more UAVs within collision reach need the whole sweep.
static __device__ __noinline__ float nearest_mixed_exact(const float4* cand, int i, int N, float px, float py) {
  float smin = __int_as_float(kInfBits);
  for (int j = 0; j < N; ++j) {
    if (j == i) continue;
    const float4 q = cand[j];
    const float s = j < i ? sq32(__fsub_rn(q.x, px), __fsub_rn(q.y, py)) : sq32(__fsub_rn(q.z, px), __fsub_rn(q.w, py));
    smin = fminf(smin, s);
  }
  return smin;
}

// One sweep over the env's other UAVs at their NEW positions (what _get_obs sees, multi_uav_world_2d.py:75), two
// neighbours per step.  It keeps the THREE smallest integer keys (distance bits with the low 5 bits replaced by the
// element number of the sweep): integer min/max only, two neighbours merged per step with the
// k-th-smallest-of-two-sorted-lists identities
//   t1' = min(t1, a)   t2' = min(t2, max(t1, a), b)   t3' = min(t3, max(t2, a), max(t1, b))       (a <= b).
// A key orders like (distance truncated to 19 mantissa bits, ring offset).  If the truncated distances of the three
// smallest keys are pairwise different, truncation cannot have reordered anything and t1, t2 are exactly the
// reference's two nearest; otherwise (two of them within 2^-18 relative, ~1e-4 of the lanes at N=32) the lane
// re-runs the exact selection.  t3 — a lower bound of the third-smallest distance — also tells the caller whether
// anybody besides the two nearest can be within collision reach.
//
// Lane i starts at the even slot s0 = i + (i & 1); element e of its sweep is ring offset k = (i & 1) + e.  Offsets
// 0 and N (the lane's own two ring slots) and anything beyond are masked with "none" keys.
template <int NT>
__device__ __forceinline__ void pair_scan(const Consts& c, const WarpScratch& ws, const Lane& L, float px, float py,
                                          int& k1, int& k2, int& t3_out) {
  const int N = NT > 0 ? NT : L.N;
  const int k0 = L.i & 1;
  const float4* row = ws.pairs + L.ring + ((L.i + 1) >> 1);
  const float2 npx = make_float2(-px, -px), npy = make_float2(-py, -py), zero = make_float2(0.f, 0.f);
  // squares and sum rounded separately, exactly as sq32().  The squares are FFMA2 with a +0 addend: a plain
  // mul.rn.f32x2 feeding add.rn.f32x2 is contracted into one FFMA2 by ptxas 12.9 (even under -fmad=false), which
  // would break the unfused np.linalg.norm order.
  auto dist2 = [&](int p) {
    const float4 q = row[p];
    const float2 dx = __fadd2_rn(make_float2(q.x, q.y), npx), dy = __fadd2_rn(make_float2(q.z, q.w), npy);
    return __fadd2_rn(__ffma2_rn(dx, dx, zero), __ffma2_rn(dy, dy, zero));
  };
  // the mask (~31) comes from the constant bank on purpose: with an opaque mask and an immediate element number the
  // key is ONE LOP3 ((s & mask) | e); as two literals it would be two
  const int mask = c.key_mask;
  auto key = [&](float sq, int e) {
    int kk = (__float_as_int(sq) & mask) | e;
    // valid iff 1 <= k0 + e <= N - 1; "none" keys lie above every real key and are pairwise unambiguous
    if (e >= N) return kInfBits + 5 * 32;
    if (e == 0) kk = k0 ? kk : kInfBits + 3 * 32;
    if (e == N - 1) kk = k0 ? kInfBits + 4 * 32 : kk;
    return kk;
  };
  int t1 = kInfBits, t2 = kInfBits + 32, t3 = kInfBits + 64;
  auto merge = [&](int ka, int kb) {
    const int a = min(ka, kb), b = max(ka, kb);
    const int m1a = max(t1, a), m2a = max(t2, a), m1b = max(t1, b);
    t3 = __vimin3_s32(t3, m2a, m1b);
    t2 = __vimin3_s32(t2, m1a, b);
    t1 = min(t1, a);
  };
  if (N > 1) {
    const int P = (N + 1) >> 1;
    if (NT > 0) {
#pragma unroll
      for (int p = 0; p < P; ++p) {
        const float2 s = dist2(p);
        merge(key(s.x, 2 * p), key(s.y, 2 * p + 1));
      }
    } else {
      for (int p = 0; p < P; ++p) {
        const float2 s = dist2(p);
        merge(key(s.x, 2 * p), key(s.y, 2 * p + 1));
      }
    }
  }
  k1 = t1 < kInfBits ? k0 + (t1 & 31) : 0;
  k2 = t2 < kInfBits ? k0 + (t2 & 31) : 0;
  t3_out = t3;
  if (((unsigned)(t1 ^ t2) < 32u) | ((unsigned)(t2 ^ t3) < 32u)) {
    const int e = nearest2_exact(ws.cand + L.base, L.i, N, px, py);
    k1 = e & 0xff;
    k2 = e >> 8;
  }
}

// The two selected neighbours, looked up by ring offset: observation features 4..9 (MultiUAVWorld2D._get_obs,
// multi_uav_world_2d.py:75-95) and, for the step, the collision distance of pass A.
// Neighbour bearings/headings are differences of float32 angles (absolute error ~2e-7 of a half-turn).
struct ObsTail {
  float2 a, b, c;  // (o4, o5) (o6, o7) (o8, o9)
};
// Observation features 4..9 from the two selected neighbours (multi_uav_world_2d.py:75-95).
__device__ __forceinline__ ObsTail obs_tail(const Consts& c, float dx1, float dy1, float dx2, float dy2, float s1, float s2,
                                            float h1, float h2, bool have1, bool have2, float th_u) {
  const float2 b = fast_atan2_pair(dy1, dx1, dy2, dx2);
  const float2 nth = make_float2(-th_u, -th_u);
  const float2 v1 = wrap_units2(__ffma2_rn(b, make_float2(c.inv_pi, c.inv_pi), nth));  // bearings relative to the heading
  const float2 v2 = wrap_units2(__fadd2_rn(make_float2(h1, h2), nth));                 // neighbour headings, relative
  const float2 d = __fmul2_rn(make_float2(sqrt_approx(s1), sqrt_approx(s2)), make_float2(c.inv_dsense, c.inv_dsense));
  ObsTail o;
  o.a.x = have1 ? d.x : 1.0f;                             // :77
  o.a.y = have1 ? v1.x : 1.0f;                            // :78-81 (no neighbour: bearing pi)
  o.b.x = have1 ? v2.x : 0.0f;                            // :82-85
  o.b.y = have2 ? d.y : 1.0f;                             // :87
  o.c.x = have2 ? v1.y : 1.0f;                            // :88-91
  o.c.y = have2 ? v2.y : 0.0f;                            // :92-95
  return o;
}

// smin (WANT_A): squared distance to the nearest other UAV as the reference's sequential sweep sees it — j < i at the
// NEW position, j > i at the OLD one (multi_uav_world_2d.py:181-210).  Only a UAV within `near` of the new position
// can be within collision reach of the old one (a UAV moves at most sqrt(2) v_max tau per step; Consts::near_key),
// so unless the third-smallest key is that close the two nearest are the only candidates.
template <int NT, bool WANT_A>
__device__ __forceinline__ ObsTail neighbours(const Consts& c, const WarpScratch& ws, const Lane& L, float px, float py,
                                              float th_u, int k1, int k2, int t3, float& smin) {
  const int N = NT > 0 ? NT : L.N;
  int j1 = L.i + k1, j2 = L.i + k2;
  const bool w1 = j1 >= N, w2 = j2 >= N;  // wrapped: j < i
  j1 -= w1 ? N : 0;
  j2 -= w2 ? N : 0;
  const float4 q1 = ws.cand[L.base + j1], q2 = ws.cand[L.base + j2];
  const float h1 = ws.th[L.base + j1], h2 = ws.th[L.base + j2];
  const float dx1 = __fsub_rn(q1.x, px), dy1 = __fsub_rn(q1.y, py), dx2 = __fsub_rn(q2.x, px), dy2 = __fsub_rn(q2.y, py);
  const float s1 = sq32(dx1, dy1), s2 = sq32(dx2, dy2);  // the exact squared distances of the two winners
  if (WANT_A) {
    const float inf = __int_as_float(kInfBits);
    float a1 = w1 ? s1 : sq32(__fsub_rn(q1.z, px), __fsub_rn(q1.w, py));
    float a2 = w2 ? s2 : sq32(__fsub_rn(q2.z, px), __fsub_rn(q2.w, py));
    a1 = k1 != 0 ? a1 : inf;
    a2 = k2 != 0 ? a2 : inf;
    smin = fminf(a1, a2);
    if (t3 <= c.near_key) smin = nearest_mixed_exact(ws.cand + L.base, L.i, N, px, py);
  }
  const bool have1 = (k1 != 0) & (s1 < c.s_dsense_lt);  // uav_agent.py:52 strict <
  const bool have2 = have1 & (k2 != 0) & (s2 < c.s_dsense_lt);
  return obs_tail(c, dx1, dy1, dx2, dy2, s1, s2, h1, h2, have1, have2, th_u);
}

// ---- small envs: one sweep for both pairwise passes ----------------------------------------------------------------------
// Each env owns a DOUBLED ring of 2N slots: slot m < N holds UAV m's (old position, new position), slot N+m holds (new,
// new).  Lane i reads slot i+k for k = 1..N-1, i.e. its ring neighbour j = (i+k) mod N, and receives as "a" exactly the
// position the reference's sequential sweep would see — OLD for j > i (not moved yet), NEW for j < i — and as "n" the NEW
// position, with no index arithmetic, no compare and no select.  A slot is laid out (a.x, n.x, a.y, n.y) so that both
// squared distances come out of five packed FP32 instructions (2 FADD2, 2 FFMA2 with a +0 addend, FADD2).
__device__ __forceinline__ void publish_mixed(const WarpScratch& ws, const Lane& L, float nx, float ny, float ox, float oy, float th_u) {
  if (L.valid) {
    const int slot = 2 * L.base + L.i;
    ws.ring()[slot] = make_float4(ox, nx, oy, ny);
    ws.ring()[slot + L.N] = make_float4(nx, nx, ny, ny);
    ws.ring_th()[slot] = th_u;
    ws.ring_th()[slot + L.N] = th_u;
  }
  __syncwarp();
}

static __device__ __noinline__ int nearest2_exact_ring(const float4* row, float px, float py, int N) {
  const float inf = __int_as_float(kInfBits);
  float s1 = inf, s2 = inf;
  int j1 = 0, j2 = 0;
  for (int k = 1; k < N; ++k) {
    const float4 q = row[k];
    const float s = sq32(__fsub_rn(q.y, px), __fsub_rn(q.w, py));
    const bool p1 = s < s1, p2 = s < s2;
    j2 = p1 ? j1 : (p2 ? k : j2);
    s2 = p1 ? s1 : (p2 ? s : s2);
    j1 = p1 ? k : j1;
    s1 = p1 ? s : s1;
  }
  return j1 | (j2 << 8);
}

// pass A (multi_uav_world_2d.py:198-210) -> smin; pass B (:75 via _get_obs) -> the ring offsets k1, k2 of the two nearest
template <int NT>
__device__ __forceinline__ void pair_scan_mixed(const Consts& c, const WarpScratch& ws, const Lane& L, float px, float py,
                                                float& smin, int& k1, int& k2) {
  constexpr int N = NT;
  const float4* row = ws.ring() + 2 * L.base + L.i;
  const float2 npx = make_float2(-px, -px), npy = make_float2(-py, -py), zero = make_float2(0.f, 0.f);
  auto dist2 = [&](int k) {  // (pass-A distance, pass-B distance) of ring neighbour k, each exactly sq32()
    const float4 q = row[k];
    const float2 dx = __fadd2_rn(make_float2(q.x, q.y), npx), dy = __fadd2_rn(make_float2(q.z, q.w), npy);
    return __fadd2_rn(__ffma2_rn(dx, dx, zero), __ffma2_rn(dy, dy, zero));
  };
  const int mask = c.key_mask;
  auto key = [mask](float sq, int k) { return (__float_as_int(sq) & mask) | k; };
  smin = __int_as_float(kInfBits);
  int t1 = kInfBits, t2 = kInfBits + 32, t3 = kInfBits + 64;
  int k = 1;
#pragma unroll
  for (; k + 1 < N; k += 2) {
    const float2 s0 = dist2(k), s1 = dist2(k + 1);
    smin = fminf(smin, fminf(s0.x, s1.x));
    const int ka = key(s0.y, k), kb = key(s1.y, k + 1);
    const int a = min(ka, kb), b = max(ka, kb);
    const int m1a = max(t1, a), m2a = max(t2, a), m1b = max(t1, b);
    t3 = __vimin3_s32(t3, m2a, m1b);
    t2 = __vimin3_s32(t2, m1a, b);
    t1 = min(t1, a);
  }
  if (k < N) {
    const float2 s0 = dist2(k);
    smin = fminf(smin, s0.x);
    const int a = key(s0.y, k);
    t3 = min(t3, max(t2, a));
    t2 = min(t2, max(t1, a));
    t1 = min(t1, a);
  }
  k1 = t1 & 31;
  k2 = t2 & 31;
  if (((unsigned)(t1 ^ t2) < 32u) | ((unsigned)(t2 ^ t3) < 32u)) {
    const int e = nearest2_exact_ring(row, px, py, N);
    k1 = e & 0xff;
    k2 = e >> 8;
  }
}

__device__ __forceinline__ ObsTail neighbours_mixed(const Consts& c, const WarpScratch& ws, const Lane& L, float px, float py,
                                                    float th_u, int k1, int k2) {
  const int slot = 2 * L.base + L.i;
  const float4 q1 = ws.ring()[slot + k1], q2 = ws.ring()[slot + k2];
  const float h1 = ws.ring_th()[slot + k1], h2 = ws.ring_th()[slot + k2];
  // both neighbours at once on the packed FP32 pipe, each element exactly as __fsub_rn / sq32 (see dist2 of pair_scan_mixed)
  const float2 dx = __fadd2_rn(make_float2(q1.y, q2.y), make_float2(-px, -px)), dy = __fadd2_rn(make_float2(q1.w, q2.w), make_float2(-py, -py));
  const float2 zero = make_float2(0.f, 0.f), s = __fadd2_rn(__ffma2_rn(dx, dx, zero), __ffma2_rn(dy, dy, zero));
  const bool have1 = (k1 != 0) & (s.x < c.s_dsense_lt);
  const bool have2 = have1 & (k2 != 0) & (s.y < c.s_dsense_lt);
  return obs_tail(c, dx.x, dy.x, dx.y, dy.y, s.x, s.y, h1, h2, have1, have2, th_u);
}

// Both pairwise passes of a step (or just the observation pass of a state at rest: old == new) for this lane's UAV:
// publish, sweep, look the two nearest up.  All lanes must call.  smin: squared distance to the nearest other UAV as the
// reference's sequential sweep sees it.
template <int NT>
__device__ __forceinline__ ObsTail scan_neighbours(const Consts& c, const WarpScratch& ws, const Lane& L, float nx, float ny,
                                                   float ox, float oy, float th_u, float& smin) {
  int k1, k2;
  if (SweepKind<NT>::kMixed) {
    publish_mixed(ws, L, nx, ny, ox, oy, th_u);
    pair_scan_mixed<NT>(c, ws, L, nx, ny, smin, k1, k2);
    return neighbours_mixed(c, ws, L, nx, ny, th_u, k1, k2);
  }
  int t3;
  publish(ws, L, nx, ny, ox, oy, th_u);
  pair_scan<NT>(c, ws, L, nx, ny, k1, k2, t3);
  return neighbours<NT, true>(c, ws, L, nx, ny, th_u, k1, k2, t3, smin);
}

// Everything the step and the observation need from a UAV's own state.
//   th_u    own heading atan2(v.y, v.x) / pi                                   (multi_uav_world_2d.py:63-64)
//   dth_u   wrap(bearing to target - heading) / pi                             (:69-72, :184-186)
//   dist    float32 distance to the target, ssq its square                      (:67)
//   vsq     |v|^2 in float64
// The heading error is ONE atan2 of the cross / dot products of heading and target direction, formed in float32
// from exactly representable differences: absolute error ~1e-7 rad, relative accuracy kept down to small angles.
struct Own {
  float th_u, dth_u, dist, ssq;
  double vsq;
};
__device__ __forceinline__ Own own_features(const Consts& c, float px, float py, float tx, float ty, double vx, double vy) {
  Own w;
  // the two differences and the two squares on the packed FP32 pipe, each element exactly as __fsub_rn / sq32 (the
  // squares as FFMA2 with a +0 addend, see pair_scan; a square is never -0)
  const float2 td = __fadd2_rn(make_float2(tx, ty), make_float2(-px, -py));
  const float tdx = td.x, tdy = td.y;
  const float2 tsq = __ffma2_rn(td, td, make_float2(0.f, 0.f));
  w.ssq = __fadd_rn(tsq.x, tsq.y);
  w.dist = __fsqrt_rn(w.ssq);
  w.vsq = sq64(vx, vy);
  const float fvx = (float)vx, fvy = (float)vy;
  // a velocity of exactly zero is common (the clipped acceleration walks v on a lattice of multiples of amax*tau
  // that contains 0, and every UAV starts at rest): atan2(0, 0) = 0, i.e. the heading points along +x
  const bool vzero = (vx == 0.0) & (vy == 0.0);
  const float hx = vzero ? 1.0f : fvx;
  const float cr = fmaf(hx, tdy, -(fvy * tdx));
  const float dt = fmaf(hx, tdx, fvy * tdy);
  const float2 ang = fast_atan2_pair(fvy, fvx, cr, dt);
  w.th_u = ang.x * c.inv_pi;
  w.dth_u = ang.y * c.inv_pi;
  // never seen in ordinary flight: a denormal-tiny non-zero velocity, or a UAV exactly on its target ->
  // the reference's own formulas in double
  if ((!vzero & (fabsf(fvx) + fabsf(fvy) < 1e-30f)) | (w.ssq == 0.0f)) {
    const float2 s = angles_slow((double)tdx, (double)tdy, vx, vy);
    w.th_u = s.x; w.dth_u = s.y;
  }
  return w;
}

__device__ __forceinline__ void obs_own(const Consts& c, const Own& w, double vsq, float2& o01, float2& o23) {
  o01 = make_float2(sqrt_approx((float)vsq) * c.inv_vm2_f, w.th_u);  // :62-64
  o23 = make_float2(w.dist * c.inv_diag, w.dth_u);                   // :67-72
}

// Observation of a state at rest (reset / observe kernels): publish, scan, build.  All lanes must call.
struct ObsRow {
  float2 o01, o23;
  ObsTail n;
};
template <int NT>
__device__ __forceinline__ ObsRow observe_state(const Consts& c, const WarpScratch& ws, const Lane& L, const Uav& u) {
  const Own w = own_features(c, u.px, u.py, u.tx, u.ty, u.vx, u.vy);
  __syncwarp();
  ObsRow r;
  obs_own(c, w, w.vsq, r.o01, r.o23);
  float unused;
  r.n = scan_neighbours<NT>(c, ws, L, u.px, u.py, u.px, u.py, w.th_u, unused);
  return r;
}

// The warp's observation rows go out as one contiguous run of 16-byte stores, staged through shared memory (a
// per-thread row is 40 bytes, which would otherwise scatter 8-byte stores 40 bytes apart).
__device__ __forceinline__ void stage_own(float* stage, int lane, float2 o01, float2 o23) {
  float2* row = reinterpret_cast<float2*>(stage) + lane * 5;
  row[0] = o01; row[1] = o23;
}
__device__ __forceinline__ void stage_neighbours(float* stage, int lane, const ObsTail& n) {
  float2* row = reinterpret_cast<float2*>(stage) + lane * 5;
  row[2] = n.a; row[3] = n.b; row[4] = n.c;
}
// all lanes; the caller has __syncwarp()ed after the last stage_* call
__device__ __forceinline__ void flush_warp_rows(const float* stage, float* g, const Lane& L);
__device__ __forceinline__ void flush_rows(const float* stage, float* gobs, const Lane& L) {
  flush_warp_rows(stage, gobs + (size_t)L.warp_m0 * 10, L);
}
// g: where the first row of this warp goes
__device__ __forceinline__ void flush_warp_rows(const float* stage, float* g, const Lane& L) {
  const int n2 = L.valid_lanes * 5;  // float2 elements to write
  if ((L.lanes_used & 1) == 0) {     // every warp's run starts on a 16-byte boundary
    const int n4 = n2 >> 1;          // <= 80
    const float4* s4 = reinterpret_cast<const float4*>(stage);
    float4* g4 = reinterpret_cast<float4*>(g);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int k = L.lane + 32 * r;
      if (k < n4) st_stream(g4 + k, s4[k]);
    }
    if ((n2 & 1) && L.lane == 0) st_stream(reinterpret_cast<float2*>(g) + (n2 - 1), reinterpret_cast<const float2*>(stage)[n2 - 1]);
  } else {
    const float2* s2 = reinterpret_cast<const float2*>(stage);
    float2* g2 = reinterpret_cast<float2*>(g);
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const int k = L.lane + 32 * r;
      if (k < n2) st_stream(g2 + k, s2[k]);
    }
  }
}
// The same stage by its shared-memory address (a 32-bit register computed once, where a loop would otherwise rebuild the
// generic pointer from the thread index every step)
__device__ __forceinline__ void sts_float2(unsigned smem_dst, float2 v) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(smem_dst), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ float2 lds_float2(unsigned smem_src) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(smem_src) : "memory");
  return v;
}
__device__ __forceinline__ float4 lds_float4(unsigned smem_src) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_src) : "memory");
  return v;
}
__device__ __forceinline__ void stage_own(unsigned stage, int lane, float2 o01, float2 o23) {
  const unsigned row = stage + lane * 40;
  sts_float2(row, o01); sts_float2(row + 8, o23);
}
__device__ __forceinline__ void stage_neighbours(unsigned stage, int lane, const ObsTail& n) {
  const unsigned row = stage + lane * 40;
  sts_float2(row + 16, n.a); sts_float2(row + 24, n.b); sts_float2(row + 32, n.c);
}
__device__ __forceinline__ void flush_warp_rows(unsigned stage, float* g, const Lane& L) {
  const int n2 = L.valid_lanes * 5;
  if ((L.lanes_used & 1) == 0) {
    const int n4 = n2 >> 1;
    float4* g4 = reinterpret_cast<float4*>(g);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int k = L.lane + 32 * r;
      if (k < n4) st_stream(g4 + k, lds_float4(stage + k * 16));
    }
    if ((n2 & 1) && L.lane == 0) st_stream(reinterpret_cast<float2*>(g) + (n2 - 1), lds_float2(stage + (n2 - 1) * 8));
  } else {
    float2* g2 = reinterpret_cast<float2*>(g);
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const int k = L.lane + 32 * r;
      if (k < n2) st_stream(g2 + k, lds_float2(stage + k * 8));
    }
  }
}
__device__ __forceinline__ void store_obs_rows(float* stage, float* gobs, const Lane& L, const ObsRow& o) {
  __syncwarp();
  stage_own(stage, L.lane, o.o01, o.o23);
  stage_neighbours(stage, L.lane, o.n);
  __syncwarp();
  flush_rows(stage, gobs, L);
}

// Start a new episode for the envs of this warp whose lanes pass do_reset (env-uniform).  Restates
// MultiUAVWorld2D.reset (multi_uav_world_2d.py:116-168): sequential rejection sampling — UAV i is re-drawn until it
// is farther than 2r from every UAV j<i, targets likewise plus farther than 2r from the UAV's own start.  The
// sequential dependency is kept (UAV `cur` is settled only after 0..cur-1), but each test runs across the lanes of
// the env at once.  All lanes of the warp must call.  `episode` is this env's episode counter BEFORE the reset.
__device__ __forceinline__ void reset_multi(const KernelArgs& a, const Lane& L, bool do_reset, unsigned episode, Uav& u) {
  const Consts& c = a.c;
  const long long env_global = c.env_base + L.env;
  if (c.reset_source == UAVCA_SOURCE_POOL && a.pool.pos != nullptr) {
    if (do_reset) {
      const long long p = (env_global + (long long)episode) % a.pool_envs;
      const long long pm = p * L.N + L.i;
      float2 pp = a.pool.pos[pm], pt = a.pool.tgt[pm];
      double2 pv = a.pool.vel[pm];
      u.px = pp.x; u.py = pp.y; u.tx = pt.x; u.ty = pt.y; u.vx = pv.x; u.vy = pv.y;
      u.init = a.pool.init[pm]; u.prev = a.pool.prev[pm]; u.flags = a.pool.flags[pm];
    }
    return;
  }
  const int N = L.N;
  // ---- start positions (:126-137)
  unsigned attempt = 0;
  float2 cand = make_float2(0.f, 0.f);
  if (do_reset) cand = draw_pair(c, env_global, episode, kStreamPos, L.i, 0u, c.lox, c.hix, c.loy, c.hiy);
  int cur = do_reset ? 1 : N;
  while (__any_sync(kFull, cur < N)) {
    const bool active = cur < N;
    const int src = L.base + (active ? cur : 0);
    const float qx = __shfl_sync(kFull, cand.x, src), qy = __shfl_sync(kFull, cand.y, src);
    const unsigned att = __shfl_sync(kFull, attempt, src);
    const bool conflict = active && (L.i < cur) && (n32(__fsub_rn(cand.x, qx), __fsub_rn(cand.y, qy)) <= c.two_r);
    const unsigned bal = __ballot_sync(kFull, conflict);
    const bool env_conflict = ((bal >> L.base) & L.envmask) != 0u;
    if (active) {
      if (env_conflict && att + 1u < kMaxResetAttempts) {
        if (L.i == cur) {
          ++attempt;
          cand = draw_pair(c, env_global, episode, kStreamPos, L.i, attempt, c.lox, c.hix, c.loy, c.hiy);
        }
      } else {
        ++cur;
      }
    }
  }
  // ---- targets (:140-153)
  float2 tg = make_float2(0.f, 0.f);
  attempt = 0;
  if (do_reset) tg = draw_pair(c, env_global, episode, kStreamTgt, L.i, 0u, c.lox, c.hix, c.loy, c.hiy);
  cur = do_reset ? 0 : N;
  while (__any_sync(kFull, cur < N)) {
    const bool active = cur < N;
    const int src = L.base + (active ? cur : 0);
    const float qx = __shfl_sync(kFull, tg.x, src), qy = __shfl_sync(kFull, tg.y, src);
    const unsigned att = __shfl_sync(kFull, attempt, src);
    bool conflict = false;
    if (active && L.i < cur) conflict = n32(__fsub_rn(tg.x, qx), __fsub_rn(tg.y, qy)) <= c.two_r;
    if (active && L.i == cur) conflict = n32(__fsub_rn(tg.x, cand.x), __fsub_rn(tg.y, cand.y)) <= c.two_r;
    const unsigned bal = __ballot_sync(kFull, conflict);
    const bool env_conflict = ((bal >> L.base) & L.envmask) != 0u;
    if (active) {
      if (env_conflict && att + 1u < kMaxResetAttempts) {
        if (L.i == cur) {
          ++attempt;
          tg = draw_pair(c, env_global, episode, kStreamTgt, L.i, attempt, c.lox, c.hix, c.loy, c.hiy);
        }
      } else {
        ++cur;
      }
    }
  }
  if (do_reset) {
    u.px = cand.x; u.py = cand.y; u.tx = tg.x; u.ty = tg.y;
    u.vx = 0.0; u.vy = 0.0; u.flags = 0u;                              // :118-123
    u.init = n32(__fsub_rn(u.tx, u.px), __fsub_rn(u.ty, u.py));        // :154
    u.prev = u.init;                                                   // :155
  }
}

// ================================================================================================================
// The step itself, independent of where the state and the I/O live.  `IO` is a policy that moves one UAV's data:
//   GlobalIO / GlobalIO64 (uavca_kernels.cu)  per-lane streaming global loads/stores, float32 / float64 actions
//   RingIO                (uavca_kernels.cu)  GlobalIO's outputs, and each transition appended to a device replay ring
//   RolloutIO / PlainRolloutIO (uavca_kernels.cu)  state in registers for K steps, outputs to [K][...] blocks
// All of them run exactly this code, so they cannot disagree on semantics.
//
//   Uav   load_uav();  float2 load_action();  int load_steps();        (load_steps: every lane, its env's counter)
//   void  loads_done();                                                (every input of this warp is in registers)
//   void  store_reward_done(float r, bool done);
//   void  put_own(float2 o01, float2 o23);  void put_neighbours(const ObsTail&);     observation row of this lane
//   void  commit_obs();  void commit_final();                          (all lanes; rows -> obs / final_obs)
//   void  store_state(const Uav&);        pos, vel, prev, flags
//   void  store_target(const Uav&);       tgt, init (reset lanes only)
//   void  store_steps(int, bool leader);  (every valid lane; the leader lane writes the env's counter)
//   void  store_reset(bool);              (env leader lanes only: the env auto-reset this step)
//   bool  wants_final();
// ================================================================================================================

// Sum of v over the N adjacent lanes of this lane's env (valid in the env's first lane).
__device__ __forceinline__ float env_sum(float v, const Lane& L) {
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const float o = __shfl_down_sync(kFull, v, off);
    v += (L.i + off < L.N) ? o : 0.0f;
  }
  return v;
}

// An env starts a new episode: its running scores join the totals over finished episodes (stats[4], stats[5]: doubles).
__device__ __forceinline__ void fold_scores(const StateView& s, int env) {
  const double2 sc = s.score[env];
  atomicAdd(reinterpret_cast<double*>(s.stats + 4), sc.x);
  atomicAdd(reinterpret_cast<double*>(s.stats + 5), sc.y);
  s.score[env] = make_double2(0.0, 0.0);
}

// UAVAgent.finish (uav_agent.py:38-42): park at 1 mm/s along the current heading (NaN -> 0 for a zero velocity)
static __device__ __forceinline__ double2 finish_velocity(double vx, double vy, double vsq) {
  const double nv = sqrt(vsq);
  double fx = __dmul_rn(__ddiv_rn(vx, nv), 0.001), fy = __dmul_rn(__ddiv_rn(vy, nv), 0.001);
  if ((fx != fx) | (fy != fy)) { fx = 0.0; fy = 0.0; }
  return make_double2(fx, fy);
}

// An I/O policy that declares `static constexpr bool kAction64 = true` hands the step FLOAT64 cartesian actions
// (`double2 load_action64()`, uavca_step_f64) instead of float32 ones; everything else in step_core is the same code.
template <class IO, class = void>
struct io_action64 { static constexpr bool value = false; };
template <class IO>
struct io_action64<IO, decltype((void)IO::kAction64)> { static constexpr bool value = IO::kAction64; };
// An I/O policy that declares `static constexpr bool kPlain = true` hands the step cartesian actions (already mapped)
// and is used only where the launch tracks no scores (Consts::track_scores == 0): neither is then tested at run time.
template <class IO, class = void>
struct io_plain { static constexpr bool value = false; };
template <class IO>
struct io_plain<IO, decltype((void)IO::kPlain)> { static constexpr bool value = IO::kPlain; };

template <int NT, class IO>
__device__ __forceinline__ void step_core(const KernelArgs& a, const WarpScratch& ws, const Lane& L, IO& io) {
  const Consts& c = a.c;
  constexpr bool kF64 = io_action64<IO>::value;
  constexpr bool kPlain = io_plain<IO>::value;

  Uav u = io.load_uav();
  float2 act = make_float2(0.f, 0.f);
  double2 act64 = make_double2(0.0, 0.0);
  if constexpr (kF64) act64 = io.load_action64();
  else act = io.load_action();
  const int steps_new = io.load_steps() + 1;  // multi_uav_world_2d.py:238
  io.loads_done();
  if constexpr (!kF64 && !kPlain) {
    if (a.io.action_mode != UAVCA_ACTION_CARTESIAN) act = map_action(act, a.io.action_mode, c);
  }

  const bool parked = (u.flags & UAVCA_FLAG_PARKED) != 0u;
  const float ox = u.px, oy = u.py;  // position before this step

  // ---- UAVAgent.step (uav_agent.py:23-36); parked UAVs do not move and report (0, 0)
  {
    double vx = u.vx, vy = u.vy;
    float px = u.px, py = u.py;
    if constexpr (kF64) integrate(act64.x, act64.y, vx, vy, px, py, c);
    else integrate((double)act.x, (double)act.y, vx, vy, px, py, c);
    if (!parked) { u.vx = vx; u.vy = vy; u.px = px; u.py = py; }
  }
  // heading, heading error to the target, distance, |v|^2 (multi_uav_world_2d.py:184-186)
  const Own w = own_features(c, u.px, u.py, u.tx, u.ty, u.vx, u.vy);
  const float dist = parked ? 0.f : w.dist;
  const float prev_d = parked ? 0.f : u.prev;

  // ---- reward shaping (:188-195).  Output only: float32 arithmetic, well inside the 1e-5 tolerance.
  float r;
  {
    const float inv_init = rcp_approx(u.init);
    const float m = fminf(c.vm2_f * inv_init, 1.0f);  // min(vm2/init, 1)
    r = fmaf(50.0f * c.inv_vm2_f, __fsub_rn(prev_d, dist), -0.01f * m);
    const float q = dist * inv_init * (1.0f / 1.5f);
    r *= (r > 0.0f) ? (1.0f - q) : (1.0f + q);
    r = fmaf(-0.01f * 3.14159274101257324f, fabsf(w.dth_u), r);
  }

  // ---- both pairwise passes: one sweep at the NEW positions for the two nearest (observation), from which the
  // collision distance of the sequential pass follows (neighbours())
  float smin;
  const ObsTail tail = scan_neighbours<NT>(c, ws, L, u.px, u.py, ox, oy, w.th_u, smin);

  // ---- collisions (:199-210), decided in squared-distance space (the thresholds already include "in sensing range")
  const bool collision = smin <= c.s_coll_le;
  r = collision ? -2.0f : r;
  const bool hard = (smin <= c.s_hard_le) & ((u.flags & (UAVCA_FLAG_PARKED | UAVCA_FLAG_COLLIDED)) == 0u) & L.valid;
  if (hard) u.flags |= UAVCA_FLAG_COLLIDED;

  // ---- done logic (:213-227)
  const bool inside = (u.px >= c.lox_f) & (u.px <= c.hix_f) & (u.py >= c.loy_f) & (u.py <= c.hiy_f);
  const bool reached = (parked ? true : (w.ssq < c.s_reach_lt)) & !collision & (w.vsq < c.reach_speed_sq);
  const bool newly_reached = reached & !parked & L.valid;
  const bool done = (reached | (!inside & (a.io.evaluate == 0))) & L.valid;
  double vsq_obs = w.vsq;
  if (reached) {
    u.flags |= UAVCA_FLAG_PARKED;
    const double2 fv = finish_velocity(u.vx, u.vy, w.vsq);
    u.vx = fv.x; u.vy = fv.y;
    r += 10.0f;
    vsq_obs = sq64(u.vx, u.vy);
  }
  u.prev = dist;  // :229

  // ---- observation (:233-235): every UAV at its new position
  {
    float2 o01, o23;
    obs_own(c, w, vsq_obs, o01, o23);
    io.put_own(o01, o23);
    io.put_neighbours(tail);
  }
  io.store_reward_done(r, done);

  // ---- per-env bookkeeping: reset decision, counters
  // reset triggers as two masks derived on the host: any done flag under rs_any_mask (bit 0 for dones[0], all
  // bits for any(dones)); every flag of the env set (rs_all_off = 0) for all(dones); the step limit (INT_MAX = none)
  // (masked to the env's own lanes: with several envs per warp the shifted ballot still carries the envs above it)
  const unsigned done_env = (__ballot_sync(kFull, done) >> L.base) & L.envmask;
  const bool rs = (((done_env & c.rs_any_mask) != 0u) | (((done_env ^ L.envmask) | c.rs_all_off) == 0u) |
                   (steps_new >= c.steps_limit)) & L.valid;
  const bool leader = L.valid & (L.i == 0);
  if (leader) io.store_reset(rs);
  // per-episode scores the training loops keep on the host (test_sac_multi.py:105: score += rewards[0];
  // :152-156: total_score += rewards[i] * (1 - dones[i])), accumulated per env when asked for
  if (!kPlain && c.track_scores) {
    const float live = env_sum((done | !L.valid) ? 0.0f : r, L);
    if (leader) {
      double2 sc = a.s.score[L.env];
      sc.x += (double)r;
      sc.y += (double)live;
      a.s.score[L.env] = sc;
    }
  }
  // a NaN / infinite reward or position (the reference zeroes some silently, uav_agent.py:40-42, and propagates the
  // rest): counted in stats[6] so that a run can assert it never happened
  const bool bad = (!(fabsf(r) <= 3.4e38f) | !(fabsf(u.px) + fabsf(u.py) <= 3.4e38f)) & L.valid;

  if (!__any_sync(kFull, rs | newly_reached | hard | bad)) {  // nothing to count, nobody resets: the common case
    io.store_steps(steps_new, leader);
    io.commit_obs();
    if (io.wants_final()) io.commit_final();
    io.store_state(u);
    return;
  }

  // ---- rare: some env of this warp counts a reach / a hard collision or starts a new episode in place
  const unsigned ev_reach = __ballot_sync(kFull, newly_reached), ev_coll = __ballot_sync(kFull, hard);
  const int reach_inc = __popc((ev_reach >> L.base) & L.envmask), coll_inc = __popc((ev_coll >> L.base) & L.envmask);
  {
    const unsigned ev_bad = __ballot_sync(kFull, bad);
    if (ev_bad != 0u && L.lane == 0) atomicAdd(a.s.stats + 6, (unsigned long long)__popc(ev_bad));
  }
  if (io.wants_final()) io.commit_final();
  if (!__any_sync(kFull, rs)) {
    io.store_steps(steps_new, leader);
    if (leader) {
      if (reach_inc) a.s.reach[L.env] += reach_inc;  // :221
      if (coll_inc) a.s.coll[L.env] += coll_inc;     // :209
    }
    io.commit_obs();
    io.store_state(u);
    return;
  }
  unsigned episode = 0;
  if (leader) episode = a.s.episode[L.env];
  episode = __shfl_sync(kFull, episode, L.base);
  if (leader) {
    if (rs) {
      if (episode > 0u) {  // fold the finished episode into the running totals
        atomicAdd(a.s.stats + 0, 1ull);
        atomicAdd(a.s.stats + 1, (unsigned long long)(a.s.reach[L.env] + reach_inc));
        atomicAdd(a.s.stats + 2, (unsigned long long)(a.s.coll[L.env] + coll_inc));
        atomicAdd(a.s.stats + 3, (unsigned long long)steps_new);
        if (c.track_scores) fold_scores(a.s, L.env);
      }
      a.s.reach[L.env] = 0; a.s.coll[L.env] = 0;  // :166-168
      a.s.episode[L.env] = episode + 1u;
    } else {
      if (reach_inc) a.s.reach[L.env] += reach_inc;
      if (coll_inc) a.s.coll[L.env] += coll_inc;
    }
  }
  io.store_steps(rs ? 0 : steps_new, leader);
  Uav nu = u;
  reset_multi(a, L, rs, episode, nu);
  const ObsRow no = observe_state<NT>(c, ws, L, nu);
  if (rs) {
    u = nu;
    io.put_own(no.o01, no.o23);
    io.put_neighbours(no.n);
  }
  io.commit_obs();
  io.store_state(u);
  if (rs) io.store_target(u);
}

}  // namespace uavca

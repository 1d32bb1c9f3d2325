// uavca_capi.cu — the C-ABI of include/uavca.h: handles, derived constants, state layout, launch plumbing.
// No torch types, no exceptions across the boundary, no CPU fallback.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "uavca_host.h"

using namespace uavca;

namespace {

thread_local std::string g_error;

int fail(int code, const std::string& msg) {
  g_error = msg;
  return code;
}
int fail_cuda(const char* what, cudaError_t e) {
  return fail(-2, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}

constexpr size_t kAlign = 256;
constexpr size_t kDmaThresholdBytes = 256u << 20;  // uavca_step_host: outputs at least this large leave by DMA (measured: 23 MB zero-copy 1.05e9 vs DMA 0.93e9 UAV-steps/s; 1.5 GB 1.12e9 vs 1.16e9)
size_t align_up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

void compute_layout(int B, int N, int float64_world, uavca_layout* L) {
  const size_t M = (size_t)B * (size_t)N;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  L->stats = take(8 * sizeof(uint64_t));
  L->pos = take(M * 2 * sizeof(float));
  L->vel = take(M * 2 * sizeof(double));
  L->tgt = take(M * 2 * sizeof(float));
  L->init = take(M * sizeof(float));
  L->prev = take(M * sizeof(float));
  L->flags = take(M);
  L->steps = take((size_t)B * sizeof(int32_t));
  L->reach = take((size_t)B * sizeof(int32_t));
  L->coll = take((size_t)B * sizeof(int32_t));
  L->episode = take((size_t)B * sizeof(uint32_t));
  L->score = take((size_t)B * 2 * sizeof(double));
  const size_t M64 = float64_world ? M : 0;  // the float64 fields exist only in that mode
  L->pos64 = take(M64 * 2 * sizeof(double));
  L->tgt64 = take(M64 * 2 * sizeof(double));
  L->init64 = take(M64 * sizeof(double));
  L->prev64 = take(M64 * sizeof(double));
  L->total_bytes = off;
}

StateView view_of(void* blob, const uavca_layout& L) {
  StateView v{};
  if (!blob) return v;
  char* p = static_cast<char*>(blob);
  v.stats = reinterpret_cast<unsigned long long*>(p + L.stats);
  v.pos = reinterpret_cast<float2*>(p + L.pos);
  v.vel = reinterpret_cast<double2*>(p + L.vel);
  v.tgt = reinterpret_cast<float2*>(p + L.tgt);
  v.init = reinterpret_cast<float*>(p + L.init);
  v.prev = reinterpret_cast<float*>(p + L.prev);
  v.flags = reinterpret_cast<uint8_t*>(p + L.flags);
  v.steps = reinterpret_cast<int*>(p + L.steps);
  v.reach = reinterpret_cast<int*>(p + L.reach);
  v.coll = reinterpret_cast<int*>(p + L.coll);
  v.episode = reinterpret_cast<unsigned*>(p + L.episode);
  v.score = reinterpret_cast<double2*>(p + L.score);
  if (L.tgt64 != L.pos64) {  // float64 world
    v.pos64 = reinterpret_cast<double2*>(p + L.pos64);
    v.tgt64 = reinterpret_cast<double2*>(p + L.tgt64);
    v.init64 = reinterpret_cast<double*>(p + L.init64);
    v.prev64 = reinterpret_cast<double*>(p + L.prev64);
  }
  return v;
}

// np.linalg.norm of a float64 2-vector as the reference's BLAS forms it (second product fused).
double n64(double x, double y) { return std::sqrt(std::fma(y, y, x * x)); }

Consts derive_consts(const uavca_config& g) {
  Consts c{};
  c.tau = g.tau;
  c.inv_tau = 1.0 / g.tau;
  c.amax = g.max_acceleration;
  c.vmax = g.max_speed;
  // least x >= 0 with fl(x / tau) >= amax (division is monotone, so the clip is decided by comparing x)
  {
    volatile double tau = g.tau;
    double x = g.max_acceleration * g.tau;
    for (int k = 0; k < 64 && x > 0 && std::nextafter(x, 0.0) / tau >= g.max_acceleration; ++k) x = std::nextafter(x, 0.0);
    for (int k = 0; k < 64 && x / tau < g.max_acceleration; ++k) x = std::nextafter(x, INFINITY);
    c.clip_x = x;
  }
  c.vm2 = n64(g.max_speed, g.max_speed);
  c.inv_vm2 = 1.0 / c.vm2;
  c.lox = -g.x_size / 2.0; c.hix = g.x_size / 2.0;
  c.loy = -g.y_size / 2.0; c.hiy = g.y_size / 2.0;
  // least s with sqrt(s) >= reach_speed:  ||v|| < reach_speed  <=>  (vx*vx + vy*vy) < s
  {
    double s = g.reach_speed * g.reach_speed;
    for (int k = 0; k < 64 && s > 0 && std::sqrt(std::nextafter(s, 0.0)) >= g.reach_speed; ++k) s = std::nextafter(s, 0.0);
    for (int k = 0; k < 64 && std::sqrt(s) < g.reach_speed; ++k) s = std::nextafter(s, INFINITY);
    c.reach_speed_sq = s;
  }
  // float32 thresholds moved to squared-distance space (sqrtf is correctly rounded and monotone)
  auto le_sq = [](float thr) {  // greatest s with sqrtf(s) <= thr
    float s = thr * thr;
    for (int k = 0; k < 64 && std::sqrt(s) > thr; ++k) s = std::nextafter(s, 0.0f);
    for (int k = 0; k < 64 && std::sqrt(std::nextafter(s, INFINITY)) <= thr; ++k) s = std::nextafter(s, INFINITY);
    return s;
  };
  auto lt_sq = [](float thr) {  // least s with sqrtf(s) >= thr  (d < thr  <=>  s < this)
    float s = thr * thr;
    for (int k = 0; k < 64 && std::sqrt(s) < thr; ++k) s = std::nextafter(s, INFINITY);
    for (int k = 0; k < 64 && s > 0 && std::sqrt(std::nextafter(s, 0.0f)) >= thr; ++k) s = std::nextafter(s, 0.0f);
    return s;
  };
  auto ceil_f = [](double v) { float f = (float)v; return ((double)f < v) ? std::nextafter(f, INFINITY) : f; };
  auto floor_f = [](double v) { float f = (float)v; return ((double)f > v) ? std::nextafter(f, -INFINITY) : f; };
  c.two_r = (float)(2.0 * g.collider_radius);
  c.two_h = (float)(2.0 * g.hard_collision_radius);
  c.dsense = (float)g.d_sense;
  c.reach_dist = (float)g.reach_distance;
  c.s_two_r_le = le_sq(c.two_r);
  c.s_two_h_le = le_sq(c.two_h);
  c.s_dsense_lt = lt_sq(c.dsense);
  {
    const float below_sense = std::nextafter(c.s_dsense_lt, -INFINITY);  // greatest s with sqrtf(s) < d_sense
    c.s_coll_le = std::fmin(c.s_two_r_le, below_sense);
    c.s_hard_le = std::fmin(c.s_two_h_le, below_sense);
  }
  c.s_reach_lt = lt_sq(c.reach_dist);
  c.two_r_d = 2.0 * g.collider_radius;
  c.two_h_d = 2.0 * g.hard_collision_radius;
  c.dsense_d = g.d_sense;
  c.reach_dist_d = g.reach_distance;
  c.lox_f = ceil_f(c.lox); c.hix_f = floor_f(c.hix);
  c.loy_f = ceil_f(c.loy); c.hiy_f = floor_f(c.hiy);
  c.vm2_floor_f = floor_f(c.vm2);
  c.vm2_f = (float)c.vm2;
  c.inv_dsense = (float)(1.0 / g.d_sense);
  const double diag = n64(g.x_size, g.y_size);
  c.inv_diag = (float)(1.0 / diag);
  c.inv_diag_d = 1.0 / diag;
  c.inv_vm2_f = (float)(1.0 / c.vm2);
  c.inv_vmax_f = (float)(1.0 / g.max_speed);
  c.inv_pi = (float)(1.0 / 3.141592653589793);
  c.polar_scale = (float)g.polar_scale;
  c.vmax_f = (float)g.max_speed;
  c.tau_f = (float)g.tau;
  c.reset_mode = g.reset_mode;
  c.max_steps = g.max_episode_steps;
  c.rs_any_mask = (g.reset_mode & UAVCA_RESET_ON_ANY_DONE) ? 0xffffffffu : ((g.reset_mode & UAVCA_RESET_ON_DONE0) ? 1u : 0u);
  c.rs_all_off = (g.reset_mode & UAVCA_RESET_ON_ALL_DONE) ? 0u : 1u;
  c.steps_limit = g.max_episode_steps > 0 ? g.max_episode_steps : 0x7fffffff;
  c.key_mask = ~31;
  {
    // Pass A tests UAV j > i at its OLD position; a UAV moves at most ||(vmax, vmax)|| * tau per step (plus the float32
    // rounding of its position), so only a UAV within `near` of lane i at the NEW positions can be within collision
    // reach at the old one.  Keys at or below near_key mark such UAVs (conservative: margins of 1 % + 2 cm).
    const double reach = std::sqrt((double)std::fmax(c.s_coll_le, c.s_hard_le));
    const double near = (reach + c.vm2 * g.tau) * 1.01 + 0.02;
    const float s = (float)(near * near);
    int bits;
    std::memcpy(&bits, &s, sizeof(bits));
    c.near_key = bits | 31;
  }
  c.reset_source = g.reset_source;
  c.circular = g.circular;
  c.single_f32_first_step = g.single_f32_first_step;
  c.track_scores = g.track_scores;
  c.seed_lo = (unsigned)(g.seed & 0xffffffffull);
  c.seed_hi = (unsigned)(g.seed >> 32);
  c.env_base = g.env_index_base;
  return c;
}

}  // namespace

struct uavca_handle {
  uavca_config cfg;
  Consts consts;
  uavca_layout layout;
  int device;
  const void* pool_blob = nullptr;
  int pool_envs = 0;
  uavca_layout pool_layout{};
  double4* ring64 = nullptr;  // reset(circular=True) table (owned): per UAV (pos.x, pos.y, tgt.x, tgt.y) in float64
  long long launches = 0;
  bool cta_pack = true;  // UAVCA_STEP_PATH=plain in the environment keeps every N <= 32 on the one-env-per-warp step kernel
  // end-to-end (host buffer) path, created lazily
  static constexpr int kHostStreams = 3;
  static constexpr int kChunks = 8;
  cudaStream_t hs[kHostStreams] = {nullptr, nullptr, nullptr};
  cudaEvent_t chunk_done[kChunks] = {};
  cudaEvent_t fork = nullptr;  // uavca_step_host: orders the internal streams after the caller's stream
  float* d_action = nullptr;
  float* d_rollout_action = nullptr;  // uavca_rollout on the general kernel: one step's Philox actions (created lazily)
  float* d_obs = nullptr;
  float* d_reward = nullptr;
  uint8_t* d_done = nullptr;
};

namespace {

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

KernelArgs make_args(const uavca_handle* h, void* state) {
  KernelArgs a{};
  a.c = h->consts;
  a.s = view_of(state, h->layout);
  a.pool = view_of(const_cast<void*>(h->pool_blob), h->pool_layout);
  a.pool_envs = h->pool_envs;
  a.ring64 = h->ring64;
  a.B = h->cfg.num_envs;
  a.N = h->cfg.num_agents;
  return a;
}

int check_handle(const uavca_handle* h) { return h ? 0 : fail(-1, "null handle"); }

// the kernels move float2 / float4 / double2 units: reject pointers that would fault instead of launching
bool misaligned(const void* p, uintptr_t a) { return p != nullptr && (reinterpret_cast<uintptr_t>(p) & (a - 1)) != 0; }
int check_step_alignment(const void* state, const void* action, const void* obs, const void* reward, const void* final_obs) {
  if (misaligned(state, 16) || misaligned(action, 8) || misaligned(obs, 16) || misaligned(reward, 4) || misaligned(final_obs, 16))
    return fail(-1, "misaligned buffer: state / obs / final_obs need 16-byte, action 8-byte, reward 4-byte alignment");
  return 0;
}

int validate_config(const uavca_config& g) {
  if (g.kind != UAVCA_KIND_MULTI && g.kind != UAVCA_KIND_SINGLE) return fail(-1, "config.kind must be UAVCA_KIND_MULTI or UAVCA_KIND_SINGLE");
  if (g.num_envs <= 0) return fail(-1, "config.num_envs must be positive");
  if (g.num_agents < 1 || g.num_agents > UAVCA_MAX_AGENTS) return fail(-1, "config.num_agents must be in 1..UAVCA_MAX_AGENTS (1024)");
  if ((long long)g.num_envs * g.num_agents > 0x7fffffffLL) return fail(-1, "num_envs * num_agents must be below 2^31 per handle (shard across handles)");
  if (g.kind == UAVCA_KIND_SINGLE && g.num_agents != 1) return fail(-1, "the single-UAV world has num_agents == 1");
  if (!(g.tau > 0) || !(g.max_speed > 0) || !(g.max_acceleration > 0)) return fail(-1, "tau, max_speed and max_acceleration must be positive");
  if (!(g.x_size > 0) || !(g.y_size > 0)) return fail(-1, "x_size and y_size must be positive");
  if (g.reset_source != UAVCA_SOURCE_PHILOX && g.reset_source != UAVCA_SOURCE_POOL) return fail(-1, "config.reset_source invalid");
  if (g.max_episode_steps < 0) return fail(-1, "config.max_episode_steps must be >= 0");
  return 0;
}

}  // namespace

extern "C" {

const char* uavca_last_error(void) { return g_error.c_str(); }
int uavca_version(void) { return UAVCA_VERSION; }

int uavca_default_config(int kind, uavca_config* cfg) {
  if (!cfg) return fail(-1, "null config");
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->kind = kind;
  cfg->num_envs = 1;
  cfg->tau = 0.02;
  cfg->max_acceleration = 5.0;
  cfg->collider_radius = 1.0;
  cfg->hard_collision_radius = 0.5;
  cfg->d_sense = 15.0;
  cfg->reach_distance = 0.5;
  cfg->reach_speed = 0.2;
  if (kind == UAVCA_KIND_SINGLE) {  // uav_world_2d.py:14
    cfg->num_agents = 1;
    cfg->x_size = 100.0; cfg->y_size = 100.0; cfg->max_speed = 12.0;
    cfg->polar_scale = 12.0;  // action_space.high[0] (test_sac.py:77)
  } else if (kind == UAVCA_KIND_MULTI) {  // multi_uav_world_2d.py:13
    cfg->num_agents = 4;
    cfg->x_size = 50.0; cfg->y_size = 50.0; cfg->max_speed = 10.0;
    cfg->polar_scale = (double)std::sqrt(200.0f);  // float32 norm of action_space.high (test_sac_multi.py:77)
  } else {
    return fail(-1, "unknown world kind");
  }
  return 0;
}

int uavca_create(const uavca_config* cfg, int device, uavca_handle** out) {
  if (!cfg || !out) return fail(-1, "null argument");
  *out = nullptr;
  if (int rc = validate_config(*cfg)) return rc;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    return fail(-3, std::string("no usable CUDA device (this library has no CPU fallback): ") + cudaGetErrorString(e));
  }
  if (device < 0 || device >= ndev) return fail(-1, "device index out of range");
  uavca_handle* h = new (std::nothrow) uavca_handle();
  if (!h) return fail(-4, "out of host memory");
  h->cfg = *cfg;
  h->consts = derive_consts(*cfg);
  h->device = device;
  compute_layout(cfg->num_envs, cfg->num_agents, cfg->kind == UAVCA_KIND_MULTI && cfg->circular, &h->layout);
  if (const char* p = std::getenv("UAVCA_STEP_PATH")) h->cta_pack = std::strcmp(p, "plain") != 0;
  if (cfg->kind == UAVCA_KIND_MULTI && cfg->circular) {
    // multi_uav_world_2d.py:157-163 with the HOST libm: the reference evaluates math.cos / math.sin (glibc) in float64,
    // and the device's cos / sin are not bit-identical to it; the ring is a table of N entries computed once here
    DeviceGuard g(device);
    const int N = cfg->num_agents;
    std::vector<double4> ring(N);
    const double pi = 3.141592653589793;
    for (int i = 0; i < N; ++i) {
      const double th = 2 * i * pi / N;
      ring[i] = make_double4(20.0 * std::cos(th), 20.0 * std::sin(th), 23.0 * std::cos(th + pi), 23.0 * std::sin(th + pi));
    }
    e = cudaMalloc(&h->ring64, sizeof(double4) * N);
    if (e == cudaSuccess) e = cudaMemcpy(h->ring64, ring.data(), sizeof(double4) * N, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { delete h; return fail_cuda("circular reset table", e); }
  }
  *out = h;
  return 0;
}

int uavca_destroy(uavca_handle* h) {
  if (!h) return 0;
  DeviceGuard g(h->device);
  if (h->ring64) cudaFree(h->ring64);
  for (auto& s : h->hs) if (s) cudaStreamDestroy(s);
  for (auto& ev : h->chunk_done) if (ev) cudaEventDestroy(ev);
  if (h->fork) cudaEventDestroy(h->fork);
  if (h->d_action) cudaFree(h->d_action);
  if (h->d_rollout_action) cudaFree(h->d_rollout_action);
  if (h->d_obs) cudaFree(h->d_obs);
  if (h->d_reward) cudaFree(h->d_reward);
  if (h->d_done) cudaFree(h->d_done);
  delete h;
  return 0;
}

int uavca_get_config(const uavca_handle* h, uavca_config* out) {
  if (int rc = check_handle(h)) return rc;
  if (!out) return fail(-1, "null argument");
  *out = h->cfg;
  return 0;
}

int uavca_state_layout(const uavca_handle* h, uavca_layout* out) {
  if (int rc = check_handle(h)) return rc;
  if (!out) return fail(-1, "null argument");
  *out = h->layout;
  return 0;
}

int uavca_pool_layout(const uavca_handle* h, int32_t pool_envs, uavca_layout* out) {
  if (int rc = check_handle(h)) return rc;
  if (!out || pool_envs <= 0) return fail(-1, "bad pool_envs / null argument");
  compute_layout(pool_envs, h->cfg.num_agents, 0, out);
  return 0;
}

int uavca_set_reset_pool(uavca_handle* h, const void* pool_state, int32_t pool_envs) {
  if (int rc = check_handle(h)) return rc;
  if (pool_state == nullptr || pool_envs <= 0) {
    h->pool_blob = nullptr; h->pool_envs = 0;
    return 0;
  }
  h->pool_blob = pool_state;
  h->pool_envs = pool_envs;
  compute_layout(pool_envs, h->cfg.num_agents, 0, &h->pool_layout);
  return 0;
}

int uavca_reset(uavca_handle* h, void* state, const uint8_t* mask, float* obs, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!state) return fail(-1, "null state");
  if (h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, state);
  a.io.obs = obs;
  cudaError_t e = h->cfg.kind == UAVCA_KIND_SINGLE ? launch_reset_single(a, mask, (cudaStream_t)stream)
                                                   : launch_reset_multi(a, mask, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_reset", e);
  h->launches += 1;
  return 0;
}

int uavca_observe(uavca_handle* h, const void* state, float* obs, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!state || !obs) return fail(-1, "null argument");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, const_cast<void*>(state));
  a.io.obs = obs;
  cudaError_t e = h->cfg.kind == UAVCA_KIND_SINGLE ? launch_observe_single(a, (cudaStream_t)stream)
                                                   : launch_observe_multi(a, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_observe", e);
  h->launches += 1;
  return 0;
}

int uavca_step_multi(uavca_handle* h, void* state, const float* action, int action_mode, int evaluate, float* obs,
                     float* reward, uint8_t* done, float* final_obs, uint8_t* reset_mask, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (h->cfg.kind != UAVCA_KIND_MULTI) return fail(-1, "uavca_step_multi on a single-UAV handle");
  if (!state || !action || !obs || !reward || !done) return fail(-1, "null argument");
  if (int rc = check_step_alignment(state, action, obs, reward, final_obs)) return rc;
  if (action_mode < 0 || action_mode > 2) return fail(-1, "bad action_mode");
  if (h->cfg.reset_mode && h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, state);
  a.io.action = reinterpret_cast<const float2*>(action);
  a.io.obs = obs; a.io.reward = reward; a.io.done = done; a.io.final_obs = final_obs; a.io.reset_mask = reset_mask;
  a.io.action_mode = action_mode; a.io.evaluate = evaluate;
  cudaError_t e = launch_step_multi(a, (cudaStream_t)stream, h->cta_pack);
  h->launches += 1;
  if (e != cudaSuccess) return fail_cuda("uavca_step_multi", e);
  return 0;
}

int uavca_step_single(uavca_handle* h, void* state, const float* action, int action_mode, float* obs, float* reward,
                      uint8_t* done, float* distance, float* final_obs, uint8_t* reset_mask, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (h->cfg.kind != UAVCA_KIND_SINGLE) return fail(-1, "uavca_step_single on a multi-UAV handle");
  if (!state || !action || !obs || !reward || !done) return fail(-1, "null argument");
  if (int rc = check_step_alignment(state, action, obs, reward, final_obs)) return rc;
  if (action_mode < 0 || action_mode > 2) return fail(-1, "bad action_mode");
  if (h->cfg.reset_mode && h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, state);
  a.io.action = reinterpret_cast<const float2*>(action);
  a.io.obs = obs; a.io.reward = reward; a.io.done = done; a.io.final_obs = final_obs; a.io.reset_mask = reset_mask;
  a.io.distance = distance; a.io.action_mode = action_mode;
  cudaError_t e = launch_step_single(a, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_step_single", e);
  h->launches += 1;
  return 0;
}

int uavca_step_f64(uavca_handle* h, void* state, const double* action, int evaluate, float* obs, float* reward, uint8_t* done,
                   float* distance, float* final_obs, uint8_t* reset_mask, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!state || !action || !obs || !reward || !done) return fail(-1, "null argument");
  if (int rc = check_step_alignment(state, nullptr, obs, reward, final_obs)) return rc;
  if (misaligned(action, 16)) return fail(-1, "misaligned buffer: float64 actions need 16-byte alignment");
  if (h->cfg.reset_mode && h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, state);
  a.io.action = nullptr;
  a.io.action64 = reinterpret_cast<const double2*>(action);
  a.io.obs = obs; a.io.reward = reward; a.io.done = done; a.io.final_obs = final_obs; a.io.reset_mask = reset_mask;
  a.io.action_mode = UAVCA_ACTION_CARTESIAN; a.io.evaluate = evaluate;
  cudaError_t e;
  if (h->cfg.kind == UAVCA_KIND_SINGLE) {
    a.io.distance = distance;
    e = launch_step_single(a, (cudaStream_t)stream);
  } else {
    e = launch_step_multi(a, (cudaStream_t)stream, h->cta_pack);  // the general one-thread-per-env kernel
  }
  h->launches += 1;
  if (e != cudaSuccess) return fail_cuda("uavca_step_f64", e);
  return 0;
}

int uavca_step_sync(uavca_handle* h, void* state, const void* action, int action_is_f64, int action_mode, int evaluate, float* obs,
                    float* reward, uint8_t* done, float* distance, float* final_obs, uint8_t* reset_mask, void* stream) {
  if (int rc = check_handle(h)) return rc;
  int rc;
  if (action_is_f64)
    rc = uavca_step_f64(h, state, static_cast<const double*>(action), evaluate, obs, reward, done, distance, final_obs, reset_mask, stream);
  else if (h->cfg.kind == UAVCA_KIND_SINGLE)
    rc = uavca_step_single(h, state, static_cast<const float*>(action), action_mode, obs, reward, done, distance, final_obs, reset_mask, stream);
  else
    rc = uavca_step_multi(h, state, static_cast<const float*>(action), action_mode, evaluate, obs, reward, done, final_obs, reset_mask, stream);
  if (rc) return rc;
  DeviceGuard g(h->device);
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_step_sync", e);
  return 0;
}

int uavca_map_action(uavca_handle* h, const float* in, int action_mode, float* out, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!in || !out) return fail(-1, "null argument");
  if (action_mode < 0 || action_mode > 2) return fail(-1, "bad action_mode");
  DeviceGuard g(h->device);
  cudaError_t e = launch_map_action(h->consts, in, out, (long long)h->cfg.num_envs * h->cfg.num_agents, action_mode,
                                    (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_map_action", e);
  h->launches += 1;
  return 0;
}

int uavca_stats(uavca_handle* h, const void* state, int64_t* out8, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!state || !out8) return fail(-1, "null argument");
  DeviceGuard g(h->device);
  StateView s = view_of(const_cast<void*>(state), h->layout);
  cudaError_t e = launch_stats(s, h->cfg.num_envs, reinterpret_cast<long long*>(out8), (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_stats", e);
  h->launches += 1;
  return 0;
}

int uavca_step_host(uavca_handle* h, void* state, const float* host_action, int action_mode, int evaluate,
                    float* host_obs, float* host_reward, uint8_t* host_done, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!state || !host_action || !host_obs || !host_reward || !host_done) return fail(-1, "null argument");
  if (action_mode < 0 || action_mode > 2) return fail(-1, "bad action_mode");
  if (h->cfg.reset_mode && h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  DeviceGuard g(h->device);
  const int B = h->cfg.num_envs, N = h->cfg.num_agents;
  const int D = h->cfg.kind == UAVCA_KIND_SINGLE ? UAVCA_OBS_DIM_SINGLE : UAVCA_OBS_DIM_MULTI;
  const size_t M = (size_t)B * N;
  cudaError_t e = cudaSuccess;
  if (!h->hs[0]) {
    for (auto& s : h->hs) {
      e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
      if (e != cudaSuccess) return fail_cuda("stream create", e);
    }
  }
  // The call is ordered after the caller's earlier work on `stream` (like every other entry point): the zero-copy
  // launch goes onto that stream itself, the copy pipelines fork their internal streams from an event recorded on it.
  cudaStream_t caller = (cudaStream_t)stream;
  if (!h->fork) {
    if ((e = cudaEventCreateWithFlags(&h->fork, cudaEventDisableTiming)) != cudaSuccess) return fail_cuda("event create", e);
  }
  // Zero-copy path: when all four host buffers are pinned (page-locked, hence mapped into the device's address
  // space under UVA) the step kernel reads the actions and writes obs/reward/done THROUGH PCIe itself — one launch,
  // no staging copies, the stores stream out as posted writes while the SMs work on the next warps.
  // UAVCA_HOST_PATH=staged forces the chunked copy pipeline below.
  auto mapped = [&](const void* p) -> void* {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
  };
  const char* hp = std::getenv("UAVCA_HOST_PATH");  // zerocopy | dma | staged: force one path (A/B measurements)
  const bool want_staged = hp && std::strcmp(hp, "staged") == 0;
  void *m_act = nullptr, *m_obs = nullptr, *m_rew = nullptr, *m_done = nullptr;
  if (!want_staged) { m_act = mapped(host_action); m_obs = mapped(host_obs); m_rew = mapped(host_reward); m_done = mapped(host_done); }
  const bool pinned = m_act && m_obs && m_rew && m_done;
  // Very large pinned batches: the copy engines stream hundreds of MB slightly faster (56 GB/s) than SM stores through
  // PCIe (47-50 GB/s), so the outputs go to device staging and leave by DMA, chunked so that H2D(k+1), step(k) and
  // D2H(k-1) overlap.  Everything smaller stays zero-copy: no copy-engine latency, no per-chunk overhead.
  const size_t out_bytes = M * ((size_t)D * sizeof(float) + sizeof(float) + 1);
  bool use_dma = pinned && out_bytes >= kDmaThresholdBytes;
  if (hp && std::strcmp(hp, "dma") == 0) use_dma = pinned;
  if (hp && std::strcmp(hp, "zerocopy") == 0) use_dma = false;
  if (pinned && !use_dma) {
    KernelArgs a = make_args(h, state);
    a.io.action = reinterpret_cast<const float2*>(m_act);
    a.io.obs = reinterpret_cast<float*>(m_obs); a.io.reward = reinterpret_cast<float*>(m_rew);
    a.io.done = reinterpret_cast<uint8_t*>(m_done);
    a.io.action_mode = action_mode; a.io.evaluate = evaluate;
    cudaStream_t st = caller;
    e = h->cfg.kind == UAVCA_KIND_SINGLE ? launch_step_single(a, st) : launch_step_multi(a, st, h->cta_pack);
    h->launches += 1;
    if (e != cudaSuccess) return fail_cuda("uavca_step_host launch", e);
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return fail_cuda("stream synchronize", e);
    return 0;
  }
  if ((e = cudaEventRecord(h->fork, caller)) != cudaSuccess) return fail_cuda("event record", e);
  for (auto& s_ : h->hs)
    if ((e = cudaStreamWaitEvent(s_, h->fork, 0)) != cudaSuccess) return fail_cuda("stream wait", e);
  if (!h->d_action) {
    if ((e = cudaMalloc(&h->d_action, M * 2 * sizeof(float))) != cudaSuccess) return fail_cuda("cudaMalloc", e);
    if ((e = cudaMalloc(&h->d_obs, M * D * sizeof(float))) != cudaSuccess) return fail_cuda("cudaMalloc", e);
    if ((e = cudaMalloc(&h->d_reward, M * sizeof(float))) != cudaSuccess) return fail_cuda("cudaMalloc", e);
    if ((e = cudaMalloc(&h->d_done, M)) != cudaSuccess) return fail_cuda("cudaMalloc", e);
    for (auto& ev : h->chunk_done)
      if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return fail_cuda("event create", e);
  }
  if (use_dma) {
    // stream 0: H2D(actions k) -> step(k) -> event k;  stream 1: wait event k -> D2H(obs k);  reward/done leave whole
    constexpr int chunks = uavca_handle::kChunks;
    long long per = ((long long)B + chunks - 1) / chunks;
    per = (per + 63) / 64 * 64;  // keeps every chunk's rows 16-byte aligned for any N
    cudaStream_t s_in = h->hs[0], s_out = h->hs[1];
    int k = 0;
    for (long long env0 = 0; env0 < B; env0 += per, ++k) {
      const long long nb = (env0 + per <= B) ? per : (B - env0);
      const size_t m0 = (size_t)env0 * N, mc = (size_t)nb * N;
      if ((e = cudaMemcpyAsync(h->d_action + m0 * 2, host_action + m0 * 2, mc * 2 * sizeof(float), cudaMemcpyHostToDevice, s_in)) != cudaSuccess)
        return fail_cuda("H2D action", e);
      KernelArgs a = make_args(h, state);
      a.s = offset_view(a.s, env0, N);
      a.c.env_base += env0;
      a.B = (int)nb;
      a.io.action = reinterpret_cast<const float2*>(h->d_action + m0 * 2);
      a.io.obs = h->d_obs + m0 * D; a.io.reward = h->d_reward + m0; a.io.done = h->d_done + m0;
      a.io.action_mode = action_mode; a.io.evaluate = evaluate;
      e = h->cfg.kind == UAVCA_KIND_SINGLE ? launch_step_single(a, s_in) : launch_step_multi(a, s_in, h->cta_pack);
      h->launches += 1;
      if (e != cudaSuccess) return fail_cuda("uavca_step_host launch", e);
      if ((e = cudaEventRecord(h->chunk_done[k], s_in)) != cudaSuccess) return fail_cuda("event record", e);
      if ((e = cudaStreamWaitEvent(s_out, h->chunk_done[k], 0)) != cudaSuccess) return fail_cuda("stream wait", e);
      if ((e = cudaMemcpyAsync(host_obs + m0 * D, h->d_obs + m0 * D, mc * D * sizeof(float), cudaMemcpyDeviceToHost, s_out)) != cudaSuccess)
        return fail_cuda("D2H obs", e);
    }
    if ((e = cudaMemcpyAsync(host_reward, h->d_reward, M * sizeof(float), cudaMemcpyDeviceToHost, s_out)) != cudaSuccess) return fail_cuda("D2H reward", e);
    if ((e = cudaMemcpyAsync(host_done, h->d_done, M, cudaMemcpyDeviceToHost, s_out)) != cudaSuccess) return fail_cuda("D2H done", e);
    if ((e = cudaStreamSynchronize(s_out)) != cudaSuccess) return fail_cuda("stream synchronize", e);
    return 0;
  }
  // Staged path (pageable host memory): chunk the env range so that H2D of chunk k+1, the step of chunk k and D2H of
  // chunk k-1 overlap
  int chunks = 8;
  long long per = ((long long)B + chunks - 1) / chunks;
  per = (per + 63) / 64 * 64;  // keeps every chunk's rows 16-byte aligned for any N
  if (per <= 0) per = 64;
  for (long long env0 = 0, k = 0; env0 < B; env0 += per, ++k) {
    const long long nb = (env0 + per <= B) ? per : (B - env0);
    const size_t m0 = (size_t)env0 * N, mc = (size_t)nb * N;
    cudaStream_t st = h->hs[k % uavca_handle::kHostStreams];
    if ((e = cudaMemcpyAsync(h->d_action + m0 * 2, host_action + m0 * 2, mc * 2 * sizeof(float), cudaMemcpyHostToDevice, st)) != cudaSuccess)
      return fail_cuda("H2D action", e);
    KernelArgs a = make_args(h, state);
    a.s = offset_view(a.s, env0, N);
    a.c.env_base += env0;
    a.B = (int)nb;
    a.io.action = reinterpret_cast<const float2*>(h->d_action + m0 * 2);
    a.io.obs = h->d_obs + m0 * D; a.io.reward = h->d_reward + m0; a.io.done = h->d_done + m0;
    a.io.action_mode = action_mode; a.io.evaluate = evaluate;
    e = h->cfg.kind == UAVCA_KIND_SINGLE ? launch_step_single(a, st) : launch_step_multi(a, st, h->cta_pack);
    h->launches += 1;
    if (e != cudaSuccess) return fail_cuda("uavca_step_host launch", e);
    if ((e = cudaMemcpyAsync(host_obs + m0 * D, h->d_obs + m0 * D, mc * D * sizeof(float), cudaMemcpyDeviceToHost, st)) != cudaSuccess)
      return fail_cuda("D2H obs", e);
    if ((e = cudaMemcpyAsync(host_reward + m0, h->d_reward + m0, mc * sizeof(float), cudaMemcpyDeviceToHost, st)) != cudaSuccess)
      return fail_cuda("D2H reward", e);
    if ((e = cudaMemcpyAsync(host_done + m0, h->d_done + m0, mc, cudaMemcpyDeviceToHost, st)) != cudaSuccess)
      return fail_cuda("D2H done", e);
  }
  for (auto& s : h->hs)
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail_cuda("stream synchronize", e);
  return 0;
}

int uavca_rollout(uavca_handle* h, void* state, int32_t K, const float* action_block, int action_mode, int evaluate,
                  uint64_t action_seed, uint64_t step0, float* obs, float* reward, uint8_t* done, float* action_out,
                  float* final_obs, uint8_t* reset_mask, float* distance, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!state || !obs || !reward || !done) return fail(-1, "null argument");
  if (K < 0) return fail(-1, "uavca_rollout: K must be >= 0");
  if (int rc = check_step_alignment(state, action_block, obs, reward, final_obs)) return rc;
  if (misaligned(action_out, 8)) return fail(-1, "misaligned buffer: action_out needs 8-byte alignment");
  if (action_mode < 0 || action_mode > 2) return fail(-1, "bad action_mode");
  if (h->cfg.reset_mode && h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  const bool single = h->cfg.kind == UAVCA_KIND_SINGLE;
  const long long M = (long long)h->cfg.num_envs * h->cfg.num_agents;
  if (!single && (h->cfg.circular || h->cfg.num_agents > 32)) {
    // The float64 world and envs wider than a warp run on the general one-thread-per-env kernel, which has no K loop: the
    // same call, K launches on the stream, every step's outputs at their [k] offsets (not a throughput path).
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (!action_block && !action_out && !h->d_rollout_action) {
      cudaError_t e = cudaMalloc(&h->d_rollout_action, (size_t)M * 2 * sizeof(float));
      if (e != cudaSuccess) return fail_cuda("uavca_rollout (action scratch)", e);
    }
    KernelArgs a = make_args(h, state);
    a.io.evaluate = evaluate;
    a.io.action_mode = (action_block == nullptr && action_mode == UAVCA_ACTION_CARTESIAN) ? UAVCA_ACTION_SCALED : action_mode;
    for (int32_t k = 0; k < K; ++k) {
      const float* act_k = action_block ? action_block + (size_t)k * M * 2 : nullptr;
      if (!act_k) {
        float* dst = action_out ? action_out + (size_t)k * M * 2 : h->d_rollout_action;
        cudaError_t e = launch_sample_actions(h->consts, dst, h->cfg.num_envs, h->cfg.num_agents, action_seed, step0 + (uint64_t)k, st);
        if (e != cudaSuccess) return fail_cuda("uavca_rollout (actions)", e);
        h->launches += 1;
        act_k = dst;
      }
      a.io.action = reinterpret_cast<const float2*>(act_k);
      a.io.obs = obs + (size_t)k * M * UAVCA_OBS_DIM_MULTI;
      a.io.reward = reward + (size_t)k * M;
      a.io.done = done + (size_t)k * M;
      a.io.final_obs = final_obs ? final_obs + (size_t)k * M * UAVCA_OBS_DIM_MULTI : nullptr;
      a.io.reset_mask = reset_mask ? reset_mask + (size_t)k * h->cfg.num_envs : nullptr;
      cudaError_t e = launch_step_multi(a, st, h->cta_pack);
      h->launches += 1;
      if (e != cudaSuccess) return fail_cuda("uavca_rollout", e);
    }
    return 0;
  }
  // the [K][...] blocks must keep every step's rows aligned for the 16-byte observation stores
  if (!single && (M * UAVCA_OBS_DIM_MULTI * sizeof(float)) % 16 != 0 && K > 1)
    return fail(-1, "uavca_rollout: num_envs * num_agents * 10 floats must be a multiple of 16 bytes for K > 1");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, state);
  a.io.obs = obs; a.io.reward = reward; a.io.done = done; a.io.final_obs = final_obs; a.io.reset_mask = reset_mask;
  a.io.distance = single ? distance : nullptr;
  a.io.evaluate = evaluate;
  // Philox actions are drawn in policy space [-1, 1)^2: "cartesian" then means the whole action box, a * max_speed
  a.io.action_mode = (action_block == nullptr && action_mode == UAVCA_ACTION_CARTESIAN) ? UAVCA_ACTION_SCALED : action_mode;
  RolloutArgs r{};
  r.K = K;
  r.action_block = reinterpret_cast<const float2*>(action_block);
  r.action_out = reinterpret_cast<float2*>(action_out);
  r.seed_lo = (unsigned)(action_seed & 0xffffffffull);
  r.seed_hi = (unsigned)(action_seed >> 32);
  r.step0 = step0;
  r.M = M;
  r.B = h->cfg.num_envs;
  cudaError_t e = single ? launch_rollout_single(a, r, (cudaStream_t)stream) : launch_rollout_multi(a, r, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_rollout", e);
  if (K > 0) h->launches += 1;
  return 0;
}

int uavca_sample_actions(uavca_handle* h, uint64_t action_seed, uint64_t step, float* out, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!out) return fail(-1, "null argument");
  if (misaligned(out, 8)) return fail(-1, "misaligned buffer: out needs 8-byte alignment");
  DeviceGuard g(h->device);
  cudaError_t e = launch_sample_actions(h->consts, out, h->cfg.num_envs, h->cfg.num_agents, action_seed, step, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_sample_actions", e);
  h->launches += 1;
  return 0;
}

static int replay_push_impl(const float* obs, const float* action, const float* reward, const float* next_obs, const uint8_t* done,
                            int64_t M, int32_t obs_dim, int32_t act_dim, float* ring_obs, float* ring_action, float* ring_reward,
                            float* ring_next_obs, float* ring_mask, int64_t capacity, int64_t head, int64_t* meta, void* stream) {
  if (!obs || !action || !reward || !next_obs || !done || !ring_obs || !ring_action || !ring_reward || !ring_next_obs || !ring_mask)
    return fail(-1, "null argument");
  if (M < 0 || obs_dim <= 0 || act_dim <= 0 || capacity <= 0) return fail(-1, "bad sizes");
  if (M > capacity) return fail(-1, "uavca_replay_push: M exceeds the ring capacity");
  if (head < 0 || head >= capacity) return fail(-1, "uavca_replay_push: head out of range");
  // the pointers decide the device (no handle here): launch where the ring lives, whatever the current device is
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, ring_obs) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(-1, "uavca_replay_push: ring_obs is not a device pointer");
  }
  DeviceGuard g(at.device);
  cudaError_t e = launch_replay_push(obs, action, reward, next_obs, done, M, obs_dim, act_dim, ring_obs, ring_action,
                                     ring_reward, ring_next_obs, ring_mask, capacity, head,
                                     reinterpret_cast<long long*>(meta), (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_replay_push", e);
  return 0;
}

int uavca_replay_push(const float* obs, const float* action, const float* reward, const float* next_obs, const uint8_t* done,
                      int64_t M, int32_t obs_dim, int32_t act_dim, float* ring_obs, float* ring_action, float* ring_reward,
                      float* ring_next_obs, float* ring_mask, int64_t capacity, int64_t head, void* stream) {
  return replay_push_impl(obs, action, reward, next_obs, done, M, obs_dim, act_dim, ring_obs, ring_action, ring_reward,
                          ring_next_obs, ring_mask, capacity, head, nullptr, stream);
}

int uavca_replay_push_dev(const float* obs, const float* action, const float* reward, const float* next_obs, const uint8_t* done,
                          int64_t M, int32_t obs_dim, int32_t act_dim, float* ring_obs, float* ring_action, float* ring_reward,
                          float* ring_next_obs, float* ring_mask, int64_t capacity, int64_t* ring_meta, void* stream) {
  if (!ring_meta) return fail(-1, "null argument");
  return replay_push_impl(obs, action, reward, next_obs, done, M, obs_dim, act_dim, ring_obs, ring_action, ring_reward,
                          ring_next_obs, ring_mask, capacity, 0, ring_meta, stream);
}

int uavca_replay_sample(const float* ring_obs, const float* ring_action, const float* ring_reward, const float* ring_next_obs,
                        const float* ring_mask, int64_t capacity, int32_t obs_dim, int32_t act_dim, const int64_t* ring_meta,
                        int64_t batch, uint64_t seed, uint64_t draw, int recency_weighted, float* out_obs, float* out_action,
                        float* out_reward, float* out_next_obs, float* out_mask, int64_t* out_index, void* stream) {
  if (!ring_obs || !ring_action || !ring_reward || !ring_next_obs || !ring_mask || !ring_meta || !out_obs || !out_action ||
      !out_reward || !out_next_obs || !out_mask)
    return fail(-1, "null argument");
  if (batch < 0 || obs_dim <= 0 || act_dim <= 0 || capacity <= 0 || capacity >= ((int64_t)1 << 32)) return fail(-1, "bad sizes");
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, ring_obs) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(-1, "uavca_replay_sample: ring_obs is not a device pointer");
  }
  DeviceGuard g(at.device);
  cudaError_t e = launch_replay_sample(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, capacity, obs_dim, act_dim,
                                       reinterpret_cast<const long long*>(ring_meta), batch, seed, draw, recency_weighted, out_obs,
                                       out_action, out_reward, out_next_obs, out_mask, reinterpret_cast<long long*>(out_index),
                                       (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_replay_sample", e);
  return 0;
}

// n-step arguments, checked before any launch: 1 <= n <= 16 (one lane of the sample's 16 per link), 1 <= stride <=
// capacity, gamma finite in [0, 1]
static int nstep_check(const char* what, int64_t capacity, int64_t stride, int32_t n, double gamma) {
  if (n < 1 || n > 16) return fail(-1, std::string(what) + ": n = " + std::to_string(n) + " is outside 1..16");
  if (stride < 1 || stride > capacity)
    return fail(-1, std::string(what) + ": stride = " + std::to_string(stride) + " is outside 1..capacity (" +
                        std::to_string(capacity) + ")");
  if (!(gamma >= 0.0 && gamma <= 1.0)) return fail(-1, std::string(what) + ": gamma must be finite and in [0, 1]");
  return 0;
}

int uavca_replay_sample_nstep(const float* ring_obs, const float* ring_action, const float* ring_reward,
                              const float* ring_next_obs, const float* ring_mask, int64_t capacity, int32_t obs_dim,
                              int32_t act_dim, const int64_t* ring_meta, int64_t batch, uint64_t seed, uint64_t draw,
                              int recency_weighted, int64_t stride, int32_t n, double gamma, float* out_obs,
                              float* out_action, float* out_reward, float* out_next_obs, float* out_discount,
                              int64_t* out_index, void* stream) {
  if (!ring_obs || !ring_action || !ring_reward || !ring_next_obs || !ring_mask || !ring_meta || !out_obs || !out_action ||
      !out_reward || !out_next_obs || !out_discount)
    return fail(-1, "null argument");
  if (batch < 0 || obs_dim <= 0 || act_dim <= 0 || capacity <= 0 || capacity >= ((int64_t)1 << 32)) return fail(-1, "bad sizes");
  if (int rc = nstep_check("uavca_replay_sample_nstep", capacity, stride, n, gamma)) return rc;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, ring_obs) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(-1, "uavca_replay_sample_nstep: ring_obs is not a device pointer");
  }
  DeviceGuard g(at.device);
  cudaError_t e = launch_replay_sample_nstep(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, capacity, obs_dim,
                                             act_dim, reinterpret_cast<const long long*>(ring_meta), batch, seed, draw,
                                             recency_weighted, stride, n, gamma, out_obs, out_action, out_reward,
                                             out_next_obs, out_discount, reinterpret_cast<long long*>(out_index),
                                             (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_replay_sample_nstep", e);
  return 0;
}

// Prioritized replay: the tree of a ring of `capacity` slots has L leaves, the least power of two >= capacity.
static int per_check_tree(const char* what, const double* tree, int64_t L, int64_t capacity, const int64_t* per_meta) {
  if (!tree || !per_meta) return fail(-1, "null argument");
  if (capacity <= 0 || capacity > UAVCA_PER_MAX_CAPACITY)
    return fail(-1, std::string(what) + ": capacity " + std::to_string(capacity) + " is outside 1..2^26");
  int64_t want = 1;
  while (want < capacity) want <<= 1;
  if (L != want)
    return fail(-1, std::string(what) + ": L = " + std::to_string(L) + ", but a ring of " + std::to_string(capacity) +
                        " slots needs L = " + std::to_string(want));
  if (misaligned(tree, 8) || misaligned(per_meta, 8)) return fail(-1, "misaligned buffer: tree and per_meta need 8-byte alignment");
  return 0;
}

static int per_device(const char* what, const void* p) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(-1, std::string(what) + ": tree is not a device pointer");
  }
  return at.device;
}

int uavca_per_sync(double* tree, int64_t L, int64_t* per_meta, const int64_t* ring_meta, int64_t capacity, void* stream) {
  if (int rc = per_check_tree("uavca_per_sync", tree, L, capacity, per_meta)) return rc;
  if (!ring_meta) return fail(-1, "null argument");
  const int dev = per_device("uavca_per_sync", tree);
  if (dev < 0) return -1;
  DeviceGuard g(dev);
  cudaError_t e = launch_per_sync(tree, L, reinterpret_cast<long long*>(per_meta), reinterpret_cast<const long long*>(ring_meta),
                                  capacity, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_per_sync", e);
  return 0;
}

int uavca_per_update(double* tree, int64_t L, int64_t capacity, int64_t* per_meta, const int64_t* index, const double* priority,
                     int64_t n, void* stream) {
  if (int rc = per_check_tree("uavca_per_update", tree, L, capacity, per_meta)) return rc;
  if (n < 0 || n > capacity) return fail(-1, "uavca_per_update: n must be in 0..capacity");
  if (n == 0) return 0;
  if (!index || !priority) return fail(-1, "null argument");
  if (misaligned(index, 8) || misaligned(priority, 8)) return fail(-1, "misaligned buffer: index and priority need 8-byte alignment");
  const int dev = per_device("uavca_per_update", tree);
  if (dev < 0) return -1;
  DeviceGuard g(dev);
  cudaError_t e = launch_per_update(tree, L, capacity, reinterpret_cast<long long*>(per_meta),
                                    reinterpret_cast<const long long*>(index), priority, n, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_per_update", e);
  return 0;
}

int uavca_per_sample(const float* ring_obs, const float* ring_action, const float* ring_reward, const float* ring_next_obs,
                     const float* ring_mask, int64_t capacity, int32_t obs_dim, int32_t act_dim, const int64_t* ring_meta,
                     double* tree, int64_t L, int64_t batch, double beta, uint64_t seed, uint64_t draw, float* out_obs,
                     float* out_action, float* out_reward, float* out_next_obs, float* out_mask, int64_t* out_index,
                     float* out_weight, void* stream) {
  if (!ring_obs || !ring_action || !ring_reward || !ring_next_obs || !ring_mask || !ring_meta || !out_obs || !out_action ||
      !out_reward || !out_next_obs || !out_mask || !out_index || !out_weight)
    return fail(-1, "null argument");
  if (!tree) return fail(-1, "null argument");
  if (int rc = per_check_tree("uavca_per_sample", tree, L, capacity, ring_meta)) return rc;
  if (batch < 0 || batch >= ((int64_t)1 << 26) || obs_dim <= 0 || act_dim <= 0) return fail(-1, "bad sizes");
  if (!std::isfinite(beta)) return fail(-1, "uavca_per_sample: beta must be finite");
  if (misaligned(out_index, 8)) return fail(-1, "misaligned buffer: out_index needs 8-byte alignment");
  const int dev = per_device("uavca_per_sample", tree);
  if (dev < 0) return -1;
  DeviceGuard g(dev);
  cudaError_t e = launch_per_sample(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, obs_dim, act_dim,
                                    reinterpret_cast<const long long*>(ring_meta), tree, L, batch, beta, seed, draw, out_obs,
                                    out_action, out_reward, out_next_obs, out_mask, reinterpret_cast<long long*>(out_index),
                                    out_weight, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_per_sample", e);
  return 0;
}

int uavca_per_sample_nstep(const float* ring_obs, const float* ring_action, const float* ring_reward,
                           const float* ring_next_obs, const float* ring_mask, int64_t capacity, int32_t obs_dim,
                           int32_t act_dim, const int64_t* ring_meta, double* tree, int64_t L, int64_t batch, double beta,
                           int64_t stride, int32_t n, double gamma, uint64_t seed, uint64_t draw, float* out_obs,
                           float* out_action, float* out_reward, float* out_next_obs, float* out_discount,
                           int64_t* out_index, float* out_weight, void* stream) {
  if (!ring_obs || !ring_action || !ring_reward || !ring_next_obs || !ring_mask || !ring_meta || !out_obs || !out_action ||
      !out_reward || !out_next_obs || !out_discount || !out_index || !out_weight)
    return fail(-1, "null argument");
  if (!tree) return fail(-1, "null argument");
  if (int rc = per_check_tree("uavca_per_sample_nstep", tree, L, capacity, ring_meta)) return rc;
  if (batch < 0 || batch >= ((int64_t)1 << 26) || obs_dim <= 0 || act_dim <= 0) return fail(-1, "bad sizes");
  if (!std::isfinite(beta)) return fail(-1, "uavca_per_sample_nstep: beta must be finite");
  if (int rc = nstep_check("uavca_per_sample_nstep", capacity, stride, n, gamma)) return rc;
  if (misaligned(out_index, 8)) return fail(-1, "misaligned buffer: out_index needs 8-byte alignment");
  const int dev = per_device("uavca_per_sample_nstep", tree);
  if (dev < 0) return -1;
  DeviceGuard g(dev);
  cudaError_t e = launch_per_sample_nstep(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, capacity, obs_dim,
                                          act_dim, reinterpret_cast<const long long*>(ring_meta), tree, L, batch, beta, stride,
                                          n, gamma, seed, draw, out_obs, out_action, out_reward, out_next_obs, out_discount,
                                          reinterpret_cast<long long*>(out_index), out_weight, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_per_sample_nstep", e);
  return 0;
}

int uavca_step_multi_replay(uavca_handle* h, void* state, const float* action, int action_mode, int evaluate,
                            const float* prev_obs, float* obs, float* reward, uint8_t* done, float* final_obs,
                            uint8_t* reset_mask, float* ring_obs, float* ring_action, float* ring_reward, float* ring_next_obs,
                            float* ring_mask, int64_t capacity, int64_t* ring_meta, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (h->cfg.kind != UAVCA_KIND_MULTI) return fail(-1, "uavca_step_multi_replay on a single-UAV handle");
  if (!state || !action || !prev_obs || !obs || !reward || !done || !ring_obs || !ring_action || !ring_reward ||
      !ring_next_obs || !ring_mask || !ring_meta)
    return fail(-1, "null argument");
  if (prev_obs == obs) return fail(-1, "uavca_step_multi_replay: prev_obs and obs must be different buffers");
  if (int rc = check_step_alignment(state, action, obs, reward, final_obs)) return rc;
  if (misaligned(prev_obs, 8) || misaligned(ring_obs, 8) || misaligned(ring_action, 8) || misaligned(ring_next_obs, 8) ||
      misaligned(ring_meta, 8))
    return fail(-1, "misaligned buffer: prev_obs and the ring arrays need 8-byte alignment");
  if (action_mode < 0 || action_mode > 2) return fail(-1, "bad action_mode");
  if (h->cfg.reset_mode && h->cfg.reset_source == UAVCA_SOURCE_POOL && !h->pool_blob) return fail(-1, "reset_source is POOL but no pool is set");
  if (h->cfg.circular || h->cfg.num_agents > 32)
    return fail(-2, "uavca_step_multi_replay serves the warp kernels (N <= 32, float32 world): use uavca_step_multi + uavca_replay_push_dev");
  const int64_t M = (int64_t)h->cfg.num_envs * h->cfg.num_agents;
  if (capacity < M) return fail(-1, "uavca_step_multi_replay: the ring is smaller than one step's transitions");
  if (capacity * 10 >= (int64_t)1 << 31) return fail(-2, "uavca_step_multi_replay: ring rows are indexed in 32 bits (capacity * 10 < 2^31)");
  DeviceGuard g(h->device);
  KernelArgs a = make_args(h, state);
  a.io.action = reinterpret_cast<const float2*>(action);
  a.io.obs = obs; a.io.reward = reward; a.io.done = done; a.io.final_obs = final_obs; a.io.reset_mask = reset_mask;
  a.io.action_mode = action_mode; a.io.evaluate = evaluate;
  RingSink r{};
  r.prev_obs = reinterpret_cast<const float2*>(prev_obs);
  r.obs = reinterpret_cast<float2*>(ring_obs); r.act = reinterpret_cast<float2*>(ring_action); r.rew = ring_reward;
  r.nxt = reinterpret_cast<float2*>(ring_next_obs); r.mask = ring_mask;
  r.meta = reinterpret_cast<long long*>(ring_meta); r.cap = (int)capacity; r.M = (int)M;
  cudaError_t e = launch_step_multi_ring(a, r, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_step_multi_replay", e);
  h->launches += 1;
  return 0;
}

int uavca_policy_act(const float* obs, int64_t M, const void* w1, const void* w2, const void* w2b, const void* w3,
                     const void* w3b, const float* noise, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                     float* action, float* head, void* stream) {
  if (!obs || !w1 || !w2 || !w2b || !w3 || !w3b || !action) return fail(-1, "null argument");
  if (M < 0) return fail(-1, "bad size");
  auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  if (!a16(w1) || !a16(w2) || !a16(w2b) || !a16(w3) || !a16(w3b) || (reinterpret_cast<uintptr_t>(obs) & 7u) ||
      (reinterpret_cast<uintptr_t>(action) & 7u) || (head && !a16(head)) || (noise && (reinterpret_cast<uintptr_t>(noise) & 7u)))
    return fail(-1, "uavca_policy_act: misaligned buffer (weights/head 16 bytes, obs/action/noise 8 bytes)");
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, obs) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(-1, "uavca_policy_act: obs is not a device pointer");
  }
  DeviceGuard g(at.device);  // no handle here: the launch goes where the buffers live
  cudaError_t e = launch_policy_act(obs, M, w1, w2, w2b, w3, w3b, noise, seed, counter,
                                    reinterpret_cast<const unsigned long long*>(counter_dev), action, head, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail_cuda("uavca_policy_act", e);
  return 0;
}

int64_t uavca_launch_count(const uavca_handle* h) { return h ? h->launches : 0; }

}  // extern "C"

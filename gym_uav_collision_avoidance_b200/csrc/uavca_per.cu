// uavca_per.cu — prioritized replay over the device ring (Schaul et al. 2016; the Ape-X regime of Horgan et al. 2018):
// a float64 sum-tree over the ring's slots, kept on the device and fed from the ring's device-side head.
//
// Layout: tree float64 [2L], L = the least power of two >= capacity; the leaf of slot s is tree[L + s]; internal node k
// (1 <= k < L) is exactly tree[2k] + tree[2k+1] (one IEEE float64 addition, left child first); tree[1] is the total.
// tree[0] is no node: it holds the CTA ticket of the multi-CTA kernels below, and is 0 between calls.  Because every node
// is one fixed-order addition of its two children the tree is a pure function of its leaves, so each kernel may form the
// nodes in any order as long as both children are final when a node is formed.
#include <cfloat>

#include "uavca_host.h"
#include "uavca_nstep.cuh"

namespace uavca {

namespace {

constexpr int kSyncThreads = 512;
constexpr int kSyncLeaves = 1024;      // leaves per CTA block of the sync kernel (2 per thread), reduced in shared memory
constexpr int kUpdateThreads = 1024;   // the update is one CTA: its steps are separated by block barriers
constexpr int kSampleThreads = 256;
constexpr int kSampleLanes = kNstepLanes;  // lanes per sample: one node each of a 4-level chunk of the descent, then the gather
constexpr unsigned long long kMark = 0xFFF0000000000000ull;  // bits of -inf: above it the leaf holds an update's marker

__device__ __forceinline__ unsigned long long* ticket(double* tree) { return reinterpret_cast<unsigned long long*>(tree); }

// ---- sync: the slots appended since the last sync take the largest priority so far ---------------------------------
// Dirty leaves form at most two runs: A = [a0, a1) and B = [0, b1) with b1 <= a0 (the wrap of A).  CTA blocks are
// aligned runs of kSyncLeaves leaves (the whole leaf level when L is smaller); block t of the list of dirty blocks takes
// A's blocks first, then B's that A does not already hold.  Each CTA writes its dirty leaves, reads the other leaves of
// its block from the tree (they do not change in this launch) and writes every node of the block's subtree from shared
// memory; the last CTA to take a ticket forms the nodes above the block roots over the dirty span, level by level.
struct SyncPlan {
  long long a0, a1, b1;          // dirty runs
  long long ablk0, nA, bblk0, nB; // dirty blocks: [ablk0, ablk0 + nA) and [bblk0, bblk0 + nB)
  long long appends, head, d;
};

__device__ __forceinline__ SyncPlan sync_plan(const long long* pm, const long long* rm, long long cap, int lb) {
  SyncPlan p;
  p.appends = rm[3];
  p.head = rm[0];
  p.d = p.appends - pm[0];
  p.a0 = p.a1 = p.b1 = 0;
  if (p.d == 1) {
    const long long h0 = pm[1];
    long long n = p.head - h0;  // (head - h0) mod capacity; 0 is a full-capacity append (an append of 0 advances nothing)
    if (n < 0) n += cap;
    if (n == 0) n = cap;
    p.a0 = h0;
    if (h0 + n <= cap) {
      p.a1 = h0 + n;
    } else {
      p.a1 = cap;
      p.b1 = h0 + n - cap;
    }
  } else if (p.d != 0) {  // more than one append (or a ring rewound under the tree): every filled slot
    p.a1 = rm[2];
  }
  p.ablk0 = p.a0 >> lb;
  p.nA = p.a1 > p.a0 ? ((p.a1 - 1) >> lb) - p.ablk0 + 1 : 0;
  p.bblk0 = 0;
  long long bend = p.b1 > 0 ? (p.b1 - 1) >> lb : -1;
  if (p.nA > 0 && bend >= p.ablk0) bend = p.ablk0 - 1;  // that block is A's: its CTA writes B's leaves there too
  p.nB = bend + 1;
  return p;
}

__global__ void __launch_bounds__(kSyncThreads) per_sync_kernel(double* tree, long long L, int D, long long* pm,
                                                                const long long* rm, long long cap) {
  __shared__ double buf[kSyncLeaves + kSyncLeaves / 2];  // one level at [0, 1024), the next at [1024, ...), alternating
  __shared__ bool last;
  const long long bl = L < kSyncLeaves ? L : kSyncLeaves;
  int lb = 0;  // levels inside a block
  while ((1ll << lb) < bl) ++lb;
  const SyncPlan p = sync_plan(pm, rm, cap, lb);
  const double pmax = __longlong_as_double(pm[2]);
  for (long long t = blockIdx.x; t < p.nA + p.nB; t += gridDim.x) {
    const long long blk = t < p.nA ? p.ablk0 + t : p.bblk0 + (t - p.nA);
    const long long s0 = blk << lb;
    for (int i = threadIdx.x; i < bl; i += kSyncThreads) {
      const long long s = s0 + i;
      const bool dirty = (s >= p.a0 && s < p.a1) || s < p.b1;
      double v;
      if (dirty) {
        v = pmax;
        tree[L + s] = v;
      } else {
        v = tree[L + s];
      }
      buf[i] = v;
    }
    for (int lev = 1; lev <= lb; ++lev) {
      __syncthreads();
      const int cur = (lev & 1) ? 0 : kSyncLeaves, nxt = kSyncLeaves - cur;
      const int w = (int)(bl >> lev);
      const long long first = (L + s0) >> lev;  // node of the block's leftmost descendant at this level
      for (int i = threadIdx.x; i < w; i += kSyncThreads) {
        const double x = __dadd_rn(buf[cur + 2 * i], buf[cur + 2 * i + 1]);
        buf[nxt + i] = x;
        tree[first + i] = x;
      }
    }
    __syncthreads();  // the buffers are reused by the next block of this CTA
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(ticket(tree), 1ull) == (unsigned long long)gridDim.x - 1ull;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // the levels above the block roots, over the dirty blocks only; B's range sits below A's and does not overlap it
  long long alo = p.ablk0, ahi = p.ablk0 + p.nA - 1, blo = p.bblk0, bhi = p.bblk0 + p.nB - 1;
  for (int lev = lb + 1; lev <= D; ++lev) {
    alo >>= 1; ahi >>= 1; blo >>= 1; bhi >>= 1;
    if (p.nA > 0 && p.nB > 0 && bhi >= alo) bhi = alo - 1;
    const long long first = L >> lev;
    const long long na = p.nA > 0 ? ahi - alo + 1 : 0, nb = p.nB > 0 && bhi >= blo ? bhi - blo + 1 : 0;
    for (long long i = threadIdx.x; i < na + nb; i += kSyncThreads) {
      const long long k = first + (i < na ? alo + i : blo + (i - na));
      tree[k] = __dadd_rn(__ldcg(tree + 2 * k), __ldcg(tree + 2 * k + 1));
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    pm[0] = p.appends;
    pm[1] = p.head;
    if (p.d != 0 && p.d != 1) pm[3] += 1;
    *ticket(tree) = 0ull;
  }
}

// ---- update: leaf index[j] = priority[j], last occurrence wins --------------------------------------------------------
// One CTA.  (1) Every entry is checked; one bad entry drops the whole update (counted in per_meta[4]).  (2) The touched
// leaves are set to kMark, (3) each entry raises its leaf to kMark + j + 1 with a 64-bit atomicMax, so the leaf ends up
// naming the last occurrence, and (4) every entry writes priority[winner] to its leaf — all duplicates write the same
// value, and an entry that finds the priority already written (bits below kMark: priorities are finite and >= 0) has
// nothing to do.  (5) The ancestors are formed 4 levels per step: an entry reads the 16 nodes of its aligned sibling
// group (one 128-byte line), reduces them in registers in the tree's own pairwise order and writes the nodes on its own
// path; entries that share a node write the same bits, formed from the same final children.
__device__ __forceinline__ double pick8(const double (&v)[16], int i) {  // v[i], i < 8, without local memory
  double x = v[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) x = i == k ? v[k] : x;
  return x;
}

__global__ void __launch_bounds__(kUpdateThreads) per_update_kernel(double* tree, long long L, int D, long long cap,
                                                                    long long* pm, const long long* idx, const double* pr,
                                                                    long long n) {
  __shared__ double wmax[kUpdateThreads / 32];
  bool bad = false;
  double mx = 0.0;
  for (long long j = threadIdx.x; j < n; j += kUpdateThreads) {
    const long long i = idx[j];
    const double p = pr[j];
    if (i < 0 || i >= cap || !(p >= 0.0 && p <= DBL_MAX)) bad = true;
    else mx = fmax(mx, p);
  }
  if (__syncthreads_or(bad)) {
    if (threadIdx.x == 0) pm[4] += 1;
    return;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(kFull, mx, o));
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = mx;
  unsigned long long* bits = reinterpret_cast<unsigned long long*>(tree + L);
  for (long long j = threadIdx.x; j < n; j += kUpdateThreads) bits[idx[j]] = kMark;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = wmax[0];
    for (int w = 1; w < kUpdateThreads / 32; ++w) m = fmax(m, wmax[w]);
    if (m > __longlong_as_double(pm[2])) pm[2] = __double_as_longlong(m);
  }
  for (long long j = threadIdx.x; j < n; j += kUpdateThreads) atomicMax(bits + idx[j], kMark + (unsigned long long)j + 1ull);
  __syncthreads();
  for (long long j = threadIdx.x; j < n; j += kUpdateThreads) {
    const long long i = idx[j];
    const unsigned long long b = __ldcg(bits + i);
    if (b > kMark) tree[L + i] = pr[b - kMark - 1ull];
  }
  for (int lev = 0; lev < D;) {
    const int r = D - lev < 4 ? D - lev : 4;
    const int width = 1 << r;
    __syncthreads();
    for (long long j = threadIdx.x; j < n; j += kUpdateThreads) {
      const long long node = (L + idx[j]) >> lev;
      const long long base = node & ~(long long)(width - 1);
      const int off = (int)(node - base);
      double v[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) v[k] = k < width ? __ldcg(tree + base + k) : 0.0;
#pragma unroll
      for (int s = 0; s < 4; ++s) {
        if (s < r) {
#pragma unroll
          for (int k = 0; k < (8 >> s); ++k) v[k] = __dadd_rn(v[2 * k], v[2 * k + 1]);
          tree[(base >> (s + 1)) + (off >> (s + 1))] = pick8(v, off >> (s + 1));
        }
      }
    }
    lev += r;
  }
}

// ---- sample: stratified draws by descent, gather, importance weights -------------------------------------------------
// 16 lanes per sample.  The descent goes 4 levels per load: lane g reads node g of the 16 descendants 4 levels below the
// current node; the nodes in between are formed again by pairwise shuffles in the tree's own order, so they equal the
// stored ones bit for bit, and the 4 decisions are taken from them.  The last CTA to finish (ticket in tree[0]) forms
// the weights, which are normalised by the largest weight of the batch.
__device__ __forceinline__ double pair_sum(double x, int d, int g, unsigned mask) {
  const double o = __shfl_xor_sync(mask, x, d, kSampleLanes);
  return (g & d) ? __dadd_rn(o, x) : __dadd_rn(x, o);  // left child first on both lanes
}

// The slot of sample j (the 16 lanes of its group: lane g, shuffle mask `mask`): stratified u on the prioritized stream
// (tag 6) at counter draw + appends so far, then the descent; slot 0 when the tree is empty.  Shared by the one-step and
// the n-step sampler, so that both draw the same slots for the same (seed, draw, appends, tree).
__device__ __forceinline__ long long per_draw_slot(const double* tree, long long L, int D, double total, const long long* rm,
                                                   long long j, long long batch, unsigned seed_lo, unsigned seed_hi,
                                                   unsigned long long draw, int g, unsigned mask) {
  long long slot = 0;
  if (total > 0.0) {
    const unsigned long long ctr = draw + (unsigned long long)rm[3];
    const uint4 r = philox_indexed(kStreamPerSample, (unsigned long long)j, ctr, seed_lo, seed_hi);
    double u = __dmul_rn(__ddiv_rn(__dadd_rn((double)j, u53(r.x, r.y)), (double)batch), total);
    long long node = 1;
    for (int left = D; left > 0;) {
      const int lv = left < 4 ? left : 4;
      const int width = 1 << lv;
      const long long base = node << lv;
      const double v = g < width ? tree[base + g] : 0.0;
      const double s1 = pair_sum(v, 1, g, mask), s2 = pair_sum(s1, 2, g, mask), s3 = pair_sum(s2, 4, g, mask);
      int pos = 0;
      for (int w = width >> 1; w >= 1; w >>= 1) {
        const double sw = w == 8 ? s3 : w == 4 ? s2 : w == 2 ? s1 : v;
        const double lft = __shfl_sync(mask, sw, pos, kSampleLanes);
        const double rgt = __shfl_sync(mask, sw, pos + w, kSampleLanes);
        if (!(u < lft) && rgt != 0.0) {  // go left if u < left or the right subtree is empty
          u = __dsub_rn(u, lft);
          pos += w;
        }
      }
      node = base + pos;
      left -= lv;
    }
    slot = node - L;
  }
  return slot;
}

// One kernel for both samplers: kNstep = false is uavca_per_sample (the drawn rows and their mask), true is
// uavca_per_sample_nstep (the n-step gather of uavca_nstep.cuh, its discount in o_mask; cap, stride, n and gamma are
// read only there).  The weight pass stays in the kernel body: as a separate function it costs the one-step instance a
// spilled pointer around the pow calls.  The last CTA to take a ticket (tree[0]) forms the weights, w_j = (size * P_j)^-beta
// with P_j = leaf / total, divided by the largest w of the batch (batch < 2^26: int indices), and gives the ticket back.
template <bool kNstep>
__global__ void __launch_bounds__(kSampleThreads) per_sample_kernel(
    const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt, const float* r_mask, long long cap, int od,
    int ad, const long long* rm, double* tree, long long L, int D, long long batch, double beta, long long stride, int n,
    double gamma, unsigned seed_lo, unsigned seed_hi, unsigned long long draw, float* o_obs, float* o_act, float* o_rew,
    float* o_nxt, float* o_mask, long long* o_idx, float* o_w) {
  __shared__ bool last;
  __shared__ double red[kSampleThreads / 32];
  const long long j = ((long long)blockIdx.x * kSampleThreads + threadIdx.x) / kSampleLanes;
  const int g = threadIdx.x % kSampleLanes;
  const unsigned mask = 0xFFFFu << (threadIdx.x & 16);
  const double total = tree[1];
  if (j < batch) {
    const long long slot = per_draw_slot(tree, L, D, total, rm, j, batch, seed_lo, seed_hi, draw, g, mask);
    if constexpr (kNstep) {
      nstep_gather(r_obs, r_act, r_rew, r_nxt, r_mask, od, ad, cap, rm[0], stride, n, gamma, slot, j, g, mask, o_obs, o_act,
                   o_rew, o_nxt, o_mask);
      if (g == 0) o_idx[j] = slot;
    } else {
      for (int k = g; k < od; k += kSampleLanes) {
        o_obs[j * od + k] = r_obs[slot * od + k];
        o_nxt[j * od + k] = r_nxt[slot * od + k];
      }
      for (int k = g; k < ad; k += kSampleLanes) o_act[j * ad + k] = r_act[slot * ad + k];
      if (g == 0) {
        o_rew[j] = r_rew[slot];
        o_mask[j] = r_mask[slot];
        o_idx[j] = slot;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(ticket(tree), 1ull) == (unsigned long long)gridDim.x - 1ull;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  const double size = (double)rm[2];
  const double* leaf = tree + L;
  const int nb = (int)batch;
  double mx = 0.0;
  if (total > 0.0) {
    for (int i = threadIdx.x; i < nb; i += kSampleThreads)
      mx = fmax(mx, pow(__dmul_rn(size, __ddiv_rn(leaf[__ldcg(o_idx + i)], total)), -beta));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(kFull, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = red[0];
    for (int w = 1; w < kSampleThreads / 32; ++w) mx = fmax(mx, red[w]);
  }
  for (int i = threadIdx.x; i < nb; i += kSampleThreads) {
    float w = 0.0f;  // an empty ring: slot 0 weighs nothing
    if (total > 0.0) w = __double2float_rn(__ddiv_rn(pow(__dmul_rn(size, __ddiv_rn(leaf[__ldcg(o_idx + i)], total)), -beta), mx));
    o_w[i] = w;
  }
  if (threadIdx.x == 0) *ticket(tree) = 0ull;
}

int log2_exact(long long L) {
  int D = 0;
  while ((1ll << D) < L) ++D;
  return D;
}

int sm_count() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
      sms <= 0)
    sms = 148;
  return sms;
}

}  // namespace

cudaError_t launch_per_sync(double* tree, long long L, long long* per_meta, const long long* ring_meta, long long capacity,
                            cudaStream_t st) {
  const long long blocks = (L + kSyncLeaves - 1) / kSyncLeaves;
  const long long cap_grid = 2ll * sm_count();
  per_sync_kernel<<<(int)(blocks < cap_grid ? blocks : cap_grid), kSyncThreads, 0, st>>>(tree, L, log2_exact(L), per_meta,
                                                                                        ring_meta, capacity);
  return cudaGetLastError();
}

cudaError_t launch_per_update(double* tree, long long L, long long capacity, long long* per_meta, const long long* index,
                              const double* priority, long long n, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  per_update_kernel<<<1, kUpdateThreads, 0, st>>>(tree, L, log2_exact(L), capacity, per_meta, index, priority, n);
  return cudaGetLastError();
}

cudaError_t launch_per_sample(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                              const float* r_mask, int obs_dim, int act_dim, const long long* ring_meta, double* tree,
                              long long L, long long batch, double beta, unsigned long long seed, unsigned long long draw,
                              float* o_obs, float* o_act, float* o_rew, float* o_nxt, float* o_mask, long long* o_idx,
                              float* o_w, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  const long long grid = (batch * kSampleLanes + kSampleThreads - 1) / kSampleThreads;
  per_sample_kernel<false><<<(int)grid, kSampleThreads, 0, st>>>(
      r_obs, r_act, r_rew, r_nxt, r_mask, 0, obs_dim, act_dim, ring_meta, tree, L, log2_exact(L), batch, beta, 0, 1, 0.0,
      (unsigned)(seed & 0xffffffffull), (unsigned)(seed >> 32), draw, o_obs, o_act, o_rew, o_nxt, o_mask, o_idx, o_w);
  return cudaGetLastError();
}

cudaError_t launch_per_sample_nstep(const float* r_obs, const float* r_act, const float* r_rew, const float* r_nxt,
                                    const float* r_mask, long long capacity, int obs_dim, int act_dim,
                                    const long long* ring_meta, double* tree, long long L, long long batch, double beta,
                                    long long stride, int n, double gamma, unsigned long long seed, unsigned long long draw,
                                    float* o_obs, float* o_act, float* o_rew, float* o_nxt, float* o_disc, long long* o_idx,
                                    float* o_w, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  const long long grid = (batch * kSampleLanes + kSampleThreads - 1) / kSampleThreads;
  per_sample_kernel<true><<<(int)grid, kSampleThreads, 0, st>>>(
      r_obs, r_act, r_rew, r_nxt, r_mask, capacity, obs_dim, act_dim, ring_meta, tree, L, log2_exact(L), batch, beta, stride,
      n, gamma, (unsigned)(seed & 0xffffffffull), (unsigned)(seed >> 32), draw, o_obs, o_act, o_rew, o_nxt, o_disc, o_idx,
      o_w);
  return cudaGetLastError();
}

}  // namespace uavca

// uavca_policy.cu — fused acting path of the shared SAC policy ("next" row 2 of SURVEY.md §8f) on the 5th-generation
// tensor cores: obs [M,10] -> relu(W1) -> relu(W2) -> (mean, log_std) -> tanh(mean + exp(log_std) * eps) in ONE kernel.
//
// Restates GaussianPolicy.forward/sample (pytorch_sac_temp/model.py:74-101) as used by SAC.select_action
// (pytorch_sac_temp/sac.py:38-44) for all M = B*N UAVs at once (every UAV shares one policy, test_sac_multi.py:90-91).
// The reference runs it as four cuBLAS GEMVs per UAV per step; batched in eager PyTorch the two hidden layers
// dominate a rollout step (~960 us of 980 us at B=16,384 x N=10 in fp32, 276 us under bf16 autocast, mostly
// elementwise traffic on the [M,256] activations).  Here the activations never leave the SM, all three layers run
// on the tensor cores and the biases ride along as one extra K step against a constant "ones" operand:
//
//   per CTA (persistent, one per SM; 16 warps: warp w owns TMEM lanes 32*(w%4).. and hidden columns 64*(w/4)..),
//   per tile of 128 rows (D = one of two 256-column TMEM accumulators, tiles alternate between them):
//     obs rows -> fp16 A1 [128x16] in smem (10 features, a 1.0 in column 10 that multiplies b1, zero padding)
//     tcgen05.mma  D[128x256] = A1 . [W1 | b1]^T                                       1 MMA  (M=128, N=256, K=16)
//     tcgen05.ld D -> relu -> fp16 -> A2 [128x256] in smem, written straight into the 128B-swizzled K-major
//                                                                         layout the MMA descriptor expects
//     tcgen05.mma  D[128x256] = A2 . W2^T   (over the layer-1 result it was computed from)   16 MMAs
//     output heads: tcgen05.ld.16x256b hands every warp its 32 rows x 64 columns of D in the register layout of a
//                   warp-level mma.sync A fragment; + b2 (fp32), relu, fp16, then 8 mma.sync.m16n8k16 per warp against
//                   W3 fragments held in registers; the four column groups of a row meet in shared memory.
//                   (Round 1 ran the heads as 17 tcgen05 MMAs of N=16 — as much tensor-pipe time as the 256-wide layer 2
//                   plus a second fp16 round trip through shared memory; the first round-2 version used packed FP32 FMAs
//                   with W3 broadcast from shared memory: 96 LDS per thread and tile, 3,200 of 7,100 cycles per tile.)
//     mean, log_std; eps ~ N(0,1) from Philox4x32-10 + Box-Muller (or caller-supplied)
//                   -> action = tanh(mean + exp(clamp(log_std)) eps)
//   Software pipeline over the CTA's tiles: while the tensor cores run layer 2 of tile i (2,250 cycles), the threads
//   compute heads + sampling of tile i-1 from the other accumulator and stage layer 1 of tile i+1, which is queued
//   behind it; only the layer-1 epilogue (350 cycles, it needs the A2 buffer layer 2 reads) leaves the tensor pipe idle.
//
// W2 (fp16, 128 KB) stays resident in shared memory for the CTA's lifetime.  The tensor-core operands (W1 | b1, W2,
// activations, W3) are fp16 with fp32 accumulation (11 significand bits, like TF32).  b2 and b3 are fp16 too (rounded on
// the host like every operand) but are added in fp32, and the second hidden layer reaches the heads unrounded (fp32).  The
// policy is the learner's side of the boundary, not part of the env-step parity contract: tests/test_acting_kernels_gpu.py
// holds the heads to a float64 emulation of exactly these rounding points (a per-row bound from the fp32 accumulation,
// ~1e-4 for O(1) heads) and to the unquantised float64 policy (a bound from the 2^-11 rounding of every fp16 operand).
#include <cuda_fp16.h>

#include <atomic>

#include "uavca_host.h"

namespace uavca {

namespace pol {

constexpr int kRows = 128;      // rows per tile = TMEM lanes
constexpr int kColGroups = 4;   // the 256 hidden columns of a row are split over 4 threads (64 each)
constexpr int kEpiThreads = kRows * kColGroups;  // 16 epilogue warps: warp w works on TMEM lanes 32*(w%4).., columns 64*(w/4)..
constexpr int kThreads = kEpiThreads + 32;       // + 1 warp that stages the observations and issues the MMAs
constexpr int kHidden = 256;
constexpr int kInPad = 16;      // obs features padded to one MMA K step
constexpr int kObs = 10;
constexpr uint32_t kTmemCols = 512;

// shared-memory carve-up (bytes; the swizzled operands need 1024-byte alignment)
constexpr int kW2Bytes = kHidden * kHidden * 2;       // 131072: 4 K-blocks x [256 rows x 128 B], 128B swizzle
constexpr int kA2Bytes = kRows * kHidden * 2;         //  65536: 4 K-blocks x [128 rows x 128 B], 128B swizzle
constexpr int kW1Bytes = kHidden * kInPad * 2;        //   8192: K = 16, no swizzle, 8x16B core matrices ([W1 | b1])
constexpr int kA1Bytes = kRows * kInPad * 2;          //   4096
constexpr int kB2fBytes = kHidden * 4;                //   1024: linear2.bias in fp32
constexpr int kW3fBytes = kHidden * 16;               //   4096: float4 per hidden unit = its weight in the four heads (fp32)
constexpr int kPartBytes = 4 * kRows * 16;            //   8192: head partials of the four column groups (float4 per row)
constexpr int kOffW2 = 0;
constexpr int kOffA2 = kOffW2 + kW2Bytes;
constexpr int kOffW1 = kOffA2 + kA2Bytes;
constexpr int kOffA1 = kOffW1 + kW1Bytes;
constexpr int kOffW3f = kOffA1 + kA1Bytes;
constexpr int kOffB2f = kOffW3f + kW3fBytes;
constexpr int kOffPart = kOffB2f + kB2fBytes;
constexpr int kOffB3 = kOffPart + kPartBytes;         // float4: the four head biases
constexpr int kOffBar = kOffB3 + 16;                  // mbarriers + tmem base
constexpr int kSmemBytes = kOffBar + 64;
constexpr int kSmemAlloc = kSmemBytes + 1024;         // slack to align the dynamic buffer to 1024 B
static_assert(kSmemAlloc <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- descriptors (cute/arch/mma_sm100_desc.hpp layouts, written out) ------------------------------------------------
// shared-memory matrix descriptor: [0,14) start>>4, [16,30) leading byte offset>>4, [32,46) stride byte offset>>4,
// [46,48) version = 1 (sm_100), [61,64) layout type (0 none, 2 = 128B swizzle)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
// instruction descriptor, kind::f16: c_format F32 (1 << 4), a/b format F16 (0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr uint32_t idesc(int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24); }

__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate, uint32_t kIdesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(kIdesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void bar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "POL_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra POL_DONE_%=;\n"
      "bra POL_WAIT_%=;\n"
      "POL_DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// 32 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 16 TMEM lanes x 64 columns in the register layout of mma.sync fragments: lane l of the warp gets, for every group j of
// 8 columns, (row l/4, columns 8j + 2(l%4) + {0,1}) in v[4j], v[4j+1] and (row l/4 + 8, same columns) in v[4j+2], v[4j+3]
__device__ __forceinline__ void tmem_ld_16x64(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// the same for 32 columns: v[4j..4j+3] = group j of 8 columns.  No wait: tmem_wait_2x16 below makes the values usable.
__device__ __forceinline__ void tmem_ld_16x32(uint32_t taddr, float (&v)[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// tcgen05.wait::ld for two loads in flight; the values pass through the statement so that no use can move above it
__device__ __forceinline__ void tmem_wait_2x16(float (&x)[16], float (&y)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(x[0]), "+f"(x[1]), "+f"(x[2]), "+f"(x[3]), "+f"(x[4]), "+f"(x[5]), "+f"(x[6]), "+f"(x[7]), "+f"(x[8]),
                 "+f"(x[9]), "+f"(x[10]), "+f"(x[11]), "+f"(x[12]), "+f"(x[13]), "+f"(x[14]), "+f"(x[15]), "+f"(y[0]),
                 "+f"(y[1]), "+f"(y[2]), "+f"(y[3]), "+f"(y[4]), "+f"(y[5]), "+f"(y[6]), "+f"(y[7]), "+f"(y[8]), "+f"(y[9]),
                 "+f"(y[10]), "+f"(y[11]), "+f"(y[12]), "+f"(y[13]), "+f"(y[14]), "+f"(y[15])
               :
               : "memory");
}
// warp-level D[16x8] += A[16x16] . B[16x8] (fp16 operands, fp32 accumulate)
__device__ __forceinline__ void mma_m16n8k16(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// (relu(x), relu(y)) as fp16x2, x in the low half: the clamp rides in the conversion (F2FP.RELU), no FMNMX
__device__ __forceinline__ uint32_t relu_pack(float x, float y) {
  uint32_t d;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(y), "f"(x));
  return d;
}
// tanh(x) = sign(x) (1 - 2 / (e^{2|x|} + 1)) on the SFU exponential and reciprocal: absolute error ~1e-7
__device__ __forceinline__ float tanh_fast(float x) {
  const float e = __expf(2.0f * fabsf(x));
  return copysignf(1.0f - __fdividef(2.0f, e + 1.0f), x);
}

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// tcgen05.wait::ld for two 32-column loads in flight; the values pass through the statement so that no use moves above it
__device__ __forceinline__ void tmem_wait_2x32(float (&x)[32], float (&y)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) asm volatile("" : "+f"(x[i]), "+f"(y[i]));
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

// byte offset of the 16-byte chunk holding elements [8c, 8c+8) of row r inside a K-major, 128B-swizzled operand
// whose K-blocks (64 halves = 128 B per row) are `block_bytes` apart: rows 128 B apart in 8-row atoms of 1024 B,
// chunk index XORed with the row inside the atom (Swizzle<3,4,3>)
__device__ __forceinline__ uint32_t sw128_chunk(int r, int c, int block_bytes) {
  return (uint32_t)((c >> 3) * block_bytes + (r >> 3) * 1024 + (r & 7) * 128 + (((c & 7) ^ (r & 7)) << 4));
}
// no-swizzle K-major operand with K = 16 (two 16-byte chunks per row): 8x16B core matrices, the two K chunks of an
// 8-row group 128 B apart (leading byte offset), 8-row groups 256 B apart (stride byte offset)
__device__ __forceinline__ uint32_t k16_chunk(int r, int c) { return (uint32_t)((r >> 3) * 256 + c * 128 + (r & 7) * 16); }

struct Args {
  const float* obs;     // [M][10]
  const __half* w1;     // [256][16]: linear1.weight in columns 0..9, linear1.bias in column 10, zeros
  const __half* w2;     // [256][256]: linear2.weight
  const __half* w2b;    // [256][16]: linear2.bias in column 0, zeros
  const __half* w3;     // [16][256]: rows 0,1 mean_linear.weight, rows 2,3 log_std_linear.weight, zeros
  const __half* w3b;    // [16][16]: the four head biases in column 0 of rows 0..3, zeros
  const float* noise;   // [M][2] standard normal draws, or nullptr -> Philox
  float* action;        // [M][2]
  float* head;          // [M][4] (mean0, mean1, log_std0, log_std1) or nullptr
  long long M;
  unsigned seed_lo, seed_hi;
  unsigned long long ctr;               // Philox call counter = ctr + *ctr_dev (kStreamPolicy layout, uavca_device.cuh)
  const unsigned long long* ctr_dev;    // nullable
};

__global__ void __launch_bounds__(kThreads, 1) policy_act_kernel(const __grid_constant__ Args a) {
  extern __shared__ unsigned char smem_raw[];
  // aligned to 1024 B by pointer arithmetic on the __shared__ array (keeps the address space: LDS / STS, not generic LD / ST)
  unsigned char* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int q = warp & 3;          // TMEM lane quarter this warp may access
  const int g = warp >> 2;         // column group
  const int r = q * 32 + lane;     // row of the tile (= TMEM lane)
  const uint32_t sbase = smem_u32(sm);
  const uint32_t bar = sbase + kOffBar;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBar + 16);

  // ---- one-time setup: TMEM, barrier, weights into shared memory in MMA layouts
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (t == 0) {
    bar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // Launched with programmatic stream serialization: everything above overlaps the tail of the previous kernel in the
  // stream; nothing that kernel (or any earlier one) may have written — weights, observations, the call counter — is read
  // before this point.  (Prefetching the weights above the wait was measured: 0.45 us of 29.6, not worth a stale-weights
  // hazard for a caller that rewrites them right before acting.)
  cudaGridDependencySynchronize();
  {
    // weights: 16-byte asynchronous copies (LDGSTS) straight into the MMA layouts.  Two groups: the small layer-1
    // operand [W1 | b1] (512 chunks) first — the first tile's layer 1 and its epilogue run while W2 (128 KB) streams in
    if (t < kEpiThreads) cp_async16(sbase + kOffW1 + k16_chunk(t >> 1, t & 1), reinterpret_cast<const uint4*>(a.w1) + t);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const uint4* w2g = reinterpret_cast<const uint4*>(a.w2);  // 256 rows x 32 chunks of 8 halves
#pragma unroll 8
    for (int idx = t; idx < kHidden * 32; idx += kThreads) {
      const int n = idx >> 5, c = idx & 31;
      cp_async16(sbase + kOffW2 + sw128_chunk(n, c, kHidden * 128), w2g + idx);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (t < kHidden) {  // fp32 tables of the head layer: W3 transposed to one float4 per hidden unit, linear2.bias
      const __half* w3 = a.w3;
      reinterpret_cast<float4*>(sm + kOffW3f)[t] = make_float4(__half2float(w3[t]), __half2float(w3[kHidden + t]),
                                                               __half2float(w3[2 * kHidden + t]), __half2float(w3[3 * kHidden + t]));
      reinterpret_cast<float*>(sm + kOffB2f)[t] = __half2float(a.w2b[t * kInPad]);
    }
    if (t == 0)
      *reinterpret_cast<float4*>(sm + kOffB3) = make_float4(__half2float(a.w3b[0]), __half2float(a.w3b[kInPad]),
                                                            __half2float(a.w3b[2 * kInPad]), __half2float(a.w3b[3 * kInPad]));
  }
  asm volatile("cp.async.wait_group 1;" ::: "memory");  // [W1 | b1] has landed; W2 is awaited before the first layer-2 MMA
  fence_async_smem();
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_slot;
  // this warp's TMEM lane quarter, first of its 64 hidden columns, as an offset from an accumulator's first column
  const uint32_t lane_off = ((uint32_t)(q * 32) << 16) + (uint32_t)(g * 64);
#ifdef UAVCA_POLICY_HEADS_MMA
  // this lane's share of the head weights as mma.sync B fragments: k-step s covers hidden units 64g + 16s .. + 15,
  // column n = lane / 4 of B is head n (rows 4..15 of the [16][256] W3 operand are zero)
  uint32_t w3frag[4][2];
#pragma unroll
  for (int s4 = 0; s4 < 4; ++s4) {
    const __half* wp = a.w3 + (lane >> 2) * kHidden + g * 64 + s4 * 16 + 2 * (lane & 3);
    w3frag[s4][0] = *reinterpret_cast<const uint32_t*>(wp);
    w3frag[s4][1] = *reinterpret_cast<const uint32_t*>(wp + 8);
  }
#endif
  const unsigned long long ctr = a.ctr + (a.ctr_dev ? *a.ctr_dev : 0ull);

  const long long tiles = (a.M + kRows - 1) / kRows;
#ifdef UAVCA_POLICY_TIMING
  long long tk[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  long long tprev = clock64();
  const long long tstart = tprev;
#define POL_TICK(i) { long long now = clock64(); tk[i] += now - tprev; tprev = now; }
#else
#define POL_TICK(i)
#endif
  // accumulator columns [col0, col0+64) of this thread's row -> relu -> fp16 -> K-block g of the A2 operand
  auto relu_to_a2 = [&](uint32_t acc) {
    float v[2][32];
    tmem_ld32_nowait(acc + lane_off, v[0]);
    tmem_ld32_nowait(acc + lane_off + 32u, v[1]);
    tmem_wait_2x32(v[0], v[1]);
    POL_TICK(6)
#pragma unroll
    for (int c = 0; c < 2; ++c) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {  // four 16-byte chunks of 8 hidden units
        uint32_t h[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) h[j] = relu_pack(v[c][k4 * 8 + 2 * j], v[c][k4 * 8 + 2 * j + 1]);
        *reinterpret_cast<uint4*>(sm + kOffA2 + sw128_chunk(r, g * 8 + c * 4 + k4, kRows * 128)) = *reinterpret_cast<const uint4*>(h);
      }
    }
  };
  // D2 = A2 . W2^T (K = 256 in 16 steps of the 128B-swizzled K-major operands)
  auto issue_layer2 = [&](uint32_t acc) {
#pragma unroll
    for (int kb = 0; kb < 4; ++kb) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {  // K = 16 halves = 32 bytes per step inside the 128-byte swizzle atom
        const uint64_t da = smem_desc(sbase + kOffA2 + kb * (kRows * 128) + ks * 32, 16, 1024, 2);
        const uint64_t db = smem_desc(sbase + kOffW2 + kb * (kHidden * 128) + ks * 32, 16, 1024, 2);
        mma_f16(acc, da, db, (uint32_t)((kb | ks) != 0), idesc(kHidden));
      }
    }
  };
#ifdef UAVCA_POLICY_HEADS_MMA
  // The output heads of this warp's 32 rows x 64 hidden units: h = relu(D + b2) in fp16 as mma.sync A fragments (the
  // 16x256b TMEM load delivers exactly that register layout), times the W3 fragments; partial (mean0, mean1, log_std0,
  // log_std1) of every row into Part[g][row].
  auto heads = [&](uint32_t acc) {
    const float2* b2p = reinterpret_cast<const float2*>(sm + kOffB2f) + g * 32 + (lane & 3);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      float v[32];
      tmem_ld_16x64(acc + lane_off + ((uint32_t)(mt * 16) << 16), v);
      float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int s4 = 0; s4 < 4; ++s4) {
        uint32_t af[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int j = 2 * s4 + h;  // group of 8 columns
          const float2 bb = b2p[4 * j];
          af[2 * h + 0] = relu_pack(v[4 * j + 0] + bb.x, v[4 * j + 1] + bb.y);  // row lane/4
          af[2 * h + 1] = relu_pack(v[4 * j + 2] + bb.x, v[4 * j + 3] + bb.y);  // row lane/4 + 8
        }
        mma_m16n8k16(c, af, w3frag[s4]);
      }
      if ((lane & 3) < 2) {  // accumulator columns 2(lane%4) + {0,1}: heads 0..3 live in lanes with lane%4 < 2
        float2* pp = reinterpret_cast<float2*>(sm + kOffPart) + ((g * kRows + q * 32 + mt * 16 + (lane >> 2)) * 2 + (lane & 3));
        pp[0] = make_float2(c[0], c[1]);
        pp[16] = make_float2(c[2], c[3]);  // 8 rows further
      }
    }
  };

#else
  // The same on the CUDA cores (the warp-level mma.sync shares the tensor pipe with tcgen05.mma and queues behind the
  // layer-2 MMAs it is meant to overlap): in the 16x256b register layout a thread holds 4 rows x 16 hidden units, so one
  // float4 of W3 per hidden unit serves 4 rows (32 LDS per thread and tile instead of 96), two heads per packed FMA;
  // the 4 lanes that share a row add up through shuffles.
  auto heads_fma = [&](uint32_t acc) {
    const float2* b2p = reinterpret_cast<const float2*>(sm + kOffB2f) + g * 32 + (lane & 3);
    const float4* w3p = reinterpret_cast<const float4*>(sm + kOffW3f) + g * 64 + 2 * (lane & 3);
    float2 s01[4], s23[4];  // (row lane/4, lane/4 + 8) of the lower 16 rows, the same of the upper 16 rows
#pragma unroll
    for (int i = 0; i < 4; ++i) s01[i] = s23[i] = make_float2(0.f, 0.f);
#pragma unroll
    for (int half = 0; half < 2; ++half) {  // 32 of the warp's 64 columns at a time, both 16-row halves of the quarter
      float v[2][16];
      tmem_ld_16x32(acc + lane_off + (uint32_t)(half * 32), v[0]);
      tmem_ld_16x32(acc + lane_off + (uint32_t)(half * 32) + (16u << 16), v[1]);
      tmem_wait_2x16(v[0], v[1]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int jj = half * 4 + j;  // group of 8 columns: this lane has hidden units 64g + 8jj + 2(lane%4) + {0,1}
        const float2 bb = b2p[4 * jj];
        const float4 wa = w3p[8 * jj], wb = w3p[8 * jj + 1];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 x = __fadd2_rn(make_float2(v[i >> 1][4 * j + 2 * (i & 1)], v[i >> 1][4 * j + 2 * (i & 1) + 1]), bb);
          const float h0 = fmaxf(x.x, 0.f), h1 = fmaxf(x.y, 0.f);
          s01[i] = __ffma2_rn(make_float2(h0, h0), make_float2(wa.x, wa.y), s01[i]);
          s23[i] = __ffma2_rn(make_float2(h0, h0), make_float2(wa.z, wa.w), s23[i]);
          s01[i] = __ffma2_rn(make_float2(h1, h1), make_float2(wb.x, wb.y), s01[i]);
          s23[i] = __ffma2_rn(make_float2(h1, h1), make_float2(wb.z, wb.w), s23[i]);
        }
      }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      // sum over the 4 lanes of a row: odd lanes end up with the upper row of the pair, and of those the lanes with
      // bit 1 set with heads 2,3 — 6 shuffles instead of 16
      const float2 lo01 = s01[2 * mt], lo23 = s23[2 * mt], hi01 = s01[2 * mt + 1], hi23 = s23[2 * mt + 1];
      const bool odd = lane & 1;
      const float2 t01 = odd ? lo01 : hi01, t23 = odd ? lo23 : hi23;  // what the partner keeps
      float2 k01 = odd ? hi01 : lo01, k23 = odd ? hi23 : lo23;
      k01.x += __shfl_xor_sync(0xffffffffu, t01.x, 1); k01.y += __shfl_xor_sync(0xffffffffu, t01.y, 1);
      k23.x += __shfl_xor_sync(0xffffffffu, t23.x, 1); k23.y += __shfl_xor_sync(0xffffffffu, t23.y, 1);
      const bool up = lane & 2;
      const float2 snd = up ? k01 : k23;
      float2 keep = up ? k23 : k01;
      keep.x += __shfl_xor_sync(0xffffffffu, snd.x, 2); keep.y += __shfl_xor_sync(0xffffffffu, snd.y, 2);
      // this lane: row lane/4 + 8 * (lane & 1), heads 2 * (lane >> 1 & 1) + {0, 1}
      float2* pp = reinterpret_cast<float2*>(sm + kOffPart) +
                   ((g * kRows + q * 32 + mt * 16 + (lane >> 2) + 8 * (lane & 1)) * 2 + ((lane >> 1) & 1));
      *pp = keep;
    }
  };
#endif

  auto issue_layer1 = [&](uint32_t acc) {
    mma_f16(acc, smem_desc(sbase + kOffA1, 128, 256, 0), smem_desc(sbase + kOffW1, 128, 256, 0), 0u, idesc(kHidden));
  };
  // barrier 1: all warps
  auto sync_all = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory"); };

  const int n_my = (int)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);  // tiles of this CTA (>= 1: grid <= tiles)
  uint32_t phase = 0;

  // Iteration `it` of the software pipeline: layer-1 epilogue and layer-2 MMAs of tile it, heads + sampling of tile
  // it-1, layer-1 operand and MMA of tile it+1.  One mbarrier: each commit covers everything issued before it.
  if (warp == kEpiThreads / 32) {
    // ================= staging / MMA warp: lane l owns rows l, l+32, l+64, l+96 of a tile (five 8-byte loads per row,
    // the same 16-byte chunks of the A1 operand the MMA reads).  A tcgen05.mma only issues when the tensor pipe's queue
    // has room (16 layer-2 MMAs block for ~1,600 cycles): that wait is this warp's alone.
    float2 o[4][kObs / 2];
    auto load_tile = [&](long long tile) {
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const long long row = tile * kRows + lane + 32 * rr;
        const bool ok = tile < tiles && row < a.M;
        const float2* gp = reinterpret_cast<const float2*>(a.obs + (ok ? row : 0) * kObs);
#pragma unroll
        for (int k = 0; k < kObs / 2; ++k) {
          o[rr][k] = make_float2(0.f, 0.f);
          // volatile: issued HERE, a whole iteration before stage_a1 consumes it (ptxas otherwise sinks the load to its use)
          if (ok) asm volatile("ld.global.cs.v2.f32 {%0, %1}, [%2];" : "=f"(o[rr][k].x), "=f"(o[rr][k].y) : "l"(gp + k));
        }
      }
    };
    auto stage_a1 = [&]() {
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const int row = lane + 32 * rr;
        __half2 h[8];
#pragma unroll
        for (int k = 0; k < 5; ++k) h[k] = __floats2half2_rn(o[rr][k].x, o[rr][k].y);
        h[5] = __floats2half2_rn(1.f, 0.f);  // the bias column
        h[6] = h[7] = __floats2half2_rn(0.f, 0.f);
        *reinterpret_cast<uint4*>(sm + kOffA1 + k16_chunk(row, 0)) = *reinterpret_cast<const uint4*>(&h[0]);
        *reinterpret_cast<uint4*>(sm + kOffA1 + k16_chunk(row, 1)) = *reinterpret_cast<const uint4*>(&h[4]);
      }
      POL_TICK(6)
      fence_async_smem();
      POL_TICK(7)
    };
    load_tile(blockIdx.x);
    stage_a1();
    load_tile((long long)blockIdx.x + gridDim.x);
    __syncwarp();
    if (lane == 0) {
      fence_after();
      issue_layer1(tmem);
      mma_commit(bar);
    }
    for (int it = 0; it <= n_my; ++it) {
      const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
      const uint32_t acc_cur = tmem + (uint32_t)((it & 1) * 256), acc_prev = tmem + (uint32_t)(((it & 1) ^ 1) * 256);
      const bool has_cur = it < n_my, has_next = it + 1 < n_my;
      bar_wait(bar, phase);  // layer 1 of tile it is complete: the A1 operand is free
      phase ^= 1u;
      POL_TICK(0)
      if (has_next) {
        stage_a1();
        load_tile(tile + 2 * (long long)gridDim.x);  // two tiles ahead: in flight for a whole iteration
      }
      if (it == 0) {  // this thread's share of W2
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        fence_async_smem();
      }
      POL_TICK(1)
      sync_all();  // the epilogue warps have turned the layer-1 result of tile it into the A2 operand
      POL_TICK(2)
      if (lane == 0 && has_cur) {
        fence_after();
        issue_layer2(acc_cur);
      }
      POL_TICK(3)
      sync_all();  // ... and are done with the other accumulator (heads of tile it-1)
      POL_TICK(4)
      if (lane == 0 && has_cur) {
        fence_after();
        if (has_next) issue_layer1(acc_prev);
        mma_commit(bar);
      }
      __syncwarp();
    }
  } else {
    // ================= epilogue warps
    for (int it = 0; it <= n_my; ++it) {
      const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
      const uint32_t acc_cur = tmem + (uint32_t)((it & 1) * 256), acc_prev = tmem + (uint32_t)(((it & 1) ^ 1) * 256);
      const bool has_cur = it < n_my, has_prev = it > 0;

      // everything issued so far is complete: layer 2 of tile it-1 (acc_prev), layer 1 of tile it (acc_cur); A2 is free
      bar_wait(bar, phase);
      phase ^= 1u;
      fence_after();
      POL_TICK(0)
      if (has_cur) {  // ---- layer 1 epilogue -> A2
        relu_to_a2(acc_cur);
        POL_TICK(7)
        if (it == 0) asm volatile("cp.async.wait_group 0;" ::: "memory");  // this thread's share of W2
        fence_async_smem();
      }
      POL_TICK(1)
      fence_before();
      sync_all();
      POL_TICK(2)
      // ---- while the tensor cores run layer 2 of tile it: the output heads of tile it-1.  The standard-normal draws of
      // its rows do not depend on the heads: the column-group-0 warps compute them first, so that the Philox / Box-Muller
      // chain interleaves with the TMEM loads and FMAs of the heads instead of standing alone on the critical path
      const long long row = (tile - gridDim.x) * kRows + r;
      const bool samples = has_prev && g == 0 && row < a.M;
      float e0 = 0.f, e1 = 0.f;
      if (samples) {
        if (a.noise) {
          const float2 z = reinterpret_cast<const float2*>(a.noise)[row];
          e0 = z.x; e1 = z.y;
        } else {  // Box-Muller on one block of the policy's Philox4x32-10 stream keyed by (seed, row, call counter)
          const uint4 rn = philox_indexed(kStreamPolicy, (unsigned long long)row, ctr, a.seed_lo, a.seed_hi);
          const float u1 = ((float)(rn.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
          const float u2 = ((float)(rn.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
          const float rad = sqrtf(-2.0f * __logf(u1));
          float sn, cs;
          __sincosf(6.28318530717958647692f * u2, &sn, &cs);
          e0 = rad * cs; e1 = rad * sn;
        }
      }
      if (has_prev) {
#if !defined(UAVCA_POLICY_HEADS_MMA)
        heads_fma(acc_prev);
#else
        heads(acc_prev);
#endif
        POL_TICK(3)
      }
      fence_before();
      sync_all();  // acc_prev may be overwritten (layer 1 of tile it+1, which the MMA warp issues now); the four column
                   // groups of every row have met in shared memory (rewritten only after the next iteration's first barrier)
      POL_TICK(4)
      if (samples) {
        // ---- sample and squash (one thread per row), while the tensor pipe runs layer 1 of the next tile
        const float4* pp = reinterpret_cast<const float4*>(sm + kOffPart) + r;
        const float4 p0 = pp[0], p1 = pp[kRows], p2 = pp[2 * kRows], p3 = pp[3 * kRows], b3 = *reinterpret_cast<const float4*>(sm + kOffB3);
        const float m0 = p0.x + p1.x + p2.x + p3.x + b3.x, m1 = p0.y + p1.y + p2.y + p3.y + b3.y;
        const float l0 = fminf(fmaxf(p0.z + p1.z + p2.z + p3.z + b3.z, -20.f), 2.f);  // LOG_SIG_MIN / LOG_SIG_MAX (model.py:6-7,79)
        const float l1 = fminf(fmaxf(p0.w + p1.w + p2.w + p3.w + b3.w, -20.f), 2.f);
        const float x0 = fmaf(__expf(l0), e0, m0), x1 = fmaf(__expf(l1), e1, m1);
        reinterpret_cast<float2*>(a.action)[row] = make_float2(tanh_fast(x0), tanh_fast(x1));  // model.py:90-91
        if (a.head) reinterpret_cast<float4*>(a.head)[row] = make_float4(m0, m1, l0, l1);
      }
    }
  }

#ifdef UAVCA_POLICY_TIMING
  POL_TICK(5)
  if ((t == 0 || t == 32 || t == kEpiThreads) && blockIdx.x == 0 && a.head) {  // an epilogue warp on SMSP 0, one on SMSP 1, the MMA warp
    float* out = a.head + (t == 0 ? 0 : t == 32 ? 12 : 24);
    for (int i = 0; i < 10; ++i) out[i] = (float)tk[i];
    out[10] = (float)(clock64() - tstart);
    out[11] = (float)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
  }
#endif
  // ---- teardown
  cudaTriggerProgrammaticLaunchCompletion();
  fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  }
}

}  // namespace pol

cudaError_t launch_policy_act(const float* obs, long long M, const void* w1, const void* w2, const void* w2b, const void* w3,
                              const void* w3b, const float* noise, unsigned long long seed, unsigned long long counter,
                              const unsigned long long* counter_dev, float* action, float* head, cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  static std::atomic<bool> configured[64];  // per device; setting the attribute twice is harmless, the flag only skips the call
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  int sms = 0;
  e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  if (dev >= 0 && dev < 64 && !configured[dev].load(std::memory_order_acquire)) {
    e = cudaFuncSetAttribute(pol::policy_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pol::kSmemAlloc);
    if (e != cudaSuccess) return e;
    configured[dev].store(true, std::memory_order_release);
  }
  pol::Args a{};
  a.obs = obs;
  a.w1 = reinterpret_cast<const __half*>(w1); a.w2 = reinterpret_cast<const __half*>(w2);
  a.w2b = reinterpret_cast<const __half*>(w2b); a.w3 = reinterpret_cast<const __half*>(w3);
  a.w3b = reinterpret_cast<const __half*>(w3b);
  a.noise = noise; a.action = action; a.head = head; a.M = M;
  a.seed_lo = (unsigned)seed; a.seed_hi = (unsigned)(seed >> 32);
  a.ctr = counter; a.ctr_dev = counter_dev;
  const long long tiles = (M + pol::kRows - 1) / pol::kRows;
  const int grid = (int)(tiles < sms ? tiles : sms);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(pol::kThreads);
  cfg.dynamicSmemBytes = pol::kSmemAlloc;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, pol::policy_act_kernel, a);
  if (e != cudaSuccess) return e;
  return cudaGetLastError();
}

}  // namespace uavca

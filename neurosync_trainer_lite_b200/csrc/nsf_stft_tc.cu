// STFT power spectrum on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM,
// operands staged by TMA into 128B-swizzled shared memory).  Replaces the rFFT inside
// librosa.feature.mfcc (reference call site: utils/audio/extraction/extract_features_utils.py:19).
//
// Maths (DESIGN.md "STFT as four small GEMMs"): two exact symmetries of the DFT kernel turn the
// F-point real DFT of a windowed frame into, per fold chain (even bins / odd bins), one GEMM for
// the real parts and one for the imaginary parts, each [frames x K] . [K x bins/2], K = F/4 + 1.
// That is 4x fewer FLOPs than the plain [frames x F] . [F x 2 bins] DFT-as-GEMM.
//
// Precision: inputs are split x = hi + lo into two fp16 values after an exact power-of-two
// scaling (per frame for the signal, 2^14 for the DFT matrix), and three products
// hi*hi + hi*lo + lo*hi are accumulated in fp32 in TMEM.  That carries ~22 mantissa bits through
// the tensor cores (fp32-class accuracy) at 3x the fp16 rate cost; a single fp16/bf16/tf32 pass
// would be 1e-2..1e-1 off on the CMVN'd features (SURVEY.md section 7.3).
//
// Kernels
//   k_tc_fold_r, k_tc_fold : signal -> folded, scaled, split fp16 operands (HBM bound, elementwise);
//                            k_tc_fold_r keeps a frame in registers (kp <= 512), k_tc_fold serves longer frames
//   k_tc_stft_mel_pair,      persistent warp-specialised TMA -> tcgen05.mma -> TMEM -> |.|^2 -> mel -> dB, one body
//   k_tc_stft_mel            on CTA pairs (cta_group::2) and on single CTAs (short K)
//   k_tc_gemm              : TMA -> tcgen05.mma -> TMEM -> |.|^2 written to HBM (NSF_DEBUG_UNFUSED_MEL, and plans
//                            whose mel filters overlap more than pairwise)
#include <cuda_fp16.h>

#include <cmath>
#include <cstring>

#include <algorithm>

#include "nsf_device_utils.cuh"
#include "nsf_stft_tc.cuh"

namespace nsf {

namespace {

constexpr int BM = 128;      // frames per tile (UMMA M)
constexpr int BN = 128;      // bins per tile   (UMMA N); Re and Im tiles sit side by side in TMEM
constexpr int BK = 64;       // K per pipeline stage: 64 fp16 = one 128-byte swizzle row
constexpr int UK = 16;       // K per tcgen05.mma for 16-bit inputs
constexpr int kStages = 3;
constexpr int kTileBytes = BM * BK * 2;             // 16 KiB, A and B tiles have the same size
constexpr int kStageBytes = 4 * kTileBytes;         // A_hi, A_lo, B_hi, B_lo
constexpr int kTmemCols = 2 * BN;                   // Re | Im accumulators, fp32
constexpr int kThreads = 192;                       // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue (k_tc_gemm)
constexpr int kFusedThreads = 320;                  // fused kernels: warps 2-5 and 6-9 share the epilogue
constexpr size_t kSmemBytes = 1024 + static_cast<size_t>(kStages) * kStageBytes + 256;

// ---- PTX wrappers --------------------------------------------------------------------------
// CTA pairs (cta_group::2): two CTAs of one cluster (same TPC) execute ONE tcgen05.mma of M = 256: each
// supplies its own 128 rows of A and HALF of the N rows of B from its own shared memory, and receives its
// 128 accumulator rows in its own TMEM.  Only the leader (cluster rank 0) issues MMAs; both issue TMA loads
// whose completion bytes land on the LEADER's mbarrier (peer bit of the shared::cluster address cleared).
// The wrappers that depend on the CTA group take it as kCtas = 1 (one CTA) or 2 (a pair).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// kCtas = 2: arrives on the leader's (even CTA's) barrier at this offset
template <int kCtas>
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  if constexpr (kCtas == 1)
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
  else
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug traps (surfacing as a CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins) {
    if (spins > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// kCtas = 2: the bytes complete on the leader's barrier at this offset
template <int kCtas>
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int32_t x, int32_t y) {
  if constexpr (kCtas == 1)
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
  else
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask),
          "r"(x), "r"(y)
        : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
template <int kCtas>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t cols) {
  if constexpr (kCtas == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int kCtas>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  if constexpr (kCtas == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, 16-bit inputs, fp32 accumulation
template <int kCtas>
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  if constexpr (kCtas == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once every previously issued tcgen05.mma of this thread has completed; kCtas = 2: on the
// barrier at this offset in BOTH CTAs
template <int kCtas>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  if constexpr (kCtas == 1)
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  else
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 16 accumulator columns of this thread's TMEM lane, asynchronously: the registers are valid only after
// tmem_wait_ld() on the same arrays.  The wait lists the registers as read-write operands so that the
// compiler cannot schedule a use in front of it.
__device__ __forceinline__ void tmem_ld_32x16_async(uint32_t taddr, float (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
        "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld(float (&a)[16], float (&b)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3]), "+f"(a[4]), "+f"(a[5]), "+f"(a[6]), "+f"(a[7]),
                 "+f"(a[8]), "+f"(a[9]), "+f"(a[10]), "+f"(a[11]), "+f"(a[12]), "+f"(a[13]), "+f"(a[14]), "+f"(a[15]),
                 "+f"(b[0]), "+f"(b[1]), "+f"(b[2]), "+f"(b[3]), "+f"(b[4]), "+f"(b[5]), "+f"(b[6]), "+f"(b[7]),
                 "+f"(b[8]), "+f"(b[9]), "+f"(b[10]), "+f"(b[11]), "+f"(b[12]), "+f"(b[13]), "+f"(b[14]), "+f"(b[15])
               :
               : "memory");
}

// One lane of a fully converged warp (elect.sync).  The MMA warp runs its loops with all 32 lanes and
// issues through the elected one: inside an `if (lane == 0)` region the compiler cannot prove that a
// single thread is active and wraps every tcgen05 instruction in an ELECT / BRA.U.ANY retry loop, which
// made instruction issue - not operand delivery - the limit of the first version of these kernels.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// K-major, 128B-swizzled operand tile: rows are 128 bytes, 8-row groups are 1024 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);   // start address, 16-byte units
  d |= static_cast<uint64_t>(1) << 16;                       // leading byte offset (unused for SW128 K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;               // stride byte offset: 8 rows * 128 B
  d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                       // SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: fp16 x fp16 -> fp32, both operands K-major
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) {
  return (1u << 4)                                  // accumulator format: F32
         | (0u << 7) | (0u << 10)                   // A, B format: F16
         | (static_cast<uint32_t>(n >> 3) << 17)    // N / 8
         | (static_cast<uint32_t>(m >> 4) << 24);   // M / 16
}

// ------------------------------------------------------------------------------------------------
// k_tc_fold: one WARP per hop-frame (grid-stride), input double-buffered per warp with TMA bulk
// copies (cp.async.bulk + mbarrier): while the warp folds frame i, the raw samples of frame
// i + stride are already landing in its second buffer, so every warp keeps ~6 KB of HBM reads in
// flight at all times.  The warp windows the frame in place (periodic Hann; zero padding at clip
// edges is filled by the lanes), tracks max|u|, then forms the folded GEMM inputs in closed form
// (nsf_plan.cpp build_fold describes the same sums as tap tables; tests check them against an FFT):
//   even F, Nh = F/2, j = 0..Nh/2:   u0 = u[j], u1 = u[j+Nh], u2 = u[Nh-j], u3 = u[F-j]
//       even bins  Re: u0+u1+u2+u3   Im: u0+u1-u2-u3      odd bins  Re: u0-u1-u2+u3   Im: u0-u1+u2-u3
//       (j == 0 or 2j == Nh is its own mirror: u0+u1 resp. u0-u1 for both parts)
//   odd F, j = 0..(F-1)/2:           Re: u[j]+u[F-j]   Im: u[j]-u[F-j]   (j == 0: u[0])
// Every folded value is bounded by 4 max|u|, which fixes the exact power-of-two scale
// (max|u| * 2^e in [2^11, 2^12), so |v| < 2^14); the scaled value is split into fp16 hi / lo and
// stored as half2 pairs.  Operand layout: plane = (chain*2 + part)*2 + hl; element
// [plane][frame][k], k contiguous.
// ------------------------------------------------------------------------------------------------
constexpr int kFoldWarps = 8;

struct Folded { float v[4]; };  // [chain*2 + part]

__device__ __forceinline__ Folded fold_at(const float* __restrict__ u, int j, int F, int Nh, int K, bool even) {
  Folded o;
  if (j >= K) { o.v[0] = o.v[1] = o.v[2] = o.v[3] = 0.0f; return o; }
  if (even) {
    const float u0 = u[j], u1 = u[j + Nh];
    const float s = u0 + u1, d = u0 - u1;
    if (j == 0 || 2 * j == Nh) {
      o.v[0] = s; o.v[1] = s; o.v[2] = d; o.v[3] = d;
    } else {
      const float u2 = u[Nh - j], u3 = u[F - j];
      const float s2 = u2 + u3, d2 = u3 - u2;
      o.v[0] = s + s2; o.v[1] = s - s2; o.v[2] = d + d2; o.v[3] = d - d2;
    }
  } else {
    const float u0 = u[j];
    if (j == 0) { o.v[0] = u0; o.v[1] = u0; }
    else { const float u1 = u[F - j]; o.v[0] = u0 + u1; o.v[1] = u0 - u1; }
    o.v[2] = 0.0f; o.v[3] = 0.0f;
  }
  return o;
}

__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// Where hop-frame g lives: its clip, the index of its first sample relative to the clip (negative /
// beyond the end = zero padding) and whether a 16-byte aligned superset of it can be bulk-copied.
struct FrameRef {
  int clip;
  int64_t base, first, len;
  const float* aligned;   // 16-byte aligned start of the bulk copy (fast path only)
  uint32_t bytes;         // multiple of 16
  int skew;               // floats between `aligned` and the frame's first sample
  bool fast;
};

// Clip descriptor of the frame run a warp is walking: refreshed only when the run enters the next clip
// (the lookup is a chain of dependent loads).
struct ClipCache { int64_t f0 = 0, f_end = -1, base = 0, len = 0; int clip = 0; };

// One int32 per hop-frame travels from the fold kernel to the GEMM epilogues: the frame's power-of-two exponent
// (|e| <= 100) in the low byte and the index of its clip above it, so the epilogue that needs the clip for the
// per-clip dB maximum does not repeat the binary search (14 dependent loads per row for a 10 000-clip batch).
__device__ __forceinline__ int32_t pack_row_info(int clip, int e2) { return (clip << 8) | (e2 & 0xff); }
__device__ __forceinline__ int row_info_exp(int32_t v) { return (v << 24) >> 24; }
__device__ __forceinline__ int row_info_clip(int32_t v) { return v >> 8; }

__device__ __forceinline__ FrameRef locate_frame(const DeviceTables& t, const BatchView& b, const float* y, int64_t g,
                                                 ClipCache& cc) {
  FrameRef r;
  if (g < cc.f0 || g >= cc.f_end) {
    const int clip = find_segment(b.frame_off, b.n_clips, g);
    cc.f0 = __ldg(b.frame_off + clip);
    cc.f_end = __ldg(b.frame_off + clip + 1);
    cc.base = __ldg(b.clip_off + clip);
    cc.len = __ldg(b.clip_off + clip + 1) - cc.base;
    cc.clip = clip;
  }
  const int64_t tf = g - cc.f0;
  r.clip = cc.clip;
  r.base = cc.base;
  r.len = cc.len;
  r.first = tf * t.H - t.pad;
  const uintptr_t addr = reinterpret_cast<uintptr_t>(y + r.base + r.first);
  const uintptr_t lo = addr & ~static_cast<uintptr_t>(15);
  const uintptr_t hi = (addr + static_cast<uintptr_t>(t.F) * 4 + 15) & ~static_cast<uintptr_t>(15);
  r.aligned = reinterpret_cast<const float*>(lo);
  r.bytes = static_cast<uint32_t>(hi - lo);
  r.skew = static_cast<int>((addr - lo) >> 2);
  r.fast = r.first >= 0 && r.first + t.F <= r.len && lo >= reinterpret_cast<uintptr_t>(y) &&
           hi <= reinterpret_cast<uintptr_t>(y + b.total_samples);
  return r;
}
__device__ __forceinline__ FrameRef locate_frame(const DeviceTables& t, const BatchView& b, const float* y, int64_t g) {
  ClipCache cc;
  return locate_frame(t, b, y, g, cc);
}

__global__ void __launch_bounds__(kFoldWarps * 32) k_tc_fold(DeviceTables t, BatchView b, const float* __restrict__ y,
                                                             __half* __restrict__ planes, int64_t plane_rows,
                                                             int32_t* __restrict__ row_exp, int buf_floats) {
  extern __shared__ __align__(16) float s_fold[];   // [F (+pad)] window, then kFoldWarps x 2 x [buf_floats] frames
  __shared__ uint64_t s_bar[kFoldWarps][2];
  const int F = t.F, kp = t.kp[0], K = t.chains == 2 ? (F / 2) / 2 + 1 : (F + 1) / 2;
  const int Nh = F / 2;
  const bool even = t.chains == 2;
  const int n_cp = 2 * t.chains;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_win = s_fold;
  float* bufs = s_fold + ((F + 3) & ~3) + static_cast<size_t>(warp) * 2 * buf_floats;
  for (int n = threadIdx.x; n < F; n += blockDim.x) s_win[n] = __ldg(t.hann_per + n);
  if (lane == 0) {
    mbar_init(&s_bar[warp][0], 1);
    mbar_init(&s_bar[warp][1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kFoldWarps;
  int64_t g = static_cast<int64_t>(blockIdx.x) * kFoldWarps + warp;
  uint32_t phase_bits = 0u;   // bit s = parity the next wait on buffer s expects
  FrameRef cur;
  if (g < b.total_frames) {
    cur = locate_frame(t, b, y, g);
    if (cur.fast && lane == 0) {
      mbar_expect_tx(&s_bar[warp][0], cur.bytes);
      bulk_load(bufs, cur.aligned, cur.bytes, &s_bar[warp][0]);
    }
  }
  for (int it = 0; g < b.total_frames; g += stride, ++it) {
    const int slot = it & 1;
    // prefetch the next frame of this warp into the other buffer
    const int64_t gn = g + stride;
    FrameRef nxt;
    nxt.fast = false;
    if (gn < b.total_frames) {
      nxt = locate_frame(t, b, y, gn);
      if (nxt.fast && lane == 0) {
        // the other buffer was last touched by this warp's generic-proxy stores two frames ago
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&s_bar[warp][slot ^ 1], nxt.bytes);
        bulk_load(bufs + (slot ^ 1) * buf_floats, nxt.aligned, nxt.bytes, &s_bar[warp][slot ^ 1]);
      }
    }
    float* u = bufs + slot * buf_floats;
    float umax = 0.0f;
    if (cur.fast) {
      mbar_wait(&s_bar[warp][slot], (phase_bits >> slot) & 1u);
      phase_bits ^= 1u << slot;
      u += cur.skew;
#pragma unroll 4
      for (int n = lane; n < F; n += 32) {
        const float v = u[n] * s_win[n];
        u[n] = v;
        umax = fmaxf(umax, fabsf(v));
      }
    } else {
      const float* src = y + cur.base + cur.first;   // zero padding (librosa stft center=True, constant)
      for (int n = lane; n < F; n += 32) {
        const int64_t i = cur.first + n;
        const float v = (i >= 0 && i < cur.len) ? __ldg(src + n) * s_win[n] : 0.0f;
        u[n] = v;
        umax = fmaxf(umax, fabsf(v));
      }
    }
    umax = warp_max(umax);     // also orders the in-place stores before the cross-lane reads below
    __syncwarp();
    // scale = 2^e with umax * 2^e in [2^11, 2^12): exact, and |folded| <= 4 umax stays below 2^14
    int e2 = 0;
    if (umax > 0.0f && umax < INFINITY) {
      e2 = 12 - (static_cast<int>((__float_as_uint(umax) >> 23) & 0xff) - 126);   // umax = m * 2^ex, m in [0.5, 1)
      e2 = max(-100, min(100, e2));
    }
    const float scale = __uint_as_float(static_cast<uint32_t>(e2 + 127) << 23);
    if (lane == 0) row_exp[g] = pack_row_info(cur.clip, e2);
    // eight planes, one half2 store each: base pointer and plane stride hoisted, the (chain, part)
    // loop fully unrolled (planes of the absent chain of an odd F are simply skipped)
    __half2* dst0 = reinterpret_cast<__half2*>(planes + g * kp) + lane;
    const int64_t pstride = plane_rows * kp / 2;           // half2 elements between planes
    for (int j = 2 * lane; j < kp; j += 64, dst0 += 32) {
      const Folded a = fold_at(u, j, F, Nh, K, even), c = fold_at(u, j + 1, F, Nh, K, even);
#pragma unroll
      for (int cp = 0; cp < 4; ++cp) {
        if (cp < n_cp) {
          const float va = a.v[cp] * scale, vc = c.v[cp] * scale;
          const __half2 hi = __floats2half2_rn(va, vc);
          const float2 back = __half22float2(hi);
          dst0[(2 * cp) * pstride] = hi;
          dst0[(2 * cp + 1) * pstride] = __floats2half2_rn(va - back.x, vc - back.y);
        }
      }
    }
    __syncwarp();
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------
// k_tc_fold_r: register-resident variant of k_tc_fold for kp <= 64 * kIt (kIt <= 8), the product path
// for every supported rate up to F = 2044.  k_tc_fold spends most of its time in the shared-memory
// pipe (window pass in place, then the fold pass re-reads everything: ~420 wavefronts per frame);
// here the frame is read from shared memory ONCE: each lane windows and folds its 2 kIt columns
// straight into registers (the periodic Hann window satisfies w[F-j] = w[j] and w[Nh-j] = w[Nh+j], so
// one float2 table entry (w[j], w[j+Nh]) windows all four taps), the warp reduces max|folded| - which
// fixes the exact power-of-two scale directly (|v| 2^e in [2^13, 2^14)) - and the scaled values are
// split and stored.  ~210 wavefronts per frame, which leaves the kernel to the HBM pipe.
// ------------------------------------------------------------------------------------------------
template <int kIt>
__global__ void __launch_bounds__(kFoldWarps * 32) k_tc_fold_r(DeviceTables t, BatchView b, const float* __restrict__ y,
                                                               __half* __restrict__ planes, int64_t plane_rows,
                                                               int32_t* __restrict__ row_exp, int buf_floats, int wp_pairs) {
  extern __shared__ __align__(16) float s_fold[];   // [wp_pairs] float2 window pairs, then kFoldWarps x 2 x [buf_floats]
  __shared__ uint64_t s_bar[kFoldWarps][2];
  const int F = t.F, kp = t.kp[0], K = t.chains == 2 ? (F / 2) / 2 + 1 : (F + 1) / 2;
  const int Nh = F / 2;
  const bool even = t.chains == 2;
  const int n_cp = 2 * t.chains;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float2* s_wp = reinterpret_cast<float2*>(s_fold);
  float* bufs = s_fold + 2 * wp_pairs + static_cast<size_t>(warp) * 2 * buf_floats;
  for (int j = threadIdx.x; j < wp_pairs; j += blockDim.x) {
    float2 w = make_float2(0.0f, 0.0f);
    if (j < K) {
      w.x = __ldg(t.hann_per + j);
      w.y = even ? __ldg(t.hann_per + j + Nh) : 0.0f;
    }
    s_wp[j] = w;
  }
  if (lane == 0) {
    mbar_init(&s_bar[warp][0], 1);
    mbar_init(&s_bar[warp][1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  // Frame order.  Few long clips (C2: 60 x 3601 frames): warps interleave frame by frame, so that at any time
  // the whole grid writes one compact region of every operand plane (measured 0.334 ms against 0.375 ms for
  // per-warp runs).  Many short clips (C5: 10 000 x 241 frames): every warp walks a contiguous run, so the
  // clip descriptor - a chain of dependent loads - is looked up once per clip instead of once per frame
  // (1.20 ms against 1.74 ms).
  const int64_t n_warps = static_cast<int64_t>(gridDim.x) * kFoldWarps;
  const int64_t widx = static_cast<int64_t>(blockIdx.x) * kFoldWarps + warp;
  const bool runs = b.n_clips > 256;
  const int64_t chunk = (b.total_frames + n_warps - 1) / n_warps;
  const int64_t g_step = runs ? 1 : n_warps;
  int64_t g = runs ? widx * chunk : widx;
  const int64_t g_end = runs ? min(g + chunk, b.total_frames) : b.total_frames;
  uint32_t phase_bits = 0u;
  ClipCache cc;
  FrameRef cur;
  if (g < g_end) {
    cur = locate_frame(t, b, y, g, cc);
    if (cur.fast && lane == 0) {
      mbar_expect_tx(&s_bar[warp][0], cur.bytes);
      bulk_load(bufs, cur.aligned, cur.bytes, &s_bar[warp][0]);
    }
  }
  const int64_t pstride = plane_rows * kp / 2;           // half2 elements between planes
  for (int it = 0; g < g_end; g += g_step, ++it) {
    const int slot = it & 1;
    const int64_t gn = g + g_step;
    FrameRef nxt;
    nxt.fast = false;
    if (gn < g_end) {
      nxt = locate_frame(t, b, y, gn, cc);
      if (nxt.fast && lane == 0) {
        // the other buffer was last read by this warp's generic-proxy loads (and edge-frame stores)
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&s_bar[warp][slot ^ 1], nxt.bytes);
        bulk_load(bufs + (slot ^ 1) * buf_floats, nxt.aligned, nxt.bytes, &s_bar[warp][slot ^ 1]);
      }
    }
    const float* u = bufs + slot * buf_floats;
    if (cur.fast) {
      mbar_wait(&s_bar[warp][slot], (phase_bits >> slot) & 1u);
      phase_bits ^= 1u << slot;
      u += cur.skew;
    } else {
      // clip edges: raw samples with the zero padding of librosa's centred STFT, staged by the lanes
      float* ub = bufs + slot * buf_floats;
      const float* src = y + cur.base + cur.first;
      for (int n = lane; n < F; n += 32) {
        const int64_t i = cur.first + n;
        ub[n] = (i >= 0 && i < cur.len) ? __ldg(src + n) : 0.0f;
      }
      __syncwarp();
    }
    // pass 1: window + fold into registers, running max of |folded|
    float v[kIt][2][4];
    float vmax = 0.0f;
#pragma unroll
    for (int q = 0; q < kIt; ++q) {
      const int j0 = 2 * lane + 64 * q;
      const float4 w = j0 < wp_pairs ? *reinterpret_cast<const float4*>(s_wp + j0) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float wj[2][2] = {{w.x, w.y}, {w.z, w.w}};
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = j0 + h;
        float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f, o3 = 0.0f;
        if (j < K) {
          if (even) {
            const float u0 = u[j] * wj[h][0], u1 = u[j + Nh] * wj[h][1];
            const float s = u0 + u1, d = u0 - u1;
            if (j == 0 || 2 * j == Nh) {
              o0 = s; o1 = s; o2 = d; o3 = d;
            } else {
              const float u2 = u[Nh - j] * wj[h][1], u3 = u[F - j] * wj[h][0];
              const float s2 = u2 + u3, d2 = u3 - u2;
              o0 = s + s2; o1 = s - s2; o2 = d + d2; o3 = d - d2;
            }
          } else {
            const float u0 = u[j] * wj[h][0];
            if (j == 0) { o0 = u0; o1 = u0; }
            else { const float u1 = u[F - j] * wj[h][0]; o0 = u0 + u1; o1 = u0 - u1; }
          }
        }
        v[q][h][0] = o0; v[q][h][1] = o1; v[q][h][2] = o2; v[q][h][3] = o3;
        vmax = fmaxf(vmax, fmaxf(fmaxf(fabsf(o0), fabsf(o1)), fmaxf(fabsf(o2), fabsf(o3))));
      }
    }
    vmax = warp_max(vmax);
    // scale = 2^e with vmax * 2^e in [2^13, 2^14): exact
    int e2 = 0;
    if (vmax > 0.0f && vmax < INFINITY) {
      e2 = 14 - (static_cast<int>((__float_as_uint(vmax) >> 23) & 0xff) - 126);   // vmax = m * 2^ex, m in [0.5, 1)
      e2 = max(-100, min(100, e2));
    }
    const float scale = __uint_as_float(static_cast<uint32_t>(e2 + 127) << 23);
    if (lane == 0) row_exp[g] = pack_row_info(cur.clip, e2);
    // pass 2: scale, split, store (eight planes, one half2 store each)
    __half2* dst0 = reinterpret_cast<__half2*>(planes + g * kp) + lane;
#pragma unroll
    for (int q = 0; q < kIt; ++q) {
      if (2 * lane + 64 * q < kp) {
#pragma unroll
        for (int cp = 0; cp < 4; ++cp) {
          if (cp < n_cp) {
            const float va = v[q][0][cp] * scale, vc = v[q][1][cp] * scale;
            const __half2 hi = __floats2half2_rn(va, vc);
            const float2 back = __half22float2(hi);
            dst0[(2 * cp) * pstride + 32 * q] = hi;
            dst0[(2 * cp + 1) * pstride + 32 * q] = __floats2half2_rn(va - back.x, vc - back.y);
          }
        }
      }
    }
    __syncwarp();
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------
// k_tc_gemm: one CTA per (bin tile, chain, frame tile).
//   warp 0    : TMA producer (one lane)   - A_hi, A_lo, B_hi, B_lo tiles per stage
//   warp 1    : TMEM allocator + tcgen05.mma issuer (one lane)
//   warps 2-5 : epilogue - tcgen05.ld Re/Im, |.|^2, undo scaling, store
// Stage schedule: part 0 (real) over all K blocks into TMEM columns [0, BN), then part 1
// (imaginary) into [BN, 2 BN).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
k_tc_gemm(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
          int64_t total_frames, int64_t plane_rows, int n_tiles, int n_chains, int kp, int np_ld, int np0,
          int np1, int col_off1, int bins_ld, const int32_t* __restrict__ row_exp, float* __restrict__ power) {
  extern __shared__ uint8_t smem_raw[];
  // 128B swizzle needs 1024-byte aligned tiles
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* tiles = smem;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // blockIdx.x = (frame tile, chain, bin tile) with the bin tile fastest, so the CTAs that re-read
  // one frame tile's operands are co-scheduled and hit in L2
  const int n_tile = blockIdx.x % n_tiles;
  const int chain = (blockIdx.x / n_tiles) % n_chains;
  const int64_t g0 = static_cast<int64_t>(blockIdx.x / (n_tiles * n_chains)) * BM;
  const int np = chain == 0 ? np0 : np1;
  const int n0 = n_tile * BN;
  if (n0 >= np) return;  // uniform per CTA: this chain has fewer bin tiles
  const int kblocks = (kp + BK - 1) / BK;
  const int iters = 2 * kblocks;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
    for (int i = 0; i < kStages; ++i) { mbar_init(full_bar + i, 1); mbar_init(empty_bar + i, 1); }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<1>(tmem_slot, kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int it = 0; it < iters; ++it) {
        const int stage = it % kStages;
        const uint32_t phase = (it / kStages) & 1;
        mbar_wait(empty_bar + stage, phase ^ 1);
        const int part = it / kblocks, kb = it - part * kblocks;
        const int cp = chain * 2 + part;
        uint8_t* st = tiles + stage * kStageBytes;
        mbar_expect_tx(full_bar + stage, kStageBytes);
        const int kx = kb * BK;
        const int64_t a_row = static_cast<int64_t>(cp * 2) * plane_rows + g0;
        tma_load_2d<1>(st + 0 * kTileBytes, &map_a, full_bar + stage, kx, static_cast<int32_t>(a_row));
        tma_load_2d<1>(st + 1 * kTileBytes, &map_a, full_bar + stage, kx, static_cast<int32_t>(a_row + plane_rows));
        const int b_row = (cp * 2) * np_ld + n0;
        tma_load_2d<1>(st + 2 * kTileBytes, &map_b, full_bar + stage, kx, b_row);
        tma_load_2d<1>(st + 3 * kTileBytes, &map_b, full_bar + stage, kx, b_row + np_ld);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BM, BN);
      for (int it = 0; it < iters; ++it) {
        const int stage = it % kStages;
        const uint32_t phase = (it / kStages) & 1;
        mbar_wait(full_bar + stage, phase);
        tcgen05_fence_after();
        const int part = it / kblocks, kb = it - part * kblocks;
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(part * BN);
        const uint32_t st = smem_u32(tiles + stage * kStageBytes);
        const int ksteps = min(BK / UK, (kp - kb * BK + UK - 1) / UK);
        for (int k = 0; k < ksteps; ++k) {
          const uint32_t koff = static_cast<uint32_t>(k * UK * 2);  // bytes along K inside the swizzle row
          const uint64_t a_hi = make_smem_desc(st + 0 * kTileBytes + koff);
          const uint64_t a_lo = make_smem_desc(st + 1 * kTileBytes + koff);
          const uint64_t b_hi = make_smem_desc(st + 2 * kTileBytes + koff);
          const uint64_t b_lo = make_smem_desc(st + 3 * kTileBytes + koff);
          umma_f16<1>(d_tmem, a_hi, b_hi, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_f16<1>(d_tmem, a_hi, b_lo, idesc, 1u);
          umma_f16<1>(d_tmem, a_lo, b_hi, idesc, 1u);
        }
        umma_commit<1>(empty_bar + stage);          // smem slot reusable once these MMAs retire
      }
      umma_commit<1>(tmem_full_bar);                // accumulators complete
    }
  } else {
    const int quarter = warp & 3;                // TMEM lane quarter this warp may access
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
    const int64_t g = g0 + quarter * 32 + lane;
    const bool row_ok = g < total_frames;
    const float sc = row_ok ? ldexpf(1.0f, -(row_info_exp(__ldg(row_exp + g)) + kTcBScaleExp)) : 0.0f;
    const int col_base = (chain == 0 ? 0 : col_off1) + n0;
    float* out_row = power + (row_ok ? g : 0) * bins_ld + col_base;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
#pragma unroll 1
    for (int j = 0; j < BN; j += 32) {
      float re[32], im[32];
      tmem_ld_32x32(lane_addr + static_cast<uint32_t>(j), re);
      tmem_ld_32x32(lane_addr + static_cast<uint32_t>(BN + j), im);
      if (row_ok) {
#pragma unroll
        for (int q = 0; q < 32; q += 4) {
          if (n0 + j + q < np) {
            float4 o;
            float a, c;
            a = re[q + 0] * sc; c = im[q + 0] * sc; o.x = fmaf(a, a, c * c);
            a = re[q + 1] * sc; c = im[q + 1] * sc; o.y = fmaf(a, a, c * c);
            a = re[q + 2] * sc; c = im[q + 2] * sc; o.z = fmaf(a, a, c * c);
            a = re[q + 3] * sc; c = im[q + 3] * sc; o.w = fmaf(a, a, c * c);
            *reinterpret_cast<float4*>(out_row + j + q) = o;
          }
        }
      }
    }
    tcgen05_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc<1>(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// Epilogue of one 128-bin sub-tile, shared by the fused kernels.  The thread owns one frame row (one TMEM
// lane) and walks 64 of the 128 Re / Im accumulator columns in chunks of 16, the TMEM loads of chunk c+1 in
// flight while chunk c is consumed.  |X|^2 is formed from the RAW accumulators; the frame's power-of-two
// scale sc2 = 2^(-2 (row_exp + 14)) is applied when a filter pair is flushed (exact, so the result does
// not depend on where the scaling happens).  A bin lies under at most two adjacent triangular filters
// (m0, m0 + 1): running sums are kept for the current pair and added to the row of the mel tile in shared
// memory when m0 changes (rows beyond the batch are pointed at a scratch row by the caller, so the hot loop
// carries no validity test).  tab: the sub-tile's table entries {bits(m0), w[m0], w[m0+1], 0} (global,
// read-only path: the 16 warp-uniform loads of chunk c+1 are issued before the arithmetic of chunk c).
// ------------------------------------------------------------------------------------------------
// Two warps share every TMEM lane quarter, each taking 64 of the 128 columns.  Their filter ranges meet in
// one place: the pair (m0, m0 + 1) that is open when the lower half ends may also be the first or second
// pair of the upper half.  The upper-half warp (kUpper) therefore keeps its first two flushes in registers
// (dm / d0 / d1) and applies them after the hand-shake with its partner (apply_deferred), so every element of
// the mel tile still receives its contributions in a fixed order.
struct MelDeferred { int m[2]; float s0[2], s1[2]; int n; };

// The 16-column chunks run as a ROLLED loop (one chunk body in the instruction stream: a fully unrolled epilogue is
// ~2400 instructions per instantiation, ncu showed 19 % of the fused kernel's stall samples as instruction-fetch
// starvation; rolling it took C2 from 0.653 to 0.641 ms and C5 from 2.13 to 2.07 ms, round 2); the chunk in flight
// lands in a second register set that is copied over the working set after the wait (32 moves per chunk).
// c_begin, c_end: the 16-column chunks this warp walks.  The callers split the LIVE chunks of the sub-tile between the
// two warps (67 of 128 columns hold bins at F = 266: chunks 0-2 and 3-4 instead of four chunks each, of which the
// upper warp's were 61 / 64 padding).
template <bool kUpper>
__device__ __forceinline__ void mel_accumulate_half(uint32_t acc_addr, const float4* __restrict__ tab,
                                                    float* my_acc, float sc2, MelDeferred& def, int c_begin, int c_end) {
  int cur_m = -1;
  float s0 = 0.0f, s1 = 0.0f;
  def.n = 0;
  auto flush = [&]() {
    if (cur_m < 0) return;
    if (kUpper && def.n == 0) {                  // (static indices: the struct stays in registers)
      def.m[0] = cur_m; def.s0[0] = s0 * sc2; def.s1[0] = s1 * sc2; def.n = 1;
    } else if (kUpper && def.n == 1) {
      def.m[1] = cur_m; def.s0[1] = s0 * sc2; def.s1[1] = s1 * sc2; def.n = 2;
    } else {
      my_acc[cur_m] += s0 * sc2;
      my_acc[cur_m + 1] += s1 * sc2;
    }
  };
  if (c_begin >= c_end) return;
  float re[16], im[16], nre[16], nim[16];
  tmem_ld_32x16_async(acc_addr + 16 * c_begin, re);
  tmem_ld_32x16_async(acc_addr + BN + 16 * c_begin, im);
  tmem_wait_ld(re, im);
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    if (c + 1 < c_end) {
      tmem_ld_32x16_async(acc_addr + 16 * (c + 1), nre);
      tmem_ld_32x16_async(acc_addr + BN + 16 * (c + 1), nim);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float4 e[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) e[q] = __ldg(tab + 16 * c + 8 * h + q);     // warp-uniform addresses: broadcast
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int m0 = __float_as_int(e[q].x);
        const float pw = fmaf(re[8 * h + q], re[8 * h + q], im[8 * h + q] * im[8 * h + q]);
        if (m0 != cur_m) {                               // uniform branch
          flush();
          cur_m = m0; s0 = 0.0f; s1 = 0.0f;
        }
        s0 = fmaf(pw, e[q].y, s0);
        s1 = fmaf(pw, e[q].z, s1);
      }
    }
    if (c + 1 < c_end) {
      tmem_wait_ld(nre, nim);
#pragma unroll
      for (int q = 0; q < 16; ++q) { re[q] = nre[q]; im[q] = nim[q]; }
    }
  }
  flush();
}
__device__ __forceinline__ void apply_deferred(float* my_acc, const MelDeferred& def) {
#pragma unroll
  for (int i = 0; i < 2; ++i)
    if (i < def.n) { my_acc[def.m[i]] += def.s0[i]; my_acc[def.m[i] + 1] += def.s1[i]; }
}
// 64-thread named barrier of the two warps that share TMEM lane quarter `quarter` (ids 1..4; 0 is __syncthreads)
__device__ __forceinline__ void pair_sync(int quarter) {
  asm volatile("bar.sync %0, 64;" ::"r"(quarter + 1) : "memory");
}

// ------------------------------------------------------------------------------------------------
// k_tc_stft_mel / k_tc_stft_mel_pair: PERSISTENT fused kernel, looping over tiles of 128 hop-frames per CTA.
// For every tile it runs the (chain, 128-bin) sub-tiles back to back; TMEM holds two 256-column
// accumulator buffers (Re | Im), so the tensor pipe works on sub-tile s+1 while the epilogue warps
// drain sub-tile s.  The epilogue never writes the power spectrum: it squares, undoes the scaling and
// accumulates the triangular mel filters straight into a [128 frames][n_mels] fp32 tile in shared
// memory (each thread owns one frame row; a bin feeds at most two adjacent filters), and after the
// last sub-tile writes 10 log10(max(1e-10, mel)) plus the per-clip dB maximum.
//   warp 0 : TMA producer      warp 1 : TMEM alloc + tcgen05.mma issuer      warps 2-9 : epilogue
//   (two warps per TMEM lane quarter, 64 of the 128 accumulator columns each)
// One body, kCtas CTAs per MMA:
//   k_tc_stft_mel       kCtas = 1, two pipeline stages.  Used for short K (fewer than four K blocks), where the
//                       pair's longer hand-off is exposed.
//   k_tc_stft_mel_pair  kCtas = 2 (product path).  With one CTA the kernel is bound by operand delivery
//                       L2 -> shared memory (every CTA streams the whole DFT matrix for each 128 frames; it sustains
//                       ~80 % of the L2 throughput cap with the tensor pipe 40 % active).  A cluster of two CTAs works
//                       on 256 frames with tcgen05.mma.cta_group::2 (M = 256): each CTA still loads its own 128 frame
//                       rows of A but only HALF of every DFT-matrix tile (64 of the 128 bin rows), the tensor cores
//                       read the other half from the peer's shared memory.  Operand bytes per CTA and stage drop from
//                       64 KB to 48 KB, which also makes room for a third pipeline stage.
// Hand-off of a pair: full[s]       leader's barrier; the leader's producer posts the bytes of BOTH CTAs, both
//                                   CTAs' TMA loads complete on it (peer bit cleared)
//                     empty[s]      per CTA; tcgen05.commit multicast from the leader's MMA thread
//                     tmem_full[b]  per CTA; tcgen05.commit multicast
//                     tmem_empty[b] leader's barrier, 16 arrivals: the eight epilogue warps of both CTAs
// ------------------------------------------------------------------------------------------------
constexpr int kMelPitch = 129;                       // floats per frame row of the mel tile
// Finished dB rows of the mel tile -> global memory, one warp per 16 consecutive frame rows (`src` = the first of them in
// the tile, `g0` its frame index).  Four rows (sixteen loads) are in flight per warp: as one load -> store pair per
// iteration the loop was pure shared-memory latency, 17 % of the single-CTA kernel's stall samples on C5
// (ncu source page of capture r02m, round 2).
__device__ __forceinline__ void store_db_rows(const float* __restrict__ src, float* __restrict__ db, int64_t g0,
                                              int64_t total_frames, int n_mels, int lane) {
  const int64_t left = total_frames - g0;
  const int rows = left >= 16 ? 16 : (left > 0 ? static_cast<int>(left) : 0);
  float* dst = db + g0 * n_mels;
  int r = 0;
  if (n_mels == 128) {
    for (; r + 4 <= rows; r += 4) {
      float v[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) v[i][j] = src[(r + i) * kMelPitch + lane + 32 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[(r + i) * 128 + lane + 32 * j] = v[i][j];
    }
  }
  for (; r < rows; ++r)
    for (int m = lane; m < n_mels; m += 32) dst[static_cast<int64_t>(r) * n_mels + m] = src[r * kMelPitch + m];
}
// BM frame rows + one scratch row (sink for rows beyond the batch), rounded so the mbarriers that follow
// stay 8-byte aligned
constexpr size_t kMelTileBytes = (static_cast<size_t>(BM + 1) * kMelPitch * sizeof(float) + 15) / 16 * 16;
// Pipeline stages and operand bytes per stage of the fused kernels: A_hi, A_lo (BM frame rows each), B_hi, B_lo
// (BN / ctas bin rows each)
__host__ __device__ constexpr int fused_stages(int ctas) { return ctas == 1 ? 2 : 3; }
__host__ __device__ constexpr int fused_stage_bytes(int ctas) { return 2 * kTileBytes + 2 * (BN / ctas) * BK * 2; }
constexpr size_t fused_smem_bytes(int ctas) {
  return 1024 + static_cast<size_t>(fused_stages(ctas)) * fused_stage_bytes(ctas) + kMelTileBytes + 256;
}
constexpr size_t kFusedSmem = fused_smem_bytes(1);
constexpr size_t kPairSmem = fused_smem_bytes(2);

template <int kCtas>
__device__ __forceinline__ void stft_mel_body(const CUtensorMap& map_a, const CUtensorMap& map_b, const DeviceTables& t,
                                              const BatchView& b, int64_t plane_rows, int kp, int np_ld,
                                              const int32_t* __restrict__ row_exp, float* __restrict__ db,
                                              uint32_t* __restrict__ dbmax_key) {
  constexpr int kFStages = fused_stages(kCtas), kFStageBytes = fused_stage_bytes(kCtas);
  constexpr int kBRows = BN / kCtas;                 // bin rows of a B tile this CTA loads
  constexpr int kTileB = kBRows * BK * 2;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment (128-byte swizzle) by OFFSETTING the shared array, not by rounding a generic pointer:
  // the compiler then keeps the shared address space and emits LDS / STS for the mel tile
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* tiles = smem;
  float* mel_acc = reinterpret_cast<float*>(smem + kFStages * kFStageBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kFStages * kFStageBytes + kMelTileBytes);
  uint64_t* empty_bar = full_bar + kFStages;
  uint64_t* tmem_full = empty_bar + kFStages;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;           // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = kCtas == 1 ? 0u : cluster_ctarank();
  const int kblocks = (kp + BK - 1) / BK;
  const int ntile[2] = {(t.np[0] + BN - 1) / BN, t.chains > 1 ? (t.np[1] + BN - 1) / BN : 0};
  const int n_sub = ntile[0] + ntile[1];
  // A unit is the kCtas * BM frames of one cluster, rank r owns frames [r BM, (r + 1) BM) of it.  Each role's loop
  // derives its first unit from blockIdx.x in its own header: hoisted above the role branches, the 64-bit start lands
  // in vector registers and the MMA issuer's loop loses its uniform (UR / BRA.U) control flow.
  const int64_t n_units = (b.total_frames + kCtas * BM - 1) / (kCtas * BM);

  if (threadIdx.x == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
    for (int i = 0; i < kFStages; ++i) { mbar_init(full_bar + i, 1); mbar_init(empty_bar + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(tmem_full + i, 1); mbar_init(tmem_empty + i, 8 * kCtas); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kCtas>(tmem_slot, 512);
  for (int i = threadIdx.x; i < BM * kMelPitch; i += blockDim.x) mel_acc[i] = 0.0f;
  tcgen05_fence_before();
  __syncthreads();
  if constexpr (kCtas == 2) cluster_sync_all();     // the peer's barriers are initialised before any remote arrive
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int64_t unit = blockIdx.x / kCtas; unit < n_units; unit += gridDim.x / kCtas) {
        const int64_t g0 = unit * kCtas * BM + static_cast<int64_t>(rank) * BM;      // this CTA's 128 frames
        for (int sub = 0; sub < n_sub; ++sub) {
          const int chain = sub < ntile[0] ? 0 : 1;
          const int n0 = (chain == 0 ? sub : sub - ntile[0]) * BN + static_cast<int>(rank) * kBRows;
          for (int part = 0; part < 2; ++part) {
            const int cp = chain * 2 + part;
            const int64_t a_row = static_cast<int64_t>(cp * 2) * plane_rows + g0;
            const int b_row = (cp * 2) * np_ld + n0;
            for (int kb = 0; kb < kblocks; ++kb, ++it) {
              const int stage = it % kFStages;
              mbar_wait(empty_bar + stage, ((it / kFStages) & 1) ^ 1);
              uint8_t* st = tiles + stage * kFStageBytes;
              if (rank == 0) mbar_expect_tx(full_bar + stage, kCtas * kFStageBytes);  // the bytes of all kCtas CTAs
              const int kx = kb * BK;
              tma_load_2d<kCtas>(st, &map_a, full_bar + stage, kx, static_cast<int32_t>(a_row));
              tma_load_2d<kCtas>(st + kTileBytes, &map_a, full_bar + stage, kx, static_cast<int32_t>(a_row + plane_rows));
              tma_load_2d<kCtas>(st + 2 * kTileBytes, &map_b, full_bar + stage, kx, b_row);
              tma_load_2d<kCtas>(st + 2 * kTileBytes + kTileB, &map_b, full_bar + stage, kx, b_row + np_ld);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // The leader issues the MMAs of its cluster.  All 32 lanes walk the schedule (and wait on the barriers) together;
    // one elected lane issues.  Descriptors of a stage are formed once; a K step of 16 fp16 = 32 bytes is +2 in the
    // address field.
    if (rank == 0) {
      constexpr uint32_t idesc = make_idesc(kCtas * BM, BN);
      uint32_t it = 0, acc_it = 0;
      for (int64_t unit = blockIdx.x / kCtas; unit < n_units; unit += gridDim.x / kCtas) {
        for (int sub = 0; sub < n_sub; ++sub, ++acc_it) {
          const uint32_t buf = acc_it & 1u;
          mbar_wait(tmem_empty + buf, ((acc_it >> 1) & 1u) ^ 1u);     // the epilogues have drained this buffer
          tcgen05_fence_after();
          for (int part = 0; part < 2; ++part) {
            const uint32_t d_tmem = tmem_base + buf * 256u + static_cast<uint32_t>(part * BN);
            for (int kb = 0; kb < kblocks; ++kb, ++it) {
              const int stage = it % kFStages;
              mbar_wait(full_bar + stage, (it / kFStages) & 1);
              tcgen05_fence_after();
              if (elect_one()) {
                const uint32_t st = smem_u32(tiles + stage * kFStageBytes);
                const uint64_t a_hi = make_smem_desc(st), a_lo = make_smem_desc(st + kTileBytes);
                const uint64_t b_hi = make_smem_desc(st + 2 * kTileBytes), b_lo = make_smem_desc(st + 2 * kTileBytes + kTileB);
                const int ksteps = min(BK / UK, (kp - kb * BK + UK - 1) / UK);
#pragma unroll
                for (int k = 0; k < BK / UK; ++k) {
                  if (k < ksteps) {
                    const uint64_t ko = static_cast<uint64_t>(k * ((UK * 2) >> 4));
                    umma_f16<kCtas>(d_tmem, a_hi + ko, b_hi + ko, idesc, (kb | k) != 0 ? 1u : 0u);
                    umma_f16<kCtas>(d_tmem, a_hi + ko, b_lo + ko, idesc, 1u);
                    umma_f16<kCtas>(d_tmem, a_lo + ko, b_hi + ko, idesc, 1u);
                  }
                }
                umma_commit<kCtas>(empty_bar + stage);
                if (part == 1 && kb == kblocks - 1) umma_commit<kCtas>(tmem_full + buf);
              }
              __syncwarp();
            }
          }
        }
      }
    }
  } else {
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const bool upper = warp >= 6;                 // warps 2-5: columns 0-63 of a sub-tile, warps 6-9: 64-127
    const int row = quarter * 32 + lane;          // frame row of the tile owned by this thread (and its partner)
    float* my_acc = mel_acc + row * kMelPitch;
    float* scratch_row = mel_acc + BM * kMelPitch;   // sink for rows beyond the batch (never read)
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    uint32_t acc_it = 0;
    for (int64_t unit = blockIdx.x / kCtas; unit < n_units; unit += gridDim.x / kCtas) {
      const int64_t tile0 = unit * kCtas * BM + static_cast<int64_t>(rank) * BM;
      const int64_t g = tile0 + row;
      const bool row_ok = g < b.total_frames;
      const int32_t row_info = row_ok ? __ldg(row_exp + g) : 0;
      const float sc2 = row_ok ? ldexpf(1.0f, -2 * (row_info_exp(row_info) + kTcBScaleExp)) : 0.0f;
      float* acc_row = row_ok ? my_acc : scratch_row;
      for (int sub = 0; sub < n_sub; ++sub, ++acc_it) {
        const int chain = sub < ntile[0] ? 0 : 1;
        const int n0 = (chain == 0 ? sub : sub - ntile[0]) * BN;
        const float4* tab = t.mel_col[chain] + n0;
        const uint32_t buf = acc_it & 1u;
        mbar_wait(tmem_full + buf, (acc_it >> 1) & 1u);
        tcgen05_fence_after();
        MelDeferred def;
        const int live_chunks = (min(BN, t.np[chain] - n0) + 15) / 16, lower_chunks = (live_chunks + 1) / 2;
        if (upper) mel_accumulate_half<true>(lane_addr + buf * 256u, tab, acc_row, sc2, def, lower_chunks, live_chunks);
        else mel_accumulate_half<false>(lane_addr + buf * 256u, tab, acc_row, sc2, def, 0, lower_chunks);
        // all TMEM reads of this warp are complete (tcgen05.wait::ld inside the routine)
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive<kCtas>(tmem_empty + buf);
        pair_sync(quarter);                        // the lower half has flushed everything
        if (upper) apply_deferred(acc_row, def);
      }
      pair_sync(quarter);                          // deferred sums are in: the rows of this quarter are complete
      // tile finished: dB (each warp its 64 mels), per-clip maximum, coalesced store, reset of the rows
      const int m_lo = upper ? t.n_mels / 2 : 0, m_hi = upper ? t.n_mels : t.n_mels / 2;
      float vmax = -INFINITY;
      int m = m_lo;
      for (; m + 8 <= m_hi; m += 8) {               // eight independent load -> log -> store chains in flight
        float v8[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v8[i] = my_acc[m + i];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          v8[i] = 10.0f * log10f(fmaxf(1e-10f, v8[i]));
          vmax = fmaxf(vmax, v8[i]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) my_acc[m + i] = v8[i];
      }
      for (; m < m_hi; ++m) {
        const float v = 10.0f * log10f(fmaxf(1e-10f, my_acc[m]));
        my_acc[m] = v;
        vmax = fmaxf(vmax, v);
      }
      pair_sync(quarter);
      const int64_t gw = tile0 + quarter * 32;          // first frame of this quarter's 32 rows
      store_db_rows(mel_acc + (quarter * 32 + (upper ? 16 : 0)) * kMelPitch, db, gw + (upper ? 16 : 0), b.total_frames,
                    t.n_mels, lane);
      pair_sync(quarter);
      for (int m = upper ? kMelPitch / 2 : 0; m < (upper ? kMelPitch : kMelPitch / 2); ++m) my_acc[m] = 0.0f;
      // the clip index was written by the fold kernel
      warp_clip_max(dbmax_key, row_ok ? row_info_clip(row_info) : -1, float_key(vmax));
    }
    tcgen05_fence_before();
  }
  __syncthreads();
  if constexpr (kCtas == 2) cluster_sync_all();     // neither CTA leaves while the pair's MMAs may still read it
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc<kCtas>(tmem_base, 512);
  }
}

__global__ void __launch_bounds__(kFusedThreads, 1)
k_tc_stft_mel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
              DeviceTables t, BatchView b, int64_t plane_rows, int kp, int np_ld,
              const int32_t* __restrict__ row_exp, float* __restrict__ db, uint32_t* __restrict__ dbmax_key) {
  stft_mel_body<1>(map_a, map_b, t, b, plane_rows, kp, np_ld, row_exp, db, dbmax_key);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFusedThreads, 1)
k_tc_stft_mel_pair(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                   DeviceTables t, BatchView b, int64_t plane_rows, int kp, int np_ld,
                   const int32_t* __restrict__ row_exp, float* __restrict__ db, uint32_t* __restrict__ dbmax_key) {
  stft_mel_body<2>(map_a, map_b, t, b, plane_rows, kp, np_ld, row_exp, db, dbmax_key);
}

// ---- host side ----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// 2-D fp16 tensor [rows][cols] (cols contiguous), box = BK x box_rows, 128B swizzle, zero OOB fill
bool encode_map(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {cols * 2};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// whole CTA-pair tiles (256 frames): the peer CTA of the last pair then never reads into the next plane
inline int64_t plane_rows_for(int64_t frames) { return (frames + 2 * BM - 1) / (2 * BM) * (2 * BM); }

}  // namespace

void build_stft_tc_blob(const Plan& p, StftTcHostBlob* blob) {
  const int kp = p.chain[0].kp;
  int np_ld = 0;
  for (int c = 0; c < p.chains; ++c) np_ld = std::max(np_ld, p.chain[c].np);
  blob->kp = kp;
  blob->np_ld = np_ld;
  blob->planes = p.chains * 4;
  std::vector<__half> h(static_cast<size_t>(blob->planes) * np_ld * kp, __float2half(0.0f));
  const double scale = std::ldexp(1.0, kTcBScaleExp);
  for (int c = 0; c < p.chains; ++c) {
    const FoldChain& ch = p.chain[c];
    for (int part = 0; part < 2; ++part)
      for (int n = 0; n < ch.nbins; ++n)
        for (int k = 0; k < ch.k; ++k) {
          const double v = ch.mat[part][static_cast<size_t>(k) * ch.np + n] * scale;
          const __half hi = __float2half_rn(static_cast<float>(v));
          const __half lo = __float2half_rn(static_cast<float>(v - static_cast<double>(__half2float(hi))));
          const size_t plane = static_cast<size_t>((c * 2 + part) * 2);
          h[((plane + 0) * np_ld + n) * kp + k] = hi;
          h[((plane + 1) * np_ld + n) * kp + k] = lo;
        }
  }
  blob->bytes.resize(h.size() * sizeof(__half));
  std::memcpy(blob->bytes.data(), h.data(), blob->bytes.size());
}

nsf_status bind_stft_tc_tables(const Plan& p, const StftTcHostBlob& blob, const void* dev_ptr,
                               StftTcTables* out) {
  out->bt = dev_ptr;
  out->kp = blob.kp;
  out->np_ld = blob.np_ld;
  out->chains = p.chains;
  out->np[0] = p.chain[0].np;
  out->np[1] = p.chains > 1 ? p.chain[1].np : 0;
  out->col_off[0] = 0;
  out->col_off[1] = p.chain[0].np;
  if (!encode_map(&out->map_b, dev_ptr, static_cast<uint64_t>(blob.planes) * blob.np_ld, blob.kp, BN)) {
    set_error("cuTensorMapEncodeTiled failed for the DFT matrix");
    return NSF_ERR_CUDA;
  }
  if (!encode_map(&out->map_b_half, dev_ptr, static_cast<uint64_t>(blob.planes) * blob.np_ld, blob.kp, BN / 2)) {
    set_error("cuTensorMapEncodeTiled failed for the DFT matrix (half tiles)");
    return NSF_ERR_CUDA;
  }
  out->ready = true;
  return NSF_OK;
}

size_t stft_tc_operand_bytes(const Plan& p, int64_t frames) {
  const int64_t rows = plane_rows_for(frames);
  const size_t planes = static_cast<size_t>(p.chains) * 4;
  // fp16 planes, then one int32 exponent per frame; both 256-byte aligned
  return (planes * rows * p.chain[0].kp * 2 + 255) / 256 * 256 + (static_cast<size_t>(rows) * 4 + 255) / 256 * 256;
}

namespace {
struct OperandView { __half* planes; int32_t* row_exp; int64_t rows; };
OperandView view_operands(const StftTcTables& tc, int64_t frames, void* operands) {
  OperandView v;
  v.rows = plane_rows_for(frames);
  v.planes = static_cast<__half*>(operands);
  const size_t plane_bytes = (static_cast<size_t>(tc.chains) * 4 * v.rows * tc.kp * 2 + 255) / 256 * 256;
  v.row_exp = reinterpret_cast<int32_t*>(static_cast<char*>(operands) + plane_bytes);
  return v;
}
}  // namespace

int launch_stft_tc_fold(cudaStream_t s, const StftTcTables& tc, const DeviceTables& t, const BatchView& b,
                        const float* y, void* operands) {
  if (!tc.ready) return -1;
  const OperandView v = view_operands(tc, b.total_frames, operands);
  const int buf_floats = ((t.F + 3) & ~3) + 8;   // frame + up to 3 floats of skew + tail, 16-byte multiple
  const int kp = tc.kp;
  const int iters = (kp + 63) / 64;
  const bool reg_path = iters <= 8;              // longer frames take the two-pass kernel k_tc_fold
  const int wp_pairs = iters * 64;               // float2 window pairs, zero beyond K
  const size_t head = reg_path ? static_cast<size_t>(2) * wp_pairs : static_cast<size_t>((t.F + 3) & ~3);
  const size_t smem = (head + static_cast<size_t>(kFoldWarps) * 2 * buf_floats) * sizeof(float);
  if (smem > 220 * 1024) return -1;
  int per_sm = static_cast<int>((224 * 1024) / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > 6 ? 6 : per_sm);
  int64_t grid = (b.total_frames + kFoldWarps - 1) / kFoldWarps;
  if (grid > kSmCount * per_sm) grid = kSmCount * per_sm;
  if (grid < 1) grid = 1;
  auto go = [&](auto kernel) {
    kernel<<<static_cast<int>(grid), kFoldWarps * 32, smem, s>>>(t, b, y, v.planes, v.rows, v.row_exp, buf_floats, wp_pairs);
    NSF_CHECK_LAUNCH();
    return 1;
  };
  if (reg_path) {
    if (iters <= 2) return go(k_tc_fold_r<2>);       // F <= 508   (16 kHz: 266, 22.05 kHz: 367 odd -> kp 192: 3)
    if (iters <= 3) return go(k_tc_fold_r<3>);
    if (iters <= 4) return go(k_tc_fold_r<4>);       // 48 kHz: F = 800, kp = 208
    if (iters <= 6) return go(k_tc_fold_r<6>);       // 88.2 kHz: F = 1470, kp = 368; 44.1 kHz: F = 735 (odd), kp = 368
    return go(k_tc_fold_r<8>);
  }
  k_tc_fold<<<static_cast<int>(grid), kFoldWarps * 32, smem, s>>>(t, b, y, v.planes, v.rows, v.row_exp, buf_floats);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_stft_tc_mel(cudaStream_t s, const StftTcTables& tc, const DeviceTables& t, const BatchView& b,
                       void* operands, float* db, uint32_t* dbmax_key) {
  if (!tc.ready || !t.mel_col_ok || t.n_mels > 128) return -1;
  const OperandView v = view_operands(tc, b.total_frames, operands);
  CUtensorMap map_a;
  if (!encode_map(&map_a, v.planes, static_cast<uint64_t>(tc.chains) * 4 * v.rows, tc.kp, BM)) return -1;
  // short K (16 kHz: two 64-column stages per accumulator) leaves the pair's longer hand-off exposed:
  // measured 3.31 vs 3.06 ms on the C5 batch, so pairs are used from four K stages on
  const int kblocks = (tc.kp + BK - 1) / BK;
  if (kblocks >= 4) {
    int64_t pairs = v.rows / (2 * BM);
    if (pairs > kSmCount / 2) pairs = kSmCount / 2;
    if (pairs < 1) pairs = 1;
    k_tc_stft_mel_pair<<<static_cast<unsigned>(2 * pairs), kFusedThreads, kPairSmem, s>>>(
        map_a, tc.map_b_half, t, b, v.rows, tc.kp, tc.np_ld, v.row_exp, db, dbmax_key);
    NSF_CHECK_LAUNCH();
    return 1;
  }
  int64_t grid = v.rows / BM;
  if (grid > kSmCount) grid = kSmCount;
  if (grid < 1) grid = 1;
  k_tc_stft_mel<<<static_cast<unsigned>(grid), kFusedThreads, kFusedSmem, s>>>(map_a, tc.map_b, t, b, v.rows, tc.kp,
                                                                             tc.np_ld, v.row_exp, db, dbmax_key);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_stft_tc_gemm(cudaStream_t s, const StftTcTables& tc, const DeviceTables& t, const BatchView& b,
                        void* operands, float* power) {
  if (!tc.ready) return -1;
  const OperandView v = view_operands(tc, b.total_frames, operands);
  CUtensorMap map_a;
  if (!encode_map(&map_a, v.planes, static_cast<uint64_t>(tc.chains) * 4 * v.rows, tc.kp, BM)) return -1;
  const int np_max = std::max(tc.np[0], tc.np[1]);
  const int n_tiles = (np_max + BN - 1) / BN;
  const int64_t grid = (v.rows / BM) * n_tiles * tc.chains;
  if (grid <= 0 || grid > 0x7fffffffLL) return -1;
  k_tc_gemm<<<static_cast<unsigned>(grid), kThreads, kSmemBytes, s>>>(
      map_a, tc.map_b, b.total_frames, v.rows, n_tiles, tc.chains, tc.kp, tc.np_ld, tc.np[0], tc.np[1],
      tc.col_off[1], t.bins_ld, v.row_exp, power);
  NSF_CHECK_LAUNCH();
  return 1;
}

// Opt-in shared-memory limits, once per device (nsf_ctx_create, after cudaSetDevice).
bool init_stft_tc_attributes() {
  bool ok = true;
  auto set = [&](auto kernel, int bytes) {
    ok = ok && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess;
  };
  set(k_tc_fold_r<2>, 220 * 1024); set(k_tc_fold_r<3>, 220 * 1024); set(k_tc_fold_r<4>, 220 * 1024);
  set(k_tc_fold_r<6>, 220 * 1024); set(k_tc_fold_r<8>, 220 * 1024); set(k_tc_fold, 220 * 1024);
  set(k_tc_stft_mel_pair, static_cast<int>(kPairSmem));
  set(k_tc_stft_mel, static_cast<int>(kFusedSmem));
  set(k_tc_gemm, static_cast<int>(kSmemBytes));
  return ok;
}

}  // namespace nsf

// K4 on the tensor pipe: normalised autocorrelation lags of every hop-frame as Hankel-structured
// warp-level MMAs (mma.sync m16n8k16, fp16 split operands, fp32 accumulation).
// Reference: utils/audio/extraction/extract_features_utils.py:54-113 (np.pad reflect, per-frame mean
// removal, np.hanning, np.correlate lags 0..187, / lag 0, edge-frame fix) and :33-44 (pair mean).
//
// Why mma.sync and not tcgen05: the work per frame is a [188 lags x F] Toeplitz matrix-VECTOR
// product - every frame has its own matrix, so there is no operand shared between frames to make
// a large GEMM of.  The 16 x 8 x 16 warp MMA is small enough to be filled by ONE frame:
//     D[i][j] += sum_k A[i][k] B[k][j],  A[i][k] = X(n0 + k + 8 i),  B[k][j] = X(n0 + k - j)
// contributes X(s + lag) X(s) with lag = 8 i + j (0..127) and s = n0 + k - j, so summing over the
// K-blocks n0 = 0, 16, 32, ... yields r[lag] for 128 lags at once; a second accumulator fed with
// the B fragments of 4 blocks earlier (a register ring) covers lags 64..191.  Both operands are
// plain reads of the (zero-extended) frame X at shifted offsets, i.e. Hankel matrices that never
// exist in memory.  A tcgen05 tile (M >= 64, N >= 8) would waste > 60 % of its MACs on lags that
// are not needed.  Measured on B200 (scripts/ubench_mma.cu): mma.sync m16n8k16 f16 553 TFLOP/s vs
// 72 TFLOP/s for fp32 FFMA.
//
// Precision: X is the mean-removed, windowed frame scaled by an exact power of two and split into
// fp16 hi + lo; hi.hi + hi.lo + lo.hi carries ~22 mantissa bits (fp32 class).  The scale cancels in
// r[lag] / r[0].
//
// Kernels (all give bit-identical rows; launch_autocorr_mma picks one):
//   k_autocorr_pipe  88.2 kHz plan (F = 1470): eight warps per SM, two frame buffers per warp, the staging of the next
//                    frame woven into the compile-time unrolled five-tile MMA loop of the current one (am_mma5_pipe)
//   k_autocorr_sym   every other frame length: every warp stages, then multiplies, its own frames (am_mma5 /
//                    am_mma5_static<17> / am_mma); NSF_AC_KERNEL=sym forces it at F = 1470
#include <cuda_fp16.h>

#include <cstdint>
#include <cstdlib>
#include <type_traits>

#include "nsf.h"
#include "nsf_device_utils.cuh"
#include "nsf_kernels.cuh"

namespace nsf {

namespace {

constexpr int kFrontMargin = 16;   // halfs of zeros before X(0)  (B reads back to X(-7))
constexpr int kBackMargin = 160;   // halfs of zeros after the last K-block (the A prefetch of one block beyond reads up to +151)
constexpr int kVals = 6;           // lags per thread that can be <= 191
constexpr int kExtraFront = 112;   // halfs of zeros in front of every warp's copies: the five-tile loop (am_mma5)
                                   // reads A fragments of the blocks m = -8 .. -1, i.e. back to X(-128)

struct AmGeom { int nblk; int nblk4; int len; };   // K-blocks that hold samples, rounded up to a multiple of 4, halfs per copy
__host__ __device__ inline AmGeom am_geom(int F) {
  AmGeom g;
  g.nblk = (F + 15) / 16;
  g.nblk4 = (g.nblk + 3) / 4 * 4;
  g.len = kFrontMargin + 16 * g.nblk4 + kBackMargin;
  return g;
}

__device__ __forceinline__ void mma_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                          uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Lag held in slot v of lane (g, t):  base = 2 t + 8 g;  {base, base+1, base+64, base+65, base+128, base+129}
__device__ __forceinline__ int lag_of(int lane, int v) {
  const int base = 2 * (lane & 3) + 8 * (lane >> 2);
  return base + (v & 1) + 64 * (v >> 1);
}

// Where the samples of one hop-frame come from.  `fast` frames lie inside their clip AND at least
// 64 n_it samples before the end of the packed signal, so their 2 x 32 x n_it loads need no bounds
// checks (what is read beyond sample F is masked: the staged window table is zero there).  All other
// frames (the two clip-edge frames of np.pad(..., mode='reflect'), the very end of a batch) take the
// checked path.
struct AmSrc {
  const float* clip;      // y + first sample of the clip
  int64_t first, len;     // index of the frame's first sample relative to the clip, clip length
  bool fast, valid;
};
__device__ __forceinline__ AmSrc am_src(const DeviceTables& t, const BatchView& b, const float* __restrict__ y,
                                        int64_t base, int64_t len, int64_t tf, int n_it) {
  AmSrc s;
  s.clip = y + base;
  s.first = tf * t.H - t.pad;
  s.len = len;
  s.fast = s.first >= 0 && s.first + t.F <= len && base + s.first + 64 * n_it <= b.total_samples;
  s.valid = true;
  return s;
}
// Element pair e = lane + 32 i of the frame: samples 2 e, 2 e + 1.
// kExact: the kernel was instantiated for exactly n_it == kIters iterations, so the `i < n_it`
// guards vanish and the unrolled iterations can be interleaved freely by the compiler.
// kWide (pipelined kernel): frames that start on an 8-byte boundary - every other frame of a clip, the hop is odd - take
// one 64-bit load per pair, half the load instructions (C2: 1.032 -> 1.020 ms; in the symmetric kernel at 128 registers
// the second code path costs more than it saves: C5 2.67 -> 2.70 ms, so it keeps the scalar loads).
template <int kIters, bool kExact, bool kWide = false>
__device__ __forceinline__ void am_issue_fast(const float* __restrict__ src, int n_it, int lane, float (&v0)[kIters],
                                              float (&v1)[kIters]) {
  const float* p = src + 2 * lane;
  if (kWide && (reinterpret_cast<uintptr_t>(src) & 7u) == 0) {      // warp-uniform
#pragma unroll
    for (int i = 0; i < kIters; ++i) {
      if (kExact || i < n_it) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(p + 64 * i));
        v0[i] = v.x;
        v1[i] = v.y;
      }
    }
    return;
  }
#pragma unroll
  for (int i = 0; i < kIters; ++i) {
    if (kExact || i < n_it) {          // warp-uniform
      v0[i] = __ldg(p + 64 * i);
      v1[i] = __ldg(p + 64 * i + 1);
    }
  }
}
// Frame held in (v0, v1) -> the four fp16 copies.
// copies: [E_hi | E_lo | O_hi | O_lo], each geo.len halfs; E[kFrontMargin + m] = X(m),
// O[kFrontMargin + m - 1] = X(m) (the one-sample shifted copy keeps odd offsets 4-byte aligned).
// hann: np.hanning(F) staged in shared memory and ZERO from F up to 64 n_it, so elements beyond the
// frame come out as exact zeros without a branch (they land in the zero margin of the copies).
// Both passes over the frame (mean / max, then window + scale + split) run out of registers and the
// hot path has no divergent or data-dependent branches.
// When `next` is a fast frame every register pair is refilled with ITS samples as soon as the pair
// has been consumed, so the next memory round trip overlaps the rest of this frame.
template <int kIters, bool kExact>
__device__ __forceinline__ void am_process(const DeviceTables& t, const float* hann, int n_it, float (&v0)[kIters],
                                           float (&v1)[kIters], __half* copies, const AmGeom& geo, int lane,
                                           const float* __restrict__ next_fast) {
  const int F = t.F;
  // pass 1: mean and max |x| (bounds |x - mean| * w, which fixes the fp16 scale)
  float sum = 0.0f, amax = 0.0f;
#pragma unroll
  for (int i = 0; i < kIters; ++i) {
    if (kExact || i < n_it) {
      const int n = 2 * (lane + 32 * i);
      const float a = n < F ? v0[i] : 0.0f, c = n + 1 < F ? v1[i] : 0.0f;
      sum += a + c;
      amax = fmaxf(amax, fmaxf(fabsf(a), fabsf(c)));
    }
  }
  sum = warp_sum(sum);
  amax = warp_max(amax);
  const float mean = sum / static_cast<float>(F);
  const float bound = amax + fabsf(mean);
  int e2 = 0;
  if (bound > 0.0f && bound < INFINITY) {
    e2 = 14 - (static_cast<int>((__float_as_uint(bound) >> 23) & 0xff) - 126);   // bound * 2^e2 in [2^13, 2^14)
    e2 = max(-100, min(100, e2));
  }
  const float scale = __uint_as_float(static_cast<uint32_t>(e2 + 127) << 23);
  // pass 2: window, scale, split.  Pair e = (X(2e), X(2e+1)) goes to the E copies as one half2 each
  // and, as two 16-bit stores, to the one-sample shifted O copies (O half m - 1 = X(m)): no second pass
  // over shared memory and no warp barrier inside the frame.
  uint32_t* e_hi = reinterpret_cast<uint32_t*>(copies) + kFrontMargin / 2 + lane;
  uint32_t* e_lo = e_hi + geo.len / 2;
  uint16_t* o_hi = reinterpret_cast<uint16_t*>(copies) + 2 * geo.len + kFrontMargin - 1 + 2 * lane;
  uint16_t* o_lo = o_hi + geo.len;
  const float2* w2 = reinterpret_cast<const float2*>(hann) + lane;
  const float* nx = next_fast + 2 * lane;
  // groups of four iterations: the four window loads of a group are issued back to back, so their
  // shared-memory latency (long when the consumers keep the pipe busy) is paid once per group
  constexpr int kGroup = 4;
#pragma unroll
  for (int i0 = 0; i0 < kIters; i0 += kGroup) {
    float2 w[kGroup];
#pragma unroll
    for (int j = 0; j < kGroup; ++j)
      if (i0 + j < kIters && (kExact || i0 + j < n_it)) w[j] = w2[32 * (i0 + j)];
#pragma unroll
    for (int j = 0; j < kGroup; ++j) {
      const int i = i0 + j;
      if (i < kIters && (kExact || i < n_it)) {
        const float x0 = (v0[i] - mean) * (w[j].x * scale);
        const float x1 = (v1[i] - mean) * (w[j].y * scale);
        if (next_fast != nullptr) {        // warp-uniform
          v0[i] = __ldg(nx + 64 * i);
          v1[i] = __ldg(nx + 64 * i + 1);
        }
        const __half2 hi = __floats2half2_rn(x0, x1);
        const float2 hf = __half22float2(hi);
        const __half2 lo = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
        const uint32_t hw = *reinterpret_cast<const uint32_t*>(&hi), lw = *reinterpret_cast<const uint32_t*>(&lo);
        e_hi[32 * i] = hw;
        e_lo[32 * i] = lw;
        o_hi[64 * i] = static_cast<uint16_t>(hw);
        o_hi[64 * i + 1] = static_cast<uint16_t>(hw >> 16);
        o_lo[64 * i] = static_cast<uint16_t>(lw);
        o_lo[64 * i + 1] = static_cast<uint16_t>(lw >> 16);
      }
    }
  }
  __syncwarp();
}

// Any frame, start to finish, without register staging: three plain passes (mean / max, window +
// split, shifted copies).  Cold path - the two clip-edge frames with np.pad(..., mode='reflect')
// indexing, the tail of a batch, and the rare edge-fix refill - kept out of line so that it
// costs the hot paths neither registers nor instruction-cache space.
__device__ __noinline__ void am_fill_simple(const DeviceTables& t, const float* hann, const AmSrc& s, __half* copies,
                                            const AmGeom& geo, int lane) {
  const int F = t.F;
  auto sample = [&](int n) -> float {
    int64_t i = s.first + n;
    if (i < 0) i = -i;
    if (i >= s.len) i = 2 * (s.len - 1) - i;
    return __ldg(s.clip + i);
  };
  // same association order as am_process (per lane: pairs e = lane, lane + 32, ...), so a frame gives
  // bit-identical results whichever path stages it (batch == single-clip determinism)
  const int n_pairs = F / 2 + 1;               // one pair beyond the frame flushes the shifted copy
  float sum = 0.0f, amax = 0.0f;
  for (int e = lane; e < n_pairs; e += 32) {
    const float a = 2 * e < F ? sample(2 * e) : 0.0f, c = 2 * e + 1 < F ? sample(2 * e + 1) : 0.0f;
    sum += a + c;
    amax = fmaxf(amax, fmaxf(fabsf(a), fabsf(c)));
  }
  sum = warp_sum(sum);
  amax = warp_max(amax);
  const float mean = sum / static_cast<float>(F);
  const float bound = amax + fabsf(mean);
  int e2 = 0;
  if (bound > 0.0f && bound < INFINITY) {
    e2 = 14 - (static_cast<int>((__float_as_uint(bound) >> 23) & 0xff) - 126);
    e2 = max(-100, min(100, e2));
  }
  const float scale = __uint_as_float(static_cast<uint32_t>(e2 + 127) << 23);
  uint32_t* e_hi = reinterpret_cast<uint32_t*>(copies) + kFrontMargin / 2;
  uint32_t* e_lo = e_hi + geo.len / 2;
  uint32_t* o_hi = e_lo + geo.len / 2;
  uint32_t* o_lo = o_hi + geo.len / 2;
  for (int e = lane; e < n_pairs; e += 32) {
    float x0 = 0.0f, x1 = 0.0f;
    if (2 * e < F) x0 = (sample(2 * e) - mean) * (hann[2 * e] * scale);
    if (2 * e + 1 < F) x1 = (sample(2 * e + 1) - mean) * (hann[2 * e + 1] * scale);
    const __half2 hi = __floats2half2_rn(x0, x1);
    const float2 hf = __half22float2(hi);
    const __half2 lo = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
    e_hi[e] = *reinterpret_cast<const uint32_t*>(&hi);
    e_lo[e] = *reinterpret_cast<const uint32_t*>(&lo);
  }
  __syncwarp();
  for (int e = lane; e < n_pairs; e += 32) {
    o_hi[e - 1] = __funnelshift_r(e_hi[e - 1], e_hi[e], 16);
    o_lo[e - 1] = __funnelshift_r(e_lo[e - 1], e_lo[e], 16);
  }
  __syncwarp();
}

__device__ __forceinline__ uint32_t am_smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
// Four 8x8 fp16 matrices in MMA fragment layout with one instruction: lane L supplies the address of
// row L % 8 of matrix L / 8 (16 bytes each) and receives elements (row lane/4, columns 2 (lane%4), +1) of
// matrix i in r[i].
__device__ __forceinline__ void ldsm_x4(uint32_t saddr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(saddr));
}

// The MMA half: normalised lags of the frame currently held in `copies` into val[0..5] (see lag_of).
// Round 2 measured three re-formulations of this loop on B200 and kept none (DESIGN.md section 3.3, gpurun logs
// r2_ab / r2d / r2h): loading each half of the A fragment once - into a register ring (1.98 ms on C2: ~20 register
// moves per K-block to assemble the fragment quads) or with plain 32-bit loads into alternating quad positions (8
// instead of 12 shared-memory wavefronts per K-block, 1.30-1.38 ms: more load INSTRUCTIONS than two ldmatrix.x4) -
// and one accumulator per MMA of a K-block (six chains instead of four: 1.282 vs 1.285 ms).  This loop: 1.25-1.29 ms.
__device__ __forceinline__ void am_mma(const __half* copies, const AmGeom& geo, int lane, float (&val)[kVals]) {
  const int g = lane >> 2, tq = lane & 3;
  const uint32_t* E_hi = reinterpret_cast<const uint32_t*>(copies);
  const uint32_t* E_lo = E_hi + geo.len / 2;
  const uint32_t* O_hi = E_lo + geo.len / 2;
  const uint32_t* O_lo = O_hi + geo.len / 2;
  // A[i][k] = X(n0 + k + 8 i): the rows of the four 8x8 blocks of the fragment are 16-byte aligned runs of
  // the E copy (rows 8 samples apart; the row blocks 8..15 start 64 samples later, the k blocks 8..15 eight
  // samples later), so ONE ldmatrix.x4 per split part loads (a0, a1, a2, a3) into four consecutive registers -
  // no register ring between K-blocks and no fragment copies (12 instead of ~20 instructions per K-block).
  const int mi = lane >> 3, mr = lane & 7;
  const uint32_t a_off = 2u * static_cast<uint32_t>(kFrontMargin + 8 * mr + (mi & 1) * 64 + (mi >> 1) * 8);
  uint32_t sa_h = am_smem_u32(copies) + a_off;                    // advances 32 bytes per K-block
  const uint32_t lo_delta = 2u * static_cast<uint32_t>(geo.len);  // E_lo - E_hi in bytes
  // B: pair at X(n0 + 2 tq - g [+8]) -> parity of g picks the copy (O index = X index - 1)
  const int boff = kFrontMargin + 2 * tq - g - (g & 1);
  const uint32_t* Bh = ((g & 1) ? O_hi : E_hi) + boff / 2;
  const uint32_t* Bl = ((g & 1) ? O_lo : E_lo) + boff / 2;

  // accumulators: tile 0 = lags 8 i + j (0..127); tile 1 is fed with the B fragments of FOUR blocks
  // earlier (64 samples), i.e. lags 64 + 8 i + j - its rows 8..15 are lags 128..191.  The main
  // (hi.hi) and the two cross products go to separate accumulators: four independent MMA chains.
  float d0[4] = {0.0f, 0.0f, 0.0f, 0.0f}, d0x[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  float d1[4] = {0.0f, 0.0f, 0.0f, 0.0f}, d1x[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  // B fragments of the last 4 K-blocks: two register sets used alternately (a group of four blocks
  // loads into one set while tile 1 reads the other), so no fragment is ever copied
  uint32_t bp[4][4], bq[4][4];                // [slot][b0h, b1h, b0l, b1l]
#pragma unroll
  for (int q = 0; q < 4; ++q) { bq[q][0] = bq[q][1] = bq[q][2] = bq[q][3] = 0u; }
  // A fragments of the current block; the next block's are requested before this block's MMAs are issued
  uint32_t ah[4], al[4];
  ldsm_x4(sa_h, ah);
  ldsm_x4(sa_h + lo_delta, al);
  // one group = 4 K-blocks; `cur` receives this group's B fragments, `old` holds the previous group's
  // nq: blocks of the group that hold samples (4, or fewer in the frame's last group: blocks beyond the frame are
  // all-zero A fragments, e.g. 3 of the 20 blocks at F = 266, and contribute nothing to either tile)
  // first (a std::true_type for the frame's first group): `old` would be the four blocks BEFORE the frame - zero
  // fragments - so the three tile-1 MMAs of each of these blocks are not issued (12 of 102 MMAs at F = 266; adding
  // exact zeros to zero accumulators, so the rows are bit-identical)
  auto group = [&](const uint32_t* pb_h, const uint32_t* pb_l, uint32_t (&cur)[4][4], const uint32_t (&old)[4][4], int nq,
                   auto first) {
    constexpr bool kTile1 = !decltype(first)::value;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (q >= nq) break;
      uint32_t nh[4], nl[4];
      sa_h += 32u;
      ldsm_x4(sa_h, nh);                       // one block beyond the last one reads the zero margin
      ldsm_x4(sa_h + lo_delta, nl);
      cur[q][0] = pb_h[8 * q]; cur[q][1] = pb_h[8 * q + 4];
      cur[q][2] = pb_l[8 * q]; cur[q][3] = pb_l[8 * q + 4];
      // the two cross products of a tile are placed four MMAs apart (dependent accumulator)
      mma_16816(d0x, ah[0], ah[1], ah[2], ah[3], cur[q][2], cur[q][3]);
      if constexpr (kTile1) mma_16816(d1x, ah[0], ah[1], ah[2], ah[3], old[q][2], old[q][3]);
      mma_16816(d0, ah[0], ah[1], ah[2], ah[3], cur[q][0], cur[q][1]);
      if constexpr (kTile1) mma_16816(d1, ah[0], ah[1], ah[2], ah[3], old[q][0], old[q][1]);
      mma_16816(d0x, al[0], al[1], al[2], al[3], cur[q][0], cur[q][1]);
      if constexpr (kTile1) mma_16816(d1x, al[0], al[1], al[2], al[3], old[q][0], old[q][1]);
#pragma unroll
      for (int i = 0; i < 4; ++i) { ah[i] = nh[i]; al[i] = nl[i]; }
    }
  };
  const uint32_t *pb_h = Bh, *pb_l = Bl;
  int left = geo.nblk;
  {
    const int nq = left < 4 ? left : 4;
    group(pb_h, pb_l, bp, bq, nq, std::true_type{});
    left -= nq;
    pb_h += 32; pb_l += 32;
  }
#pragma unroll 1
  for (; left >= 8; left -= 8) {
    group(pb_h, pb_l, bq, bp, 4, std::false_type{});
    group(pb_h + 32, pb_l + 32, bp, bq, 4, std::false_type{});
    pb_h += 64; pb_l += 64;
  }
  if (left >= 4) {
    group(pb_h, pb_l, bq, bp, 4, std::false_type{});
    if (left > 4) group(pb_h + 32, pb_l + 32, bp, bq, left - 4, std::false_type{});
  } else if (left) {
    group(pb_h, pb_l, bq, bp, left, std::false_type{});
  }
  // tile 0: c0,c1 = lags base, base+1; c2,c3 = base+64, base+65.  tile 1: c2,c3 = base+128, base+129.
  val[0] = d0[0] + d0x[0]; val[1] = d0[1] + d0x[1]; val[2] = d0[2] + d0x[2]; val[3] = d0[3] + d0x[3];
  val[4] = d1[2] + d1x[2]; val[5] = d1[3] + d1x[3];
  const float r0 = __shfl_sync(0xffffffffu, val[0], 0);  // lag 0 lives in lane 0
  if (r0 != 0.0f) {
    const float inv = __fdiv_rn(1.0f, r0);
#pragma unroll
    for (int v = 0; v < kVals; ++v) val[v] *= inv;
  }
  __syncwarp();
}

// Final step of the five-tile loops: the three cross-correlation tiles folded onto lags 0 .. 191, r[lag] / r[0].
__device__ __forceinline__ void am_mma5_finish(const float (&hh0)[4], const float (&hh1)[4], const float (&cA)[4],
                                               const float (&cB)[4], const float (&cC)[4], int lane, float (&val)[kVals]) {
  // Lane (g, tq) holds rows g (c0, c1) and g + 8 (c2, c3), columns 2 tq, 2 tq + 1 of every tile.  With u = 8 g + 2 tq + e:
  //   hh0: u, 64 + u    hh1: (64 + u), 128 + u    cA: -64 + u, u    cB: 64 + u, 128 + u    cC: -192 + u, -128 + u
  // C[-(64 k + u)] = entry 64 - u of the tile that starts at -64 (k + 1): for odd u that is lane 31 - L (same e), for
  // even u lane 32 - L - and for L = 0 (u = 0) the first entry of the NEXT tile, which lane 0 holds itself.
  const int src_e = (32 - lane) & 31, src_o = 31 - lane;
  float n0e = __shfl_sync(0xffffffffu, cA[0], src_e), n0o = __shfl_sync(0xffffffffu, cA[1], src_o);
  float n1e = __shfl_sync(0xffffffffu, cC[2], src_e), n1o = __shfl_sync(0xffffffffu, cC[3], src_o);
  float n2e = __shfl_sync(0xffffffffu, cC[0], src_e), n2o = __shfl_sync(0xffffffffu, cC[1], src_o);
  if (lane == 0) { n0e = cA[2]; n1e = cA[0]; n2e = cC[2]; }
  val[0] = hh0[0] + (cA[2] + n0e); val[1] = hh0[1] + (cA[3] + n0o);
  val[2] = hh0[2] + (cB[0] + n1e); val[3] = hh0[3] + (cB[1] + n1o);
  val[4] = hh1[2] + (cB[2] + n2e); val[5] = hh1[3] + (cB[3] + n2o);
  const float r0 = __shfl_sync(0xffffffffu, val[0], 0);  // lag 0 lives in lane 0
  if (r0 != 0.0f) {
    const float inv = __fdiv_rn(1.0f, r0);
#pragma unroll
    for (int v = 0; v < kVals; ++v) val[v] *= inv;
  }
  __syncwarp();
}

// Five MMAs per K-block instead of six (round 2, the product loop).  With x = h + l (fp16 each)
//     r[lag] = HH[lag] + C[lag] + C[-lag],   HH[lag] = sum_s h(s + lag) h(s),   C[lag] = sum_s h(s + lag) l(s),
// because sum_s l(s + lag) h(s) = C[-lag]: the two cross products are ONE cross-correlation seen at both signs of the
// lag.  am_mma computes them as two products of two tiles each (A_h x B_l and A_l x B_h: 4 MMAs for 2 x 256 lag slots
// of which 2 x 188 are used); here C[-192 .. 191] comes from THREE tiles that all take the A_h fragment of the block:
//     tile (A_h(m), B_p(m'))  ->  lags 16 (m - m') + 8 i + j
//     cC: B_l(m + 12) -> [-192, -65]     cA: B_l(m + 4) -> [-64, 63]     cB: B_l(m - 4) -> [64, 191]
// (383 of 384 slots used) next to hh0: B_h(m) -> [0, 127] and hh1: B_h(m - 4) -> [64, 191] as before.  The A_l
// fragment is never loaded: one ldmatrix.x4 and four 32-bit loads per five MMAs (8 shared-memory wavefronts per block
// instead of 12).  The B_l fragments live in a ring of sixteen blocks (loaded twelve blocks ahead of their A block,
// last used four blocks behind it), the B_h fragments in a ring of eight; both rings are indexed by compile-time
// constants inside a body unrolled sixteen times, so nothing is ever copied.  Blocks m = -8 .. -1 (A rows that start
// before the frame but end inside it) only feed cC and cA and read zeros from kExtraFront; the tiles whose B block lies
// beyond the frame are skipped at the far end, so a frame costs 5 nblk - 12 MMAs.
__device__ __forceinline__ void am_mma5(const __half* copies, const AmGeom& geo, int lane, float (&val)[kVals]) {
  const int g = lane >> 2, tq = lane & 3;
  const uint32_t* E_hi = reinterpret_cast<const uint32_t*>(copies);
  const uint32_t* E_lo = E_hi + geo.len / 2;
  const uint32_t* O_hi = E_lo + geo.len / 2;
  const uint32_t* O_lo = O_hi + geo.len / 2;
  const int mi = lane >> 3, mr = lane & 7;
  const uint32_t a_off = 2u * static_cast<uint32_t>(kFrontMargin + 8 * mr + (mi & 1) * 64 + (mi >> 1) * 8);
  const uint32_t sa0 = am_smem_u32(copies) + a_off;               // A_h(0); block m is 32 m bytes further
  const int boff = kFrontMargin + 2 * tq - g - (g & 1);
  const uint32_t* Bh = ((g & 1) ? O_hi : E_hi) + boff / 2;        // block m': words 8 m' (k = 2 tq, +1) and 8 m' + 4 (k + 8)
  const uint32_t* Bl = ((g & 1) ? O_lo : E_lo) + boff / 2;
  const int nblk = geo.nblk;

  float hh0[4] = {0.0f, 0.0f, 0.0f, 0.0f}, hh1[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  float cA[4] = {0.0f, 0.0f, 0.0f, 0.0f}, cB[4] = {0.0f, 0.0f, 0.0f, 0.0f}, cC[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  uint32_t bh[8][2], bl[16][2];                 // slot = block index mod 8 / mod 16
#pragma unroll
  for (int q = 4; q < 8; ++q) bh[q][0] = bh[q][1] = 0u;          // B_h(-4 .. -1): zeros
#pragma unroll
  for (int q = 12; q < 16; ++q) bl[q][0] = bl[q][1] = 0u;        // B_l(-4 .. -1): zeros
#pragma unroll
  for (int q = 0; q < 4; ++q) { bl[q][0] = Bl[8 * q]; bl[q][1] = Bl[8 * q + 4]; }   // B_l(0 .. 3) (zero margin beyond the frame)
#pragma unroll
  for (int q = 0; q < 4; ++q) bh[q][0] = bh[q][1] = 0u;          // overwritten before use; keeps the compiler quiet
#pragma unroll
  for (int q = 4; q < 12; ++q) bl[q][0] = bl[q][1] = 0u;

  uint32_t a[4], an[4];
  // lead-in: m = -8 .. -1
  ldsm_x4(sa0 - 32u * 8u, a);
#pragma unroll
  for (int q = 8; q < 16; ++q) {
    const int m = q - 16;
    ldsm_x4(sa0 + static_cast<uint32_t>(32 * (m + 1)), an);      // m = -1 prefetches A_h(0)
    if (m + 12 < nblk) {
      bl[(q + 12) & 15][0] = Bl[8 * (m + 12)];
      bl[(q + 12) & 15][1] = Bl[8 * (m + 12) + 4];
    }
    if (m >= -4 && m + 4 < nblk) mma_16816(cA, a[0], a[1], a[2], a[3], bl[(q + 4) & 15][0], bl[(q + 4) & 15][1]);
    if (m + 12 < nblk) mma_16816(cC, a[0], a[1], a[2], a[3], bl[(q + 12) & 15][0], bl[(q + 12) & 15][1]);
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = an[i];
  }
  // main loop: groups of sixteen blocks; `fast` groups need no range checks
  uint32_t sa = sa0;                                              // address of A_h(m0)
#pragma unroll 1
  for (int m0 = 0; m0 < nblk; m0 += 16, sa += 32u * 16u) {
    const uint32_t* pbh = Bh + 8 * m0;
    const uint32_t* pbl = Bl + 8 * m0;
    if (m0 + 27 < nblk) {
#pragma unroll
      for (int q = 0; q < 16; ++q) {
        ldsm_x4(sa + static_cast<uint32_t>(32 * (q + 1)), an);
        bh[q & 7][0] = pbh[8 * q]; bh[q & 7][1] = pbh[8 * q + 4];
        mma_16816(cB, a[0], a[1], a[2], a[3], bl[(q + 12) & 15][0], bl[(q + 12) & 15][1]);   // B_l(m - 4)
        bl[(q + 12) & 15][0] = pbl[8 * (q + 12)]; bl[(q + 12) & 15][1] = pbl[8 * (q + 12) + 4];   // <- B_l(m + 12)
        mma_16816(hh1, a[0], a[1], a[2], a[3], bh[(q + 4) & 7][0], bh[(q + 4) & 7][1]);      // B_h(m - 4)
        mma_16816(cA, a[0], a[1], a[2], a[3], bl[(q + 4) & 15][0], bl[(q + 4) & 15][1]);     // B_l(m + 4)
        mma_16816(hh0, a[0], a[1], a[2], a[3], bh[q & 7][0], bh[q & 7][1]);                  // B_h(m)
        mma_16816(cC, a[0], a[1], a[2], a[3], bl[(q + 12) & 15][0], bl[(q + 12) & 15][1]);   // B_l(m + 12)
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = an[i];
      }
    } else {
#pragma unroll
      for (int q = 0; q < 16; ++q) {
        const int m = m0 + q;
        if (m >= nblk) break;
        ldsm_x4(sa + static_cast<uint32_t>(32 * (q + 1)), an);    // one block beyond the last reads the zero margin
        bh[q & 7][0] = pbh[8 * q]; bh[q & 7][1] = pbh[8 * q + 4];
        mma_16816(cB, a[0], a[1], a[2], a[3], bl[(q + 12) & 15][0], bl[(q + 12) & 15][1]);
        if (m + 12 < nblk) { bl[(q + 12) & 15][0] = pbl[8 * (q + 12)]; bl[(q + 12) & 15][1] = pbl[8 * (q + 12) + 4]; }
        mma_16816(hh1, a[0], a[1], a[2], a[3], bh[(q + 4) & 7][0], bh[(q + 4) & 7][1]);
        if (m + 4 < nblk) mma_16816(cA, a[0], a[1], a[2], a[3], bl[(q + 4) & 15][0], bl[(q + 4) & 15][1]);
        mma_16816(hh0, a[0], a[1], a[2], a[3], bh[q & 7][0], bh[q & 7][1]);
        if (m + 12 < nblk) mma_16816(cC, a[0], a[1], a[2], a[3], bl[(q + 12) & 15][0], bl[(q + 12) & 15][1]);
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = an[i];
      }
    }
  }
  am_mma5_finish(hh0, hh1, cA, cB, cC, lane, val);
}

// am_mma5 with the number of K-blocks known at compile time (F = 266: seventeen), unrolled completely: every range check
// of the lead-in and of the far end resolves at compile time, the rings are indexed by constants, and the tiles whose B
// block lies before the frame (cB, hh1 for m < 4: zero fragments) are not issued either - 5 NBLK - 12 MMAs and one
// ldmatrix.x4 + at most four 32-bit loads per block, no loop control.  Same products into the same accumulators in the
// same order as am_mma5 (the skipped MMAs add exact zeros), so the rows are identical.  Used where the generic loop's
// lead-in and checks cost more than the MMAs it saves over the six-MMA loop (short frames; launch_autocorr_mma).
template <int NBLK>
__device__ __forceinline__ void am_mma5_static(const __half* copies, const AmGeom& geo, int lane, float (&val)[kVals]) {
  static_assert(NBLK >= 13 && NBLK <= 24, "unrolled loop: short frames only");
  const int g = lane >> 2, tq = lane & 3;
  const uint32_t* E_hi = reinterpret_cast<const uint32_t*>(copies);
  const uint32_t* E_lo = E_hi + geo.len / 2;
  const uint32_t* O_hi = E_lo + geo.len / 2;
  const uint32_t* O_lo = O_hi + geo.len / 2;
  const int mi = lane >> 3, mr = lane & 7;
  const uint32_t a_off = 2u * static_cast<uint32_t>(kFrontMargin + 8 * mr + (mi & 1) * 64 + (mi >> 1) * 8);
  const uint32_t sa0 = am_smem_u32(copies) + a_off;
  const int boff = kFrontMargin + 2 * tq - g - (g & 1);
  const uint32_t* Bh = ((g & 1) ? O_hi : E_hi) + boff / 2;
  const uint32_t* Bl = ((g & 1) ? O_lo : E_lo) + boff / 2;
  float hh0[4] = {0.0f, 0.0f, 0.0f, 0.0f}, hh1[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  float cA[4] = {0.0f, 0.0f, 0.0f, 0.0f}, cB[4] = {0.0f, 0.0f, 0.0f, 0.0f}, cC[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  uint32_t bh[8][2], bl[16][2];                 // slot = block index mod 8 / mod 16
#pragma unroll
  for (int q = 0; q < 8; ++q) bh[q][0] = bh[q][1] = 0u;
#pragma unroll
  for (int q = 0; q < 16; ++q) bl[q][0] = bl[q][1] = 0u;
#pragma unroll
  for (int q = 0; q < 4; ++q) { bl[q][0] = Bl[8 * q]; bl[q][1] = Bl[8 * q + 4]; }   // B_l(0 .. 3)
  uint32_t a[4], an[4];
  ldsm_x4(sa0 - 32u * 8u, a);
#pragma unroll
  for (int m = -8; m < NBLK; ++m) {
    ldsm_x4(sa0 + static_cast<uint32_t>(32 * (m + 1)), an);      // the block beyond the last reads the zero margin
    if (m >= 0) { bh[m & 7][0] = Bh[8 * m]; bh[m & 7][1] = Bh[8 * m + 4]; }
    if (m >= 4) mma_16816(cB, a[0], a[1], a[2], a[3], bl[(m - 4) & 15][0], bl[(m - 4) & 15][1]);            // B_l(m - 4)
    if (m + 12 < NBLK) { bl[(m + 12) & 15][0] = Bl[8 * (m + 12)]; bl[(m + 12) & 15][1] = Bl[8 * (m + 12) + 4]; }
    if (m >= 4) mma_16816(hh1, a[0], a[1], a[2], a[3], bh[(m - 4) & 7][0], bh[(m - 4) & 7][1]);             // B_h(m - 4)
    if (m >= -4 && m + 4 < NBLK) mma_16816(cA, a[0], a[1], a[2], a[3], bl[(m + 4) & 15][0], bl[(m + 4) & 15][1]);
    if (m >= 0) mma_16816(hh0, a[0], a[1], a[2], a[3], bh[m & 7][0], bh[m & 7][1]);                         // B_h(m)
    if (m + 12 < NBLK) mma_16816(cC, a[0], a[1], a[2], a[3], bl[(m + 12) & 15][0], bl[(m + 12) & 15][1]);   // B_l(m + 12)
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = an[i];
  }
  am_mma5_finish(hh0, hh1, cA, cB, cC, lane, val);
}

// ------------------------------------------------------------------------------------------------
// Software-pipelined frame (round 2, k_autocorr_pipe): the five-tile loop of the frame held in `copies`, unrolled at
// compile time like am_mma5_static, with the STAGING of the warp's next frame woven into it.  The next frame's raw
// samples are already in flight into (v0, v1) when the loop starts (am_issue_fast); pass 1 (mean, max |x|, scale) runs
// after block kPass1, one pass-2 iteration (window, scale, split, six shared stores into `next_copies`) every
// kStride blocks from block kPass2 on.  ptxas schedules the two independent instruction streams into one another, so
// a warp never leaves the MMA loop: the phase trace of the symmetric kernel (scripts/ac_trace.py, B200) showed a warp
// spending 5.3 k of its 21.5 k cycles per frame staging, the tensor pipe 66 % active although the loop alone sustains
// 88 % (scripts/ubench_ac5.cu).  Same staging arithmetic as am_process and the same MMAs into the same accumulators
// in the same order as am_mma5 / am_mma5_static: the rows are bit-identical to the symmetric kernel's.
// kIters must be the exact iteration count of the frame length (n_it == kIters), which also makes the `n < F` guards
// of pass 1 compile-time true for every iteration but the last.
template <int NBLK, int kIters>
__device__ __forceinline__ void am_mma5_pipe(const __half* copies, const AmGeom& geo, int lane, float (&val)[kVals],
                                             const DeviceTables& t, const float* hann, float (&v0)[kIters],
                                             float (&v1)[kIters], __half* next_copies) {
  constexpr int kPass1 = NBLK >= 40 ? 12 : 5;           // block after which the loads are consumed
  constexpr int kPass2 = kPass1 + 2;                    // block of the first pass-2 iteration
  constexpr int kStride = (NBLK - 2 - kPass2) / kIters > 0 ? (NBLK - 2 - kPass2) / kIters : 1;
  static_assert(kPass2 + kStride * (kIters - 1) < NBLK, "every staging iteration must fall inside the loop");
  const int g = lane >> 2, tq = lane & 3;
  const uint32_t* E_hi = reinterpret_cast<const uint32_t*>(copies);
  const uint32_t* E_lo = E_hi + geo.len / 2;
  const uint32_t* O_hi = E_lo + geo.len / 2;
  const uint32_t* O_lo = O_hi + geo.len / 2;
  const int mi = lane >> 3, mr = lane & 7;
  const uint32_t a_off = 2u * static_cast<uint32_t>(kFrontMargin + 8 * mr + (mi & 1) * 64 + (mi >> 1) * 8);
  const uint32_t sa0 = am_smem_u32(copies) + a_off;
  const int boff = kFrontMargin + 2 * tq - g - (g & 1);
  const uint32_t* Bh = ((g & 1) ? O_hi : E_hi) + boff / 2;
  const uint32_t* Bl = ((g & 1) ? O_lo : E_lo) + boff / 2;
  float hh0[4] = {0.0f, 0.0f, 0.0f, 0.0f}, hh1[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  float cA[4] = {0.0f, 0.0f, 0.0f, 0.0f}, cB[4] = {0.0f, 0.0f, 0.0f, 0.0f}, cC[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  uint32_t bh[8][2], bl[16][2];                 // slot = block index mod 8 / mod 16
#pragma unroll
  for (int q = 0; q < 8; ++q) bh[q][0] = bh[q][1] = 0u;
#pragma unroll
  for (int q = 0; q < 16; ++q) bl[q][0] = bl[q][1] = 0u;
#pragma unroll
  for (int q = 0; q < 4; ++q) { bl[q][0] = Bl[8 * q]; bl[q][1] = Bl[8 * q + 4]; }   // B_l(0 .. 3)
  // staging state of the next frame
  const int F = t.F;
  float mean = 0.0f, scale = 1.0f;
  uint32_t* e_hi = reinterpret_cast<uint32_t*>(next_copies) + kFrontMargin / 2 + lane;
  uint32_t* e_lo = e_hi + geo.len / 2;
  uint16_t* o_hi = reinterpret_cast<uint16_t*>(next_copies) + 2 * geo.len + kFrontMargin - 1 + 2 * lane;
  uint16_t* o_lo = o_hi + geo.len;
  const float2* w2 = reinterpret_cast<const float2*>(hann) + lane;
  uint32_t a[4], an[4];
  ldsm_x4(sa0 - 32u * 8u, a);
#pragma unroll
  for (int m = -8; m < NBLK; ++m) {
    ldsm_x4(sa0 + static_cast<uint32_t>(32 * (m + 1)), an);      // the block beyond the last reads the zero margin
    if (m >= 0) { bh[m & 7][0] = Bh[8 * m]; bh[m & 7][1] = Bh[8 * m + 4]; }
    if (m >= 4) mma_16816(cB, a[0], a[1], a[2], a[3], bl[(m - 4) & 15][0], bl[(m - 4) & 15][1]);            // B_l(m - 4)
    if (m + 12 < NBLK) { bl[(m + 12) & 15][0] = Bl[8 * (m + 12)]; bl[(m + 12) & 15][1] = Bl[8 * (m + 12) + 4]; }
    if (m >= 4) mma_16816(hh1, a[0], a[1], a[2], a[3], bh[(m - 4) & 7][0], bh[(m - 4) & 7][1]);             // B_h(m - 4)
    if (m >= -4 && m + 4 < NBLK) mma_16816(cA, a[0], a[1], a[2], a[3], bl[(m + 4) & 15][0], bl[(m + 4) & 15][1]);
    if (m >= 0) mma_16816(hh0, a[0], a[1], a[2], a[3], bh[m & 7][0], bh[m & 7][1]);                         // B_h(m)
    if (m + 12 < NBLK) mma_16816(cC, a[0], a[1], a[2], a[3], bl[(m + 12) & 15][0], bl[(m + 12) & 15][1]);   // B_l(m + 12)
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = an[i];
    if (m == kPass1) {
      // pass 1 of am_process: mean and max |x| of the next frame, the exact power-of-two scale
      float sum = 0.0f, amax = 0.0f;
#pragma unroll
      for (int i = 0; i < kIters; ++i) {
        const int n = 2 * (lane + 32 * i);
        const float x = (i < kIters - 1 || n < F) ? v0[i] : 0.0f, c = (i < kIters - 1 || n + 1 < F) ? v1[i] : 0.0f;
        sum += x + c;
        amax = fmaxf(amax, fmaxf(fabsf(x), fabsf(c)));
      }
      sum = warp_sum(sum);
      amax = warp_max(amax);
      mean = sum / static_cast<float>(F);
      const float bound = amax + fabsf(mean);
      int e2 = 0;
      if (bound > 0.0f && bound < INFINITY) {
        e2 = 14 - (static_cast<int>((__float_as_uint(bound) >> 23) & 0xff) - 126);
        e2 = max(-100, min(100, e2));
      }
      scale = __uint_as_float(static_cast<uint32_t>(e2 + 127) << 23);
    }
    if (m >= kPass2 && (m - kPass2) % kStride == 0 && (m - kPass2) / kStride < kIters) {
      // one pass-2 iteration of am_process
      const int i = (m - kPass2) / kStride;
      const float2 w = w2[32 * i];
      const float x0 = (v0[i] - mean) * (w.x * scale);
      const float x1 = (v1[i] - mean) * (w.y * scale);
      const __half2 hi = __floats2half2_rn(x0, x1);
      const float2 hf = __half22float2(hi);
      const __half2 lo = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
      const uint32_t hw = *reinterpret_cast<const uint32_t*>(&hi), lw = *reinterpret_cast<const uint32_t*>(&lo);
      e_hi[32 * i] = hw;
      e_lo[32 * i] = lw;
      o_hi[64 * i] = static_cast<uint16_t>(hw);
      o_hi[64 * i + 1] = static_cast<uint16_t>(hw >> 16);
      o_lo[64 * i] = static_cast<uint16_t>(lw);
      o_lo[64 * i + 1] = static_cast<uint16_t>(lw >> 16);
    }
  }
  am_mma5_finish(hh0, hh1, cA, cB, cC, lane, val);     // ends with __syncwarp: the staged frame is visible to the warp
}

__device__ __forceinline__ bool am_all_small(const float (&val)[kVals], int lane, int n_lags, float thr) {
  bool small = true;
#pragma unroll
  for (int v = 0; v < kVals; ++v) {
    const int lag = lag_of(lane, v);
    if (lag >= 1 && lag <= n_lags && !(fabsf(val[v]) < thr)) small = false;
  }
  return __all_sync(0xffffffffu, small);
}

// ------------------------------------------------------------------------------------------------
// Symmetric kernel: every warp stages AND multiplies its own frames (one frame buffer per warp, no mbarriers).
// Round 1's warp-specialised producer / consumer pairs kept two MMA warps per scheduler busy and two producer warps
// idle two thirds of the time (ncu, round 2: 25 % of all stall samples were producers spinning on `empty`), and
// whenever both MMA warps of a scheduler waited for a fragment or a hand-off at the same moment the tensor pipe idled
// (67 % active).  Here the same sixteen warps per SM all issue MMAs, each in its own phase of the stage / multiply
// cycle, so on average two to three warps per scheduler have MMAs ready while the others convert their next frame.
// Same shared-memory footprint (sixteen frame buffers per SM), same registers, same arithmetic in the same order as
// the pairs: bit-identical rows.
// ------------------------------------------------------------------------------------------------
constexpr int kSymWarps = 8;       // per block, two blocks per SM

#ifdef NSF_AC_TRACE
// Debug build only (scripts/build_variant.sh ... -DNSF_AC_TRACE): per warp, the SM clock at the start of the staging
// half, the start and the end of the MMA loop of its first kTraceFrames frames; read back with nsf_debug_ac_trace.
constexpr int kTraceFrames = 40;
__device__ long long g_ac_trace[296 * 8 * kTraceFrames * 3];
__device__ int g_ac_smid[296];
#endif

// kFive: the five-tile loop am_mma5 (product path) instead of the six-MMA loop am_mma (NSF_AC_LOOP=six, validation).
template <int kIters, bool kExact, bool kFive>
__global__ void __launch_bounds__(kSymWarps * 32, 2) k_autocorr_sym(DeviceTables t, BatchView b,
                                                                    const float* __restrict__ y, bool reduce,
                                                                    float* __restrict__ out, int64_t out_ld, int col0) {
  extern __shared__ __align__(16) __half s_am[];
  const AmGeom geo = am_geom(t.F);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_warps = static_cast<int>(blockDim.x >> 5);
  const size_t region = kExtraFront + 4 * static_cast<size_t>(geo.len);   // halfs per warp: [zeros | E_hi | E_lo | O_hi | O_lo]
  __half* copies = s_am + static_cast<size_t>(warp) * region + kExtraFront;
  float* hann = reinterpret_cast<float*>(s_am + static_cast<size_t>(n_warps) * region);
  const int n_it = (t.F / 2 + 1 + 31) / 32;
  for (int n = threadIdx.x; n < 64 * n_it; n += blockDim.x) hann[n] = n < t.F ? __ldg(t.hann_sym + n) : 0.0f;
  // zero once: the margins are never written again, the frame region is rewritten per frame
  for (int i = lane; i < static_cast<int>(region / 2); i += 32) reinterpret_cast<uint32_t*>(copies - kExtraFront)[i] = 0u;
  __syncthreads();
  const int64_t n_warps_total = static_cast<int64_t>(gridDim.x) * n_warps;
  const int64_t chunk = (b.total_rows + n_warps_total - 1) / n_warps_total;
  const int64_t r_begin = (static_cast<int64_t>(blockIdx.x) * n_warps + warp) * chunk;
  const int64_t r_end = min(r_begin + chunk, b.total_rows);
  int64_t base = 0, len = 0, clip_row0 = 0, clip_row_end = -1;
  int T = 0, tf_lo = 0, tf_hi = 0;      // frames of the clip; its `fast` frames (am_src) are tf_lo <= tf < tf_hi
  // the MMA half of a frame: six-MMA loop, five-tile loop, or (F = 266, the 16 kHz plan: seventeen K-blocks) the
  // five-tile loop unrolled at compile time
  auto run_mma = [&](float (&val)[kVals]) {
    if constexpr (kFive) {
      if constexpr (kIters == 5 && kExact) {
        if (geo.nblk == 17) { am_mma5_static<17>(copies, geo, lane, val); return; }
      }
      am_mma5(copies, geo, lane, val);
    } else {
      am_mma(copies, geo, lane, val);
    }
  };
#ifdef NSF_AC_TRACE
  int trace_i = 0;
  if (threadIdx.x == 0 && blockIdx.x < 296) { int sm; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); g_ac_smid[blockIdx.x] = sm; }
#endif
  for (int64_t r = r_begin; r < r_end; ++r) {
    if (r >= clip_row_end) {
      const int clip = find_segment(b.row_off, b.n_clips, r);
      base = __ldg(b.clip_off + clip);
      len = __ldg(b.clip_off + clip + 1) - base;
      T = static_cast<int>(__ldg(b.frame_off + clip + 1) - __ldg(b.frame_off + clip));
      clip_row0 = __ldg(b.row_off + clip);
      clip_row_end = __ldg(b.row_off + clip + 1);
      // fast frames (inside the clip, 64 n_it samples before the end of the packed signal): tf_lo <= tf < tf_hi,
      // derived once per clip so that a frame costs two comparisons and one 32 x 32 -> 64 bit product
      const int64_t in_clip = len - t.F + t.pad, in_batch = b.total_samples - base - 64 * static_cast<int64_t>(n_it) + t.pad;
      const int64_t last = min(in_clip, in_batch);          // tf H <= last
      tf_lo = (t.pad + t.H - 1) / t.H;
      tf_hi = last >= 0 ? static_cast<int>(min(last / t.H, static_cast<int64_t>(T))) + 1 : 0;
    }
    const int lr = static_cast<int>(r - clip_row0);
    const int tf0 = reduce ? 2 * lr : lr;
    const int n_frames = (reduce && tf0 + 1 < T) ? 2 : 1;   // odd T: the last row passes through
    float acc[kVals];
#pragma unroll
    for (int v = 0; v < kVals; ++v) acc[v] = 0.0f;
    for (int f = 0; f < n_frames; ++f) {
      const int tf = tf0 + f;
      const bool fast = tf >= tf_lo && tf < tf_hi;
#ifdef NSF_AC_TRACE
      const bool tr = lane == 0 && trace_i < kTraceFrames && blockIdx.x < 296 && warp < 8;
      long long* trp = g_ac_trace + ((static_cast<size_t>(blockIdx.x) * 8 + warp) * kTraceFrames + trace_i) * 3;
      if (tr) trp[0] = clock64();
#endif
      if (fast) {
        float v0[kIters], v1[kIters];
        am_issue_fast<kIters, kExact>(y + base + (static_cast<int64_t>(tf) * t.H - t.pad), n_it, lane, v0, v1);
        am_process<kIters, kExact>(t, hann, n_it, v0, v1, copies, geo, lane, nullptr);
      } else {
        am_fill_simple(t, hann, am_src(t, b, y, base, len, tf, n_it), copies, geo, lane);
      }                                                   // both end with __syncwarp
#ifdef NSF_AC_TRACE
      if (tr) trp[1] = clock64();
#endif
      float val[kVals];
      run_mma(val);                                       // ends with __syncwarp: the buffer may be rewritten
#ifdef NSF_AC_TRACE
      if (tr) trp[2] = clock64();
      ++trace_i;
#endif
      if (T > 1 && (tf == 0 || tf == T - 1) && am_all_small(val, lane, t.n_lags, t.edge_thr)) {
        am_fill_simple(t, hann, am_src(t, b, y, base, len, tf == 0 ? 1 : T - 2, n_it), copies, geo, lane);
        run_mma(val);
      }
#pragma unroll
      for (int v = 0; v < kVals; ++v) acc[v] += val[v];
    }
    const float wgt = n_frames == 2 ? 0.5f : 1.0f;
    float* o = out + r * out_ld + col0;
#pragma unroll
    for (int v = 0; v < kVals; ++v) {
      const int lag = lag_of(lane, v);
      if (lag >= 1 && lag <= t.n_lags) o[lag - 1] = acc[v] * wgt;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Software-pipelined kernel (round 2, product path for the 88.2 kHz plan: F = 1470, 92 K-blocks): eight warps per SM,
// each with TWO frame buffers and up to 255 registers.  While a warp runs the MMA loop of frame n out of one buffer it
// converts frame n + 1 - whose raw samples were requested before the loop started and wait in registers - into the
// other (am_mma5_pipe), so every warp issues MMAs all the time and the staging instructions fill the issue slots the
// tensor pipe leaves free.  Same shared-memory footprint as the symmetric kernel (sixteen frame buffers per SM), same
// arithmetic in the same order: bit-identical rows (tests/test_gpu_round2.py::test_autocorr_kernels_agree).
// Cold paths (clip-edge frames with reflect padding, the end of the batch, the edge-frame fix) are staged by
// am_fill_simple outside the loop and multiplied by the generic am_mma5.
// ------------------------------------------------------------------------------------------------
constexpr int kPipeWarps = 8;      // per block, one block per SM

// One hop-frame of a warp's row run: output row, frame index inside its clip, position inside the row's frame pair.
// `crossed`: the frame is the first one of the next clip (the clip state of the enumeration has moved on).
struct AmFrame {
  int64_t r;
  int tf, n_frames, f;
  bool valid, crossed;
};

template <int kIters, int NBLK, int kWarps, int kBlocksPerSm>
__global__ void __launch_bounds__(kWarps * 32, kBlocksPerSm) k_autocorr_pipe(DeviceTables t, BatchView b,
                                                                      const float* __restrict__ y, bool reduce,
                                                                      float* __restrict__ out, int64_t out_ld, int col0) {
  extern __shared__ __align__(16) __half s_am[];
  const AmGeom geo = am_geom(t.F);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_warps = static_cast<int>(blockDim.x >> 5);
  const size_t region = kExtraFront + 4 * static_cast<size_t>(geo.len);   // halfs per buffer: [zeros | E_hi | E_lo | O_hi | O_lo]
  __half* buf0 = s_am + static_cast<size_t>(2 * warp) * region + kExtraFront;
  __half* buf1 = buf0 + region;
  float* hann = reinterpret_cast<float*>(s_am + static_cast<size_t>(2 * n_warps) * region);
  constexpr int n_it = kIters;
  for (int n = threadIdx.x; n < 64 * n_it; n += blockDim.x) hann[n] = n < t.F ? __ldg(t.hann_sym + n) : 0.0f;
  // zero once: the margins are never written again, the frame regions are rewritten per frame
  for (int i = lane; i < static_cast<int>(region); i += 32) reinterpret_cast<uint32_t*>(buf0 - kExtraFront)[i] = 0u;
  __syncthreads();
  const int64_t n_warps_total = static_cast<int64_t>(gridDim.x) * n_warps;
  const int64_t chunk = (b.total_rows + n_warps_total - 1) / n_warps_total;
  const int64_t r_begin = (static_cast<int64_t>(blockIdx.x) * n_warps + warp) * chunk;
  const int64_t r_end = min(r_begin + chunk, b.total_rows);
  // Frame enumeration of the warp's row run with one frame of look-ahead.  Inside a clip the next frame is an
  // increment: the clip state - and the range [tf_lo, tf_hi) of its `fast` frames (am_src: inside the clip and 64 n_it
  // samples before the end of the packed signal) - is derived once per clip; the clip before is kept for the edge
  // fix of its last frame, which is handled after the enumeration has moved on.
  int64_t base = 0, len = 0, clip_row0 = 0, clip_row_end = -1, pbase = 0, plen = 0;
  int T = 0, pT = 0, tf_lo = 0, tf_hi = 0;
  auto open_clip = [&](int64_t r) {
    pbase = base; plen = len; pT = T;
    const int clip = find_segment(b.row_off, b.n_clips, r);
    base = __ldg(b.clip_off + clip);
    len = __ldg(b.clip_off + clip + 1) - base;
    T = static_cast<int>(__ldg(b.frame_off + clip + 1) - __ldg(b.frame_off + clip));
    clip_row0 = __ldg(b.row_off + clip);
    clip_row_end = __ldg(b.row_off + clip + 1);
    const int64_t in_clip = len - t.F + t.pad, in_batch = b.total_samples - base - 64 * n_it + t.pad;
    const int64_t last = min(in_clip, in_batch);          // tf H <= last
    tf_lo = (t.pad + t.H - 1) / t.H;
    tf_hi = last >= 0 ? static_cast<int>(min(last / t.H, static_cast<int64_t>(T))) + 1 : 0;
  };
  auto first_frame = [&]() -> AmFrame {
    AmFrame fr;
    fr.r = r_begin; fr.tf = 0; fr.n_frames = 1; fr.f = 0; fr.crossed = false;
    fr.valid = r_begin < r_end;
    if (fr.valid) {
      open_clip(r_begin);
      const int64_t lr = r_begin - clip_row0;
      fr.tf = static_cast<int>(reduce ? 2 * lr : lr);
      fr.n_frames = (reduce && fr.tf + 1 < T) ? 2 : 1;     // odd T: the last row passes through
    }
    return fr;
  };
  auto next_frame = [&](const AmFrame& prev) -> AmFrame {
    AmFrame fr = prev;
    fr.crossed = false;
    if (prev.f + 1 < prev.n_frames) { fr.f = prev.f + 1; fr.tf = prev.tf + 1; return fr; }
    fr.r = prev.r + 1;
    fr.f = 0;
    if (fr.r >= r_end) { fr.valid = false; return fr; }
    if (fr.r >= clip_row_end) {
      open_clip(fr.r);
      fr.crossed = true;
      const int64_t lr = fr.r - clip_row0;
      fr.tf = static_cast<int>(reduce ? 2 * lr : lr);
    } else {
      fr.tf = prev.tf + 1;
    }
    fr.n_frames = (reduce && fr.tf + 1 < T) ? 2 : 1;
    return fr;
  };
  AmFrame cur = first_frame();
  if (cur.valid) {                                     // prologue: the first frame is staged on its own
    const AmSrc src = am_src(t, b, y, base, len, cur.tf, n_it);
    if (src.fast) {
      float v0[kIters], v1[kIters];
      am_issue_fast<kIters, true>(src.clip + src.first, n_it, lane, v0, v1);
      am_process<kIters, true>(t, hann, n_it, v0, v1, buf0, geo, lane, nullptr);
    } else {
      am_fill_simple(t, hann, src, buf0, geo, lane);
    }
  }
  int p = 0;
  float acc[kVals];
#pragma unroll
  for (int v = 0; v < kVals; ++v) acc[v] = 0.0f;
  while (cur.valid) {
    __half* copies = p ? buf1 : buf0;
    __half* next_copies = p ? buf0 : buf1;
    const AmFrame nxt = next_frame(cur);               // may move the clip state on (nxt.crossed)
    const bool nfast = nxt.valid && nxt.tf >= tf_lo && nxt.tf < tf_hi;
    float val[kVals];
    if (nfast) {
      float v0[kIters], v1[kIters];
      am_issue_fast<kIters, true, true>(y + base + (static_cast<int64_t>(nxt.tf) * t.H - t.pad), n_it, lane, v0, v1);
      am_mma5_pipe<NBLK, kIters>(copies, geo, lane, val, t, hann, v0, v1, next_copies);
    } else {
      am_mma5(copies, geo, lane, val);
      if (nxt.valid) am_fill_simple(t, hann, am_src(t, b, y, base, len, nxt.tf, n_it), next_copies, geo, lane);
    }
    // fix_edge_frames_autocorr: a near-silent first (last) frame takes the values of frame 1 (T-2); rare
    const bool moved = nxt.valid && nxt.crossed;       // cur belongs to the clip before
    const int cT = moved ? pT : T;
    if (cT > 1 && (cur.tf == 0 || cur.tf == cT - 1) && am_all_small(val, lane, t.n_lags, t.edge_thr)) {
      am_fill_simple(t, hann, am_src(t, b, y, moved ? pbase : base, moved ? plen : len, cur.tf == 0 ? 1 : cT - 2, n_it),
                     copies, geo, lane);
      am_mma5(copies, geo, lane, val);
    }
#pragma unroll
    for (int v = 0; v < kVals; ++v) acc[v] += val[v];
    if (cur.f == cur.n_frames - 1) {
      const float wgt = cur.n_frames == 2 ? 0.5f : 1.0f;
      float* o = out + cur.r * out_ld + col0;
#pragma unroll
      for (int v = 0; v < kVals; ++v) {
        const int lag = lag_of(lane, v);
        if (lag >= 1 && lag <= t.n_lags) o[lag - 1] = acc[v] * wgt;
        acc[v] = 0.0f;
      }
    }
    cur = nxt;
    p ^= 1;
  }
}

}  // namespace

int launch_autocorr_mma(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* y,
                        bool reduce, float* out, int64_t out_ld, int col0) {
  const AmGeom geo = am_geom(t.F);
  if (t.n_lags > 191) return -1;
  const int iters = (t.F / 2 + 1 + 31) / 32;      // register-staging iterations the frame needs
  const size_t hann_bytes = static_cast<size_t>(64) * iters * sizeof(float);   // np.hanning(F), zero padded
  // MMA loop of the symmetric kernel: the five-tile loop (am_mma5) for frames of at least 44 K-blocks (F >= 689:
  // 44.1 kHz and up), where most blocks run in its unchecked body; the six-MMA loop (am_mma) for short frames, where the
  // eight lead-in blocks and the range checks of the five-tile loop cost more than the MMAs it saves (B200, F = 266:
  // 3.35 vs 3.12 ms on C5; F = 1470: 1.11 vs 1.24 ms on C2).  NSF_AC_LOOP=five / six forces one (validation, A/B).
  static const int loop_env = [] {
    const char* v = std::getenv("NSF_AC_LOOP");
    return v == nullptr ? 0 : (v[0] == 's' ? 6 : (v[0] == 'f' ? 5 : 0));
  }();
  // F = 266 (iters == 5, seventeen K-blocks) has the five-tile loop unrolled at compile time (am_mma5_static), which
  // has neither the lead-in overhead nor the checks
  const bool static_five = iters == 5 && geo.nblk == 17;
  const bool use_six = loop_env == 6 || (loop_env == 0 && geo.nblk < 44 && !static_five);
  // symmetric kernel: as many warps per block as fit twice per SM (eight up to F ~ 1530, fewer for long frames);
  // two blocks of 113 KB (+ 1 KB reserved each) are what an SM's 228 KB hold
  int warps = kSymWarps;
  size_t smem = 0;
  for (; warps >= 1; --warps) {
    smem = static_cast<size_t>(warps) * (kExtraFront + 4 * static_cast<size_t>(geo.len)) * sizeof(__half) + hann_bytes;
    if (smem <= (warps > 2 ? 113 : 220) * 1024) break;      // long frames: one block per SM
  }
  if (warps < 1) return -1;
  // Software-pipelined kernel (k_autocorr_pipe): the 88.2 kHz plan (23 staging iterations, 92 K-blocks).
  // NSF_AC_KERNEL=sym selects the symmetric kernel instead (validation; bit-identical rows)
  static const bool no_pipe = [] {
    const char* v = std::getenv("NSF_AC_KERNEL");
    return v != nullptr && v[0] == 's';
  }();
  // Short frames stay on the symmetric kernel: at F = 266 (16 kHz) the pipelined kernel is bit-identical but SLOWER
  // (B200, C5: 2.93 ms at twelve warps per SM / 168 registers with one or two frames of look-ahead, 3.10 - 4.70 ms at
  // sixteen warps / 128 registers, against 2.68 ms; profiles/experiments/README.md section 8)
  const bool pipe23 = iters == 23 && geo.nblk == 92;
  if (!no_pipe && loop_env != 6 && pipe23) {
    const size_t region = kExtraFront + 4 * static_cast<size_t>(geo.len);
    const size_t pipe_smem = static_cast<size_t>(2 * kPipeWarps) * region * sizeof(__half) + hann_bytes;
    int64_t pgrid = (b.total_rows + kPipeWarps - 1) / kPipeWarps;
    if (pgrid > kSmCount) pgrid = kSmCount;
    if (pgrid < 1) pgrid = 1;
    k_autocorr_pipe<23, 92, kPipeWarps, 1><<<static_cast<int>(pgrid), kPipeWarps * 32, pipe_smem, s>>>(t, b, y, reduce, out, out_ld, col0);
    NSF_CHECK_LAUNCH();
    return 1;
  }
  const int per_sm = smem <= 113 * 1024 ? 2 : 1;
  int64_t grid = (b.total_rows + warps - 1) / warps;
  if (grid > static_cast<int64_t>(kSmCount) * per_sm) grid = static_cast<int64_t>(kSmCount) * per_sm;
  if (grid < 1) grid = 1;
  const int threads = warps * 32;
  auto go = [&](auto k_five, auto k_six) {
    if (use_six) k_six<<<static_cast<int>(grid), threads, smem, s>>>(t, b, y, reduce, out, out_ld, col0);
    else k_five<<<static_cast<int>(grid), threads, smem, s>>>(t, b, y, reduce, out, out_ld, col0);
    NSF_CHECK_LAUNCH();
    return 1;
  };
#define NSF_AC_GO(IT, EX) go(k_autocorr_sym<IT, EX, true>, k_autocorr_sym<IT, EX, false>)
  if (iters == 23) return NSF_AC_GO(23, true);    // 88.2 kHz: F = 1470
  if (iters == 5) return NSF_AC_GO(5, true);      // 16 kHz: F = 266
  if (iters <= 6) return NSF_AC_GO(6, false);     // F <= 382   (22.05 kHz: 367)
  if (iters <= 12) return NSF_AC_GO(12, false);   // F <= 766   (44.1 kHz: 735)
  if (iters <= 24) return NSF_AC_GO(24, false);   // F <= 1534  (48 kHz: 800)
  if (iters <= 40) return NSF_AC_GO(40, false);   // F <= 2558
  return NSF_AC_GO(66, false);                    // F <= 4096  (plan limit)
#undef NSF_AC_GO
}

// Opt-in shared-memory limit of every instantiation, once per device (called by nsf_ctx_create after
// cudaSetDevice; the attribute is per device and a process may drive several).
bool init_autocorr_mma_attributes() {
  bool ok = true;
  auto set = [&](auto kernel) {
    ok = ok && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) == cudaSuccess;
  };
#define NSF_AC_SET(IT, EX) set(k_autocorr_sym<IT, EX, true>); set(k_autocorr_sym<IT, EX, false>)
  NSF_AC_SET(23, true); NSF_AC_SET(5, true); NSF_AC_SET(6, false); NSF_AC_SET(12, false);
  NSF_AC_SET(24, false); NSF_AC_SET(40, false); NSF_AC_SET(66, false);
#undef NSF_AC_SET
  set(k_autocorr_pipe<23, 92, kPipeWarps, 1>);
  return ok;
}

}  // namespace nsf

#ifdef NSF_AC_TRACE
extern "C" __attribute__((visibility("default"))) int nsf_debug_ac_trace(long long* trace, int* smid) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(trace, nsf::g_ac_trace, sizeof(nsf::g_ac_trace)) != cudaSuccess) return -1;
  if (cudaMemcpyFromSymbol(smid, nsf::g_ac_smid, sizeof(nsf::g_ac_smid)) != cudaSuccess) return -1;
  return nsf::kTraceFrames;
}
#endif

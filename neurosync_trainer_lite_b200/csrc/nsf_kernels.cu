// Bandwidth- and FMA-bound kernels of the feature front-end (sm_100a).
//
//   k_absmax / k_normalize   utils/audio/load_audio.py:12-14       (HBM bound)
//   k_fold32 / k_dft_simt    validation-only fp32 STFT path (NSF_DEBUG_SIMT_DFT); the product path
//                            is the tcgen05 kernel in nsf_stft_tc.cu
//   k_mel_db                 mel projection (sparse: 1.5 % of the 128 x 736 basis is non-zero),
//                            10 log10(max(1e-10, .)), per-clip max       (HBM bound)
//   k_dct_sum                top_db floor, DCT-II to n_mfcc, CMVN moments (sum x, sum x^2 in f64)
//   k_delta_reduce           CMVN, Savitzky-Golay delta / delta-delta, pair reduction
//   k_autocorr               reflect-pad framing, DC removal, np.hanning, 188 lags, normalise,
//                            edge fix, pair reduction  (fp32 FMA bound; extract_features_utils.py:54-113)
//   k_smooth                 smooth_features (extract_features_utils.py:47-51)
//   k_collect_rows           collect_features augmentation (dataset/data_processing.py:126-197)
#include <cuda_fp16.h>

#include "nsf.h"
#include "nsf_device_utils.cuh"
#include <cstdlib>

#include "nsf_kernels.cuh"

namespace nsf {

namespace {

template <typename T> __device__ __forceinline__ float decode_pcm(T v);
template <> __device__ __forceinline__ float decode_pcm<float>(float v) { return v; }
template <> __device__ __forceinline__ float decode_pcm<int16_t>(int16_t v) {
  return static_cast<float>(v) * (1.0f / 32768.0f);  // exact: soundfile's int16 -> float32
}

// ------------------------------------------------------------------------------------------------
// K0: per-clip max|y|.  Each block owns a fixed chunk of the packed signal and walks the clips
// that intersect it; one atomicMax per (block, clip).
// ------------------------------------------------------------------------------------------------
constexpr int kChunk = 16384;

// 16-byte vectors of the PCM stream (8 int16 or 4 float32 samples); kVec = false is the scalar form for caller
// pointers that are not 16-byte aligned.
template <typename T> struct PcmVec;
template <> struct PcmVec<int16_t> {
  static constexpr int kN = 8;
  static __device__ __forceinline__ void load(const int16_t* p, float (&v)[8]) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = decode_pcm<int16_t>(static_cast<int16_t>(w[i] & 0xffffu));
      v[2 * i + 1] = decode_pcm<int16_t>(static_cast<int16_t>(w[i] >> 16));
    }
  }
};
template <> struct PcmVec<float> {
  static constexpr int kN = 4;
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
};

// [s, e) of the packed signal as scalar head, 16-byte aligned vector body, scalar tail (indices relative to the
// array, whose base is 16-byte aligned when kVec)
template <typename T, bool kVec>
struct PcmSpan {
  int64_t head_end, body_end;     // [s, head_end) scalar, [head_end, body_end) vectors, [body_end, e) scalar
  __device__ __forceinline__ PcmSpan(int64_t s, int64_t e) {
    constexpr int n = PcmVec<T>::kN;
    if (kVec) {
      head_end = min(e, (s + n - 1) / n * n);
      body_end = max(head_end, e / n * n);
    } else {
      head_end = e;
      body_end = e;
    }
  }
};

template <typename T, bool kVec>
__global__ void __launch_bounds__(256) k_absmax(const T* __restrict__ pcm, BatchView b,
                                                uint32_t* __restrict__ peak_bits) {
  __shared__ float s_part[8];
  constexpr int n = PcmVec<T>::kN;
  for (int64_t c0 = static_cast<int64_t>(blockIdx.x) * kChunk; c0 < b.total_samples; c0 += static_cast<int64_t>(gridDim.x) * kChunk) {
  const int64_t c1 = min(c0 + kChunk, b.total_samples);
  int clip = find_segment(b.clip_off, b.n_clips, c0);
  int64_t s = c0;
  while (s < c1) {
    const int64_t e = min(c1, __ldg(b.clip_off + clip + 1));
    const PcmSpan<T, kVec> sp(s, e);
    float m = 0.0f;
    for (int64_t i = s + threadIdx.x; i < sp.head_end; i += blockDim.x) m = fmaxf(m, fabsf(decode_pcm<T>(pcm[i])));
    for (int64_t i = sp.head_end + static_cast<int64_t>(threadIdx.x) * n; i < sp.body_end; i += static_cast<int64_t>(blockDim.x) * n) {
      float v[n];
      PcmVec<T>::load(pcm + i, v);
#pragma unroll
      for (int k = 0; k < n; ++k) m = fmaxf(m, fabsf(v[k]));
    }
    for (int64_t i = sp.body_end + threadIdx.x; i < e; i += blockDim.x) m = fmaxf(m, fabsf(decode_pcm<T>(pcm[i])));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
      float r = s_part[0];
      for (int w = 1; w < 8; ++w) r = fmaxf(r, s_part[w]);
      atomicMax(peak_bits + clip, __float_as_uint(r));  // r >= 0: bit order == value order
    }
    __syncthreads();
    s = e;
    ++clip;
  }
  }
}

template <typename T, bool kVec>
__global__ void __launch_bounds__(256) k_normalize(const T* __restrict__ pcm, BatchView b,
                                                   const uint32_t* __restrict__ peak_bits,
                                                   bool use_peak, float* __restrict__ y) {
  constexpr int n = PcmVec<T>::kN;
  for (int64_t c0 = static_cast<int64_t>(blockIdx.x) * kChunk; c0 < b.total_samples; c0 += static_cast<int64_t>(gridDim.x) * kChunk) {
  const int64_t c1 = min(c0 + kChunk, b.total_samples);
  int clip = find_segment(b.clip_off, b.n_clips, c0);
  int64_t s = c0;
  while (s < c1) {
    const int64_t e = min(c1, __ldg(b.clip_off + clip + 1));
    const float peak = use_peak ? __uint_as_float(__ldg(peak_bits + clip)) : 0.0f;
    const bool div = peak > 0.0f;
    const PcmSpan<T, kVec> sp(s, e);
    // IEEE division: bit-identical to numpy's float32 y / max_val
    auto one = [&](int64_t i) { const float v = decode_pcm<T>(pcm[i]); y[i] = div ? __fdiv_rn(v, peak) : v; };
    for (int64_t i = s + threadIdx.x; i < sp.head_end; i += blockDim.x) one(i);
    for (int64_t i = sp.head_end + static_cast<int64_t>(threadIdx.x) * n; i < sp.body_end; i += static_cast<int64_t>(blockDim.x) * n) {
      float v[n];
      PcmVec<T>::load(pcm + i, v);
      if (div) {
#pragma unroll
        for (int k = 0; k < n; ++k) v[k] = __fdiv_rn(v[k], peak);
      }
#pragma unroll
      for (int k = 0; k < n; k += 4)                      // i is a multiple of n >= 4: 16-byte aligned stores
        *reinterpret_cast<float4*>(y + i + k) = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
    }
    for (int64_t i = sp.body_end + threadIdx.x; i < e; i += blockDim.x) one(i);
    s = e;
    ++clip;
  }
  }
}

// ------------------------------------------------------------------------------------------------
// Validation STFT path, fp32 on CUDA cores: fold (signed 4-tap gather) + small GEMMs + |.|^2
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_fold32(DeviceTables t, BatchView b,
                                                const float* __restrict__ y,
                                                float* __restrict__ a32) {
  extern __shared__ float s_x[];  // [F]
  for (int64_t g = blockIdx.x; g < b.total_frames; g += gridDim.x) {
    const int clip = find_segment(b.frame_off, b.n_clips, g);
    const int64_t tf = g - __ldg(b.frame_off + clip);
    const int64_t base = __ldg(b.clip_off + clip);
    const int64_t len = __ldg(b.clip_off + clip + 1) - base;
    const int64_t first = tf * t.H - t.pad;  // zero padding (librosa stft center=True, constant)
    for (int n = threadIdx.x; n < t.F; n += blockDim.x) {
      const int64_t i = first + n;
      s_x[n] = (i >= 0 && i < len) ? __ldg(y + base + i) : 0.0f;
    }
    __syncthreads();
    for (int c = 0; c < t.chains; ++c) {
      const int kp = t.kp[c];
      for (int e = threadIdx.x; e < 2 * kp; e += blockDim.x) {
        const int part = e / kp, j = e - part * kp;
        float acc = 0.0f;
#pragma unroll
        for (int tap = 0; tap < 4; ++tap) {
          const int o = (part * 4 + tap) * kp + j;
          acc = fmaf(__ldg(t.tap_coef[c] + o), s_x[__ldg(t.tap_idx[c] + o)], acc);
        }
        a32[(static_cast<int64_t>(c * 2 + part) * b.total_frames + g) * kp + j] = acc;
      }
    }
    __syncthreads();
  }
}

// 64 frames x 64 bins per block, both Re and Im accumulators, K chunks of 16.
__global__ void __launch_bounds__(256) k_dft_simt(DeviceTables t, BatchView b,
                                                  const float* __restrict__ a32,
                                                  float* __restrict__ power) {
  const int c = blockIdx.z;
  const int kp = t.kp[c], np = t.np[c], nb = t.nbins[c];
  const int n0 = blockIdx.y * 64;
  if (n0 >= np) return;
  const int64_t g0 = static_cast<int64_t>(blockIdx.x) * 64;
  __shared__ float As[2][16][64 + 4];
  __shared__ float Bs[2][16][64];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[2][4][4] = {};
  const float* A0 = a32 + static_cast<int64_t>(c * 2 + 0) * b.total_frames * kp;
  const float* A1 = a32 + static_cast<int64_t>(c * 2 + 1) * b.total_frames * kp;
  for (int k0 = 0; k0 < kp; k0 += 16) {
    for (int e = threadIdx.x; e < 64 * 16; e += 256) {
      const int r = e >> 4, kk = e & 15;
      const int64_t g = g0 + r;
      const bool ok = g < b.total_frames;
      As[0][kk][r] = ok ? A0[g * kp + k0 + kk] : 0.0f;
      As[1][kk][r] = ok ? A1[g * kp + k0 + kk] : 0.0f;
    }
    for (int e = threadIdx.x; e < 16 * 64; e += 256) {
      const int kk = e >> 6, n = e & 63;
      const bool ok = (n0 + n) < np;
      Bs[0][kk][n] = ok ? __ldg(t.mat32[c][0] + static_cast<int64_t>(k0 + kk) * np + n0 + n) : 0.0f;
      Bs[1][kk][n] = ok ? __ldg(t.mat32[c][1] + static_cast<int64_t>(k0 + kk) * np + n0 + n) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[2][4], bb[2][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        a[0][i] = As[0][kk][ty * 4 + i];
        a[1][i] = As[1][kk][ty * 4 + i];
        bb[0][i] = Bs[0][kk][tx * 4 + i];
        bb[1][i] = Bs[1][kk][tx * 4 + i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[0][i][j] = fmaf(a[0][i], bb[0][j], acc[0][i][j]);
          acc[1][i][j] = fmaf(a[1][i], bb[1][j], acc[1][i][j]);
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t g = g0 + ty * 4 + i;
    if (g >= b.total_frames) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = n0 + tx * 4 + j;
      if (m < nb) {
        const float re = acc[0][i][j], im = acc[1][i][j];
        power[g * t.bins_ld + t.col_off[c] + m] = fmaf(re, re, im * im);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K1c: sparse mel projection + dB + per-clip dB max.  A block owns 32 consecutive hop-frames: the
// power tile is transposed into shared memory ([column][frame], pitch 33) so that LANES ARE FRAMES:
// every shared load is conflict-free and every filter weight is a warp-uniform (broadcast) load.
// Warp w accumulates mels [16 w, 16 w + 16); each filter is one contiguous column run per fold chain.
// ------------------------------------------------------------------------------------------------
constexpr int kMelWarps = 8;
constexpr int kMelFrames = 32;
constexpr int kMelPitch = kMelFrames + 1;
constexpr int kMelPerWarp = 16;                    // n_mels <= 128
__global__ void __launch_bounds__(kMelWarps * 32) k_mel_db(DeviceTables t, BatchView b,
                                                           const float* __restrict__ power,
                                                           float* __restrict__ db,
                                                           uint32_t* __restrict__ dbmax_key, int chain_cols) {
  extern __shared__ float s_mel[];                 // [chain_cols][33] power^T of one chain, then [32][n_mels + 1] dB
  __shared__ uint32_t s_max[kMelFrames];
  float* s_pow = s_mel;
  float* s_out = s_mel + static_cast<size_t>(chain_cols) * kMelPitch;
  const int out_pitch = t.n_mels + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_tiles = (b.total_frames + kMelFrames - 1) / kMelFrames;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t g0 = tile * kMelFrames;
    const int nf = static_cast<int>(min(static_cast<int64_t>(kMelFrames), b.total_frames - g0));
    if (threadIdx.x < kMelFrames) s_max[threadIdx.x] = 0u;
    float acc[kMelPerWarp];
#pragma unroll
    for (int q = 0; q < kMelPerWarp; ++q) acc[q] = 0.0f;
    for (int c = 0; c < t.chains; ++c) {
      const int c0 = t.col_off[c], nc = t.np[c];
      __syncthreads();                              // previous chain / tile fully consumed
      for (int f = warp; f < kMelFrames; f += kMelWarps) {
        const float* src = power + (g0 + f) * t.bins_ld + c0;
        if (f < nf) {
          // 12 independent 128-byte requests per warp in flight, then the transposing stores
          for (int k0 = lane; k0 < nc; k0 += 32 * 12) {
            float v[12];
#pragma unroll
            for (int q = 0; q < 12; ++q) v[q] = (k0 + 32 * q < nc) ? __ldg(src + k0 + 32 * q) : 0.0f;
#pragma unroll
            for (int q = 0; q < 12; ++q)
              if (k0 + 32 * q < nc) s_pow[(k0 + 32 * q) * kMelPitch + f] = v[q];
          }
        } else {
          for (int k = lane; k < nc; k += 32) s_pow[k * kMelPitch + f] = 0.0f;
        }
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < kMelPerWarp; ++q) {
        const int m = q * kMelWarps + warp;     // interleaved: long (high) filters spread over warps
        if (m < t.n_mels) {
          const int e = c * t.n_mels + m;
          const int ln = __ldg(t.mel_len + e);
          const float* w = t.mel_w + __ldg(t.mel_ptr + e);
          const float* col = s_pow + static_cast<size_t>(__ldg(t.mel_start + e) - c0) * kMelPitch + lane;
          float a = acc[q];
#pragma unroll 4
          for (int i = 0; i < ln; ++i) a = fmaf(__ldg(w + i), col[i * kMelPitch], a);
          acc[q] = a;
        }
      }
    }
    float vmax = -INFINITY;
#pragma unroll
    for (int q = 0; q < kMelPerWarp; ++q) {
      const int m = q * kMelWarps + warp;
      if (m < t.n_mels) {
        const float v = 10.0f * log10f(fmaxf(1e-10f, acc[q]));
        s_out[lane * out_pitch + m] = v;
        vmax = fmaxf(vmax, v);
      }
    }
    if (lane < nf && warp < t.n_mels) atomicMax(&s_max[lane], float_key(vmax));
    __syncthreads();
    // coalesced dB rows out
    for (int f = warp; f < nf; f += kMelWarps)
      for (int m = lane; m < t.n_mels; m += 32) db[(g0 + f) * t.n_mels + m] = s_out[f * out_pitch + m];
    if (warp == 0)   // one global atomic per tile, unless the tile spans clips
      warp_clip_max(dbmax_key, lane < nf ? find_segment(b.frame_off, b.n_clips, g0 + lane) : -1, s_max[lane]);
  }
}

// ------------------------------------------------------------------------------------------------
// K2: top_db floor + DCT-II (first n_mfcc) + per-clip moments.  LANES ARE FRAMES: a warp transposes
// a tile of 32 dB rows into shared memory (coalesced 128-byte reads, pitch 33), then every lane runs
// the DCT of its own frame - per mel one conflict-free shared load of the dB value and KP/4 broadcast
// 128-bit loads of the coefficient row feed KP FFMAs.  MFCC rows leave through shared memory as one
// contiguous, fully coalesced block; sum x and sum x^2 are warp-reduced per tile and added in f64.
// ------------------------------------------------------------------------------------------------
constexpr int kDctWarps = 4;
constexpr int kDctPitch = 33;

template <int KP>
__global__ void __launch_bounds__(kDctWarps * 32) k_dct_sum(DeviceTables t, BatchView b,
                                                            const float* __restrict__ db,
                                                            const uint32_t* __restrict__ dbmax_key,
                                                            float* __restrict__ mfcc_raw,
                                                            double* __restrict__ sum,
                                                            double* __restrict__ sumsq) {
  extern __shared__ __align__(16) float s_dctk[];   // [n_mels][KP] coefficients, then kDctWarps x [n_mels][33]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_c = s_dctk;
  float* s_t = s_dctk + t.n_mels * KP + static_cast<size_t>(warp) * t.n_mels * kDctPitch;
  for (int i = threadIdx.x; i < t.n_mels * KP; i += blockDim.x) {
    const int m = i / KP, k = i - m * KP;
    s_c[i] = __ldg(t.dct_t + m * 32 + k);          // dct_t is [m][32], zero padded beyond n_mfcc
  }
  __syncthreads();
  const int64_t n_tiles = (b.total_frames + 31) / 32;
  for (int64_t tile = static_cast<int64_t>(blockIdx.x) * kDctWarps + warp; tile < n_tiles;
       tile += static_cast<int64_t>(gridDim.x) * kDctWarps) {
    const int64_t g0 = tile * 32;
    const int nf = static_cast<int>(min(static_cast<int64_t>(32), b.total_frames - g0));
    const bool valid = lane < nf;
    const int clip = valid ? find_segment(b.frame_off, b.n_clips, g0 + lane) : -1;
    const float floor_db = valid ? key_float(__ldg(dbmax_key + clip)) - 80.0f : 0.0f;
    // transposing load, 8 rows (up to 32 independent 128-byte requests per warp) at a time
    for (int f0 = 0; f0 < 32; f0 += 8) {
      float v[8][4];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int m = lane + 32 * j;
          v[r][j] = (f0 + r < nf && m < t.n_mels) ? __ldg(db + (g0 + f0 + r) * t.n_mels + m) : 0.0f;
        }
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int m = lane + 32 * j;
          if (m < t.n_mels) s_t[m * kDctPitch + f0 + r] = v[r][j];
        }
    }
    __syncwarp();
    float acc[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) acc[k] = 0.0f;
#pragma unroll 2
    for (int m = 0; m < t.n_mels; ++m) {
      const float x = fmaxf(s_t[m * kDctPitch + lane], floor_db);
      const float4* c4 = reinterpret_cast<const float4*>(s_c + m * KP);
#pragma unroll
      for (int k4 = 0; k4 < KP / 4; ++k4) {
        const float4 c = c4[k4];
        acc[4 * k4 + 0] = fmaf(c.x, x, acc[4 * k4 + 0]);
        acc[4 * k4 + 1] = fmaf(c.y, x, acc[4 * k4 + 1]);
        acc[4 * k4 + 2] = fmaf(c.z, x, acc[4 * k4 + 2]);
        acc[4 * k4 + 3] = fmaf(c.w, x, acc[4 * k4 + 3]);
      }
    }
    __syncwarp();
    // MFCC rows of the tile are one contiguous block of nf * n_mfcc floats
    float* s_o = s_t;
#pragma unroll
    for (int k = 0; k < KP; ++k)
      if (k < t.n_mfcc) s_o[lane * t.n_mfcc + k] = acc[k];
    __syncwarp();
    for (int i = lane; i < nf * t.n_mfcc; i += 32) mfcc_raw[g0 * t.n_mfcc + i] = s_o[i];
    // moments
    const int first_clip = __shfl_sync(0xffffffffu, clip, 0);
    const bool uniform = __all_sync(0xffffffffu, clip == first_clip || clip < 0);
    if (uniform) {
      // float64 reductions: the mean of a constant channel must come out exact (silence -> all-zero rows)
      double my_s = 0.0, my_q = 0.0;
#pragma unroll
      for (int k = 0; k < KP; ++k) {
        if (k < t.n_mfcc) {
          const double a = valid ? static_cast<double>(acc[k]) : 0.0;
          double ts = a, tq = a * a;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            ts += __shfl_xor_sync(0xffffffffu, ts, o);
            tq += __shfl_xor_sync(0xffffffffu, tq, o);
          }
          if (lane == k) { my_s = ts; my_q = tq; }
        }
      }
      if (lane < t.n_mfcc && first_clip >= 0) {
        atomicAdd(sum + static_cast<int64_t>(first_clip) * t.n_mfcc + lane, my_s);
        atomicAdd(sumsq + static_cast<int64_t>(first_clip) * t.n_mfcc + lane, my_q);
      }
    } else if (valid) {                              // tile straddles a clip boundary: per-frame adds
#pragma unroll
      for (int k = 0; k < KP; ++k)
        if (k < t.n_mfcc) {
          const double a = static_cast<double>(acc[k]);
          atomicAdd(sum + static_cast<int64_t>(clip) * t.n_mfcc + k, a);
          atomicAdd(sumsq + static_cast<int64_t>(clip) * t.n_mfcc + k, a * a);
        }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// K2 (product variant): the same arithmetic with LANES = FRAMES and NO transposition tile.  Each lane
// reads its own dB row with 128-bit loads (a warp request touches 32 rows; the seven later requests
// to the same 128-byte lines hit in L1, which is nearly all free here because the kernel needs only
// 15 KB of shared memory) and feeds KP FFMAs per mel from broadcast 128-bit coefficient loads.  Without
// the 17 KB tile per warp the SM holds 16 warps instead of 8, which is what hides the memory latency
// (k_dct_sum: 0.131 ms on C2, long-scoreboard bound).  Accumulation order over the mels is identical
// to k_dct_sum, so the MFCCs are bit-identical; the per-clip moments are summed over the 32 frames of a
// tile by lane k (float64, one column each) from the staged output rows.
// ------------------------------------------------------------------------------------------------
constexpr int kDct2Warps = 8;

template <int KP>
__global__ void __launch_bounds__(kDct2Warps * 32, 2) k_dct_rows(DeviceTables t, BatchView b,
                                                                 const float* __restrict__ db,
                                                                 const uint32_t* __restrict__ dbmax_key,
                                                                 float* __restrict__ mfcc_raw,
                                                                 double* __restrict__ sum,
                                                                 double* __restrict__ sumsq) {
  extern __shared__ __align__(16) float s_dctk[];   // [n_mels][KP] coefficients, then kDct2Warps x [32][n_mfcc]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_c = s_dctk;
  float* s_o = s_dctk + t.n_mels * KP + static_cast<size_t>(warp) * 32 * t.n_mfcc;
  for (int i = threadIdx.x; i < t.n_mels * KP; i += blockDim.x) {
    const int m = i / KP, k = i - m * KP;
    s_c[i] = __ldg(t.dct_t + m * 32 + k);          // dct_t is [m][32], zero padded beyond n_mfcc
  }
  __syncthreads();
  const int64_t n_tiles = (b.total_frames + 31) / 32;
  const int nq = t.n_mels >> 2;                     // n_mels is a multiple of 4 (checked by the launcher)
  for (int64_t tile = static_cast<int64_t>(blockIdx.x) * kDct2Warps + warp; tile < n_tiles;
       tile += static_cast<int64_t>(gridDim.x) * kDct2Warps) {
    const int64_t g0 = tile * 32;
    const int nf = static_cast<int>(min(static_cast<int64_t>(32), b.total_frames - g0));
    const bool valid = lane < nf;
    const int clip = valid ? find_segment(b.frame_off, b.n_clips, g0 + lane) : -1;
    const float floor_db = valid ? key_float(__ldg(dbmax_key + clip)) - 80.0f : 0.0f;
    const float4* row = reinterpret_cast<const float4*>(db + (g0 + (valid ? lane : 0)) * t.n_mels);
    float acc[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) acc[k] = 0.0f;
#pragma unroll 1
    for (int q0 = 0; q0 < nq; q0 += 4) {
      float4 x4[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) x4[u] = q0 + u < nq ? __ldg(row + q0 + u) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (q0 + u < nq) {
          const float xs[4] = {x4[u].x, x4[u].y, x4[u].z, x4[u].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float x = fmaxf(xs[e], floor_db);
            const float4* c4 = reinterpret_cast<const float4*>(s_c + (4 * (q0 + u) + e) * KP);
#pragma unroll
            for (int k4 = 0; k4 < KP / 4; ++k4) {
              const float4 c = c4[k4];
              acc[4 * k4 + 0] = fmaf(c.x, x, acc[4 * k4 + 0]);
              acc[4 * k4 + 1] = fmaf(c.y, x, acc[4 * k4 + 1]);
              acc[4 * k4 + 2] = fmaf(c.z, x, acc[4 * k4 + 2]);
              acc[4 * k4 + 3] = fmaf(c.w, x, acc[4 * k4 + 3]);
            }
          }
        }
      }
    }
    // MFCC rows of the tile are one contiguous block of nf * n_mfcc floats: stage, then coalesced stores
#pragma unroll
    for (int k = 0; k < KP; ++k)
      if (k < t.n_mfcc) s_o[lane * t.n_mfcc + k] = valid ? acc[k] : 0.0f;
    __syncwarp();
    for (int i = lane; i < nf * t.n_mfcc; i += 32) mfcc_raw[g0 * t.n_mfcc + i] = s_o[i];
    // moments
    const int first_clip = __shfl_sync(0xffffffffu, clip, 0);
    const bool uniform = __all_sync(0xffffffffu, clip == first_clip || clip < 0);
    if (uniform) {
      // float64 sums: the mean of a constant channel must come out exact (silence -> all-zero rows)
      if (lane < t.n_mfcc && first_clip >= 0) {
        double ts = 0.0, tq = 0.0;
        for (int f = 0; f < nf; ++f) {
          const double a = static_cast<double>(s_o[f * t.n_mfcc + lane]);
          ts += a;
          tq = fma(a, a, tq);
        }
        atomicAdd(sum + static_cast<int64_t>(first_clip) * t.n_mfcc + lane, ts);
        atomicAdd(sumsq + static_cast<int64_t>(first_clip) * t.n_mfcc + lane, tq);
      }
    } else if (valid) {                              // tile straddles a clip boundary: per-frame adds
#pragma unroll
      for (int k = 0; k < KP; ++k)
        if (k < t.n_mfcc) {
          const double a = static_cast<double>(acc[k]);
          atomicAdd(sum + static_cast<int64_t>(clip) * t.n_mfcc + k, a);
          atomicAdd(sumsq + static_cast<int64_t>(clip) * t.n_mfcc + k, a * a);
        }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// K2 on the tensor pipe: the DCT-II of the default shape (128 mels -> 23 coefficients) as warp-level MMAs
// (mma.sync m16n8k16, fp16 split operands, fp32 accumulation).  north_star lists the DCT among the dense contractions
// that belong on tensor cores; as FFMAs it costs 2944 instructions per frame (round 2's constant-bank FFMA kernel:
// issue bound at 0.46 of the HBM roofline), as MMAs 4.5 per frame: [32 frames x 128] x [128 x 24] per warp tile =
// 8 k-steps x 2 row tiles x 3 column tiles x 3 split products.
//   A  floored dB rows, CENTRED per row: x' = max(x, clip_max - 80) - (clip_max - 40) lies in [-40, 40], so the fp16
//      hi + lo split carries 2^-22 x 64 = 1.5e-5 of absolute error per element instead of 3e-5 at |x| ~ 100.  The
//      offset only reaches coefficient 0 (the other DCT rows sum to zero) and is added back there in float32.
//   B  the DCT matrix scaled by 2^10 (exact), pre-split on the host into hi / lo and laid out in fragment order
//      (one 64-bit shared-memory load per lane, k-step, column tile and part).
// hi.hi + hi.lo + lo.hi: fp32-class like the other split GEMMs of the path.  Staging, store and the float64 CMVN
// moments are those of k_dct_rows.
// ------------------------------------------------------------------------------------------------
constexpr int kDctMmaFragWords = 8 * 3 * 2 * 32 * 2;      // [k-step][column tile][hi, lo][lane] x {b0, b1}
constexpr float kDctMmaScale = 1024.0f;

__device__ __forceinline__ void dct_mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// (x0, x1) -> packed fp16 hi pair and lo pair
__device__ __forceinline__ void dct_split(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

__global__ void __launch_bounds__(kDct2Warps * 32, 3) k_dct_mma(const uint2* __restrict__ frag, BatchView b,
                                                                const float* __restrict__ db,
                                                                const uint32_t* __restrict__ dbmax_key,
                                                                float* __restrict__ mfcc_raw,
                                                                double* __restrict__ sum, double* __restrict__ sumsq) {
  constexpr int NM = kDctMmaMels, NC = kDctMmaMfcc;
  __shared__ uint2 s_frag[kDctMmaFragWords / 2];
  __shared__ float s_stage[kDct2Warps * 32 * NC];
  for (int i = threadIdx.x; i < kDctMmaFragWords / 2; i += blockDim.x) s_frag[i] = __ldg(frag + i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, tq = lane & 3;
  float* s_o = s_stage + warp * 32 * NC;
  const int64_t n_tiles = (b.total_frames + 31) / 32;
  for (int64_t tile = static_cast<int64_t>(blockIdx.x) * kDct2Warps + warp; tile < n_tiles;
       tile += static_cast<int64_t>(gridDim.x) * kDct2Warps) {
    const int64_t g0 = tile * 32;
    const int nf = static_cast<int>(min(static_cast<int64_t>(32), b.total_frames - g0));
    const bool valid = lane < nf;
    const int clip = valid ? find_segment(b.frame_off, b.n_clips, g0 + lane) : -1;
    const float floor_db = valid ? key_float(__ldg(dbmax_key + clip)) - 80.0f : 0.0f;   // of row `lane`
    // the four rows this lane feeds: g, g + 8 (row tile 0), g + 16, g + 24 (row tile 1)
    float fl[4];
    const float* rowp[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int r = g + 8 * q;
      fl[q] = __shfl_sync(0xffffffffu, floor_db, r);
      rowp[q] = db + (g0 + (r < nf ? r : 0)) * NM + 2 * tq;     // rows beyond the batch re-read row 0 (discarded)
    }
    float acc[2][3][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 3; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[mt][nt][c] = 0.0f;
#pragma unroll
    for (int ks = 0; ks < NM / 16; ++ks) {
      uint32_t ah[2][4], al[2][4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 x0 = __ldg(reinterpret_cast<const float2*>(rowp[q] + 16 * ks));        // k = 2 tq, 2 tq + 1
        const float2 x1 = __ldg(reinterpret_cast<const float2*>(rowp[q] + 16 * ks + 8));    // k + 8
        const float off = fl[q] + 40.0f;
        const int mt = q >> 1, h = q & 1;        // fragment registers: a0 = (row g, k), a1 = (row g+8, k), a2 / a3 = k + 8
        dct_split(fmaxf(x0.x, fl[q]) - off, fmaxf(x0.y, fl[q]) - off, ah[mt][h], al[mt][h]);
        dct_split(fmaxf(x1.x, fl[q]) - off, fmaxf(x1.y, fl[q]) - off, ah[mt][h + 2], al[mt][h + 2]);
      }
#pragma unroll
      for (int nt = 0; nt < 3; ++nt) {
        const uint2 bh = s_frag[((ks * 3 + nt) * 2 + 0) * 32 + lane];
        const uint2 bl = s_frag[((ks * 3 + nt) * 2 + 1) * 32 + lane];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          dct_mma_16816(acc[mt][nt], ah[mt], bh.x, bh.y);
          dct_mma_16816(acc[mt][nt], ah[mt], bl.x, bl.y);
          dct_mma_16816(acc[mt][nt], al[mt], bh.x, bh.y);
        }
      }
    }
    // accumulator (c0, c1) = (row g, columns 2 tq, 2 tq + 1) of the column tile, (c2, c3) = row g + 8
    const float inv_scale = 1.0f / kDctMmaScale;
    const float sum_row0 = 11.313708498984761f;                // sum_m D[0][m] = 128 / sqrt(128)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 3; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int q = 2 * mt + (c >> 1);
          const int row = g + 8 * q, col = 8 * nt + 2 * tq + (c & 1);
          float v = acc[mt][nt][c] * inv_scale;
          if (col == 0) v = fmaf(fl[q] + 40.0f, sum_row0, v);
          if (col < NC) s_o[row * NC + col] = row < nf ? v : 0.0f;
        }
    __syncwarp();
    for (int i = lane; i < nf * NC; i += 32) mfcc_raw[g0 * NC + i] = s_o[i];
    const int first_clip = __shfl_sync(0xffffffffu, clip, 0);
    const bool uniform = __all_sync(0xffffffffu, clip == first_clip || clip < 0);
    if (uniform) {
      if (lane < NC && first_clip >= 0) {
        double ts = 0.0, tq2 = 0.0;
        for (int f = 0; f < nf; ++f) {
          const double a = static_cast<double>(s_o[f * NC + lane]);
          ts += a;
          tq2 = fma(a, a, tq2);
        }
        atomicAdd(sum + static_cast<int64_t>(first_clip) * NC + lane, ts);
        atomicAdd(sumsq + static_cast<int64_t>(first_clip) * NC + lane, tq2);
      }
    } else if (valid) {
      for (int k = 0; k < NC; ++k) {
        const double a = static_cast<double>(s_o[lane * NC + k]);
        atomicAdd(sum + static_cast<int64_t>(clip) * NC + k, a);
        atomicAdd(sumsq + static_cast<int64_t>(clip) * NC + k, a * a);
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// K3: CMVN -> Savitzky-Golay delta / delta-delta (width 9, edges = value at frame 4 / T-5)
//     -> pair reduction.  Thread per (output row, channel).
//     extract_features_utils.py:5-8,21-27,33-44; librosa.feature.delta == scipy savgol 'interp'.
// ------------------------------------------------------------------------------------------------
// Savitzky-Golay taps on nine consecutive frames x[0..8]:
//   delta  = sum k x[k] / 60,  delta2 = [28 7 -8 -17 -20 -17 -8 7 28] . x / 462
__device__ __forceinline__ float sg_d1(const float* x) {
  return (4.0f * (x[8] - x[0]) + 3.0f * (x[7] - x[1]) + 2.0f * (x[6] - x[2]) + (x[5] - x[3])) * (1.0f / 60.0f);
}
__device__ __forceinline__ float sg_d2(const float* x) {
  return (28.0f * (x[0] + x[8]) + 7.0f * (x[1] + x[7]) - 8.0f * (x[2] + x[6]) - 17.0f * (x[3] + x[5]) -
          20.0f * x[4]) * (1.0f / 462.0f);
}

// One warp per output row, lanes over channels.  CMVN is affine and the filters are linear, so the
// deltas are taken on the mean-centred values and scaled by 1 / (sigma + 1e-10) once; the two frames of a row
// share nine of their ten taps, so an interior row costs ten coalesced loads per lane.
__global__ void __launch_bounds__(256, 3) k_delta_reduce(BatchView b, const float* __restrict__ in, int C,
                                                         int in_ld, const double* __restrict__ sum,
                                                         const double* __restrict__ sumsq, bool cmvn,
                                                         bool deltas, bool reduce,
                                                         float* __restrict__ out, int64_t out_ld,
                                                         int col0) {
  const int rows_per_block = blockDim.x / 32;
  const int lane = threadIdx.x & 31, wr = threadIdx.x >> 5;
  // every warp owns a CONTIGUOUS run of rows: consecutive rows share eight of their ten taps (L1 hits)
  // and almost always the clip, so the float64 CMVN constants of a (clip, channel) are formed once per
  // run instead of once per row
  const int64_t n_warps = static_cast<int64_t>(gridDim.x) * rows_per_block;
  const int64_t chunk = (b.total_rows + n_warps - 1) / n_warps;
  const int64_t r_begin = (static_cast<int64_t>(blockIdx.x) * rows_per_block + wr) * chunk;
  const int64_t r_end = min(r_begin + chunk, b.total_rows);
  int cached_clip = -1;
  float cached_mu = 0.0f, cached_inv = 1.0f;       // channel `lane` of cached_clip
  float win[10];                                   // frames win_ta-4 .. win_ta+5 of clip win_clip, channel `lane`
  int win_clip = -1;
  int64_t win_ta = 0;
#pragma unroll
  for (int k = 0; k < 10; ++k) win[k] = 0.0f;
  // clip of the current row: looked up only when the run crosses into the next clip (the lookup is a chain
  // of dependent loads - most of a row's latency when it is repeated per row)
  int clip = -1;
  int64_t f0 = 0, T = 0, clip_row0 = 0, clip_row_end = -1;
  double inv_T = 0.0;                              // 1 / T of the current clip (a float64 division: once per clip, not per row)
  for (int64_t r = r_begin; r < r_end; ++r) {
    if (r >= clip_row_end) {
      clip = find_segment(b.row_off, b.n_clips, r);
      f0 = __ldg(b.frame_off + clip);
      T = __ldg(b.frame_off + clip + 1) - f0;
      clip_row0 = __ldg(b.row_off + clip);
      clip_row_end = __ldg(b.row_off + clip + 1);
      inv_T = cmvn ? 1.0 / static_cast<double>(T) : 0.0;
    }
    const int64_t lr = r - clip_row0;
    const int64_t ta = reduce ? 2 * lr : lr;
    const bool pair = reduce && (ta + 1 < T);
    // window centres (edges replicate the value at frame 4 / T-5: savgol mode='interp')
    const int64_t ca = min(max(ta, static_cast<int64_t>(4)), T - 5);
    const int64_t cb = min(max(ta + 1, static_cast<int64_t>(4)), T - 5);
    const bool shared_taps = pair && cb == ca + 1;
    // Fast path (MFCC block: C <= 32, deltas, pair reduction): an interior row's two windows are the ten
    // consecutive frames ta-4 .. ta+5, and the next row's are the same ten shifted by two - the lane keeps
    // them in registers and fetches only the two new frames per row.  Same arithmetic, same order as below.
    const bool interior = deltas && pair && C <= 32 && ta >= 4 && ta + 1 <= T - 5;
    // Four interior rows at once when the window continues and rows r .. r + 3 are all interior rows of this run: the
    // eight frames they add are requested together.  One row at a time keeps two 92-byte loads in flight per warp -
    // ~5 KB per SM, i.e. memory-level parallelism, not bandwidth or arithmetic, set the kernel's time (half of its
    // stall samples on the first use of the two loads; requesting them one row ahead changed 3 %).  Same arithmetic
    // per row in the same order: identical rows.
    if (interior && win_clip == clip && win_ta + 2 == ta && r + 3 < r_end && ta + 12 <= T) {
      const int ch = lane;
      if (ch < C) {
        const float mu = cmvn ? cached_mu : 0.0f, inv = cmvn ? cached_inv : 1.0f;    // win_clip == clip: constants are cached
        const float* p = in + (f0 + ta - 4) * in_ld + ch;
        float w[16];                                  // frames ta - 4 .. ta + 11, centred
#pragma unroll
        for (int k = 0; k < 8; ++k) w[8 + k] = __ldg(p + (8 + k) * in_ld);
#pragma unroll
        for (int k = 0; k < 8; ++k) w[k] = win[k + 2];
#pragma unroll
        for (int k = 8; k < 16; ++k) w[k] -= mu;
        float* o = out + r * out_ld + col0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float* x = w + 2 * j;
          const float va = 0.5f * (x[4] * inv + x[5] * inv);
          const float d1 = 0.5f * (sg_d1(x) + sg_d1(x + 1)) * inv;
          const float d2 = 0.5f * (sg_d2(x) + sg_d2(x + 1)) * inv;
          o[j * out_ld + ch] = va;
          o[j * out_ld + C + ch] = d1;
          o[j * out_ld + 2 * C + ch] = d2;
        }
#pragma unroll
        for (int k = 0; k < 10; ++k) win[k] = w[6 + k];
      }
      win_ta = ta + 6;
      r += 3;
      continue;
    }
    if (interior) {
      const int ch = lane;
      if (ch < C) {
        float mu = 0.0f, inv = 1.0f;
        if (cmvn) {
          if (clip == cached_clip) {
            mu = cached_mu;
            inv = cached_inv;
          } else {
            const double m = __ldg(sum + static_cast<int64_t>(clip) * C + ch) * inv_T;
            const double var = fmax(0.0, fma(__ldg(sumsq + static_cast<int64_t>(clip) * C + ch), inv_T, -m * m));
            mu = static_cast<float>(m);
            inv = __fdiv_rn(1.0f, sqrtf(static_cast<float>(var)) + 1e-10f);
            cached_mu = mu; cached_inv = inv;
          }
        }
        // the window holds CENTRED values (x - mu, formed once when a frame is loaded: constants give exact 0);
        // it is dropped whenever the clip - and with it mu - changes
        const float* p = in + (f0 + ta - 4) * in_ld + ch;
        if (win_clip == clip && win_ta + 2 == ta) {
#pragma unroll
          for (int k = 0; k < 8; ++k) win[k] = win[k + 2];
          win[8] = __ldg(p + 8 * in_ld) - mu;
          win[9] = __ldg(p + 9 * in_ld) - mu;
        } else {
#pragma unroll
          for (int k = 0; k < 10; ++k) win[k] = __ldg(p + k * in_ld) - mu;
        }
        const float va = 0.5f * (win[4] * inv + win[5] * inv);
        const float d1 = 0.5f * (sg_d1(win) + sg_d1(win + 1)) * inv;
        const float d2 = 0.5f * (sg_d2(win) + sg_d2(win + 1)) * inv;
        float* o = out + r * out_ld + col0;
        o[ch] = va;
        o[C + ch] = d1;
        o[2 * C + ch] = d2;
      }
      win_clip = clip;
      win_ta = ta;
      cached_clip = clip;
      continue;
    }
    win_clip = -1;
    for (int ch = lane; ch < C; ch += 32) {
      float mu = 0.0f, inv = 1.0f;
      if (cmvn) {
        if (ch == lane && clip == cached_clip) {
          mu = cached_mu;
          inv = cached_inv;
        } else {
          const double m = __ldg(sum + static_cast<int64_t>(clip) * C + ch) * inv_T;
          // population variance from the float64 moments (sum x, sum x^2) of the float32 values
          const double var = fmax(0.0, fma(__ldg(sumsq + static_cast<int64_t>(clip) * C + ch), inv_T, -m * m));
          mu = static_cast<float>(m);
          inv = __fdiv_rn(1.0f, sqrtf(static_cast<float>(var)) + 1e-10f);   // float32 std + 1e-10
          if (ch == lane) { cached_mu = mu; cached_inv = inv; }
        }
      }
      const float* col = in + f0 * in_ld + ch;
      float va = (__ldg(col + ta * in_ld) - mu) * inv, d1 = 0.0f, d2 = 0.0f;
      if (pair) va = 0.5f * (va + (__ldg(col + (ta + 1) * in_ld) - mu) * inv);
      if (deltas) {
        float xa[9];
        const float* pa = col + (ca - 4) * in_ld;
#pragma unroll
        for (int k = 0; k < 9; ++k) xa[k] = __ldg(pa + k * in_ld) - mu;   // centred: constants give exact 0
        d1 = sg_d1(xa);
        d2 = sg_d2(xa);
        if (pair) {
          float xb[9];
          if (shared_taps) {                         // interior row: nine of the ten taps are shared
#pragma unroll
            for (int k = 0; k < 8; ++k) xb[k] = xa[k + 1];
            xb[8] = __ldg(pa + 9 * in_ld) - mu;
          } else if (cb == ca) {                     // both frames clamp to the same edge window
#pragma unroll
            for (int k = 0; k < 9; ++k) xb[k] = xa[k];
          } else {
            const float* pb = col + (cb - 4) * in_ld;
#pragma unroll
            for (int k = 0; k < 9; ++k) xb[k] = __ldg(pb + k * in_ld) - mu;
          }
          d1 = 0.5f * (d1 + sg_d1(xb));
          d2 = 0.5f * (d2 + sg_d2(xb));
        }
        d1 *= inv;
        d2 *= inv;
      }
      float* o = out + r * out_ld + col0;
      o[ch] = va;
      if (deltas) {
        o[C + ch] = d1;
        o[2 * C + ch] = d2;
      }
    }
    cached_clip = clip;
  }
}

// ------------------------------------------------------------------------------------------------
// K4: autocorrelation.  One warp per output row (frame pair).  The mean-removed, Hann-windowed
// frame lives in shared memory; lane (g, q) accumulates 12 lags [12q, 12q+12) over half of the
// frame (g) with a sliding register window: 48 FMAs per two 128-bit shared loads.
// ------------------------------------------------------------------------------------------------
constexpr int kAcWarps = 8;
constexpr int kAcLagsPerLane = 12;
constexpr int kAcTail = 16 * kAcLagsPerLane + 16;  // zero tail so x[n + lag] never leaves the row

struct AcGeom { int half; int row_floats; };  // half = samples per n-group (multiple of 16)
__host__ __device__ inline AcGeom ac_geom(int F) {
  AcGeom g;
  g.half = (((F + 1) / 2) + 15) / 16 * 16;
  g.row_floats = 2 * g.half + kAcTail;
  return g;
}

// Computes normalised lags of hop-frame tf into acc[0..11] of lanes with g == 0 (lag = 12 q + j);
// returns r[0]-normalised values; lane (0,0)'s acc[0] is lag 0 (== 1 or 0).
__device__ __forceinline__ void autocorr_frame(const DeviceTables& t, const float* __restrict__ y,
                                               int64_t base, int64_t len, int64_t tf, float* xs,
                                               const float* __restrict__ hann, const AcGeom& geo, int lane,
                                               float (&acc)[kAcLagsPerLane]) {
  const int F = t.F;
  const int64_t first = tf * t.H - t.pad;
  // pass 1: load with np.pad(..., mode='reflect') indexing, accumulate the mean
  float part = 0.0f;
  if (first >= 0 && first + F <= len) {          // interior frame: plain coalesced loads, 16 in flight
    const float* src = y + base + first;
    for (int n0 = lane; n0 < F; n0 += 32 * 8) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = (n0 + 32 * k < F) ? __ldg(src + n0 + 32 * k) : 0.0f;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (n0 + 32 * k < F) { xs[n0 + 32 * k] = v[k]; part += v[k]; }
    }
  } else {
    for (int n = lane; n < F; n += 32) {
      int64_t i = first + n;
      if (i < 0) i = -i;
      if (i >= len) i = 2 * (len - 1) - i;
      const float v = __ldg(y + base + i);
      xs[n] = v;
      part += v;
    }
  }
  const float mean = warp_sum(part) / static_cast<float>(F);
  __syncwarp();
#pragma unroll 4
  for (int n = lane; n < F; n += 32) xs[n] = (xs[n] - mean) * __ldg(hann + n);
  for (int n = F + lane; n < geo.row_floats; n += 32) xs[n] = 0.0f;
  __syncwarp();

  const int g = lane >> 4, q = lane & 15;
#pragma unroll
  for (int j = 0; j < kAcLagsPerLane; ++j) acc[j] = 0.0f;
  const float* xa = xs + g * geo.half;                 // x[n]
  const float* xw = xa + q * kAcLagsPerLane;           // x[n + lag0 + ...], 16-byte aligned
  float4 w[4];
  w[0] = *reinterpret_cast<const float4*>(xw);
  w[1] = *reinterpret_cast<const float4*>(xw + 4);
  w[2] = *reinterpret_cast<const float4*>(xw + 8);
  for (int n = 0; n < geo.half; n += 16) {
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      const float4 a = *reinterpret_cast<const float4*>(xa + n + 4 * s);
      w[(s + 3) & 3] = *reinterpret_cast<const float4*>(xw + n + 4 * s + 12);
      const float av[4] = {a.x, a.y, a.z, a.w};
      float wv[16];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 ww = w[(s + k) & 3];
        wv[4 * k + 0] = ww.x; wv[4 * k + 1] = ww.y; wv[4 * k + 2] = ww.z; wv[4 * k + 3] = ww.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < kAcLagsPerLane; ++j) acc[j] = fmaf(av[i], wv[i + j], acc[j]);
    }
  }
  // combine the two n-groups, normalise by lag 0 when it is non-zero
#pragma unroll
  for (int j = 0; j < kAcLagsPerLane; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
  const float r0 = __shfl_sync(0xffffffffu, acc[0], 0);
  if (r0 != 0.0f) {
    const float inv = __fdiv_rn(1.0f, r0);       // one division per frame; the products are within 1 ulp
#pragma unroll
    for (int j = 0; j < kAcLagsPerLane; ++j) acc[j] *= inv;
  }
  __syncwarp();
}

// true when every kept coefficient (lags 1..n_lags) is below the 1e-7 threshold
__device__ __forceinline__ bool ac_all_small(const float (&acc)[kAcLagsPerLane], int lane, int n_lags, float thr) {
  const int q = lane & 15;
  bool small = true;
#pragma unroll
  for (int j = 0; j < kAcLagsPerLane; ++j) {
    const int lag = q * kAcLagsPerLane + j;
    if (lag >= 1 && lag <= n_lags && !(fabsf(acc[j]) < thr)) small = false;
  }
  return __all_sync(0xffffffffu, small);
}

__global__ void __launch_bounds__(kAcWarps * 32, 4) k_autocorr(DeviceTables t, BatchView b,
                                                            const float* __restrict__ y, bool reduce,
                                                            float* __restrict__ out, int64_t out_ld,
                                                            int col0) {
  extern __shared__ __align__(16) float s_ac[];
  const AcGeom geo = ac_geom(t.F);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* xs = s_ac + static_cast<size_t>(warp) * geo.row_floats;
  const float* hann = t.hann_sym;                                        // L1-resident read-only table
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * kAcWarps + warp; r < b.total_rows;
       r += static_cast<int64_t>(gridDim.x) * kAcWarps) {
    const int clip = find_segment(b.row_off, b.n_clips, r);
    const int64_t base = __ldg(b.clip_off + clip);
    const int64_t len = __ldg(b.clip_off + clip + 1) - base;
    const int64_t T = __ldg(b.frame_off + clip + 1) - __ldg(b.frame_off + clip);
    const int64_t lr = r - __ldg(b.row_off + clip);
    float va[kAcLagsPerLane], vb[kAcLagsPerLane];
    if (reduce) {
      const int64_t ta = 2 * lr;
      const bool pair = ta + 1 < T;
      autocorr_frame(t, y, base, len, ta, xs, hann, geo, lane, va);
      if (pair) {
        autocorr_frame(t, y, base, len, ta + 1, xs, hann, geo, lane, vb);
        // fix_edge_frames_autocorr: first frame copies frame 1, last frame copies frame T-2
        if (ta == 0 && ac_all_small(va, lane, t.n_lags, t.edge_thr)) {
#pragma unroll
          for (int j = 0; j < kAcLagsPerLane; ++j) va[j] = vb[j];
        }
        if (ta + 1 == T - 1 && ac_all_small(vb, lane, t.n_lags, t.edge_thr)) {
#pragma unroll
          for (int j = 0; j < kAcLagsPerLane; ++j) vb[j] = va[j];
        }
#pragma unroll
        for (int j = 0; j < kAcLagsPerLane; ++j) va[j] = 0.5f * (va[j] + vb[j]);
      } else if (ta == T - 1 && ac_all_small(va, lane, t.n_lags, t.edge_thr)) {
        autocorr_frame(t, y, base, len, T - 2, xs, hann, geo, lane, va);  // odd T: last row passes through
      }
    } else {
      autocorr_frame(t, y, base, len, lr, xs, hann, geo, lane, va);
      if (lr == 0 && ac_all_small(va, lane, t.n_lags, t.edge_thr)) {
        autocorr_frame(t, y, base, len, 1, xs, hann, geo, lane, va);
      } else if (lr == T - 1 && ac_all_small(va, lane, t.n_lags, t.edge_thr)) {
        autocorr_frame(t, y, base, len, T - 2, xs, hann, geo, lane, va);
      }
    }
    if (lane < 16) {
      float* o = out + r * out_ld + col0;
#pragma unroll
      for (int j = 0; j < kAcLagsPerLane; ++j) {
        const int lag = lane * kAcLagsPerLane + j;
        if (lag >= 1 && lag <= t.n_lags) o[lag - 1] = va[j];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// smooth_features: row i <- (row i-1 + row i) / 2 inside each clip (from the original rows)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_smooth(BatchView b, const float* __restrict__ in,
                                                int64_t in_ld, int cols, float* __restrict__ out,
                                                int64_t out_ld) {
  for (int64_t r = blockIdx.x; r < b.total_rows; r += gridDim.x) {
    const int clip = find_segment(b.row_off, b.n_clips, r);
    const bool first = (r == __ldg(b.row_off + clip));
    for (int c = threadIdx.x; c < cols; c += blockDim.x) {
      const float cur = in[r * in_ld + c];
      out[r * out_ld + c] = first ? cur : (in[(r - 1) * in_ld + c] + cur) * 0.5f;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// collect_features augmentation.  One warp per output row, every warp walking short runs of consecutive rows;
// the row's provenance (which version, blend weights) is resolved once, then the lanes stream the 256 + 61 columns.
// ------------------------------------------------------------------------------------------------
// np.linspace(start, stop, n)[i] exactly as numpy evaluates it (arange * step + start, endpoint set)
__device__ __forceinline__ double linspace_at(double start, double stop, int64_t n, int64_t i) {
  if (n == 1) return start;
  if (i == n - 1) return stop;
  const double step = (stop - start) / static_cast<double>(n - 1);
  return __dadd_rn(__dmul_rn(static_cast<double>(i), step), start);
}

// value of version `ver` at its row j, column c, for source matrix `src` (rows [s0, s0+n))
// ver 0: original, 1: fast rows[::2], 2: slow = interpolate_slower (+ smoothing when smooth_slow)
template <typename T>
__device__ __forceinline__ T version_value(const T* __restrict__ src, int64_t ld, int ver, int64_t j,
                                           int c, bool smooth_slow) {
  auto at = [&](int64_t row) { return src[row * ld + c]; };
  auto slow = [&](int64_t k) -> T {
    if ((k & 1) == 0) return at(k >> 1);
    return mul_rn(add_rn(at(k >> 1), at((k >> 1) + 1)), static_cast<T>(0.5));
  };
  if (ver == 0) return at(j);
  if (ver == 1) return at(2 * j);
  if (!smooth_slow || j == 0) return slow(j);
  return mul_rn(add_rn(slow(j - 1), slow(j)), static_cast<T>(0.5));  // smooth_facial_data
}

// float4 form of version_value for the float32 audio block (256 columns): four columns per lane and load,
// the same operations in the same order per component.
__device__ __forceinline__ float4 add4(float4 a, float4 b) {
  return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}
__device__ __forceinline__ float4 mul4(float4 a, float s) {
  return make_float4(__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s), __fmul_rn(a.w, s));
}
__device__ __forceinline__ float4 mul4s(float s, float4 a) {      // scalar first, like mul_rn(w, val)
  return make_float4(__fmul_rn(s, a.x), __fmul_rn(s, a.y), __fmul_rn(s, a.z), __fmul_rn(s, a.w));
}
__device__ __forceinline__ float4 version_value4(const float* __restrict__ src, int64_t ld, int ver, int64_t j,
                                                 int c4, bool smooth_slow) {
  auto at = [&](int64_t row) { return __ldg(reinterpret_cast<const float4*>(src + row * ld) + c4); };
  auto slow = [&](int64_t k) -> float4 {
    if ((k & 1) == 0) return at(k >> 1);
    return mul4(add4(at(k >> 1), at((k >> 1) + 1)), 0.5f);
  };
  if (ver == 0) return at(j);
  if (ver == 1) return at(2 * j);
  if (!smooth_slow || j == 0) return slow(j);
  return mul4(add4(slow(j - 1), slow(j)), 0.5f);
}

// The stack geometry of a clip (trim offsets, version lengths, blend zones) is derived once per clip and kept in
// registers - round 1's block-per-row kernel recomputed it, behind a chain of dependent loads, with all 128 threads
// of a block for every single row - and the lanes stream the 256 + 61 columns of the row with fully coalesced
// 128-byte requests.  add_rn / mul_rn, linspace_at and version_value keep the float64 variant bit-exact.
constexpr int kCollectRun = 4;      // consecutive rows per warp and tile
template <typename T>
__global__ void __launch_bounds__(256, 5) k_collect_rows(CollectView v, const T* __restrict__ audio, int a_cols,
                                                      const T* __restrict__ facial, int f_cols,
                                                      T* __restrict__ out_audio, T* __restrict__ out_facial) {
  const int lane = threadIdx.x & 31, wr = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  // Row order: the grid sweeps the output in TILES of wpb x kCollectRun consecutive rows (block b takes tiles b,
  // b + gridDim.x, ...; a warp takes kCollectRun consecutive rows of the tile), so at any time all resident warps
  // read and write ONE compact region (~25 MB) of each stream.  With one long run per warp (round 1 / early round 2)
  // the 5 920 resident warps touched 5 920 x 4 scattered 1 KB rows at a time: every access opened its own DRAM
  // page and the kernel sat at 30 % of the DRAM peak with all stalls on the loads (ncu, round 2).
  const int64_t tile_rows = static_cast<int64_t>(wpb) * kCollectRun;
  const int64_t n_tiles = (v.total_out_rows + tile_rows - 1) / tile_rows;
  int64_t clip_o0 = 0, clip_o_end = -1, a0 = 0, f0 = 0;
  int ver[3] = {0, 0, 0};
  int nv = 0;
  int64_t len_before[3] = {0, 0, 0}, nb[3] = {0, 0, 0};
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
  for (int64_t r = tile * tile_rows + static_cast<int64_t>(wr) * kCollectRun,
               r_end = min(r + kCollectRun, v.total_out_rows); r < r_end; ++r) {
    if (r >= clip_o_end || r < clip_o0) {
      const int clip = find_segment(v.o_off, v.n_clips, r);
      clip_o0 = __ldg(v.o_off + clip);
      clip_o_end = __ldg(v.o_off + clip + 1);
      a0 = __ldg(v.a_off + clip);
      f0 = __ldg(v.f_off + clip);
      const int64_t na = __ldg(v.a_off + clip + 1) - a0, nf = __ldg(v.f_off + clip + 1) - f0;
      // centre-trim the longer stream (data_processing.py:126-145)
      if (na > nf) a0 += (na - nf) / 2; else if (nf > na) f0 += (nf - na) / 2;
      const int64_t n = min(na, nf);
      // version lengths and blend zones (stack_with_blend, data_processing.py:179-197)
      int64_t vlen[3];
      nv = 0;
      ver[nv] = 0; vlen[nv++] = n;
      if (v.flags & NSF_COLLECT_FAST) { ver[nv] = 1; vlen[nv++] = (n + 1) / 2; }
      if (v.flags & NSF_COLLECT_SLOW) { ver[nv] = 2; vlen[nv++] = n > 0 ? 2 * n - 1 : 0; }
      const bool blend = (v.flags & NSF_COLLECT_BLEND) != 0;
      int64_t total = vlen[0];
      len_before[0] = 0; nb[0] = 0;
      for (int i = 1; i < nv; ++i) {
        int64_t k = blend ? min(min(static_cast<int64_t>(v.blend_frames), total), vlen[i]) : 0;
        if (k < 0) k = 0;
        len_before[i] = total; nb[i] = k;
        total += vlen[i] - k;
      }
    }
    const int64_t p = r - clip_o0;
    // Resolve row p by walking from the last stacked version down.  Level i of the stack is
    //   [ result_{i-1}[: L-k] | w1*result_{i-1}[L-k+q] + w2*V_i[q], q < k | V_i[k:] ],  L = len(result_{i-1})
    // so a row is one "terminal" version row plus at most two enclosing cross-fades.
    int term_ver = ver[0];
    int64_t term_row = p;
    int n_blend = 0, blend_level[2] = {0, 0};
    int64_t blend_q[2] = {0, 0};
    for (int level = nv - 1; level >= 1; --level) {
      const int64_t L = len_before[level], k = nb[level];
      if (p >= L) { term_ver = ver[level]; term_row = p - L + k; break; }
      if (p >= L - k) { blend_level[n_blend] = level; blend_q[n_blend] = p - (L - k); ++n_blend; }
    }
    if (sizeof(T) == 4 && n_blend == 0 && a_cols == 256 && f_cols <= 64) {
      // Rows outside the cross-fade zones (all but 2 x blend_frames per clip) of the float32 default shape: every
      // value is a fixed expression of at most TWO adjacent source rows of its stream -
      //   original / fast: at(r)        slow, odd row k: (at(k/2) + at(k/2 + 1)) / 2
      //   facial slow rows also carry smooth_facial_data: (slow(j-1) + slow(j)) / 2, again rows (j-1)/2 and (j-1)/2 + 1
      // so the row's eight loads (two float4 columns and two facial columns from two rows each) are issued back to
      // back and the warp pays ONE memory round trip per row instead of one per column group (ncu, round 2: 7 k cycles
      // per row, 30 % of the DRAM peak).  Same operations in the same order as version_value / version_value4.
      const float* asrc = reinterpret_cast<const float*>(audio) + a0 * 256;
      const float* fsrc = reinterpret_cast<const float*>(facial) + f0 * f_cols;
      int64_t ra = term_row, rf = term_row;      // first source row of the audio / facial expression
      int a_kind = 0, f_kind = 0;                // 0: at(r)   1: (at(r) + at(r+1)) / 2   facial 2, 3: smoothed slow rows
      if (term_ver == 1) { ra = 2 * term_row; rf = ra; }
      if (term_ver == 2) {
        ra = term_row >> 1;
        a_kind = static_cast<int>(term_row & 1);
        if (term_row == 0) { rf = 0; f_kind = 0; }
        else if (term_row & 1) { rf = term_row >> 1; f_kind = 2; }     // (at(p) + (at(p) + at(p+1)) / 2) / 2
        else { rf = (term_row >> 1) - 1; f_kind = 3; }                 // ((at(q-1) + at(q)) / 2 + at(q)) / 2
      }
      const float4* a_r0 = reinterpret_cast<const float4*>(asrc + ra * 256);
      const float4* a_r1 = reinterpret_cast<const float4*>(asrc + (ra + (a_kind ? 1 : 0)) * 256);
      const float* f_r0 = fsrc + rf * f_cols;
      const float* f_r1 = fsrc + (rf + (f_kind ? 1 : 0)) * f_cols;
      const int fc0 = lane, fc1 = lane + 32;
      const float4 x0 = __ldg(a_r0 + lane), x1 = __ldg(a_r0 + lane + 32);
      const float4 y0 = __ldg(a_r1 + lane), y1 = __ldg(a_r1 + lane + 32);
      const float p0 = fc0 < f_cols ? __ldg(f_r0 + fc0) : 0.0f, p1 = fc1 < f_cols ? __ldg(f_r0 + fc1) : 0.0f;
      const float q0 = fc0 < f_cols ? __ldg(f_r1 + fc0) : 0.0f, q1 = fc1 < f_cols ? __ldg(f_r1 + fc1) : 0.0f;
      float4* adst = reinterpret_cast<float4*>(reinterpret_cast<float*>(out_audio) + r * 256);
      adst[lane] = a_kind ? mul4(add4(x0, y0), 0.5f) : x0;
      adst[lane + 32] = a_kind ? mul4(add4(x1, y1), 0.5f) : x1;
      auto fexpr = [&](float u, float w) -> float {
        if (f_kind == 0) return u;
        const float h = __fmul_rn(__fadd_rn(u, w), 0.5f);
        if (f_kind == 1) return h;
        return f_kind == 2 ? __fmul_rn(__fadd_rn(u, h), 0.5f) : __fmul_rn(__fadd_rn(h, w), 0.5f);
      };
      float* fdst = reinterpret_cast<float*>(out_facial) + r * f_cols;
      if (fc0 < f_cols) fdst[fc0] = fexpr(p0, q0);
      if (fc1 < f_cols) fdst[fc1] = fexpr(p1, q1);
      continue;
    }
    T w1[2] = {static_cast<T>(0), static_cast<T>(0)}, w2[2] = {static_cast<T>(0), static_cast<T>(0)};
    for (int bi = 0; bi < n_blend; ++bi) {
      w1[bi] = static_cast<T>(linspace_at(1.0, 0.0, nb[blend_level[bi]], blend_q[bi]));
      w2[bi] = static_cast<T>(linspace_at(0.0, 1.0, nb[blend_level[bi]], blend_q[bi]));
    }
    auto row_out = [&](const T* src, int64_t ld, int cols, bool smooth_slow, T* dst) {
      for (int c = lane; c < cols; c += 32) {
        T val = version_value<T>(src, ld, term_ver, term_row, c, smooth_slow);
        for (int bi = n_blend - 1; bi >= 0; --bi) {
          const T nv_val = version_value<T>(src, ld, ver[blend_level[bi]], blend_q[bi], c, smooth_slow);
          val = add_rn(mul_rn(w1[bi], val), mul_rn(w2[bi], nv_val));
        }
        dst[c] = val;
      }
    };
    if (sizeof(T) == 4 && (a_cols & 3) == 0) {
      // float32 audio block: 16 bytes per lane and request (a row of 256 columns is two warp requests)
      const float* src = reinterpret_cast<const float*>(audio) + a0 * a_cols;
      float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(out_audio) + r * a_cols);
      for (int c4 = lane; c4 < (a_cols >> 2); c4 += 32) {
        float4 val = version_value4(src, a_cols, term_ver, term_row, c4, false);
        for (int bi = n_blend - 1; bi >= 0; --bi) {
          const float4 nv_val = version_value4(src, a_cols, ver[blend_level[bi]], blend_q[bi], c4, false);
          val = add4(mul4s(static_cast<float>(w1[bi]), val), mul4s(static_cast<float>(w2[bi]), nv_val));
        }
        dst[c4] = val;
      }
    } else {
      row_out(audio + a0 * a_cols, a_cols, a_cols, false, out_audio + r * a_cols);
    }
    row_out(facial + f0 * f_cols, f_cols, f_cols, true, out_facial + r * f_cols);
  }
}


// ------------------------------------------------------------------------------------------------
// Stand-alone row helpers with the reference's rounding order (templated float / double).
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_rows_op(int op, const T* __restrict__ a, int64_t na,
                                                 const T* __restrict__ b, int64_t nb, int cols,
                                                 int64_t k, T* __restrict__ out, int64_t out_rows) {
  const int64_t total = out_rows * cols;
  for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
       e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = e / cols;
    const int c = static_cast<int>(e - r * cols);
    T v;
    if (op == NSF_ROWS_INTERP_SLOWER) {
      v = (r & 1) ? mul_rn(add_rn(a[(r >> 1) * cols + c], a[((r >> 1) + 1) * cols + c]), static_cast<T>(0.5))
                  : a[(r >> 1) * cols + c];
    } else if (op == NSF_ROWS_SMOOTH) {
      v = r == 0 ? a[c] : mul_rn(add_rn(a[(r - 1) * cols + c], a[r * cols + c]), static_cast<T>(0.5));
    } else {  // NSF_ROWS_BLEND_STACK
      if (r < na - k) v = a[r * cols + c];
      else if (r < na) {
        const int64_t q = r - (na - k);
        const T w1 = static_cast<T>(linspace_at(1.0, 0.0, k, q));
        const T w2 = static_cast<T>(linspace_at(0.0, 1.0, k, q));
        v = add_rn(mul_rn(w1, a[r * cols + c]), mul_rn(w2, b[q * cols + c]));
      } else v = b[(r - na + k) * cols + c];
    }
    out[e] = v;
  }
}

// one block per channel: float64 moments sum x and sum x^2
__global__ void __launch_bounds__(256) k_col_stats(const float* __restrict__ in, int64_t T, int C,
                                                   double* __restrict__ sum, double* __restrict__ sumsq) {
  const int c = blockIdx.x;
  double acc = 0.0, acc2 = 0.0;
  for (int64_t t = threadIdx.x; t < T; t += blockDim.x) {
    const double v = static_cast<double>(in[t * C + c]);
    acc += v;
    acc2 = fma(v, v, acc2);
  }
  const double tot = block_sum<256>(acc);
  const double sq = block_sum<256>(acc2);
  if (threadIdx.x == 0) { sum[c] = tot; sumsq[c] = sq; }
}

// fix_edge_frames_autocorr on a frame-major [T][C] matrix, single block
__global__ void __launch_bounds__(256) k_edge_fix(float* __restrict__ d, int64_t T, int C, float thr) {
  __shared__ int s_big[2];
  if (threadIdx.x < 2) s_big[threadIdx.x] = 0;
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    if (!(fabsf(d[c]) < thr)) s_big[0] = 1;
    if (!(fabsf(d[(T - 1) * C + c]) < thr)) s_big[1] = 1;
  }
  __syncthreads();
  const bool fix_first = s_big[0] == 0, fix_last = s_big[1] == 0;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    if (fix_first) d[c] = d[C + c];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    if (fix_last) d[(T - 1) * C + c] = d[(T - 2) * C + c];
  }
}

// ---- inference-side chunker (utils/audio/processing/audio_processing.py:14-23, 33-48, 50-112) ---------------
// Chunk k covers feature rows [k stride, k stride + frame), stride = frame - overlap; a chunk that runs past the
// last row is completed with np.pad(..., mode='reflect') of ITS OWN rows (period 2 m - 2 for m valid rows, a single
// row repeats).  One thread per (chunk row, float4 of columns): pure data movement.
__global__ void __launch_bounds__(256) k_chunk_gather(const float* __restrict__ rows, int64_t n_rows, int cols, int64_t ld,
                                                      int frame, int stride, int64_t n_chunks, float* __restrict__ out) {
  const int64_t total = n_chunks * frame * cols;
  for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
       e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(e % cols);
    const int64_t cr = e / cols;
    const int j = static_cast<int>(cr % frame);
    const int64_t k = cr / frame;
    const int64_t s = k * stride;
    const int64_t m = min(static_cast<int64_t>(frame), n_rows - s);     // valid rows of this chunk (>= 1)
    int64_t idx = j;
    if (idx >= m) {
      if (m == 1) idx = 0;
      else {
        const int64_t period = 2 * m - 2;
        idx %= period;
        if (idx >= m) idx = period - idx;
      }
    }
    out[e] = __ldg(rows + (s + idx) * ld + c);
  }
}

// Output row r of process_audio_features: the decoded rows of the chunks that cover r, folded in chunk order with
// blend_chunks' cross-fade  (1 - i/n) * accumulated + (i/n) * chunk[i]  (the Python-float weights rounded to float32
// first, separate multiply and add - NumPy's arithmetic), then `[:, :scale_cols] /= divisor`.
__global__ void __launch_bounds__(256) k_chunk_blend(const float* __restrict__ dec, int64_t n_rows, int cols, int frame,
                                                     int stride, int overlap, int64_t n_chunks, int scale_cols,
                                                     float divisor, float* __restrict__ out) {
  const int64_t total = n_rows * cols;
  for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
       e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(e % cols);
    const int64_t r = e / cols;
    int64_t k_hi = r / stride;
    if (k_hi > n_chunks - 1) k_hi = n_chunks - 1;
    int64_t k_lo = r - frame + 1 <= 0 ? 0 : (r - frame + 1 + stride - 1) / stride;
    float v = __ldg(dec + (k_lo * frame + (r - k_lo * stride)) * cols + c);
    for (int64_t k = k_lo + 1; k <= k_hi; ++k) {
      const int64_t s = k * stride;
      const int64_t len_k = min(static_cast<int64_t>(frame), n_rows - s);
      const int64_t l_prev = min(n_rows, s - stride + frame);           // rows accumulated before chunk k
      const int64_t n = min(min(static_cast<int64_t>(overlap), l_prev), len_k);
      const int64_t i = r - s;                                          // l_prev - n == s (checked on the host)
      const float x = __ldg(dec + (k * frame + i) * cols + c);
      if (i < n) {
        const double alpha = static_cast<double>(i) / static_cast<double>(n);
        const float w1 = static_cast<float>(1.0 - alpha), w2 = static_cast<float>(alpha);
        v = __fadd_rn(__fmul_rn(w1, v), __fmul_rn(w2, x));
      } else {
        v = x;
      }
    }
    if (c < scale_cols) v = __fdiv_rn(v, divisor);
    out[e] = v;
  }
}

// ---- training windows (dataset/dataset.py:58-98, _WindowedClip) --------------------------------------------
// One stream (audio or facial) of a resolved window: output row r reads rows[base + r] while r < seg; past seg it
// mirrors (rows[base + 2 seg - 1 - r], the tail window; a one-row segment repeats, as torch broadcasts it) or is zero
// (a regular window past the stream's end).
struct WinStream {
  int64_t base;
  int32_t seg, reflect;
};

__device__ __forceinline__ int64_t win_src(const WinStream& s, int r) {
  if (r < s.seg) return s.base + r;
  if (!s.reflect) return -1;
  return s.seg == 1 ? s.base : s.base + 2 * s.seg - 1 - r;
}

template <int V> struct WinVec;
template <> struct WinVec<1> {
  using T = float;
  static __device__ __forceinline__ T zero() { return 0.0f; }
};
template <> struct WinVec<4> {
  using T = float4;
  static __device__ __forceinline__ T zero() { return make_float4(0.0f, 0.0f, 0.0f, 0.0f); }
};

constexpr int kWinThreads = 256, kWinUnroll = 8;

// `n_rows` rows of one stream of the block's tile into the contiguous `out`, V floats per access: every thread issues
// up to kWinUnroll independent loads before its first store (a 32-row tile of 256 float4 columns is exactly one round).
template <int V>
__device__ __forceinline__ void win_copy(const float* __restrict__ rows, int cols, const WinStream& s, int r0, int n_rows,
                                         float* __restrict__ out) {
  using T = typename WinVec<V>::T;
  const int cv = cols / V;
  const int total = n_rows * cv;
  for (int e0 = threadIdx.x; e0 < total; e0 += kWinThreads * kWinUnroll) {
    T v[kWinUnroll];
#pragma unroll
    for (int u = 0; u < kWinUnroll; ++u) {
      const int e = e0 + u * kWinThreads;
      v[u] = WinVec<V>::zero();
      if (e < total) {
        const int r = e / cv;
        const int64_t src = win_src(s, r0 + r);
        if (src >= 0) v[u] = __ldg(reinterpret_cast<const T*>(rows + src * cols) + (e - r * cv));
      }
    }
#pragma unroll
    for (int u = 0; u < kWinUnroll; ++u) {
      const int e = e0 + u * kWinThreads;
      if (e < total) reinterpret_cast<T*>(out)[e] = v[u];
    }
  }
}

// Block b copies rows [r0, r0 + kWindowTileRows) of output window b / tiles.  Thread 0 resolves the window to its clip
// (find_segment over the window offsets) and to the two streams' sources once; the copy itself is pure data movement.
// V = 4: audio rows as float4 (cols % 4 == 0 and 16-byte aligned bases); facial rows are always scalar (61 columns,
// 244-byte rows), read by consecutive threads.
template <int V>
__global__ void __launch_bounds__(kWinThreads) k_window_gather(WindowView v, int tiles, const float* __restrict__ audio,
                                                               int a_cols, const float* __restrict__ facial, int f_cols,
                                                               float* __restrict__ out_a, float* __restrict__ out_f) {
  __shared__ WinStream s_st[2];
  const int64_t k = blockIdx.x / tiles;
  const int r0 = static_cast<int>(blockIdx.x % tiles) * kWindowTileRows;
  const int n_rows = min(kWindowTileRows, v.window - r0);
  if (threadIdx.x == 0) {
    const int64_t idx = v.index[k];
    const int lo = find_segment(v.w_off, v.n_clips, idx);   // every clip has >= 1 window
    const int64_t j = idx - __ldg(v.w_off + lo);
    const int64_t a0 = __ldg(v.a_off + lo), f0 = __ldg(v.f_off + lo);
    const int64_t na = __ldg(v.a_off + lo + 1) - a0, nf = __ldg(v.f_off + lo + 1) - f0;
    const int64_t top = max(na, nf), w = v.window;
    const bool tail = j >= top - w + 1;
    const int64_t start = tail ? top - w : j;
    // regular: rows of the stream left from `start`, at most a window (zero past them); tail: min(top, n) - start,
    // at least half a window (validated on the host)
    const int64_t seg_a = max(int64_t(0), min(w, min(top, na) - start));
    const int64_t seg_f = max(int64_t(0), min(w, min(top, nf) - start));
    s_st[0] = WinStream{a0 + start, static_cast<int32_t>(seg_a), tail ? 1 : 0};
    s_st[1] = WinStream{f0 + start, static_cast<int32_t>(seg_f), tail ? 1 : 0};
  }
  __syncthreads();
  const WinStream sa = s_st[0], sf = s_st[1];
  const int64_t out_row = k * v.window + r0;
  win_copy<V>(audio, a_cols, sa, r0, n_rows, out_a + out_row * a_cols);
  win_copy<1>(facial, f_cols, sf, r0, n_rows, out_f + out_row * f_cols);
}

int grid_for(int64_t items, int per_block, int max_blocks) {
  int64_t g = (items + per_block - 1) / per_block;
  if (g < 1) g = 1;
  if (g > max_blocks) g = max_blocks;
  return static_cast<int>(g);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// launchers (return number of kernels launched, or -1 on launch error)
// ------------------------------------------------------------------------------------------------
// 16-byte vector loads / stores need 16-byte aligned array bases (library arenas always are; caller-owned device
// pointers of the stream-ordered entry points may not be: those take the scalar instantiation)
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// max_blocks > 0 caps the grid (the kernels stride over the 16 K-sample chunks).  The pipelined host entry points
// pass a cap: these two kernels are pure HBM streams, and whenever a kernel saturates HBM the copy engine's upload of
// the NEXT clip group stalls - measured on C2 end to end (int16 host PCM -> host rows, B200): 6.45 ms with the grid
// capped at 74 / 148 blocks against 6.78 ms uncapped, although the uncapped kernels are 3x shorter (round 2,
// profiles/experiments/README.md).  Device-resident callers run them uncapped.
int launch_absmax(cudaStream_t s, const void* pcm, int fmt, const BatchView& b, uint32_t* peak_bits, int max_blocks) {
  if (b.total_samples == 0) return 0;
  int grid = static_cast<int>((b.total_samples + kChunk - 1) / kChunk);
  if (max_blocks > 0 && grid > max_blocks) grid = max_blocks;
  const bool vec = aligned16(pcm);
  if (fmt == NSF_PCM_I16) {
    if (vec) k_absmax<int16_t, true><<<grid, 256, 0, s>>>(static_cast<const int16_t*>(pcm), b, peak_bits);
    else k_absmax<int16_t, false><<<grid, 256, 0, s>>>(static_cast<const int16_t*>(pcm), b, peak_bits);
  } else {
    if (vec) k_absmax<float, true><<<grid, 256, 0, s>>>(static_cast<const float*>(pcm), b, peak_bits);
    else k_absmax<float, false><<<grid, 256, 0, s>>>(static_cast<const float*>(pcm), b, peak_bits);
  }
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_normalize(cudaStream_t s, const void* pcm, int fmt, const BatchView& b,
                     const uint32_t* peak_bits, bool use_peak, float* y, int max_blocks) {
  if (b.total_samples == 0) return 0;
  int grid = static_cast<int>((b.total_samples + kChunk - 1) / kChunk);
  if (max_blocks > 0 && grid > max_blocks) grid = max_blocks;
  const bool vec = aligned16(pcm) && aligned16(y);
  if (fmt == NSF_PCM_I16) {
    if (vec) k_normalize<int16_t, true><<<grid, 256, 0, s>>>(static_cast<const int16_t*>(pcm), b, peak_bits, use_peak, y);
    else k_normalize<int16_t, false><<<grid, 256, 0, s>>>(static_cast<const int16_t*>(pcm), b, peak_bits, use_peak, y);
  } else {
    if (vec) k_normalize<float, true><<<grid, 256, 0, s>>>(static_cast<const float*>(pcm), b, peak_bits, use_peak, y);
    else k_normalize<float, false><<<grid, 256, 0, s>>>(static_cast<const float*>(pcm), b, peak_bits, use_peak, y);
  }
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_fold32(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* y, float* a32) {
  const int grid = grid_for(b.total_frames, 1, kSmCount * 8);
  k_fold32<<<grid, 256, t.F * sizeof(float), s>>>(t, b, y, a32);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_dft_simt(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* a32,
                    float* power) {
  const int np_max = t.np[0] > t.np[1] ? t.np[0] : t.np[1];
  dim3 grid(static_cast<unsigned>((b.total_frames + 63) / 64), (np_max + 63) / 64, t.chains);
  k_dft_simt<<<grid, 256, 0, s>>>(t, b, a32, power);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_mel_db(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* power,
                  float* db, uint32_t* dbmax_key) {
  if (t.n_mels > kMelWarps * kMelPerWarp) return -1;
  const int chain_cols = t.np[0] > t.np[1] ? t.np[0] : t.np[1];
  const size_t smem = (static_cast<size_t>(chain_cols) * kMelPitch + kMelFrames * (t.n_mels + 1)) * sizeof(float);
  if (smem > 200 * 1024) return -1;
  int per_sm = static_cast<int>((220 * 1024) / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm);
  const int grid = grid_for((b.total_frames + kMelFrames - 1) / kMelFrames, 1, kSmCount * per_sm);
  k_mel_db<<<grid, kMelWarps * 32, smem, s>>>(t, b, power, db, dbmax_key, chain_cols);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_dct_sum(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* db,
                   const uint32_t* dbmax_key, float* mfcc_raw, double* sum, double* sumsq) {
  if (t.n_mels > 128 || t.n_mfcc > 32) return -1;
  const int kp = t.n_mfcc <= 24 ? 24 : 32;
  // default shape: the tensor-pipe kernel.  NSF_DCT_SMEM=1 keeps the shared-memory coefficient kernels for the
  // default shape too (the FFMA reference of test_dct_mma_kernel_agrees_with_ffma_kernel)
  static const bool force_smem = std::getenv("NSF_DCT_SMEM") != nullptr;
  if (t.dct_frag && !force_smem && t.n_mels == kDctMmaMels && t.n_mfcc == kDctMmaMfcc) {
    const int grid_m = grid_for((b.total_frames + 31) / 32, kDct2Warps, kSmCount * 3);
    k_dct_mma<<<grid_m, kDct2Warps * 32, 0, s>>>(t.dct_frag, b, db, dbmax_key, mfcc_raw, sum, sumsq);
    NSF_CHECK_LAUNCH();
    return 1;
  }
  // k_dct_rows reads 16-byte aligned rows; mel counts that are not a multiple of 4 take the transposing-tile kernel
  if ((t.n_mels & 3) == 0) {
    const size_t smem2 = (static_cast<size_t>(t.n_mels) * kp + static_cast<size_t>(kDct2Warps) * 32 * t.n_mfcc) * sizeof(float);
    const int grid2 = grid_for((b.total_frames + 31) / 32, kDct2Warps, kSmCount * 2);
    if (kp == 24) k_dct_rows<24><<<grid2, kDct2Warps * 32, smem2, s>>>(t, b, db, dbmax_key, mfcc_raw, sum, sumsq);
    else k_dct_rows<32><<<grid2, kDct2Warps * 32, smem2, s>>>(t, b, db, dbmax_key, mfcc_raw, sum, sumsq);
    NSF_CHECK_LAUNCH();
    return 1;
  }
  const size_t smem = (static_cast<size_t>(t.n_mels) * kp + static_cast<size_t>(kDctWarps) * t.n_mels * kDctPitch) * sizeof(float);
  const int grid = grid_for((b.total_frames + 31) / 32, kDctWarps, kSmCount * 2);
  if (kp == 24) {
    k_dct_sum<24><<<grid, kDctWarps * 32, smem, s>>>(t, b, db, dbmax_key, mfcc_raw, sum, sumsq);
  } else {
    k_dct_sum<32><<<grid, kDctWarps * 32, smem, s>>>(t, b, db, dbmax_key, mfcc_raw, sum, sumsq);
  }
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_delta_reduce(cudaStream_t s, const BatchView& b, const float* in, int C, int in_ld,
                        const double* sum, const double* sumsq, bool cmvn, bool deltas, bool reduce,
                        float* out, int64_t out_ld, int col0) {
  // one wave of resident blocks (three per SM): the first row of a warp's run costs several times an interior row
  // (clip lookup, float64 CMVN constants, ten window loads), so runs are as long as the grid allows
  const int grid = grid_for(b.total_rows, 8, kSmCount * 3);
  k_delta_reduce<<<grid, 256, 0, s>>>(b, in, C, in_ld, sum, sumsq, cmvn, deltas, reduce, out, out_ld, col0);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_autocorr(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* y,
                    bool reduce, float* out, int64_t out_ld, int col0) {
  const AcGeom geo = ac_geom(t.F);
  const size_t smem = static_cast<size_t>(kAcWarps) * geo.row_floats * sizeof(float);
  if (smem > 200 * 1024) return -1;
  int per_sm = static_cast<int>((220 * 1024) / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  const int grid = grid_for(b.total_rows, kAcWarps, kSmCount * per_sm);
  k_autocorr<<<grid, kAcWarps * 32, smem, s>>>(t, b, y, reduce, out, out_ld, col0);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_smooth(cudaStream_t s, const BatchView& b, const float* in, int64_t in_ld, int cols,
                  float* out, int64_t out_ld) {
  const int grid = grid_for(b.total_rows, 1, kSmCount * 16);
  k_smooth<<<grid, 256, 0, s>>>(b, in, in_ld, cols, out, out_ld);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_collect(cudaStream_t s, int dtype, const CollectView& v, const void* audio, int a_cols,
                   const void* facial, int f_cols, void* out_audio, void* out_facial) {
  if (v.total_out_rows == 0) return 0;
  // one wave of resident blocks (48 registers: five blocks of 256 threads per SM), >= 8 rows per warp when there are
  // enough: with 8 blocks per SM the second wave ran 60 % full (ncu: 1.6 waves)
  const int grid = grid_for(v.total_out_rows, 8 * 8, kSmCount * 5);
  if (dtype == NSF_F64)
    k_collect_rows<double><<<grid, 256, 0, s>>>(v, static_cast<const double*>(audio), a_cols,
                                                static_cast<const double*>(facial), f_cols,
                                                static_cast<double*>(out_audio), static_cast<double*>(out_facial));
  else
    k_collect_rows<float><<<grid, 256, 0, s>>>(v, static_cast<const float*>(audio), a_cols,
                                               static_cast<const float*>(facial), f_cols,
                                               static_cast<float*>(out_audio), static_cast<float*>(out_facial));
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_rows_op(cudaStream_t s, int op, int dtype, const void* a, int64_t na, const void* b, int64_t nb,
                   int cols, int64_t k_blend, void* out, int64_t out_rows) {
  if (out_rows <= 0) return 0;
  const int grid = grid_for(out_rows * cols, 256 * 4, kSmCount * 16);
  if (dtype == NSF_F64)
    k_rows_op<double><<<grid, 256, 0, s>>>(op, static_cast<const double*>(a), na, static_cast<const double*>(b),
                                          nb, cols, k_blend, static_cast<double*>(out), out_rows);
  else
    k_rows_op<float><<<grid, 256, 0, s>>>(op, static_cast<const float*>(a), na, static_cast<const float*>(b), nb,
                                         cols, k_blend, static_cast<float*>(out), out_rows);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_col_stats(cudaStream_t s, const float* in, int64_t T, int C, double* sum, double* sumsq) {
  k_col_stats<<<C, 256, 0, s>>>(in, T, C, sum, sumsq);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_edge_fix(cudaStream_t s, float* data, int64_t T, int C, float zero_threshold) {
  k_edge_fix<<<1, 256, 0, s>>>(data, T, C, zero_threshold);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_chunk_gather(cudaStream_t s, const float* rows, int64_t n_rows, int cols, int64_t ld, int frame, int overlap,
                        int64_t n_chunks, float* out) {
  const int grid = grid_for(n_chunks * frame * cols, 256, kSmCount * 8);
  k_chunk_gather<<<grid, 256, 0, s>>>(rows, n_rows, cols, ld, frame, frame - overlap, n_chunks, out);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_chunk_blend(cudaStream_t s, const float* decoded, int64_t n_rows, int cols, int frame, int overlap,
                       int64_t n_chunks, int scale_cols, float divisor, float* out) {
  const int grid = grid_for(n_rows * cols, 256, kSmCount * 8);
  k_chunk_blend<<<grid, 256, 0, s>>>(decoded, n_rows, cols, frame, frame - overlap, overlap, n_chunks, scale_cols, divisor, out);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_window_gather(cudaStream_t s, const WindowView& v, const float* audio, int a_cols, const float* facial,
                         int f_cols, float* out_a, float* out_f) {
  if (v.n <= 0) return 0;
  const int tiles = (v.window + kWindowTileRows - 1) / kWindowTileRows;
  const unsigned blocks = static_cast<unsigned>(v.n * tiles);   // <= INT32_MAX (checked by nsf_window_gather)
  if (a_cols % 4 == 0 && aligned16(audio) && aligned16(out_a))
    k_window_gather<4><<<blocks, kWinThreads, 0, s>>>(v, tiles, audio, a_cols, facial, f_cols, out_a, out_f);
  else
    k_window_gather<1><<<blocks, kWinThreads, 0, s>>>(v, tiles, audio, a_cols, facial, f_cols, out_a, out_f);
  NSF_CHECK_LAUNCH();
  return 1;
}

// Opt-in shared-memory limits of the kernels in this file, once per device (nsf_ctx_create, after
// cudaSetDevice): the attribute is per device and a process may drive several.
bool init_kernel_attributes() {
  bool ok = true;
  auto set = [&](auto kernel, int bytes) {
    ok = ok && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess;
  };
  set(k_mel_db, 200 * 1024);
  set(k_dct_sum<24>, 100 * 1024);
  set(k_dct_sum<32>, 100 * 1024);
  set(k_autocorr, 200 * 1024);
  return ok;
}

}  // namespace nsf


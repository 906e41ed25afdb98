// WAV conversion kernels: decode + channel downmix (+ polyphase resampling) of a ragged batch of clips.
// See nsf_convert_* in include/nsf.h for the contract; every result is bit-identical to decode_wav followed by
// the float64 polyphase filter of nsf_resample_host.
#include <cstdint>

#include "nsf.h"
#include "nsf_kernels.cuh"

#define NSF_CHECK_LAUNCH() \
  do { if (cudaGetLastError() != cudaSuccess) return -1; } while (0)

namespace nsf {
namespace {

// One sample of a clip, decoded exactly as decode_wav does it (float32 IEEE arithmetic, no contraction possible:
// there is no multiply feeding an add).  8- and 24-bit samples may sit at any byte address; the wider containers
// are aligned (checked on the host before any launch).
__device__ __forceinline__ float decode_sample(const uint8_t* p, int enc) {
  switch (enc) {
    case NSF_ENC_U8: return (static_cast<float>(*p) - 128.0f) / 128.0f;
    case NSF_ENC_I16: return static_cast<float>(*reinterpret_cast<const int16_t*>(p)) / 32768.0f;
    case NSF_ENC_I24: {
      const int32_t v = static_cast<int32_t>(p[0]) | (static_cast<int32_t>(p[1]) << 8) |
                        (static_cast<int32_t>(static_cast<int8_t>(p[2])) << 16);
      return __double2float_rn(static_cast<double>(v) / 8388608.0);
    }
    case NSF_ENC_I32:
      return __double2float_rn(static_cast<double>(*reinterpret_cast<const int32_t*>(p)) / 2147483648.0);
    case NSF_ENC_F32: return *reinterpret_cast<const float*>(p);
    default: return __double2float_rn(*reinterpret_cast<const double*>(p));
  }
}

// NumPy's pairwise float32 sum (pairwise_sum of numpy/_core/src/umath/loops_utils.h.src) over n samples `stride`
// bytes apart: below 8 a left-to-right sum from 0, up to 128 eight interleaved partial sums combined as
// ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)) then the remainder, above that the sum of two halves split at
// a multiple of 8 (pairwise_sum_big).
__device__ __forceinline__ float pairwise_leaf(const uint8_t* p, int n, int stride, int enc) {
  if (n < 8) {
    float res = 0.0f;
    for (int i = 0; i < n; ++i) res += decode_sample(p + static_cast<int64_t>(i) * stride, enc);
    return res;
  }
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = decode_sample(p + static_cast<int64_t>(j) * stride, enc);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] += decode_sample(p + static_cast<int64_t>(i + j) * stride, enc);
  }
  float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res += decode_sample(p + static_cast<int64_t>(i) * stride, enc);
  return res;
}

// n > 128: NumPy's recursion pw(a, n) = pw(a, n2) + pw(a + n2, n - n2), n2 = n / 2 - (n / 2) % 8, walked with an
// explicit stack (left half first, one float add per split).  Depth 12 covers the 65535 channels of a WAV header.
__device__ __noinline__ float pairwise_sum_big(const uint8_t* p, int n, int stride, int enc) {
  struct Node { int off, n, state; float left; };
  Node st[12];
  int top = 0;
  st[0] = Node{0, n, 0, 0.0f};
  float ret = 0.0f;
  while (top >= 0) {
    Node& f = st[top];
    if (f.n <= 128) { ret = pairwise_leaf(p + static_cast<int64_t>(f.off) * stride, f.n, stride, enc); --top; continue; }
    int n2 = f.n / 2;
    n2 -= n2 % 8;
    if (f.state == 0) { f.state = 1; st[++top] = Node{f.off, n2, 0, 0.0f}; }
    else if (f.state == 1) { f.left = ret; f.state = 2; st[++top] = Node{f.off + n2, f.n - n2, 0, 0.0f}; }
    else { ret = f.left + ret; --top; }
  }
  return ret;
}

// Frame n of a clip as decode_wav returns it: the sample itself for mono, else
// x.reshape(-1, channels).mean(axis=1, dtype=float32) = (0 + pairwise sum) / channels.
__device__ __forceinline__ float decode_frame(const uint8_t* clip, int64_t n, int enc, int channels, int bps) {
  const uint8_t* p = clip + n * channels * bps;
  if (channels == 1) return decode_sample(p, enc);
  const float s = 0.0f + (channels <= 128 ? pairwise_leaf(p, channels, bps, enc) : pairwise_sum_big(p, channels, bps, enc));
  return s / static_cast<float>(channels);
}

__device__ __forceinline__ int find_clip(const ConvClip* c, int n, int64_t tile) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (c[mid].tile0 <= tile) lo = mid; else hi = mid - 1;
  }
  return lo;
}

}  // namespace

// Same-rate clips: decode + downmix only.  kConvDecodeTile frames per block.
__global__ void __launch_bounds__(256) k_convert_decode(const ConvClip* __restrict__ clips, int n_clips,
                                                        const uint8_t* __restrict__ payload, float* __restrict__ out) {
  const ConvClip c = clips[find_clip(clips, n_clips, blockIdx.x)];
  const int64_t f0 = (blockIdx.x - c.tile0) * kConvDecodeTile;
  const int64_t f1 = min(f0 + kConvDecodeTile, c.frames);
  const uint8_t* src = payload + c.byte_off;
  for (int64_t f = f0 + threadIdx.x; f < f1; f += blockDim.x)
    out[c.out_off + f] = decode_frame(src, f, c.enc, c.channels, c.bps);
}

// Resampled clips.  out[j] = sum_{k < kmax} taps[k][phase(j)] x[n_hi(j) - k], t = (j + n_pre_remove) down - n_pre_pad,
// n_hi = t / up, phase = t mod up - one float64 FMA chain per output in ascending k, rounded once to float32.
// A block owns S * R consecutive outputs (S a multiple of `up`, R <= kConvMaxReps): thread slot i computes the R
// outputs j0 + i + r S, which share one phase, so every tap it loads feeds R FMAs; neighbouring slots hold
// neighbouring phases, which the k-major table keeps in one short row.  The block first decodes its
// whole input window into shared memory as float64 (each input frame decoded and downmixed once per block, not once
// per tap), with zeros outside [0, frames): fma(h, +0, acc) == acc for the finite taps and the never-negative-zero
// accumulator, so the zeros drop exactly the terms the reference skips (n < 0, n >= n_in).
__global__ void __launch_bounds__(256) k_convert_resample(const ConvClip* __restrict__ clips, int n_clips,
                                                          const uint8_t* __restrict__ payload,
                                                          float* __restrict__ out) {
  extern __shared__ double s_x[];
  const ConvClip c = clips[find_clip(clips, n_clips, blockIdx.x)];
  const int64_t span = static_cast<int64_t>(c.slots) * c.reps;
  const int64_t j0 = (blockIdx.x - c.tile0) * span;
  const int64_t lo = ((j0 + c.n_pre_remove) * c.down - c.n_pre_pad) / c.up - (c.kmax - 1);
  const int64_t hi = ((j0 + span - 1 + c.n_pre_remove) * c.down - c.n_pre_pad) / c.up;
  const int w_len = static_cast<int>(hi - lo + 1);
  const uint8_t* src = payload + c.byte_off;
  for (int w = threadIdx.x; w < w_len; w += blockDim.x) {
    const int64_t n = lo + w;
    s_x[w] = (n >= 0 && n < c.frames) ? static_cast<double>(decode_frame(src, n, c.enc, c.channels, c.bps)) : 0.0;
  }
  __syncthreads();
  const int kmax = c.kmax, reps = c.reps;
  const int64_t rep_in = static_cast<int64_t>(c.slots / c.up) * c.down;   // input step between r and r + 1
  for (int i = threadIdx.x; i < c.slots; i += blockDim.x) {
    const int64_t t = (j0 + i + c.n_pre_remove) * c.down - c.n_pre_pad;
    const int64_t n_hi = t / c.up;
    const double* h = c.taps + (t - n_hi * c.up);                        // k-major: tap k at h[k up]
    const double* x = s_x + (n_hi - lo);
    double acc[kConvMaxReps];
#pragma unroll
    for (int r = 0; r < kConvMaxReps; ++r) acc[r] = 0.0;
    for (int k = 0; k < kmax; ++k) {
      const double tap = __ldg(h + static_cast<int64_t>(k) * c.up);
#pragma unroll
      for (int r = 0; r < kConvMaxReps; ++r)
        if (r < reps) acc[r] = fma(tap, x[r * rep_in - k], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < kConvMaxReps; ++r) {
      const int64_t j = j0 + i + static_cast<int64_t>(r) * c.slots;
      if (r < reps && j < c.n_out) out[c.out_off + j] = static_cast<float>(acc[r]);
    }
  }
}

int launch_convert(cudaStream_t s, bool resample, const ConvClip* clips_dev, int n_clips, int64_t tiles,
                   size_t smem_bytes, const void* payload, float* out) {
  if (n_clips <= 0 || tiles <= 0) return 0;
  if (resample)
    k_convert_resample<<<static_cast<unsigned>(tiles), 256, smem_bytes, s>>>(
        clips_dev, n_clips, static_cast<const uint8_t*>(payload), out);
  else
    k_convert_decode<<<static_cast<unsigned>(tiles), 256, 0, s>>>(clips_dev, n_clips,
                                                                  static_cast<const uint8_t*>(payload), out);
  NSF_CHECK_LAUNCH();
  return 1;
}

bool init_convert_attributes() {
  return cudaFuncSetAttribute(k_convert_resample, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              static_cast<int>(kConvMaxSmem)) == cudaSuccess;
}

}  // namespace nsf

// Small device helpers shared by the kernel translation units.
#ifndef NSF_DEVICE_UTILS_CUH_
#define NSF_DEVICE_UTILS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

namespace nsf {

// Largest c in [0, n) with off[c] <= g (off is a non-decreasing prefix sum, off[0] == 0, g < off[n]).
// Batches are usually clips of (nearly) equal length, so the proportional guess c = g n / off[n] is
// probed first - two independent loads instead of log2(n) dependent ones (14 for the 10 000-clip
// batches) - and only a miss falls back to the bisection, on the side of the guess that holds g.
__device__ __forceinline__ int find_segment(const int64_t* __restrict__ off, int n, int64_t g) {
  int lo = 0, hi = n;  // invariant: off[lo] <= g < off[hi]
  if (n > 2) {
    const int64_t total = __ldg(off + n);
    int c = total > 0 ? static_cast<int>(static_cast<double>(g) * static_cast<double>(n) / static_cast<double>(total)) : 0;
    c = c < 0 ? 0 : (c > n - 1 ? n - 1 : c);
    const int64_t a = __ldg(off + c), e = __ldg(off + c + 1);
    if (a <= g) {
      if (g < e) return c;
      lo = c + 1;          // off[c + 1] <= g
    } else {
      hi = c;              // g < off[c]
    }
  }
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(off + mid) <= g) lo = mid; else hi = mid;
  }
  return lo;
}

// Largest i in [0, n) with key(i) <= x (key non-decreasing in i), 0 when there is none: the search over an array of
// descriptors sorted by one of their fields, e.g. last_le(n, x, [&](int i) { return clips[i].tile0; }).
template <typename Key>
__device__ __forceinline__ int last_le(int n, int64_t x, Key key) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (key(mid) <= x) lo = mid; else hi = mid - 1;
  }
  return lo;
}

template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += y;
  }
  return v;
}

// Exclusive prefix sum of x over the kThreads threads of the block, in thread order; *total <- the block's sum.  Ends
// with the barrier that frees its shared slots, so the next call (or any reuse of memory the caller wrote before it)
// needs no barrier of its own.
template <int kThreads, typename T>
__device__ __forceinline__ T block_exclusive_scan(T x, T* total) {
  __shared__ T s_warp[kThreads / 32];
  const int warp = threadIdx.x >> 5;
  const T incl = warp_inclusive_scan(x);
  if ((threadIdx.x & 31) == 31) s_warp[warp] = incl;
  __syncthreads();
  T before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    const T s = s_warp[w];
    before += w < warp ? s : T(0);
    all += s;
  }
  __syncthreads();
  *total = all;
  return before + incl - x;
}

// Sum of v over the kThreads threads of the block, seen by every thread: a warp xor tree, then the warp totals added in
// warp order (a fixed order, so a float sum is reproducible).  Ends with the barrier that frees its shared slots.
template <int kThreads, typename T>
__device__ __forceinline__ T block_sum(T v) {
  __shared__ T s_warp[kThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
  __syncthreads();
  T r = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) r += s_warp[w];
  __syncthreads();
  return r;
}

// One block of kThreads threads: start[t] = count[0] + ... + count[t - 1] for t < n; returns the total.  Each thread
// sums a contiguous run of tiles, the block scans the run sums, and each thread writes its run's starts.
template <int kThreads>
__device__ __forceinline__ int64_t scan_counts(const int32_t* __restrict__ count, int64_t n,
                                               int64_t* __restrict__ start) {
  const int64_t per = (n + kThreads - 1) / kThreads;
  const int64_t a = min(n, per * threadIdx.x), b = min(n, a + per);
  int64_t sum = 0;
  for (int64_t t = a; t < b; ++t) sum += count[t];
  int64_t total;
  int64_t run = block_exclusive_scan<kThreads>(sum, &total);
  for (int64_t t = a; t < b; ++t) { start[t] = run; run += count[t]; }
  return total;
}

// IEEE operations each rounded once to nearest, for code that must match a reference's float or double arithmetic
// operation for operation: nvcc never contracts these into an FMA.  The host build is the plain operation.
#ifdef __CUDA_ARCH__
__host__ __device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__host__ __device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__host__ __device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__host__ __device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__host__ __device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__host__ __device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
#else
__host__ __device__ __forceinline__ float add_rn(float a, float b) { return a + b; }
__host__ __device__ __forceinline__ float mul_rn(float a, float b) { return a * b; }
__host__ __device__ __forceinline__ float div_rn(float a, float b) { return a / b; }
__host__ __device__ __forceinline__ double add_rn(double a, double b) { return a + b; }
__host__ __device__ __forceinline__ double mul_rn(double a, double b) { return a * b; }
__host__ __device__ __forceinline__ double div_rn(double a, double b) { return a / b; }
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// order-preserving float -> uint32 key (so atomicMax works for negative dB values); 0 = "-inf"
__device__ __forceinline__ uint32_t float_key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// max_key[clip] = max(max_key[clip], key) for every lane of a converged warp; clip < 0: the lane has no value.  A warp
// whose lanes share one clip (the usual case: clips are far longer than 32 frames) reduces first and makes one atomic.
__device__ __forceinline__ void warp_clip_max(uint32_t* __restrict__ max_key, int clip, uint32_t key) {
  const int first_clip = __shfl_sync(0xffffffffu, clip, 0);
  if (__all_sync(0xffffffffu, clip == first_clip || clip < 0)) {
    uint32_t k = clip >= 0 ? key : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) k = max(k, __shfl_xor_sync(0xffffffffu, k, o));
    if ((threadIdx.x & 31) == 0 && first_clip >= 0) atomicMax(max_key + first_clip, k);
  } else if (clip >= 0) {
    atomicMax(max_key + clip, key);
  }
}

}  // namespace nsf
#endif  // NSF_DEVICE_UTILS_CUH_

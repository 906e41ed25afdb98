// CSV text of packed feature rows: byte for byte what pandas writes for DataFrame(rows.astype(float64))
// .to_csv(index=False), the reference's audio_features.csv cache (dataset/data_processing.py:115-120).  See
// nsf_format_csv_host in include/nsf.h for the contract.
//
// Every finite field is Python's repr(float(v)): the shortest decimal that rounds back to the double and, among
// those of that length, the one nearest the exact value (Schubfach, R. Giulietti 2020, in the form of A. Bolz's
// schubfach_64), positional for 1e-4 <= |v| < 1e16 with ".0" on integers, else d.ddd e+XX.  NaN is an empty field
// ("" when it is the row's only field, as Python's csv writer quotes a lone empty field), infinities are inf / -inf.
//
// Two kernels per file group: k_csv_lengths gives each row's byte count (the host turns the counts into row
// positions), k_csv_write formats each row again, places the fields with a block scan in shared memory and stores
// the row in 16-byte words.  Recomputing the digits is cheaper than a round trip of per-value lengths through HBM.
#include <cstdint>
#include <cstring>

#include "nsf.h"
#include "nsf_internal.h"
#include "nsf_kernels.cuh"

#define NSF_CHECK_LAUNCH() \
  do { if (cudaGetLastError() != cudaSuccess) return -1; } while (0)

namespace nsf {
namespace {

struct Pow10 { uint64_t hi, lo; };
constexpr int kPow10Min = -292;
// Read per lane from global memory through the read-only cache: the lanes of a warp index different entries, which
// __constant__ memory would serialise.
__device__ const Pow10 d_pow10[] = {
#include "nsf_csv_pow10.inc"
};
const Pow10 h_pow10[] = {
#include "nsf_csv_pow10.inc"
};

constexpr int kCsvThreads = 256;   // one column tile of a row per pass of a block
constexpr int kCsvFieldMax = 25;   // longest field (-1.2345678901234567e-308) and its separator

enum : uint32_t { kFinite = 0, kNan = 1, kInf = 2 };

// A field before its characters: |value| = digits * 10^(exp10 - n + 1), digits with n digits and no trailing zero.
struct Field {
  uint64_t digits;
  int32_t n, exp10, len;   // len: characters of the field, separator excluded
  uint32_t kind;
  bool neg;
};

__host__ __device__ __forceinline__ uint64_t double_bits(double v) {
#ifdef __CUDA_ARCH__
  return static_cast<uint64_t>(__double_as_longlong(v));
#else
  uint64_t b;
  std::memcpy(&b, &v, sizeof(b));
  return b;
#endif
}

__host__ __device__ __forceinline__ Pow10 pow10_entry(int e) {
#ifdef __CUDA_ARCH__
  const Pow10* p = d_pow10 + (e - kPow10Min);
  return {__ldg(&p->hi), __ldg(&p->lo)};
#else
  return h_pow10[e - kPow10Min];
#endif
}

// floor(g cp / 2^128) with its lowest bit set when the discarded fraction is not (nearly) zero: rounding to odd.
__host__ __device__ __forceinline__ uint64_t round_to_odd(Pow10 g, uint64_t cp) {
#ifdef __CUDA_ARCH__
  const uint64_t x_hi = __umul64hi(g.lo, cp), y_hi = __umul64hi(g.hi, cp), y_lo = g.hi * cp;
#else
  const unsigned __int128 x = static_cast<unsigned __int128>(g.lo) * cp, y = static_cast<unsigned __int128>(g.hi) * cp;
  const uint64_t x_hi = static_cast<uint64_t>(x >> 64), y_hi = static_cast<uint64_t>(y >> 64), y_lo = static_cast<uint64_t>(y);
#endif
  const uint64_t z = y_lo + x_hi;
  const uint64_t z1 = y_hi + (z < y_lo);
  return z1 | (z > 1);
}

// Shortest decimal d * 10^k of the positive double with biased exponent `be` and fraction `m` (be, m not both 0).
__host__ __device__ __forceinline__ void shortest(uint64_t m, uint32_t be, uint64_t* d, int* k) {
  uint64_t c;
  int q;
  if (be != 0) {
    c = (uint64_t(1) << 52) | m;
    q = static_cast<int>(be) - 1075;
    if (q <= 0 && q > -53 && (c & ((uint64_t(1) << -q) - 1)) == 0) {   // an integer below 2^53: its own digits
      *d = c >> -q;
      *k = 0;
      return;
    }
  } else {
    c = m;
    q = -1074;
  }
  const bool even = (c & 1) == 0;
  const bool lower_closer = m == 0 && be > 1;
  const uint64_t cbl = 4 * c - 2 + lower_closer, cb = 4 * c, cbr = 4 * c + 2;
  // floor(log10(2^q)), or floor(log10(3/4 2^q)) when the lower neighbour is closer; then 1 <= h <= 4
  const int kk = (q * 1262611 - (lower_closer ? 524031 : 0)) >> 22;
  const int h = q + ((-kk * 1741647) >> 19) + 1;
  const Pow10 g = pow10_entry(-kk);
  const uint64_t vbl = round_to_odd(g, cbl << h), vb = round_to_odd(g, cb << h), vbr = round_to_odd(g, cbr << h);
  const uint64_t lower = vbl + !even, upper = vbr - !even;
  const uint64_t s = vb / 4;
  if (s >= 10) {   // one digit fewer: at most one of its two candidates lies in the rounding interval
    const uint64_t sp = s / 10;
    const bool up_in = lower <= 40 * sp, wp_in = 40 * sp + 40 <= upper;
    if (up_in != wp_in) {
      *d = sp + wp_in;
      *k = kk + 1;
      return;
    }
  }
  const bool u_in = lower <= 4 * s, w_in = 4 * s + 4 <= upper;
  if (u_in != w_in) {
    *d = s + w_in;
    *k = kk;
    return;
  }
  const uint64_t mid = 4 * s + 2;
  *d = s + (vb > mid || (vb == mid && (s & 1) != 0));
  *k = kk;
}

__host__ __device__ __forceinline__ Field make_field(double v) {
  Field f;
  const uint64_t bits = double_bits(v);
  const uint64_t m = bits & ((uint64_t(1) << 52) - 1);
  const uint32_t be = static_cast<uint32_t>(bits >> 52) & 0x7ff;
  f.neg = (bits >> 63) != 0;
  f.digits = 0;
  f.n = 1;
  f.exp10 = 0;
  if (be == 0x7ff) {
    f.kind = m ? kNan : kInf;
    f.neg = f.neg && !m;
    f.len = m ? 0 : 3 + f.neg;
    return f;
  }
  f.kind = kFinite;
  uint64_t d = 0;
  int k = 0;
  if (be != 0 || m != 0) {
    shortest(m, be, &d, &k);
    while (d % 10 == 0) { d /= 10; ++k; }
  }
  int n = 1;
  for (uint64_t p = 10; n < 19 && d >= p; p *= 10) ++n;
  const int e = k + n - 1;
  f.digits = d;
  f.n = n;
  f.exp10 = e;
  if (e < -4 || e >= 16) f.len = n + (n > 1) + 2 + ((e <= -100 || e >= 100) ? 3 : 2);   // d[.ddd]e+XX
  else if (e >= n - 1) f.len = e + 3;                                                     // ddd000.0
  else if (e < 0) f.len = n + 1 - e;                                                      // 0.000ddd
  else f.len = n + 1;                                                                     // dd.ddd
  f.len += f.neg;
  return f;
}

// n decimal digits of d at p[0 .. n-1]
__host__ __device__ __forceinline__ void put_digits(char* p, uint64_t d, int n) {
  int i = n - 1;
  if (n > 8) {
    const uint64_t hi = d / 100000000u;
    uint32_t lo = static_cast<uint32_t>(d - hi * 100000000u);
    for (int j = 0; j < 8; ++j, --i) { p[i] = static_cast<char>('0' + lo % 10); lo /= 10; }
    d = hi;
  }
  uint32_t x = static_cast<uint32_t>(d);
  for (; i >= 0; --i) { p[i] = static_cast<char>('0' + x % 10); x /= 10; }
}

// The f.len characters of a field at p (nothing for NaN).
__host__ __device__ __forceinline__ void put_field(const Field& f, char* p) {
  if (f.kind == kNan) return;
  if (f.neg) *p++ = '-';
  if (f.kind == kInf) { p[0] = 'i'; p[1] = 'n'; p[2] = 'f'; return; }
  const int n = f.n, e = f.exp10;
  if (e < -4 || e >= 16) {
    put_digits(p + 1, f.digits, n);
    p[0] = p[1];
    int i = 1;
    if (n > 1) { p[1] = '.'; i = n + 1; }
    p[i++] = 'e';
    p[i++] = e < 0 ? '-' : '+';
    int a = e < 0 ? -e : e;
    if (a >= 100) { p[i++] = static_cast<char>('0' + a / 100); a %= 100; }
    p[i++] = static_cast<char>('0' + a / 10);
    p[i] = static_cast<char>('0' + a % 10);
  } else if (e >= n - 1) {
    put_digits(p, f.digits, n);
    for (int i = n; i <= e; ++i) p[i] = '0';
    p[e + 1] = '.';
    p[e + 2] = '0';
  } else if (e < 0) {
    p[0] = '0';
    p[1] = '.';
    for (int i = 0; i < -e - 1; ++i) p[2 + i] = '0';
    put_digits(p + 1 - e, f.digits, n);
  } else {
    put_digits(p + 1, f.digits, n);
    for (int i = 0; i <= e; ++i) p[i] = p[i + 1];
    p[e + 1] = '.';
  }
}

// Bytes of a field and its separator in a row of `cols` fields: a lone NaN field is written "".
__device__ __forceinline__ int field_bytes(const Field& f, int cols) {
  return (f.kind == kNan && cols == 1 ? 2 : f.len) + 1;
}

// Offset of column label c in the header line "0,1,...,cols-1\n".
__host__ __device__ __forceinline__ int64_t header_pos(int64_t c) {
  int64_t pos = 0, lo = 0, hi = 10;
  int digits = 1;
  while (c >= hi) { pos += (hi - lo) * (digits + 1); lo = hi; hi *= 10; ++digits; }
  return pos + (c - lo) * (digits + 1);
}

__device__ __forceinline__ double csv_value(const float* p) { return static_cast<double>(__ldg(p)); }
__device__ __forceinline__ double csv_value(const double* p) { return __ldg(p); }

// Block reduction / exclusive scan helpers over kCsvThreads threads.
__device__ __forceinline__ int warp_inclusive_scan(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// One block per row: row_len[r] = bytes of row r, separators and newline included.
template <typename T>
__global__ void __launch_bounds__(kCsvThreads) k_csv_lengths(const T* __restrict__ rows, int cols,
                                                             int64_t* __restrict__ row_len) {
  __shared__ int64_t s_warp[kCsvThreads / 32];
  const T* row = rows + static_cast<int64_t>(blockIdx.x) * cols;
  int64_t sum = 0;
  for (int c = threadIdx.x; c < cols; c += kCsvThreads) sum += field_bytes(make_field(csv_value(row + c)), cols);
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t t = 0;
#pragma unroll
    for (int w = 0; w < kCsvThreads / 32; ++w) t += s_warp[w];
    row_len[blockIdx.x] = t;
  }
}

// Blocks [0, n_rows): row b at text + start[b].  Blocks [n_rows, n_rows + n_files): the header of file b - n_rows
// at text + start[b].  A row goes tile by tile (kCsvThreads columns): the fields are placed by a block scan into
// shared memory, congruent to their global address modulo 16, and leave as aligned 16-byte words; only the first
// and last word of a tile, shared with the neighbouring text, are stored byte by byte.
template <typename T>
__global__ void __launch_bounds__(kCsvThreads) k_csv_write(const T* __restrict__ rows, int64_t n_rows, int cols,
                                                           const int64_t* __restrict__ start, char* __restrict__ text) {
  __shared__ __align__(16) char s_buf[kCsvThreads * kCsvFieldMax + 16];
  __shared__ int s_warp[kCsvThreads / 32];
  const int64_t b = blockIdx.x;
  int64_t pos = start[b];
  if (b >= n_rows) {
    for (int c = threadIdx.x; c < cols; c += kCsvThreads) {
      char* p = text + pos + header_pos(c);
      int digits = 1;
      for (int v = c; v >= 10; v /= 10) ++digits;
      for (int i = digits - 1, v = c; i >= 0; --i, v /= 10) p[i] = static_cast<char>('0' + v % 10);
      p[digits] = c == cols - 1 ? '\n' : ',';
    }
    return;
  }
  const T* row = rows + b * cols;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c0 = 0; c0 < cols; c0 += kCsvThreads) {
    const int c = c0 + static_cast<int>(threadIdx.x);
    Field f{};
    int len = 0;
    if (c < cols) {
      f = make_field(csv_value(row + c));
      len = field_bytes(f, cols);
    }
    const int incl = warp_inclusive_scan(len, lane);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kCsvThreads / 32; ++w) {
      const int t = s_warp[w];
      before += w < warp ? t : 0;
      total += t;
    }
    const int head = static_cast<int>(pos & 15);
    if (c < cols) {
      char* p = s_buf + head + before + incl - len;
      if (f.kind == kNan && cols == 1) { p[0] = '"'; p[1] = '"'; }
      else put_field(f, p);
      p[len - 1] = c == cols - 1 ? '\n' : ',';
    }
    __syncthreads();
    char* base = text + (pos - head);
    const int end = head + total;
    for (int w = threadIdx.x; w < (end + 15) / 16; w += kCsvThreads) {
      const int lo = w * 16;
      if (lo >= head && lo + 16 <= end) {
        *reinterpret_cast<uint4*>(base + lo) = *reinterpret_cast<const uint4*>(s_buf + lo);
      } else {
        for (int i = max(lo, head); i < min(lo + 16, end); ++i) base[i] = s_buf[i];
      }
    }
    pos += total;
    __syncthreads();   // s_buf and s_warp are the next tile's
  }
}

}  // namespace

int64_t csv_header_bytes(int cols) { return header_pos(cols); }

int launch_csv_lengths(cudaStream_t s, int dtype, const void* rows, int64_t n_rows, int cols, int64_t* row_len) {
  if (n_rows <= 0) return 0;
  const unsigned grid = static_cast<unsigned>(n_rows);
  if (dtype == NSF_F64)
    k_csv_lengths<double><<<grid, kCsvThreads, 0, s>>>(static_cast<const double*>(rows), cols, row_len);
  else
    k_csv_lengths<float><<<grid, kCsvThreads, 0, s>>>(static_cast<const float*>(rows), cols, row_len);
  NSF_CHECK_LAUNCH();
  return 1;
}

int launch_csv_write(cudaStream_t s, int dtype, const void* rows, int64_t n_rows, int cols, int32_t n_files,
                     const int64_t* start, char* text) {
  if (n_rows + n_files <= 0) return 0;
  const unsigned grid = static_cast<unsigned>(n_rows + n_files);
  if (dtype == NSF_F64)
    k_csv_write<double><<<grid, kCsvThreads, 0, s>>>(static_cast<const double*>(rows), n_rows, cols, start, text);
  else
    k_csv_write<float><<<grid, kCsvThreads, 0, s>>>(static_cast<const float*>(rows), n_rows, cols, start, text);
  NSF_CHECK_LAUNCH();
  return 1;
}

}  // namespace nsf

extern "C" {

int64_t nsf_csv_bytes_bound(int64_t n_rows, int32_t cols, int32_t n_files) {
  if (n_rows < 0 || cols < 1 || n_files < 0) return -1;
  return n_rows * cols * nsf::kCsvFieldMax + n_files * nsf::csv_header_bytes(cols);
}

nsf_status nsf_format_check(const double* values, int64_t n, char* out, int32_t* lengths) {
  if (!values || !out || !lengths || n < 0) { nsf::set_error("nsf_format_check: bad argument"); return NSF_ERR_BAD_ARG; }
  for (int64_t i = 0; i < n; ++i) {
    const nsf::Field f = nsf::make_field(values[i]);
    nsf::put_field(f, out + 32 * i);
    lengths[i] = f.len;
  }
  return NSF_OK;
}

}  // extern "C"

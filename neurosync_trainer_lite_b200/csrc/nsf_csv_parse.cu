// CSV text -> rows: value for value what pd.read_csv(path).drop(columns=...).values holds, for the files whose
// text stays inside the grammar below (the reference's facial CSVs and its audio_features.csv cache,
// dataset/data_processing.py:112-123).  See nsf_csv_parse in include/nsf.h for the contract.
//
// A number field is pandas' precise_xstrtod restated with the same IEEE double operations in the same order (it is
// not correctly rounded, so a correct parser would differ from the reference's reads): up to 17 mantissa digits
// accumulated as number * 10 + d, the rest counted into the decimal exponent, then one multiplication or division
// by the double literal 1e<k> (two divisions below 1e-308).  The first 15 digits accumulate in a uint64_t, where
// every intermediate is exact, as it is in the double chain; digits 16 and 17 continue in doubles.  nvcc would
// contract number * 10 + d into a DFMA (--fmad=true), which rounds once instead of twice: the device code spells
// every operation with mul_rn / add_rn / div_rn (nsf_device_utils.cuh).
//
// Kernels of one parse call (the row-offsets call runs the first two):
//   k_csv_count   one block per text tile (16 KB, never across a file boundary): data rows starting in the tile
//   k_csv_scan    one block: exclusive scan of the tile counts -> first row of each tile, per-file row offsets
//   k_csv_starts  one block per tile: the byte position of every data row, in order
//   k_csv_fields  one warp per row: the row in windows of 32 lanes x 16 bytes through shared memory, separators
//                 by per-lane byte masks and a warp scan, fields round-robin over the lanes
//   k_csv_int_zero  one block per file: pandas types an all-integer column as int64, whose -0 is +0
// The parse call rescans the text for the row positions rather than keeping them between the two calls: a pass
// over the text costs less than holding the positions, the same trade nsf_csv.cu makes for its digits.
#include <algorithm>
#include <cstdint>
#include <cstring>

#include "nsf.h"
#include "nsf_device_utils.cuh"
#include "nsf_internal.h"
#include "nsf_kernels.cuh"

namespace nsf {
namespace {

__device__ const double d_e10[] = {
#include "nsf_csv_e10.inc"
};
const double h_e10[] = {
#include "nsf_csv_e10.inc"
};

constexpr int kTileThreads = 256;                 // 64 bytes per thread
constexpr int kScanThreads = 1024;
constexpr int kFieldWarps = 8;                    // warps (rows in flight) per block of k_csv_fields
constexpr int kWin = 512;                         // bytes of a row window: 32 lanes x 16
constexpr int kFieldMax = 40;                     // longest number field accepted
// per (file, column) flags of k_csv_fields
constexpr uint32_t kNonInt = 1, kNegZeroInt = 2;

__host__ __device__ __forceinline__ double e10(int k) {
#ifdef __CUDA_ARCH__
  return __ldg(d_e10 + k);
#else
  return h_e10[k];
#endif
}
__host__ __device__ __forceinline__ double from_bits(uint64_t b) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(static_cast<long long>(b));
#else
  double v;
  std::memcpy(&v, &b, sizeof(v));
  return v;
#endif
}
__host__ __device__ __forceinline__ bool is_digit(char c) { return c >= '0' && c <= '9'; }

// Why a field is outside the number grammar: a quote or a '\r' changes how pandas splits the line, anything else is a
// field pandas would not read as a number.
__host__ __device__ __forceinline__ uint32_t field_fault(const char* p, int n) {
  for (int k = 0; k < n; ++k)
    if (p[k] == '"' || p[k] == '\r') return NSF_CSV_BAD_LINE;
  return NSF_CSV_BAD_FIELD;
}

// One field p[0 .. n) -> *v, returns its NSF_CSV_KIND_*.  For an unaccepted field *why holds the NSF_CSV_BAD_* bit.
__host__ __device__ __forceinline__ int parse_field(const char* p, int n, double* v, uint32_t* why) {
  *v = 0.0;
  *why = 0;
  if (n == 0) { *v = from_bits(0x7ff8000000000000ull); return NSF_CSV_KIND_EMPTY; }
  int i = 0;
  const bool neg = p[0] == '-';
  if (neg || p[0] == '+') i = 1;
  if (n - i == 3 && p[0] != '+' && p[i] == 'i' && p[i + 1] == 'n' && p[i + 2] == 'f') {
    *v = from_bits(neg ? 0xfff0000000000000ull : 0x7ff0000000000000ull);
    return NSF_CSV_KIND_INF;
  }
  if (n > kFieldMax) { *why = field_fault(p, n); return NSF_CSV_KIND_BAD; }
  uint64_t acc = 0;
  double number = 0.0;
  int nd = 0, ndig = 0, exponent = 0, ndec = 0;
  bool integer = true;
  // digit d of the mantissa: number = number * 10 + d while fewer than 17 digits are in
  auto push = [&](int d) {
    if (nd < 15) {
      acc = acc * 10 + static_cast<uint64_t>(d);
    } else {
      if (nd == 15) number = static_cast<double>(acc);
      number = add_rn(mul_rn(number, 10.0), static_cast<double>(d));
    }
    ++nd;
  };
  for (; i < n && is_digit(p[i]); ++i, ++ndig) {
    if (nd < 17) push(p[i] - '0');
    else ++exponent;
  }
  if (i < n && p[i] == '.') {
    integer = false;
    for (++i; i < n && is_digit(p[i]); ++i, ++ndig)
      if (nd < 17) { push(p[i] - '0'); ++ndec; }
    exponent -= ndec;
  }
  if (nd <= 15) number = static_cast<double>(acc);
  if (ndig == 0) { *why = field_fault(p, n); return NSF_CSV_KIND_BAD; }
  if (neg) number = -number;
  if (i < n && (p[i] == 'e' || p[i] == 'E')) {
    integer = false;
    ++i;
    const bool eneg = i < n && p[i] == '-';
    if (i < n && (p[i] == '-' || p[i] == '+')) ++i;
    int en = 0, ed = 0;
    for (; i < n && is_digit(p[i]); ++i, ++ed) {
      en = en * 10 + (p[i] - '0');
      if (en > 99999) { *why = NSF_CSV_BAD_FIELD; return NSF_CSV_KIND_BAD; }
    }
    if (ed == 0) { *why = field_fault(p, n); return NSF_CSV_KIND_BAD; }
    exponent += eneg ? -en : en;
  }
  if (i != n) { *why = field_fault(p, n); return NSF_CSV_KIND_BAD; }
  // pandas types a column of integer literals as int64; beyond 15 digits its value is no longer the double's
  if (integer && ndig > 15) { *why = NSF_CSV_BAD_INT; return NSF_CSV_KIND_BAD; }
  if (exponent > 308) { *why = NSF_CSV_BAD_FIELD; return NSF_CSV_KIND_BAD; }
  if (exponent > 0) number = mul_rn(number, e10(exponent));
  else if (exponent < -308) number = exponent < -616 ? 0.0 : div_rn(div_rn(number, e10(-308 - exponent)), e10(308));
  else number = div_rn(number, e10(-exponent));
  if (number == from_bits(0x7ff0000000000000ull) || number == from_bits(0xfff0000000000000ull)) { *why = NSF_CSV_BAD_FIELD; return NSF_CSV_KIND_BAD; }
  *v = number;
  return integer ? NSF_CSV_KIND_INTEGER : NSF_CSV_KIND_NUMBER;
}

// Byte p of file [fb, fe) as the row index sees it: '\n' at fe (a last line without its newline ends there),
// 0 outside the file.
__device__ __forceinline__ uint32_t text_byte(const char* text, int64_t p, int64_t fb, int64_t fe) {
  if (p == fe) return '\n';
  return (p >= fb && p < fe) ? static_cast<uint8_t>(__ldg(text + p)) : 0u;
}

// 16 bytes at the 16-aligned position w, bytes at or past `fe` read as '\n' and bytes before `fb` as 0; one 16-byte
// load when the word lies inside [fb, fe).
__device__ __forceinline__ uint4 load_word(const char* text, int64_t w, int64_t fb, int64_t fe) {
  if (w >= fb && w + 16 <= fe) return __ldg(reinterpret_cast<const uint4*>(text + w));
  uint32_t r[4] = {0, 0, 0, 0};
  for (int k = 0; k < 16; ++k) {
    const int64_t p = w + k;
    const uint32_t c = p >= fe ? '\n' : (p >= fb ? static_cast<uint8_t>(__ldg(text + p)) : 0u);
    r[k >> 2] |= c << (8 * (k & 3));
  }
  return make_uint4(r[0], r[1], r[2], r[3]);
}

__device__ __forceinline__ uint32_t byte_of(const uint4& w, int k) {
  const uint32_t x = k < 4 ? w.x : k < 8 ? w.y : k < 12 ? w.z : w.w;
  return (x >> (8 * (k & 3))) & 0xffu;
}

struct Tile { int64_t fb, fe, lo, hi; int file; };   // file bytes, tile bytes [lo, hi)

__device__ __forceinline__ Tile tile_of(const CsvView& v, int64_t t) {
  Tile r;
  r.file = find_segment(v.tile_off, v.n_files, t);
  r.fb = __ldg(v.text_off + r.file);
  r.fe = __ldg(v.text_off + r.file + 1);
  const int64_t a = (r.fb / kCsvTile + (t - __ldg(v.tile_off + r.file))) * kCsvTile;
  r.lo = max(r.fb, a);
  r.hi = min(r.fe, a + kCsvTile);
  return r;
}

// Bit k: byte base + k (k < 64) starts a data row - the first byte of a line after the header line that is not
// blank (empty once a '\r' before its '\n' is dropped) - and lies in [lo, hi).
__device__ __forceinline__ uint64_t row_starts(const char* text, const Tile& t, int64_t base) {
  if (base + 64 <= t.lo || base >= t.hi) return 0;
  uint64_t nl = 0, cr = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint4 w = load_word(text, base + 16 * q, t.fb, t.fe);
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t c = byte_of(w, k);
      nl |= static_cast<uint64_t>(c == '\n') << (16 * q + k);
      cr |= static_cast<uint64_t>(c == '\r') << (16 * q + k);
    }
  }
  const uint64_t prev = text_byte(text, base - 1, t.fb, t.fe) == '\n';
  const uint64_t next = text_byte(text, base + 64, t.fb, t.fe) == '\n';
  const uint64_t start = (nl << 1) | prev;
  const uint64_t blank = nl | (cr & ((nl >> 1) | (next << 63)));
  uint64_t valid = ~uint64_t(0);
  if (t.lo > base) valid &= ~uint64_t(0) << (t.lo - base);
  if (t.hi < base + 64) valid &= ~uint64_t(0) >> (base + 64 - t.hi);
  return start & ~blank & valid;
}

__global__ void __launch_bounds__(kTileThreads) k_csv_count(CsvView v, int32_t* __restrict__ tile_rows) {
  const Tile t = tile_of(v, blockIdx.x);
  const int64_t base = t.lo / kCsvTile * kCsvTile + 64 * threadIdx.x;
  const int c = block_sum<kTileThreads>(__popcll(row_starts(v.text, t, base)));
  if (threadIdx.x == 0) tile_rows[blockIdx.x] = c;
}

// One block: tile_start[t] = data rows before tile t (n_tiles + 1 entries); row_off[i] = rows before file i.  With
// `given`, a file whose row count differs from the caller's row offsets is marked NSF_CSV_BAD_ROWS.
__global__ void __launch_bounds__(kScanThreads) k_csv_scan(CsvView v, const int32_t* __restrict__ tile_rows,
                                                           int64_t* __restrict__ tile_start, int64_t* __restrict__ row_off,
                                                           const int64_t* __restrict__ given, uint32_t* __restrict__ status) {
  const int64_t n = v.n_tiles, total = scan_counts<kScanThreads>(tile_rows, n, tile_start);
  if (threadIdx.x == 0) tile_start[n] = total;
  __syncthreads();
  for (int i = threadIdx.x; i <= v.n_files; i += kScanThreads) {
    const int64_t r = tile_start[__ldg(v.tile_off + i)];
    if (row_off) row_off[i] = r;
    if (given && r != __ldg(given + i)) {
      if (i < v.n_files) atomicOr(status + i, NSF_CSV_BAD_ROWS);
      if (i > 0) atomicOr(status + i - 1, NSF_CSV_BAD_ROWS);
    }
  }
}

// row_start[r] = byte position of data row r, for r < n_rows.
__global__ void __launch_bounds__(kTileThreads) k_csv_starts(CsvView v, const int64_t* __restrict__ tile_start,
                                                             int64_t n_rows, int64_t* __restrict__ row_start) {
  const Tile t = tile_of(v, blockIdx.x);
  const int64_t base = t.lo / kCsvTile * kCsvTile + 64 * threadIdx.x;
  uint64_t m = row_starts(v.text, t, base);
  int64_t total;
  int64_t r = tile_start[blockIdx.x] + block_exclusive_scan<kTileThreads>(int64_t(__popcll(m)), &total);
  for (; m; m &= m - 1, ++r)
    if (r < n_rows) row_start[r] = base + __ffsll(static_cast<long long>(m)) - 1;
}

template <typename T> __device__ __forceinline__ T out_value(double x);
template <> __device__ __forceinline__ float out_value<float>(double x) { return __double2float_rn(x); }
template <> __device__ __forceinline__ double out_value<double>(double x) { return x; }

// One warp per row (grid-stride).  A window holds 512 bytes from the 16-byte word of the first unfinished field;
// every field whose separator (',' or the line end) lies in the window is parsed by one lane, and the next window
// starts after the last separator.  A window without a separator holds a field longer than any accepted one.
template <typename T>
__global__ void __launch_bounds__(32 * kFieldWarps) k_csv_fields(CsvView v, const int64_t* __restrict__ row_start,
                                                                 T* __restrict__ out, int64_t out_ld,
                                                                 uint32_t* __restrict__ col_flags,
                                                                 uint32_t* __restrict__ status) {
  __shared__ __align__(16) char s_win[kFieldWarps][kWin];
  __shared__ int16_t s_term[kFieldWarps][kWin];
  const int lane = threadIdx.x & 31, wb = threadIdx.x >> 5;
  char* win = s_win[wb];
  int16_t* term = s_term[wb];
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * kFieldWarps + wb; r < v.n_rows;
       r += static_cast<int64_t>(gridDim.x) * kFieldWarps) {
    const int f = find_segment(v.row_off, v.n_files, r);
    const int64_t fb = __ldg(v.text_off + f), fe = __ldg(v.text_off + f + 1);
    int64_t cur = row_start[r];
    uint32_t bad = 0;
    if (cur <= fb || cur >= fe) bad = NSF_CSV_BAD_ROWS;    // only with row offsets that do not match the text
    T* orow = out + r * out_ld;
    int col0 = 0;
    while (!bad) {
      const int64_t base = cur & ~int64_t(15);
      const uint4 w = load_word(v.text, base + 16 * lane, fb, fe);
      *reinterpret_cast<uint4*>(win + 16 * lane) = w;
      uint32_t comma = 0, nl = 0;
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const uint32_t c = byte_of(w, k);
        const bool live = base + 16 * lane + k >= cur;
        comma |= static_cast<uint32_t>(live && c == ',') << k;
        nl |= static_cast<uint32_t>(live && c == '\n') << k;
      }
      const uint32_t nl_lanes = __ballot_sync(0xffffffffu, nl != 0);
      int end = kWin;                                      // window offset of the line end, kWin if not in it
      if (nl_lanes) {
        const int l = __ffs(nl_lanes) - 1;
        end = 16 * l + __ffs(__shfl_sync(0xffffffffu, nl, l)) - 1;
      }
      const int mine = end - 16 * lane;                    // separators of this lane: bytes before `end`, and `end`
      uint32_t tm = comma & (mine >= 16 ? 0xffffu : mine <= 0 ? 0u : (1u << mine) - 1);
      if (mine >= 0 && mine < 16) tm |= 1u << mine;
      const int cnt = __popc(tm);
      const int incl = warp_inclusive_scan(cnt);
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      for (int k = incl - cnt; tm; tm &= tm - 1, ++k) term[k] = static_cast<int16_t>(16 * lane + __ffs(tm) - 1);
      __syncwarp();
      if (total == 0) { bad = NSF_CSV_BAD_FIELD; break; }
      const bool line_end = end < kWin;
      for (int k = lane; k < total; k += 32) {
        const int col = col0 + k;
        if (col >= v.cols) { bad |= NSF_CSV_BAD_SHAPE; break; }
        const int a = k == 0 ? static_cast<int>(cur - base) : term[k - 1] + 1;
        int b = term[k];
        if (line_end && k == total - 1 && b > a && win[b - 1] == '\r') --b;
        const int oc = __ldg(v.out_col + col);
        if (oc < 0) {   // a dropped field is not parsed, only checked for what changes the tokenisation
          for (int i = a; i < b; ++i) {
            const uint8_t c = static_cast<uint8_t>(win[i]);
            if (c == '"' || c == '\r') bad |= NSF_CSV_BAD_LINE;
            else if (c < 0x20 || c >= 0x80) bad |= NSF_CSV_BAD_FIELD;
          }
          continue;
        }
        double x;
        uint32_t why;
        const int kind = parse_field(win + a, b - a, &x, &why);
        if (kind == NSF_CSV_KIND_BAD) { bad |= why; continue; }
        orow[oc] = out_value<T>(x);
        const uint32_t fl = kind != NSF_CSV_KIND_INTEGER ? kNonInt : (x == 0.0 && signbit(x)) ? kNegZeroInt : 0u;
        uint32_t* pf = col_flags + static_cast<int64_t>(f) * v.cols + col;
        if (fl && (__ldcg(pf) & fl) != fl) atomicOr(pf, fl);
      }
      __syncwarp();
      if (line_end) {
        if (col0 + total != v.cols) bad |= NSF_CSV_BAD_SHAPE;
        break;
      }
      col0 += total;
      if (col0 >= v.cols) bad |= NSF_CSV_BAD_SHAPE;       // another field follows
      cur = base + term[total - 1] + 1;
      bad = __reduce_or_sync(0xffffffffu, bad);
      __syncwarp();                                      // term[] is read above before the next window rewrites it
    }
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0 && bad) atomicOr(status + f, bad);
    __syncwarp();
  }
}

// One block per file.  A column whose every field is an integer literal is int64 in pandas, so its -0 is +0.  A -0
// literal in a column that also holds other fields has the sign of whatever type pandas' chunked reader (low_memory)
// gave the chunk it fell in, which depends on the file's size: such a file is not accepted.
template <typename T>
__global__ void __launch_bounds__(256) k_csv_int_zero(CsvView v, T* __restrict__ out, int64_t out_ld,
                                                      const uint32_t* __restrict__ col_flags,
                                                      uint32_t* __restrict__ status) {
  const int f = blockIdx.x;
  const int64_t r0 = __ldg(v.row_off + f), r1 = __ldg(v.row_off + f + 1);
  for (int c = 0; c < v.cols; ++c) {
    const uint32_t fl = col_flags[static_cast<int64_t>(f) * v.cols + c];
    const int oc = __ldg(v.out_col + c);
    if (oc < 0 || !(fl & kNegZeroInt)) continue;
    if (fl & kNonInt) {
      if (threadIdx.x == 0) atomicOr(status + f, NSF_CSV_BAD_INT);
      continue;
    }
    for (int64_t r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
      T* p = out + r * out_ld + oc;
      if (*p == T(0)) *p = T(0);
    }
  }
}

}  // namespace

int64_t csv_tiles(int64_t begin, int64_t end) {
  return end > begin ? (end - 1) / kCsvTile - begin / kCsvTile + 1 : 0;
}

int launch_csv_row_offsets(cudaStream_t s, const CsvView& v, int32_t* tile_rows, int64_t* tile_start, int64_t* row_off) {
  if (v.n_tiles > 0) {
    k_csv_count<<<static_cast<unsigned>(v.n_tiles), kTileThreads, 0, s>>>(v, tile_rows);
    NSF_CHECK_LAUNCH();
  }
  k_csv_scan<<<1, kScanThreads, 0, s>>>(v, tile_rows, tile_start, row_off, nullptr, nullptr);
  NSF_CHECK_LAUNCH();
  return v.n_tiles > 0 ? 2 : 1;
}

int launch_csv_parse(cudaStream_t s, const CsvView& v, int dtype, int32_t* tile_rows, int64_t* tile_start,
                     int64_t* row_start, uint32_t* col_flags, void* out, int64_t out_ld, uint32_t* status) {
  int m = 0;
  if (v.n_tiles > 0) {
    k_csv_count<<<static_cast<unsigned>(v.n_tiles), kTileThreads, 0, s>>>(v, tile_rows);
    NSF_CHECK_LAUNCH();
    ++m;
  }
  k_csv_scan<<<1, kScanThreads, 0, s>>>(v, tile_rows, tile_start, nullptr, v.row_off, status);
  NSF_CHECK_LAUNCH();
  ++m;
  if (v.n_rows == 0 || v.n_tiles == 0) return m;   // (rows without text: the scan has marked every file)
  k_csv_starts<<<static_cast<unsigned>(v.n_tiles), kTileThreads, 0, s>>>(v, tile_start, v.n_rows, row_start);
  NSF_CHECK_LAUNCH();
  const int64_t blocks = std::min<int64_t>((v.n_rows + kFieldWarps - 1) / kFieldWarps, int64_t(kSmCount) * 8);
  if (dtype == NSF_F64) {
    k_csv_fields<double><<<static_cast<unsigned>(blocks), 32 * kFieldWarps, 0, s>>>(
        v, row_start, static_cast<double*>(out), out_ld, col_flags, status);
    NSF_CHECK_LAUNCH();
    k_csv_int_zero<double><<<v.n_files, 256, 0, s>>>(v, static_cast<double*>(out), out_ld, col_flags, status);
  } else {
    k_csv_fields<float><<<static_cast<unsigned>(blocks), 32 * kFieldWarps, 0, s>>>(
        v, row_start, static_cast<float*>(out), out_ld, col_flags, status);
    NSF_CHECK_LAUNCH();
    k_csv_int_zero<float><<<v.n_files, 256, 0, s>>>(v, static_cast<float*>(out), out_ld, col_flags, status);
  }
  NSF_CHECK_LAUNCH();
  return m + 3;
}

}  // namespace nsf

extern "C" {

nsf_status nsf_parse_check(const char* text, const int64_t* field_offsets, int64_t n, double* values, int32_t* kinds) {
  if (!text || !field_offsets || !values || !kinds || n < 0) { nsf::set_error("nsf_parse_check: bad argument"); return NSF_ERR_BAD_ARG; }
  for (int64_t i = 0; i < n; ++i)
    if (field_offsets[i + 1] < field_offsets[i]) { nsf::set_error("nsf_parse_check: offsets must be non-decreasing"); return NSF_ERR_BAD_ARG; }
  for (int64_t i = 0; i < n; ++i) {
    const int64_t len = field_offsets[i + 1] - field_offsets[i];
    uint32_t why;
    // any length above kFieldMax is unaccepted alike; the clamp keeps it an int
    kinds[i] = nsf::parse_field(text + field_offsets[i], static_cast<int>(len > 64 ? 64 : len), values + i, &why);
  }
  return NSF_OK;
}

}  // extern "C"

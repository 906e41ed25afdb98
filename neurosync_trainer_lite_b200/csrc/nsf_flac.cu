// FLAC frame decoding (RFC 9639) behind nsf_flac_decode_host; see include/nsf.h for the contract.  The metadata blocks
// are parsed on the host (load_audio.flac_layout); the frames are found and decoded here.
//
// Frames carry no index, so their positions come from the data: every byte pair 0xFF 0xF8/0xF9 whose header parses and
// passes its CRC-8 is a candidate.  Kernels of one stream group:
//   k_flac_count      one block per kFlacScanTile scan positions: candidates in the tile
//   k_flac_scan       one block: exclusive scan of the tile counts, and the candidate total
//   k_flac_write      one block per tile: the candidates' scan positions, in byte order (no atomics)
//   k_flac_parse      one thread per candidate: decodes the frame bit by bit without keeping samples, records where
//                     it ends, whether its CRC-16 matches and where each subframe starts
// The host then walks each stream's frame chain over the candidate table (the first frame at the stream's first byte,
// each next one where the previous ended), so a false sync inside compressed data never reaches the output, and
// uploads the kept frames:
//   k_flac_decode     one thread per kept (frame, channel): residual + FIXED / LPC recurrence in int64, wasted bits
//   k_flac_interleave one thread per output frame: inter-channel decorrelation, WAV container bytes
// The bit reader, header parser and frame decoder are __host__ __device__: nsf_flac_check runs them on the CPU.
#include <cstdint>
#include <cstring>

#include "nsf.h"
#include "nsf_internal.h"
#include "nsf_kernels.cuh"

#define NSF_CHECK_LAUNCH() \
  do { if (cudaGetLastError() != cudaSuccess) return -1; } while (0)

#define HD __host__ __device__ __forceinline__

namespace nsf {
namespace {

constexpr int kParseThreads = 64;
constexpr int kMaxLpcOrder = 32;

HD int clz64(uint64_t v) {
#ifdef __CUDA_ARCH__
  return __clzll(static_cast<long long>(v));
#else
  return __builtin_clzll(v);
#endif
}

// CRC-8 (poly 0x07, init 0) of a header: at most 16 bytes, bitwise.
HD uint8_t crc8(const uint8_t* p, int n) {
  uint32_t c = 0;
  for (int i = 0; i < n; ++i) {
    c ^= p[i];
    for (int b = 0; b < 8; ++b) c = (c & 0x80) ? ((c << 1) ^ 0x07) & 0xFF : (c << 1) & 0xFF;
  }
  return static_cast<uint8_t>(c);
}
// Entry b of the CRC-16 (poly 0x8005, init 0, not reflected) byte table.
HD uint16_t crc16_entry(uint32_t b) {
  uint32_t c = b << 8;
  for (int i = 0; i < 8; ++i) c = (c & 0x8000) ? ((c << 1) ^ 0x8005) & 0xFFFF : (c << 1) & 0xFFFF;
  return static_cast<uint16_t>(c);
}

// Big-endian bit reader over bytes [.., end) of `p`: a 64-bit cache holding `nbits` valid bits at its top.  A read past
// `end` sets `bad` and yields zeros, so a corrupt or false frame never reads outside its stream.
struct BitReader {
  const uint8_t* p;
  int64_t byte, end;
  uint64_t cache;
  int nbits;
  bool bad;
  HD void init(const uint8_t* base, int64_t first_byte, int64_t end_byte) {
    p = base; byte = first_byte; end = end_byte; cache = 0; nbits = 0; bad = false;
  }
  HD void refill() {
    while (nbits <= 56 && byte < end) { cache |= static_cast<uint64_t>(p[byte++]) << (56 - nbits); nbits += 8; }
  }
  HD uint32_t bits(int n) {     // 0 <= n <= 32
    if (n == 0) return 0;
    if (nbits < n) { refill(); if (nbits < n) { bad = true; cache = 0; nbits = 0; return 0; } }
    const uint32_t v = static_cast<uint32_t>(cache >> (64 - n));
    cache = n == 64 ? 0 : cache << n;
    nbits -= n;
    return v;
  }
  HD int32_t sbits(int n) {     // two's complement of n bits, 0 <= n <= 32
    if (n == 0) return 0;
    const uint32_t v = bits(n);
    return n == 32 ? static_cast<int32_t>(v) : static_cast<int32_t>(v << (32 - n)) >> (32 - n);
  }
  HD uint32_t unary() {         // zeros up to the next one (consumed); the zero count, capped at 2^32 - 1
    uint64_t q = 0;
    for (;;) {
      if (nbits == 0) { refill(); if (nbits == 0) { bad = true; return 0; } }
      if (cache == 0) { q += nbits; nbits = 0; if (q > 0xFFFFFFFFull) { bad = true; return 0; } continue; }
      const int z = clz64(cache);
      q += z;
      cache = z + 1 >= 64 ? 0 : cache << (z + 1);
      nbits -= z + 1;
      return q > 0xFFFFFFFFull ? 0xFFFFFFFFu : static_cast<uint32_t>(q);
    }
  }
  HD void align() { const int r = nbits & 7; cache = r ? cache << r : cache; nbits -= r; }
  HD int64_t bitpos() const { return byte * 8 - nbits; }
};

struct Header {
  int64_t number;
  int32_t block, rate, bits, assignment, channels, variable, length, fields;   // fields: NSF_FLAC_* of the field codes
};

// The frame header at d[pos]: NSF_FLAC_OK when the sync code, the coded number and the CRC-8 are right (the field codes
// are judged separately, in h->fields).  si_rate / si_bits stand in for the codes that defer to STREAMINFO.
HD int parse_header(const uint8_t* d, int64_t pos, int64_t end, int32_t si_rate, int32_t si_bits, Header* h) {
  if (pos + 2 > end) return NSF_FLAC_TRUNCATED;
  if (d[pos] != 0xFF || (d[pos + 1] & 0xFE) != 0xF8) return NSF_FLAC_NO_SYNC;
  if (pos + 5 > end) return NSF_FLAC_TRUNCATED;
  h->variable = d[pos + 1] & 1;
  const int bs_code = d[pos + 2] >> 4, sr_code = d[pos + 2] & 15, ch_code = d[pos + 3] >> 4;
  const int ss_code = (d[pos + 3] >> 1) & 7, zero = d[pos + 3] & 1;
  // coded number, UTF-8 style: at most 6 bytes (36 bits) for a frame number, 7 for a sample number
  int64_t q = pos + 4;
  const uint32_t c0 = d[q++];
  int extra;
  uint64_t v;
  if (c0 < 0x80) { extra = 0; v = c0; }
  else if ((c0 & 0xE0) == 0xC0) { extra = 1; v = c0 & 0x1F; }
  else if ((c0 & 0xF0) == 0xE0) { extra = 2; v = c0 & 0x0F; }
  else if ((c0 & 0xF8) == 0xF0) { extra = 3; v = c0 & 0x07; }
  else if ((c0 & 0xFC) == 0xF8) { extra = 4; v = c0 & 0x03; }
  else if ((c0 & 0xFE) == 0xFC) { extra = 5; v = c0 & 0x01; }
  else if (c0 == 0xFE) { extra = 6; v = 0; }
  else return NSF_FLAC_BAD_NUMBER;
  if (extra == 6 && !h->variable) return NSF_FLAC_BAD_NUMBER;
  if (q + extra > end) return NSF_FLAC_TRUNCATED;
  for (int i = 0; i < extra; ++i) {
    const uint32_t c = d[q++];
    if ((c & 0xC0) != 0x80) return NSF_FLAC_BAD_NUMBER;
    v = (v << 6) | (c & 0x3F);
  }
  h->number = static_cast<int64_t>(v);
  const int bs_bytes = bs_code == 6 ? 1 : bs_code == 7 ? 2 : 0;
  const int sr_bytes = sr_code == 12 ? 1 : (sr_code == 13 || sr_code == 14) ? 2 : 0;
  if (q + bs_bytes + sr_bytes + 1 > end) return NSF_FLAC_TRUNCATED;
  uint32_t bs_raw = 0, sr_raw = 0;
  for (int i = 0; i < bs_bytes; ++i) bs_raw = (bs_raw << 8) | d[q++];
  for (int i = 0; i < sr_bytes; ++i) sr_raw = (sr_raw << 8) | d[q++];
  if (crc8(d + pos, static_cast<int>(q - pos)) != d[q]) return NSF_FLAC_BAD_CRC8;
  h->length = static_cast<int32_t>(q + 1 - pos);
  // field codes
  int fields = zero ? NSF_FLAC_RESERVED : NSF_FLAC_OK;
  if (bs_code == 0) { fields = NSF_FLAC_RESERVED; h->block = 0; }
  else if (bs_code == 1) h->block = 192;
  else if (bs_code <= 5) h->block = 576 << (bs_code - 2);
  else if (bs_code <= 7) h->block = static_cast<int32_t>(bs_raw) + 1;
  else h->block = 256 << (bs_code - 8);
  if (h->block > 65535) fields = NSF_FLAC_RESERVED;
  const int32_t rates[12] = {0, 88200, 176400, 192000, 8000, 16000, 22050, 24000, 32000, 44100, 48000, 96000};
  if (sr_code == 0) h->rate = si_rate;
  else if (sr_code < 12) h->rate = rates[sr_code];
  else if (sr_code == 12) h->rate = static_cast<int32_t>(sr_raw) * 1000;
  else if (sr_code == 13) h->rate = static_cast<int32_t>(sr_raw);
  else if (sr_code == 14) h->rate = static_cast<int32_t>(sr_raw) * 10;
  else { h->rate = 0; fields = NSF_FLAC_RESERVED; }
  h->assignment = ch_code;
  if (ch_code < 8) h->channels = ch_code + 1;
  else if (ch_code <= 10) h->channels = 2;
  else { h->channels = 0; fields = NSF_FLAC_RESERVED; }
  const int32_t sizes[8] = {0, 8, 12, 0, 16, 20, 24, 32};
  if (ss_code == 0) h->bits = si_bits;
  else if (ss_code == 3) { h->bits = 0; fields = NSF_FLAC_RESERVED; }
  else h->bits = sizes[ss_code];
  h->fields = fields;
  return NSF_FLAC_OK;
}

// Rice-coded residual of a subframe: block - order values into res (NULL: parsed and checked only).
HD int read_residual(BitReader& br, int block, int order, int32_t* res) {
  const uint32_t method = br.bits(2);
  if (method >= 2) return br.bad ? NSF_FLAC_TRUNCATED : NSF_FLAC_RESERVED;
  const int pbits = method ? 5 : 4;
  const uint32_t escape = (1u << pbits) - 1;
  const int po = static_cast<int>(br.bits(4));
  if (br.bad) return NSF_FLAC_TRUNCATED;
  const int parts = 1 << po, psz = block >> po;
  if ((block & (parts - 1)) != 0 || psz < order) return NSF_FLAC_PARTITION;
  int i = 0;
  for (int part = 0; part < parts; ++part) {
    const int n = part == 0 ? psz - order : psz;
    const uint32_t k = br.bits(pbits);
    if (k == escape) {
      const int w = static_cast<int>(br.bits(5));
      for (int j = 0; j < n; ++j, ++i) {
        const int32_t v = br.sbits(w);
        if (res) res[i] = v;
      }
    } else {
      for (int j = 0; j < n; ++j, ++i) {
        const uint64_t u = (static_cast<uint64_t>(br.unary()) << k) | br.bits(static_cast<int>(k));
        if (u > 0xFFFFFFFFull) return br.bad ? NSF_FLAC_TRUNCATED : NSF_FLAC_RANGE;
        const uint32_t u32 = static_cast<uint32_t>(u);
        if (res) res[i] = static_cast<int32_t>((u32 >> 1) ^ (0u - (u32 & 1)));
      }
    }
    if (br.bad) return NSF_FLAC_TRUNCATED;
  }
  return NSF_FLAC_OK;
}

// One subframe of `bps` bits (side channel included) and `block` samples: decoded into out[0, block) when out != NULL,
// else parsed and checked only.
HD int read_subframe(BitReader& br, int bps, int block, int32_t* out) {
  const uint32_t zero = br.bits(1), type = br.bits(6), wasted_flag = br.bits(1);
  if (br.bad) return NSF_FLAC_TRUNCATED;
  if (zero) return NSF_FLAC_RESERVED;
  int wasted = 0;
  if (wasted_flag) {
    const uint32_t k = br.unary();
    if (br.bad) return NSF_FLAC_TRUNCATED;
    if (k + 1 >= static_cast<uint32_t>(bps)) return NSF_FLAC_WASTED;
    wasted = static_cast<int>(k) + 1;
  }
  bps -= wasted;
  if (type == 0) {                                       // CONSTANT
    const int32_t v = br.sbits(bps);
    if (br.bad) return NSF_FLAC_TRUNCATED;
    if (out) for (int i = 0; i < block; ++i) out[i] = v;
  } else if (type == 1) {                                // VERBATIM
    for (int i = 0; i < block; ++i) {
      const int32_t v = br.sbits(bps);
      if (out) out[i] = v;
    }
    if (br.bad) return NSF_FLAC_TRUNCATED;
  } else if (type >= 8 && type <= 12) {                  // FIXED, order 0..4
    const int order = static_cast<int>(type) - 8;
    if (order > block) return NSF_FLAC_PARTITION;
    for (int i = 0; i < order; ++i) {
      const int32_t v = br.sbits(bps);
      if (out) out[i] = v;
    }
    const int st = read_residual(br, block, order, out ? out + order : nullptr);
    if (st != NSF_FLAC_OK) return st;
    if (out) {
      for (int i = order; i < block; ++i) {
        int64_t pred = 0;
        switch (order) {
          case 1: pred = out[i - 1]; break;
          case 2: pred = 2 * int64_t(out[i - 1]) - out[i - 2]; break;
          case 3: pred = 3 * int64_t(out[i - 1]) - 3 * int64_t(out[i - 2]) + out[i - 3]; break;
          case 4: pred = 4 * int64_t(out[i - 1]) - 6 * int64_t(out[i - 2]) + 4 * int64_t(out[i - 3]) - out[i - 4]; break;
          default: break;
        }
        out[i] = static_cast<int32_t>(pred + out[i]);
      }
    }
  } else if (type >= 32) {                               // LPC, order 1..32
    const int order = static_cast<int>(type) - 31;
    if (order > block) return NSF_FLAC_PARTITION;
    for (int i = 0; i < order; ++i) {
      const int32_t v = br.sbits(bps);
      if (out) out[i] = v;
    }
    const int precision = static_cast<int>(br.bits(4)) + 1;
    const int shift = br.sbits(5);
    if (br.bad) return NSF_FLAC_TRUNCATED;
    if (precision == 16) return NSF_FLAC_RESERVED;
    if (shift < 0) return NSF_FLAC_LPC_SHIFT;
    int32_t coef[kMaxLpcOrder];
    for (int j = 0; j < order; ++j) coef[j] = br.sbits(precision);
    const int st = read_residual(br, block, order, out ? out + order : nullptr);
    if (st != NSF_FLAC_OK) return st;
    if (out) {
      for (int i = order; i < block; ++i) {
        int64_t sum = 0;
        for (int j = 0; j < order; ++j) sum += static_cast<int64_t>(coef[j]) * out[i - 1 - j];
        out[i] = static_cast<int32_t>(out[i] + (sum >> shift));
      }
    }
  } else {
    return NSF_FLAC_RESERVED;
  }
  if (out && wasted)
    for (int i = 0; i < block; ++i) out[i] = static_cast<int32_t>(static_cast<uint32_t>(out[i]) << wasted);
  return NSF_FLAC_OK;
}

// Bits of channel c's subframe: the side channel of a stereo decorrelation carries one bit more.
HD int subframe_bits(int bits, int assignment, int c) {
  return bits + ((assignment == 8 && c == 1) || (assignment == 9 && c == 0) || (assignment == 10 && c == 1) ? 1 : 0);
}

// Left and right of a decorrelated stereo pair (a, b) = (channel 0, channel 1).
HD void decorrelate(int assignment, int32_t a, int32_t b, int32_t* l, int32_t* r) {
  const int64_t x = a, y = b;
  if (assignment == 8) { *l = a; *r = static_cast<int32_t>(x - y); }            // left/side
  else if (assignment == 9) { *l = static_cast<int32_t>(x + y); *r = b; }       // side/right
  else if (assignment == 10) {                                                  // mid/side
    const int64_t mid = x * 2 + (y & 1);
    *l = static_cast<int32_t>((mid + y) >> 1);
    *r = static_cast<int32_t>((mid - y) >> 1);
  } else { *l = a; *r = b; }
}

// The frame at d[pos] of stream `st` (bytes before st.end): header, every subframe (decoded into
// out[c * block + i] when out != NULL, before decorrelation), padding and CRC-16.  The candidate's fields are filled
// as far as the decode got; the status is the first failure, NSF_FLAC_OK for a good frame.
HD int decode_frame(const uint8_t* d, int64_t pos, const FlacStream& st, const uint16_t* crc_tab, FlacCand* fc,
                    int32_t* out) {
  Header h;
  fc->start = pos;
  fc->end = pos;
  fc->number = 0; fc->block = 0; fc->assignment = 0;
  int status = parse_header(d, pos, st.end, st.sample_rate, st.bits, &h);
  if (status != NSF_FLAC_OK) return fc->status = status;
  fc->number = h.number;
  fc->block = h.block;
  fc->assignment = h.assignment | (h.variable << 4);
  if (h.fields != NSF_FLAC_OK) return fc->status = h.fields;
  if (h.channels != st.channels) return fc->status = NSF_FLAC_CHANNELS;
  if (h.bits != st.bits) return fc->status = NSF_FLAC_BITS;
  if (h.rate != st.sample_rate) return fc->status = NSF_FLAC_RATE;
  if (h.block > st.max_block) return fc->status = NSF_FLAC_BLOCK;
  BitReader br;
  br.init(d, pos + h.length, st.end);
  for (int c = 0; c < h.channels; ++c) {
    fc->sub_bit[c] = static_cast<uint32_t>(br.bitpos() - pos * 8);
    status = read_subframe(br, subframe_bits(h.bits, h.assignment, c), h.block, out ? out + c * h.block : nullptr);
    if (status != NSF_FLAC_OK) return fc->status = status;
  }
  br.align();
  const int64_t crc_at = br.bitpos() / 8;
  const uint32_t stored = br.bits(16);
  if (br.bad) return fc->status = NSF_FLAC_TRUNCATED;
  fc->end = crc_at + 2;
  uint32_t crc = 0;
  for (int64_t i = pos; i < crc_at; ++i) crc = ((crc << 8) & 0xFFFF) ^ crc_tab[((crc >> 8) ^ d[i]) & 0xFF];
  return fc->status = (crc == stored ? NSF_FLAC_OK : NSF_FLAC_BAD_CRC16);
}

// Stream owning scan position p (streams sorted by scan0).
__device__ __forceinline__ int find_stream(const FlacStream* s, int n, int64_t p) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (s[mid].scan0 <= p) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Is scan position p a candidate: a sync code whose header parses and passes its CRC-8?
__device__ __forceinline__ bool is_candidate(const FlacStream* streams, int n, const uint8_t* d, int64_t p) {
  const FlacStream& st = streams[find_stream(streams, n, p)];
  const int64_t pos = st.begin + (p - st.scan0);
  if (d[pos] != 0xFF) return false;
  Header h;
  return parse_header(d, pos, st.end, st.sample_rate, st.bits, &h) == NSF_FLAC_OK;
}

}  // namespace

__global__ void __launch_bounds__(256) k_flac_count(const FlacStream* __restrict__ streams, int n, int64_t total,
                                                    const uint8_t* __restrict__ d, int32_t* __restrict__ blk_count) {
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kFlacScanTile;
  int count = 0;
  for (int i = 0; i < kFlacScanTile; i += 256) {
    const int64_t p = base + i + threadIdx.x;
    count += __syncthreads_count(p < total && is_candidate(streams, n, d, p));
  }
  if (threadIdx.x == 0) blk_count[blockIdx.x] = count;
}

// Exclusive scan of the tile counts by one block of 1024 threads: each thread owns a contiguous run of tiles.
__global__ void __launch_bounds__(1024) k_flac_scan(const int32_t* __restrict__ blk_count, int64_t n_blk,
                                                    int64_t* __restrict__ blk_off, int64_t* __restrict__ cand_total) {
  __shared__ int64_t s[1024];
  const int64_t per = (n_blk + 1023) / 1024, b0 = threadIdx.x * per, b1 = min(b0 + per, n_blk);
  int64_t sum = 0;
  for (int64_t b = b0; b < b1; ++b) sum += blk_count[b];
  s[threadIdx.x] = sum;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    const int64_t v = threadIdx.x >= off ? s[threadIdx.x - off] : 0;
    __syncthreads();
    s[threadIdx.x] += v;
    __syncthreads();
  }
  int64_t run = s[threadIdx.x] - sum;
  for (int64_t b = b0; b < b1; ++b) { blk_off[b] = run; run += blk_count[b]; }
  if (threadIdx.x == 1023) *cand_total = s[1023];
}

// The candidates of a tile at blk_off[tile] + their rank in byte order (position rows of 256, warps in order).
__global__ void __launch_bounds__(256) k_flac_write(const FlacStream* __restrict__ streams, int n, int64_t total,
                                                    const uint8_t* __restrict__ d, const int64_t* __restrict__ blk_off,
                                                    int64_t* __restrict__ cand_pos, int64_t cap) {
  __shared__ int warp_count[8];
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kFlacScanTile;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t next = blk_off[blockIdx.x];
  for (int i = 0; i < kFlacScanTile; i += 256) {
    const int64_t p = base + i + threadIdx.x;
    const bool hit = p < total && is_candidate(streams, n, d, p);
    const unsigned ballot = __ballot_sync(0xFFFFFFFFu, hit);
    if (lane == 0) warp_count[warp] = __popc(ballot);
    __syncthreads();
    int before = 0, row = 0;
    for (int w = 0; w < 8; ++w) { before += w < warp ? warp_count[w] : 0; row += warp_count[w]; }
    if (hit) {
      const int64_t idx = next + before + __popc(ballot & ((1u << lane) - 1));
      if (idx < cap) cand_pos[idx] = p;
    }
    next += row;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kParseThreads) k_flac_parse(const FlacStream* __restrict__ streams, int n,
                                                              const uint8_t* __restrict__ d,
                                                              const int64_t* __restrict__ cand_total,
                                                              const int64_t* __restrict__ cand_pos,
                                                              FlacCand* __restrict__ cand, int64_t cap) {
  __shared__ uint16_t crc_tab[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = crc16_entry(i);
  __syncthreads();
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= min(*cand_total, cap)) return;
  const int64_t p = cand_pos[i];
  const int s = find_stream(streams, n, p);
  FlacCand fc;
  fc.stream = s;
  decode_frame(d, streams[s].begin + (p - streams[s].scan0), streams[s], crc_tab, &fc, nullptr);
  cand[i] = fc;
}

// One thread per (kept frame, channel): the subframe decoded into its scratch rows.  The frame parsed cleanly in
// k_flac_parse, so the reads stay inside the frame.
__global__ void __launch_bounds__(128) k_flac_decode(const FlacStream* __restrict__ streams,
                                                     const FlacCand* __restrict__ cand, const FlacKept* __restrict__ kept,
                                                     int n_kept, int max_channels, const uint8_t* __restrict__ d,
                                                     int32_t* __restrict__ scratch) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t k = t / max_channels;
  const int c = static_cast<int>(t % max_channels);
  if (k >= n_kept) return;
  const FlacKept kf = kept[k];
  const FlacStream& st = streams[kf.stream];
  if (c >= st.channels) return;
  const FlacCand& fc = cand[kf.cand];
  BitReader br;
  const int64_t bit = fc.start * 8 + fc.sub_bit[c];
  br.init(d, bit >> 3, fc.end);
  br.bits(static_cast<int>(bit & 7));
  read_subframe(br, subframe_bits(st.bits, fc.assignment & 15, c), fc.block, scratch + kf.scratch0 +
                static_cast<int64_t>(c) * fc.block);
}

// One thread per output frame g of the group: kept frame by binary search over g0, decorrelation, container bytes.
__global__ void __launch_bounds__(256) k_flac_interleave(const FlacStream* __restrict__ streams,
                                                         const FlacCand* __restrict__ cand,
                                                         const FlacKept* __restrict__ kept, int n_kept, int64_t n_out,
                                                         const int32_t* __restrict__ scratch, uint8_t* __restrict__ out) {
  const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (g >= n_out) return;
  int lo = 0, hi = n_kept - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (kept[mid].g0 <= g) lo = mid; else hi = mid - 1;
  }
  const FlacKept kf = kept[lo];
  const FlacStream& st = streams[kf.stream];
  const int block = cand[kf.cand].block, assignment = cand[kf.cand].assignment & 15;
  const int64_t i = g - kf.g0;
  const int32_t* s = scratch + kf.scratch0 + i;
  const int cb = st.bits >> 3;
  uint8_t* o = out + st.out0 + (kf.first + i) * st.channels * cb;
  int32_t l = s[0], r = 0;
  if (st.channels == 2) decorrelate(assignment, s[0], s[block], &l, &r);
  for (int c = 0; c < st.channels; ++c) {
    const uint32_t v = static_cast<uint32_t>(c == 0 ? l : c == 1 && st.channels == 2 ? r : s[static_cast<int64_t>(c) * block]);
    if (cb == 1) o[c] = static_cast<uint8_t>(v + 128);
    else {
      for (int b = 0; b < cb; ++b) o[c * cb + b] = static_cast<uint8_t>(v >> (8 * b));
    }
  }
}

int launch_flac_scan_parse(cudaStream_t s, const FlacStream* streams, int n_streams, int64_t scan_total,
                           const uint8_t* payload, int32_t* blk_count, int64_t* blk_off, int64_t* cand_total,
                           int64_t* cand_pos, FlacCand* cand, int64_t cap) {
  const int64_t n_blk = (scan_total + kFlacScanTile - 1) / kFlacScanTile;
  if (n_blk <= 0 || n_blk > INT32_MAX || cap <= 0) return -1;
  k_flac_count<<<static_cast<unsigned>(n_blk), 256, 0, s>>>(streams, n_streams, scan_total, payload, blk_count);
  NSF_CHECK_LAUNCH();
  k_flac_scan<<<1, 1024, 0, s>>>(blk_count, n_blk, blk_off, cand_total);
  NSF_CHECK_LAUNCH();
  k_flac_write<<<static_cast<unsigned>(n_blk), 256, 0, s>>>(streams, n_streams, scan_total, payload, blk_off, cand_pos,
                                                            cap);
  NSF_CHECK_LAUNCH();
  k_flac_parse<<<static_cast<unsigned>((cap + kParseThreads - 1) / kParseThreads), kParseThreads, 0, s>>>(
      streams, n_streams, payload, cand_total, cand_pos, cand, cap);
  NSF_CHECK_LAUNCH();
  return 4;
}

int launch_flac_decode(cudaStream_t s, const FlacStream* streams, const FlacCand* cand, const FlacKept* kept,
                       int n_kept, int max_channels, int64_t out_frames, const uint8_t* payload, int32_t* scratch,
                       uint8_t* out) {
  if (n_kept <= 0 || out_frames <= 0) return 0;
  const int64_t threads = static_cast<int64_t>(n_kept) * max_channels;
  k_flac_decode<<<static_cast<unsigned>((threads + 127) / 128), 128, 0, s>>>(streams, cand, kept, n_kept, max_channels,
                                                                              payload, scratch);
  NSF_CHECK_LAUNCH();
  k_flac_interleave<<<static_cast<unsigned>((out_frames + 255) / 256), 256, 0, s>>>(streams, cand, kept, n_kept,
                                                                                    out_frames, scratch, out);
  NSF_CHECK_LAUNCH();
  return 2;
}

int flac_header_status(const uint8_t* payload, int64_t pos, int64_t end) {
  Header h;
  return parse_header(payload, pos, end, 0, 0, &h);
}

const char* flac_status_text(int status) {
  switch (status) {
    case NSF_FLAC_OK: return "ok";
    case NSF_FLAC_NO_SYNC: return "no frame sync code";
    case NSF_FLAC_TRUNCATED: return "truncated frame";
    case NSF_FLAC_BAD_NUMBER: return "malformed coded number";
    case NSF_FLAC_BAD_CRC8: return "header CRC-8 mismatch";
    case NSF_FLAC_RESERVED: return "reserved code";
    case NSF_FLAC_CHANNELS: return "channel count disagrees with STREAMINFO";
    case NSF_FLAC_BITS: return "bits per sample disagree with STREAMINFO";
    case NSF_FLAC_RATE: return "sample rate disagrees with STREAMINFO";
    case NSF_FLAC_BLOCK: return "block size above the STREAMINFO maximum";
    case NSF_FLAC_WASTED: return "wasted bits leave no sample bits";
    case NSF_FLAC_LPC_SHIFT: return "negative LPC shift";
    case NSF_FLAC_PARTITION: return "residual partitions do not fit the block";
    case NSF_FLAC_RANGE: return "residual outside 32 bits";
    case NSF_FLAC_BAD_CRC16: return "frame CRC-16 mismatch";
    default: return "unknown status";
  }
}

}  // namespace nsf

extern "C" {

nsf_status nsf_flac_check(const void* payload, const nsf_flac_source* src, nsf_flac_frame* frame, int32_t* samples,
                          int64_t capacity) {
  if (!payload || !src || !frame || src->byte_offset < 0 || src->byte_length < 0 || src->channels < 1 ||
      src->channels > 8 || src->max_block < 1) {
    nsf::set_error("nsf_flac_check: bad argument");
    return NSF_ERR_BAD_ARG;
  }
  static uint16_t tab[256];
  static const bool tab_ready = [] { for (uint32_t b = 0; b < 256; ++b) tab[b] = nsf::crc16_entry(b); return true; }();
  (void)tab_ready;
  const uint8_t* d = static_cast<const uint8_t*>(payload);
  nsf::FlacStream st{src->byte_offset, src->byte_offset + src->byte_length, 0, 0, src->channels, src->bits,
                     src->sample_rate, src->max_block};
  nsf::FlacCand fc;
  std::memset(&fc, 0, sizeof fc);
  nsf::decode_frame(d, src->byte_offset, st, tab, &fc, nullptr);
  nsf::Header h;
  std::memset(&h, 0, sizeof h);
  const int hs = nsf::parse_header(d, src->byte_offset, st.end, src->sample_rate, src->bits, &h);
  std::memset(frame, 0, sizeof *frame);
  frame->end = fc.end;
  frame->status = fc.status;
  frame->crc8_ok = hs == NSF_FLAC_OK;
  frame->crc16_ok = fc.status == NSF_FLAC_OK;   // 0 also when the decode stopped before the CRC-16
  if (hs == NSF_FLAC_OK) {
    frame->number = h.number; frame->block = h.block; frame->sample_rate = h.rate; frame->bits = h.bits;
    frame->assignment = h.assignment; frame->channels = h.channels; frame->variable = h.variable;
  }
  if (samples && fc.status == NSF_FLAC_OK) {
    const int block = fc.block, ch = src->channels;
    if (capacity < static_cast<int64_t>(ch) * block) { nsf::set_error("nsf_flac_check: capacity below channels * block"); return NSF_ERR_BAD_ARG; }
    nsf::decode_frame(d, src->byte_offset, st, tab, &fc, samples);
    if (ch == 2)
      for (int i = 0; i < block; ++i) nsf::decorrelate(fc.assignment & 15, samples[i], samples[block + i], samples + i, samples + block + i);
  }
  return NSF_OK;
}

}  // extern "C"

// C ABI over the kernels: contexts, workspace carving, the batched extraction pipeline and the
// host-buffer (H2D -> kernels -> D2H) pipeline.  See include/nsf.h for the contract.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cuda_fp16.h>

#include "nsf.h"
#include "nsf_internal.h"
#include "nsf_kernels.cuh"
#include "nsf_stft_tc.cuh"

namespace nsf {

namespace {

constexpr int kStages = 8;

std::string cuda_msg(const char* what, cudaError_t e) {
  return std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
}

#define NSF_CUDA(call)                                  \
  do {                                                  \
    cudaError_t e__ = (call);                           \
    if (e__ != cudaSuccess) {                           \
      set_error(cuda_msg(#call, e__));                  \
      return NSF_ERR_CUDA;                              \
    }                                                   \
  } while (0)

// Runs a launcher (its kernel count, or < 0 when a launch failed) and counts its kernels in ctx->launches.
#define NSF_LAUNCH(ctx, call)                           \
  do {                                                  \
    const int n__ = (call);                             \
    if (n__ < 0) {                                      \
      set_error(cuda_msg(#call, cudaGetLastError()));   \
      return NSF_ERR_CUDA;                              \
    }                                                   \
    (ctx)->launches += n__;                             \
  } while (0)

nsf_status check_pcm_format(int32_t pcm_format) {
  if (pcm_format != NSF_PCM_F32 && pcm_format != NSF_PCM_I16) { set_error("unknown pcm_format"); return NSF_ERR_BAD_ARG; }
  return NSF_OK;
}

nsf_status check_dtype(const char* fn, int32_t dtype) {
  if (dtype != NSF_F32 && dtype != NSF_F64) { set_error(std::string(fn) + ": bad dtype"); return NSF_ERR_BAD_ARG; }
  return NSF_OK;
}

// off[0..n]: "<what> must be non-decreasing" unless every entry is >= the one before it.
nsf_status check_nondecreasing(const std::string& what, const int64_t* off, int64_t n) {
  for (int64_t i = 0; i < n; ++i)
    if (off[i + 1] < off[i]) { set_error(what + " must be non-decreasing"); return NSF_ERR_BAD_ARG; }
  return NSF_OK;
}

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Bump allocator over a caller-provided (or context-owned) device buffer.
struct Carver {
  char* base;
  size_t cap, used = 0;
  bool ok = true;
  Carver(void* b, size_t c) : base(static_cast<char*>(b)), cap(c) {}
  template <typename T> T* take(size_t count) {
    const size_t bytes = align_up(count * sizeof(T));
    if (used + bytes > cap) { ok = false; used += bytes; return nullptr; }
    T* p = reinterpret_cast<T*>(base + used);
    used += bytes;
    return p;
  }
};

struct Sizes {
  int64_t total_samples, frames_ub, rows_ub;
  int32_t n_clips;
};

// One layout function used both for sizing (base == nullptr) and carving.
struct Layout {
  int64_t* clip_off; int64_t* frame_off; int64_t* row_off;
  uint32_t* peak_bits; uint32_t* dbmax_key; double* sum; double* sumsq;
  float* y; float* a32; float* power; float* db; float* mfcc_raw; float* ac_raw; float* tmp_out;
  void* tc_a;  // tcgen05 path: folded fp16 hi/lo operands
  size_t zero_begin, zero_bytes;  // region that must be cleared before each batch
};

size_t plan_layout(const Plan& p, const Sizes& z, uint32_t flags, bool need_y, void* base, size_t cap,
                   Layout* L, bool* ok) {
  Carver c(base ? base : reinterpret_cast<void*>(0x1000), base ? cap : ~size_t(0) >> 1);
  const size_t n1 = static_cast<size_t>(z.n_clips) + 1;
  L->clip_off = c.take<int64_t>(3 * n1);   // one block, one upload: [clip_off | frame_off | row_off]
  L->frame_off = L->clip_off ? L->clip_off + n1 : nullptr;
  L->row_off = L->clip_off ? L->clip_off + 2 * n1 : nullptr;
  L->zero_begin = c.used;
  L->peak_bits = c.take<uint32_t>(z.n_clips);
  L->dbmax_key = c.take<uint32_t>(z.n_clips);
  L->sum = c.take<double>(static_cast<size_t>(z.n_clips) * p.n_mfcc);
  L->sumsq = c.take<double>(static_cast<size_t>(z.n_clips) * p.n_mfcc);
  L->zero_bytes = c.used - L->zero_begin;
  L->y = need_y ? c.take<float>(z.total_samples) : nullptr;
  const int bins_ld = p.chain[0].np + (p.chains > 1 ? p.chain[1].np : 0);
  L->a32 = nullptr;
  L->tc_a = nullptr;
  if (flags & NSF_DEBUG_SIMT_DFT) {
    size_t kp_total = 0;
    for (int ch = 0; ch < p.chains; ++ch) kp_total += 2 * static_cast<size_t>(p.chain[ch].kp);
    L->a32 = c.take<float>(kp_total * z.frames_ub);
  } else {
    L->tc_a = c.take<char>(stft_tc_operand_bytes(p, z.frames_ub));
  }
  L->power = c.take<float>(static_cast<size_t>(z.frames_ub) * bins_ld);
  L->db = c.take<float>(static_cast<size_t>(z.frames_ub) * p.n_mels);
  L->mfcc_raw = c.take<float>(static_cast<size_t>(z.frames_ub) * p.n_mfcc);
  L->ac_raw = (flags & NSF_AC_DELTAS) && !(flags & NSF_NO_AUTOCORR)
                  ? c.take<float>(static_cast<size_t>(z.frames_ub) * p.n_lags) : nullptr;
  const int cols = p.n_mfcc * 3 + p.n_lags * 3;
  L->tmp_out = (flags & NSF_SMOOTH) ? c.take<float>(static_cast<size_t>(z.rows_ub) * cols) : nullptr;
  if (ok) *ok = c.ok;
  return c.used;
}

}  // namespace

struct Arena {
  void* ptr = nullptr;
  size_t bytes = 0;
  nsf_status reserve(size_t need) {
    if (need <= bytes) return NSF_OK;
    if (ptr) { cudaFree(ptr); ptr = nullptr; bytes = 0; }
    const size_t want = align_up(need + need / 8, 1 << 20);
    NSF_CUDA(cudaMalloc(&ptr, want));
    bytes = want;
    return NSF_OK;
  }
  void release() { if (ptr) cudaFree(ptr); ptr = nullptr; bytes = 0; }
};

struct PinnedArena {
  void* ptr = nullptr;
  size_t bytes = 0;
  nsf_status reserve(size_t need) {
    if (need <= bytes) return NSF_OK;
    if (ptr) { cudaFreeHost(ptr); ptr = nullptr; bytes = 0; }
    const size_t want = align_up(need + need / 4, 1 << 16);
    NSF_CUDA(cudaHostAlloc(&ptr, want, cudaHostAllocDefault));
    bytes = want;
    return NSF_OK;
  }
  void release() { if (ptr) cudaFreeHost(ptr); ptr = nullptr; bytes = 0; }
};

// Host pipeline: clip groups rotate over three slots (stream + arenas each), so the upload of group g+1, the
// kernels of group g and the download of group g-1 overlap without the upload engine ever waiting for a
// download to release its slot.  The first groups are small (the pipeline fills after a short upload instead of
// a large one), later groups carry up to 8 Mi samples: measured on C2 (r2_ab.jsonl) 8 / 16 / 24 / 32 Mi give
// 6.5 / 7.0 / 7.1 / 7.1 ms per int16 step against a bare-copy ceiling of 6.1 ms - the tail (kernels + download of
// the LAST group) and the bubble before the first kernels shrink with the group.
constexpr int kSlots = 3;
constexpr int64_t kGroupSamples = int64_t(8) << 20;        // ~32 MB of float32 PCM per in-flight group
constexpr int64_t kFirstGroupSamples = int64_t(6) << 20;   // groups 0 and 1
// NSF_GROUP_MI / NSF_FIRST_MI (Mi samples) override the two budgets for pipeline experiments
inline int64_t env_mi(const char* name, int64_t dflt) {
  const char* v = std::getenv(name);
  const long n = v ? std::atol(v) : 0;
  return n > 0 ? (int64_t(n) << 20) : dflt;
}
inline int64_t group_budget(int turn) {
  static const int64_t big = env_mi("NSF_GROUP_MI", kGroupSamples), first = env_mi("NSF_FIRST_MI", kFirstGroupSamples);
  return turn < 2 ? first : big;
}
// (Tapering the last groups - a third of the remaining samples each, so that the kernels and the download that follow
// the final upload belong to one small group - was measured in round 2 and made the pass SLOWER, 6.83 against 6.77 ms
// on C2: every extra group costs more than the shorter tail saves.)
// Grid caps of the two front-end kernels inside the pipelined passes (nsf_kernels.cu, launch_absmax).
constexpr int kPipelinedAbsmaxBlocks = 74, kPipelinedNormalizeBlocks = 148;

struct Slot {  // one in-flight clip group of the host pipeline
  cudaStream_t stream = nullptr;
  Arena in[2], out[3], work;   // device: the group's inputs, its results, kernel workspace
  // pinned twins of `in` / `out` for pageable caller buffers: an input is gathered into stage_in[i] before its
  // upload, a result comes back through stage_out[i]; `pending` lists the copy-outs owed to the caller's buffers
  PinnedArena stage_in[2], stage_out[3];
  struct CopyOut { void* dst; const void* src; size_t dst_pitch, width; int64_t rows; };   // rows of `width` bytes
  CopyOut pending[3];
  int n_pending = 0;
};

// Ring of pinned descriptor staging buffers.  A stream-ordered call writes its (tiny) descriptor arrays into
// the next ring entry, enqueues the upload and records the entry's event; the entry is reused kDescRing calls
// later, so the host only ever waits when that many calls' descriptor uploads are still outstanding.
constexpr int kDescRing = 8;
struct DescEntry {
  PinnedArena mem;
  Arena dev;              // device copy of the entry, for calls whose descriptors have no other home (convert, collect, windows)
  cudaEvent_t copied = nullptr;
  bool pending = false;
};

// Polyphase filter of one (rate pair, quality), k-major [kmax][up], resident on the device (nsf_convert_*).
struct TapTable {
  int orig = 0, target = 0, quality = 0;
  int up = 1, down = 1, n_pre_pad = 0, n_pre_remove = 0, kmax = 0;
  Arena mem;
};

// Host-side descriptor arrays of a batch (kept in the context: no heap traffic per call after the first).
struct HostDesc {
  std::vector<int64_t> clip_off, frame_off, row_off;
  int64_t total_samples = 0, total_frames = 0, total_rows = 0;
};

}  // namespace nsf

struct nsf_ctx {
  const nsf_plan* plan = nullptr;
  int device = 0;
  nsf::DeviceTables tables{};
  nsf::StftTcTables tc{};
  nsf::Arena table_mem;
  nsf::DescEntry desc[nsf::kDescRing];
  int desc_next = 0;
  nsf::HostDesc hd_batch, hd_all;   // scratch of nsf_extract_batch / the host pipelines
  float edge_zero_threshold = 1e-7f;   // fix_edge_frames_autocorr(zero_threshold=1e-7)
  int resample_quality = NSF_RESAMPLE_HQ;
  nsf::Slot slot[nsf::kSlots];
  int64_t launches = 0;
  bool profiling = false;
  cudaEvent_t stage_ev[nsf::kStages + 1] = {};
  bool stage_valid = false;
  std::vector<nsf::TapTable*> tap_tables;   // filter cache of the conversion calls, one per (rate pair, quality)
  std::vector<nsf::ConvClip> conv_clips;    // scratch of convert_enqueue
  std::vector<nsf_pcm_source> conv_src;     // scratch of nsf_convert_host (one group's rebased descriptors)
  std::vector<int64_t> conv_off, conv_group_off;
};

namespace nsf {
namespace {

nsf_status upload_tables(nsf_ctx* ctx) {
  const Plan& p = ctx->plan->p;
  // pack everything into one host blob, one cudaMalloc, one copy
  std::vector<char> blob;
  auto put = [&](const void* src, size_t bytes) {
    const size_t off = align_up(blob.size());
    blob.resize(off + bytes);
    std::memcpy(blob.data() + off, src, bytes);
    return off;
  };
  size_t off_tap_idx[2] = {}, off_tap_coef[2] = {}, off_mat[2][2] = {};
  std::vector<float> m32;
  for (int c = 0; c < p.chains; ++c) {
    const FoldChain& ch = p.chain[c];
    off_tap_idx[c] = put(ch.tap_idx.data(), ch.tap_idx.size() * sizeof(int32_t));
    off_tap_coef[c] = put(ch.tap_coef.data(), ch.tap_coef.size() * sizeof(float));
    for (int part = 0; part < 2; ++part) {
      m32.assign(ch.mat[part].begin(), ch.mat[part].end());
      off_mat[c][part] = put(m32.data(), m32.size() * sizeof(float));
    }
  }
  const size_t off_hann = put(p.hann_sym.data(), p.hann_sym.size() * sizeof(float));
  const size_t off_hann_per = put(p.hann_per.data(), p.hann_per.size() * sizeof(float));
  // sparse mel runs in the chain-major power layout: natural bin k lives at column
  // col_off[chain(k)] + index-within-chain(k); a filter's contiguous bin range becomes one run of
  // consecutive columns per chain
  int col_off[2] = {0, p.chain[0].np};
  std::vector<int32_t> run_start(static_cast<size_t>(p.chains) * p.n_mels, 0),
      run_len(run_start.size(), 0), run_ptr(run_start.size(), 0);
  std::vector<float> melw;
  for (int c = 0; c < p.chains; ++c)
    for (int m = 0; m < p.n_mels; ++m) {
      const size_t e = static_cast<size_t>(c) * p.n_mels + m;
      run_ptr[e] = static_cast<int32_t>(melw.size());
      const int lo = p.mel_start[m], hi = lo + p.mel_len[m];  // natural bins [lo, hi)
      bool first = true;
      for (int idx = 0; idx < p.chain[c].nbins; ++idx) {
        const int k = p.chain[c].bin[idx];
        if (k < lo || k >= hi) continue;
        if (first) { run_start[e] = col_off[c] + idx; first = false; }
        melw.push_back(p.mel_dense[static_cast<size_t>(m) * p.bins + k]);
        ++run_len[e];
      }
    }
  if (melw.empty()) melw.push_back(0.0f);
  const size_t off_ms = put(run_start.data(), run_start.size() * sizeof(int32_t));
  const size_t off_ml = put(run_len.data(), run_len.size() * sizeof(int32_t));
  const size_t off_mp = put(run_ptr.data(), run_ptr.size() * sizeof(int32_t));
  const size_t off_mw = put(melw.data(), melw.size() * sizeof(float));
  std::vector<float> dct_t(static_cast<size_t>(p.n_mels) * 32, 0.0f);
  for (int k = 0; k < p.n_mfcc; ++k)
    for (int m = 0; m < p.n_mels; ++m) dct_t[static_cast<size_t>(m) * 32 + k] = p.dct[static_cast<size_t>(k) * p.n_mels + m];
  const size_t off_dct = put(dct_t.data(), dct_t.size() * sizeof(float));
  // k_dct_mma: B[k][n] = 2^10 dct[n][k] (n < n_mfcc, else 0) split into fp16 hi + lo, in m16n8k16 fragment order:
  // lane (g, tq) of k-step ks, column tile nt holds b0 = (k = 16 ks + 2 tq, + 1; n = 8 nt + g), b1 = (k + 8, k + 9)
  std::vector<uint32_t> dct_frag;
  const bool dct_frag_ok = p.n_mels == kDctMmaMels && p.n_mfcc == kDctMmaMfcc;
  if (dct_frag_ok) {
    dct_frag.assign(static_cast<size_t>(8) * 3 * 2 * 32 * 2, 0u);
    auto half_bits = [](float v) { const __half h = __float2half_rn(v); uint16_t u; std::memcpy(&u, &h, 2); return u; };
    auto half_val = [](float v) { return __half2float(__float2half_rn(v)); };
    for (int ks = 0; ks < 8; ++ks)
      for (int nt = 0; nt < 3; ++nt)
        for (int lane = 0; lane < 32; ++lane) {
          const int g = lane >> 2, tq = lane & 3, n = 8 * nt + g;
          for (int reg = 0; reg < 2; ++reg) {
            uint32_t hi = 0, lo = 0;
            for (int e = 0; e < 2; ++e) {
              const int k = 16 * ks + 2 * tq + 8 * reg + e;
              const float v = n < p.n_mfcc ? p.dct[static_cast<size_t>(n) * p.n_mels + k] * 1024.0f : 0.0f;
              const float vh = half_val(v);
              hi |= static_cast<uint32_t>(half_bits(v)) << (16 * e);
              lo |= static_cast<uint32_t>(half_bits(v - vh)) << (16 * e);
            }
            dct_frag[((static_cast<size_t>(ks * 3 + nt) * 2 + 0) * 32 + lane) * 2 + reg] = hi;
            dct_frag[((static_cast<size_t>(ks * 3 + nt) * 2 + 1) * 32 + lane) * 2 + reg] = lo;
          }
        }
  }
  const size_t off_dct_frag = dct_frag_ok ? put(dct_frag.data(), dct_frag.size() * sizeof(uint32_t)) : 0;
  // column -> (first filter, two weights) table for the fused mel epilogue of the tcgen05 kernel
  size_t off_melcol[2] = {0, 0};
  int mel_col_ok = 1;
  for (int c = 0; c < p.chains; ++c) {
    const int ncols = (p.chain[c].np + 127) / 128 * 128;
    std::vector<float> tab(static_cast<size_t>(ncols) * 4, 0.0f);
    for (int idx = 0; idx < p.chain[c].nbins; ++idx) {
      const int k = p.chain[c].bin[idx];
      int m0 = -1, count = 0, last = -1;
      for (int m = 0; m < p.n_mels; ++m)
        if (p.mel_dense[static_cast<size_t>(m) * p.bins + k] != 0.0f) { if (m0 < 0) m0 = m; last = m; ++count; }
      if (count > 2 || (count == 2 && last != m0 + 1)) mel_col_ok = 0;
      if (m0 < 0) m0 = 0;
      if (m0 > p.n_mels - 2) m0 = p.n_mels - 2 < 0 ? 0 : p.n_mels - 2;
      int32_t bits = m0;
      float fb;
      std::memcpy(&fb, &bits, 4);
      tab[4 * static_cast<size_t>(idx) + 0] = fb;
      tab[4 * static_cast<size_t>(idx) + 1] = p.mel_dense[static_cast<size_t>(m0) * p.bins + k];
      tab[4 * static_cast<size_t>(idx) + 2] = m0 + 1 < p.n_mels ? p.mel_dense[static_cast<size_t>(m0 + 1) * p.bins + k] : 0.0f;
    }
    off_melcol[c] = put(tab.data(), tab.size() * sizeof(float));
  }
  if (p.n_mels < 2) mel_col_ok = 0;
  StftTcHostBlob tcblob;
  build_stft_tc_blob(p, &tcblob);
  const size_t off_tc = put(tcblob.bytes.data(), tcblob.bytes.size());

  nsf_status st = ctx->table_mem.reserve(blob.size());
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaMemcpy(ctx->table_mem.ptr, blob.data(), blob.size(), cudaMemcpyHostToDevice));
  char* base = static_cast<char*>(ctx->table_mem.ptr);
  DeviceTables& t = ctx->tables;
  t.F = p.F; t.H = p.H; t.pad = p.pad; t.bins = p.bins;
  t.edge_thr = ctx->edge_zero_threshold;
  t.bins_ld = p.chain[0].np + (p.chains > 1 ? p.chain[1].np : 0);
  t.col_off[0] = col_off[0]; t.col_off[1] = col_off[1];
  t.n_mfcc = p.n_mfcc; t.n_mels = p.n_mels; t.n_lags = p.n_lags; t.chains = p.chains;
  for (int c = 0; c < 2; ++c) {
    t.kp[c] = t.np[c] = t.nbins[c] = 0;
    t.tap_idx[c] = nullptr; t.tap_coef[c] = nullptr;
    t.mat32[c][0] = t.mat32[c][1] = nullptr;
  }
  for (int c = 0; c < p.chains; ++c) {
    t.kp[c] = p.chain[c].kp; t.np[c] = p.chain[c].np; t.nbins[c] = p.chain[c].nbins;
    t.tap_idx[c] = reinterpret_cast<const int32_t*>(base + off_tap_idx[c]);
    t.tap_coef[c] = reinterpret_cast<const float*>(base + off_tap_coef[c]);
    t.mat32[c][0] = reinterpret_cast<const float*>(base + off_mat[c][0]);
    t.mat32[c][1] = reinterpret_cast<const float*>(base + off_mat[c][1]);
  }
  t.hann_sym = reinterpret_cast<const float*>(base + off_hann);
  t.hann_per = reinterpret_cast<const float*>(base + off_hann_per);
  t.mel_start = reinterpret_cast<const int32_t*>(base + off_ms);
  t.mel_len = reinterpret_cast<const int32_t*>(base + off_ml);
  t.mel_ptr = reinterpret_cast<const int32_t*>(base + off_mp);
  t.mel_w = reinterpret_cast<const float*>(base + off_mw);
  t.dct_t = reinterpret_cast<const float*>(base + off_dct);
  t.dct_frag = dct_frag_ok ? reinterpret_cast<const uint2*>(base + off_dct_frag) : nullptr;
  t.mel_col[0] = reinterpret_cast<const float4*>(base + off_melcol[0]);
  t.mel_col[1] = p.chains > 1 ? reinterpret_cast<const float4*>(base + off_melcol[1]) : nullptr;
  t.mel_col_ok = mel_col_ok;
  return bind_stft_tc_tables(p, tcblob, base + off_tc, &ctx->tc);
}

// Next entry of the descriptor ring with room for `bytes`; waits only if the entry's previous upload (issued
// kDescRing calls ago) has not run yet.
nsf_status desc_acquire(nsf_ctx* ctx, size_t bytes, DescEntry** out) {
  DescEntry& d = ctx->desc[ctx->desc_next];
  ctx->desc_next = (ctx->desc_next + 1) % kDescRing;
  if (d.pending) { NSF_CUDA(cudaEventSynchronize(d.copied)); d.pending = false; }
  if (bytes > d.mem.bytes) {
    // a larger batch geometry than any seen so far: grow EVERY entry now (cudaHostAlloc synchronises the
    // device), so that the following calls of the same size find their entries ready
    for (auto& e : ctx->desc) {
      if (e.pending) { NSF_CUDA(cudaEventSynchronize(e.copied)); e.pending = false; }
      const nsf_status st = e.mem.reserve(bytes);
      if (st != NSF_OK) return st;
    }
  }
  *out = &d;
  return NSF_OK;
}
// One descriptor block through the ring: fill(host) writes `bytes` into the next entry's pinned memory, and their upload
// is queued on `s` to `dst`, or, when dst is NULL, to the entry's own device copy, reserved at dev_bytes >= bytes (a call
// may keep device scratch behind its block).  The caller commits the entry once nothing on `s` reads it any more.
template <typename Fill>
nsf_status desc_upload(nsf_ctx* ctx, cudaStream_t s, size_t bytes, void* dst, size_t dev_bytes, DescEntry** out,
                       Fill&& fill) {
  DescEntry* de = nullptr;
  nsf_status st = desc_acquire(ctx, bytes, &de);
  if (st != NSF_OK) return st;
  if (!dst) {
    if ((st = de->dev.reserve(dev_bytes)) != NSF_OK) return st;
    dst = de->dev.ptr;
  }
  fill(de->mem.ptr);
  NSF_CUDA(cudaMemcpyAsync(dst, de->mem.ptr, bytes, cudaMemcpyHostToDevice, s));
  *out = de;
  return NSF_OK;
}
nsf_status desc_commit(DescEntry* d, cudaStream_t s) {
  NSF_CUDA(cudaEventRecord(d->copied, s));
  d->pending = true;
  return NSF_OK;
}

// Host-side descriptor build + validation shared by the device and host entry points.
nsf_status build_desc(const Plan& p, const int64_t* clip_offsets, int32_t n_clips, uint32_t flags,
                      const int64_t* out_row_offsets, HostDesc* d) {
  if ((flags & NSF_NO_MFCC) && (flags & NSF_NO_AUTOCORR)) {
    set_error("NSF_NO_MFCC | NSF_NO_AUTOCORR leaves nothing to compute"); return NSF_ERR_BAD_ARG;
  }
  // pad_signal=False exists for the autocorrelation branch only (librosa's STFT always centre-pads)
  if ((flags & NSF_AC_NO_PAD) && !(flags & NSF_NO_MFCC)) {
    set_error("NSF_AC_NO_PAD needs NSF_NO_MFCC: only the autocorrelation branch has a pad_signal switch");
    return NSF_ERR_UNSUPPORTED;
  }
  if (!clip_offsets || n_clips <= 0) {
    set_error("clip_offsets is NULL or n_clips <= 0");
    return NSF_ERR_BAD_ARG;
  }
  const nsf_status st = check_nondecreasing("clip_offsets", clip_offsets, n_clips);
  if (st != NSF_OK) return st;
  d->clip_off.resize(n_clips + 1);
  d->frame_off.resize(n_clips + 1);
  d->row_off.resize(n_clips + 1);
  const int64_t origin = clip_offsets[0];
  d->frame_off[0] = 0;
  d->row_off[0] = out_row_offsets ? out_row_offsets[0] : 0;
  for (int i = 0; i < n_clips; ++i) {
    const int64_t len = clip_offsets[i + 1] - clip_offsets[i];
    int64_t R;
    const int64_t T = clip_frames(len, p.F, p.H, flags, &R);
    // librosa.feature.delta(width=9) raises below 9 frames; the edge fix and reflect padding need
    // 2 frames and F/2 + 1 samples.  (The 9-frame *guard* of extract_features.py:16 counts
    // un-padded frames and belongs to the caller: see nsf_guard_frames.)
    const bool any_delta = (!(flags & NSF_NO_DELTAS) && !(flags & NSF_NO_MFCC)) ||
                           ((flags & NSF_AC_DELTAS) && !(flags & NSF_NO_AUTOCORR));
    const int64_t need = any_delta ? kMinGuardFrames : ((flags & NSF_AC_NO_PAD) ? 1 : 2);
    if (T < need || len <= p.F / 2) {
      char buf[160];
      std::snprintf(buf, sizeof buf, "clip %d is too short: %lld hop-frames, required: %lld", i,
                    static_cast<long long>(T), static_cast<long long>(need));
      set_error(buf);
      return NSF_ERR_TOO_SHORT;
    }
    d->clip_off[i] = clip_offsets[i] - origin;
    d->frame_off[i + 1] = d->frame_off[i] + T;
    if (out_row_offsets) {
      if (out_row_offsets[i + 1] - out_row_offsets[i] != R) {
        set_error("out_row_offsets is not the prefix sum of the per-clip row counts");
        return NSF_ERR_BAD_ARG;
      }
      d->row_off[i + 1] = out_row_offsets[i + 1];
    } else {
      d->row_off[i + 1] = d->row_off[i] + R;
    }
  }
  d->clip_off[n_clips] = clip_offsets[n_clips] - origin;
  d->total_samples = d->clip_off[n_clips];
  d->total_frames = d->frame_off[n_clips];
  d->total_rows = d->row_off[n_clips] - d->row_off[0];
  return NSF_OK;
}

struct StageTimer {
  nsf_ctx* ctx; cudaStream_t s; int next = 0;
  void mark(int stage) {
    if (!ctx->profiling) return;
    while (next <= stage) cudaEventRecord(ctx->stage_ev[next++], s);
  }
  void finish() {
    if (!ctx->profiling) return;
    while (next <= kStages) cudaEventRecord(ctx->stage_ev[next++], s);
    ctx->stage_valid = true;
  }
};

// ---- host-buffer pipeline ------------------------------------------------------------------------
nsf_status ensure_slot(Slot* sl) {
  if (!sl->stream) NSF_CUDA(cudaStreamCreateWithFlags(&sl->stream, cudaStreamNonBlocking));
  return NSF_OK;
}

// Is `p` memory the copy engines can reach directly (cudaHostAlloc / cudaHostRegister / managed)?  Pageable
// buffers are staged through the slot's pinned arenas so that uploads and downloads stay asynchronous.
bool dma_reachable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// memcpy split over a few threads once it is large enough to be bound by one core's copy bandwidth.
void host_copy(void* dst, const void* src, size_t bytes) {
  constexpr size_t kChunk = size_t(8) << 20;
  unsigned hw = std::thread::hardware_concurrency();
  size_t n = bytes / kChunk;
  if (n > 8) n = 8;
  if (hw && n > hw) n = hw;
  if (n < 2) { std::memcpy(dst, src, bytes); return; }
  const size_t part = (bytes / n + 63) & ~size_t(63);
  std::vector<std::thread> th;
  th.reserve(n - 1);
  for (size_t i = 1; i < n; ++i) {
    const size_t off = i * part;
    if (off >= bytes) break;
    const size_t len = std::min(part, bytes - off);
    th.emplace_back([=] { std::memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off, len); });
  }
  std::memcpy(dst, src, std::min(part, bytes));
  for (auto& t : th) t.join();
}

// Waits for the slot's stream, then makes the copy-outs it owes to pageable caller buffers.
nsf_status drain_slot(Slot* sl) {
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  for (int i = 0; i < sl->n_pending; ++i) {
    const Slot::CopyOut& c = sl->pending[i];
    if (c.dst_pitch == c.width) {
      host_copy(c.dst, c.src, c.width * static_cast<size_t>(c.rows));
    } else {
      for (int64_t r = 0; r < c.rows; ++r)
        std::memcpy(static_cast<char*>(c.dst) + r * c.dst_pitch, static_cast<const char*>(c.src) + r * c.width, c.width);
    }
  }
  sl->n_pending = 0;
  return NSF_OK;
}

// Queues the copy of `bytes` of caller memory into the slot's device input i (reserved by the caller).  Pageable
// memory is first gathered into the pinned stage_in[i] by the host, so that the copy itself stays asynchronous.
nsf_status upload(Slot* sl, int i, const void* src, size_t bytes, bool dma) {
  if (!dma) {
    const nsf_status st = sl->stage_in[i].reserve(bytes);
    if (st != NSF_OK) return st;
    host_copy(sl->stage_in[i].ptr, src, bytes);
    src = sl->stage_in[i].ptr;
  }
  NSF_CUDA(cudaMemcpyAsync(sl->in[i].ptr, src, bytes, cudaMemcpyHostToDevice, sl->stream));
  return NSF_OK;
}

// Queues the copy of the slot's device output i, `rows` packed rows of `width` bytes, to caller memory whose rows
// start `dst_pitch` bytes apart.  The copy engine writes page-locked memory itself; pageable memory gets the rows
// from the pinned stage_out[i] when the slot drains.
nsf_status download(Slot* sl, int i, void* dst, size_t dst_pitch, size_t width, int64_t rows, bool dma) {
  const size_t bytes = width * static_cast<size_t>(rows);
  if (dma && dst_pitch == width) {
    NSF_CUDA(cudaMemcpyAsync(dst, sl->out[i].ptr, bytes, cudaMemcpyDeviceToHost, sl->stream));
  } else if (dma) {
    NSF_CUDA(cudaMemcpy2DAsync(dst, dst_pitch, sl->out[i].ptr, width, width, rows, cudaMemcpyDeviceToHost, sl->stream));
  } else {
    const nsf_status st = sl->stage_out[i].reserve(bytes);
    if (st != NSF_OK) return st;
    NSF_CUDA(cudaMemcpyAsync(sl->stage_out[i].ptr, sl->out[i].ptr, bytes, cudaMemcpyDeviceToHost, sl->stream));
    sl->pending[sl->n_pending++] = Slot::CopyOut{dst, sl->stage_out[i].ptr, dst_pitch, width, rows};
  }
  return NSF_OK;
}

// Runs a host call as clip groups.  cost[0..n] is a prefix sum over the n clips; a group is the longest run of clips
// [first, last) with cost[last] - cost[first] <= group_budget(turn), and at least one clip.  Groups rotate over the
// slots, and a slot drains before it takes its next group, so the upload of group g + 1, the kernels of group g and
// the download of group g - 1 overlap.  body(first, last, slot) reserves the slot's arenas and queues the group's
// uploads, kernels and downloads.  Every slot drains before the call returns: the caller's buffers are final on
// success and no copy into them is still running on error.  On error the owed copy-outs are dropped and the first
// error is returned.
template <typename Body>
nsf_status run_groups(nsf_ctx* ctx, const int64_t* cost, int32_t n, Body&& body) {
  nsf_status st = NSF_OK;
  for (int first = 0, turn = 0; first < n && st == NSF_OK; ++turn) {
    int last = first + 1;
    while (last < n && cost[last + 1] - cost[first] <= group_budget(turn)) ++last;
    Slot* sl = &ctx->slot[turn % kSlots];
    if ((st = ensure_slot(sl)) == NSF_OK && (st = drain_slot(sl)) == NSF_OK) st = body(first, last, sl);
    first = last;
  }
  for (auto& sl : ctx->slot) {
    if (!sl.stream) continue;
    if (st == NSF_OK) { st = drain_slot(&sl); continue; }
    sl.n_pending = 0;
    cudaStreamSynchronize(sl.stream);   // the first error is the one reported
  }
  return st;
}

// A synchronous host call as one group of run_groups: body(slot) reserves the slot's arenas and queues the uploads,
// kernels and downloads.
template <typename Body>
nsf_status run_once(nsf_ctx* ctx, Body&& body) {
  const int64_t cost[2] = {0, 0};
  return run_groups(ctx, cost, 1, [&](int, int, Slot* sl) { return body(sl); });
}

// The body of nsf_extract_batch.  absmax_blocks / normalize_blocks cap the grids of the two front-end kernels (0: no
// cap); the pipelined host passes cap them to stay off the copy engine's HBM share.
nsf_status extract_enqueue(nsf_ctx* ctx, cudaStream_t s, const void* pcm_dev, int32_t pcm_format,
                           const int64_t* clip_offsets_host, int32_t n_clips, uint32_t flags, float* out_dev,
                           int64_t out_ld, const int64_t* out_row_offsets_host, float* y_norm_dev, void* workspace_dev,
                           int64_t workspace_bytes, int absmax_blocks, int normalize_blocks) {
  if (!ctx || !pcm_dev || !out_dev || !workspace_dev) { set_error("nsf_extract_batch: NULL argument"); return NSF_ERR_BAD_ARG; }
  nsf_status st = check_pcm_format(pcm_format);
  if (st != NSF_OK) return st;
  const Plan& p = ctx->plan->p;
  const int cols = nsf_feature_cols(ctx->plan, flags);
  if (out_ld < cols) { set_error("out_ld smaller than the feature width"); return NSF_ERR_BAD_ARG; }
  if (workspace_bytes <= 0) { set_error("workspace_bytes must be positive; size it with nsf_workspace_bytes()"); return NSF_ERR_WORKSPACE; }
  HostDesc& hd = ctx->hd_batch;
  if ((st = build_desc(p, clip_offsets_host, n_clips, flags, out_row_offsets_host, &hd)) != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));

  const bool normalize = (flags & NSF_PEAK_NORMALIZE) != 0;
  const bool need_y = normalize || pcm_format == NSF_PCM_I16;
  Sizes z;
  z.total_samples = hd.total_samples; z.n_clips = n_clips;
  z.frames_ub = hd.total_frames; z.rows_ub = hd.total_rows;
  Layout L;
  bool fits = false;
  // 256-byte align the caller's pointer
  char* wbase = reinterpret_cast<char*>(align_up(reinterpret_cast<size_t>(workspace_dev)));
  const size_t wslack = static_cast<size_t>(wbase - static_cast<char*>(workspace_dev));
  if (static_cast<size_t>(workspace_bytes) <= wslack) { set_error("workspace too small; size it with nsf_workspace_bytes()"); return NSF_ERR_WORKSPACE; }
  const size_t wcap = static_cast<size_t>(workspace_bytes) - wslack;
  plan_layout(p, z, flags, need_y && !y_norm_dev, wbase, wcap, &L, &fits);
  if (!fits) { set_error("workspace too small; size it with nsf_workspace_bytes()"); return NSF_ERR_WORKSPACE; }

  // descriptors: next entry of the pinned ring -> workspace, one stream-ordered upload, no host wait
  const size_t n1 = static_cast<size_t>(n_clips) + 1;
  const int64_t row_origin = hd.row_off[0];
  DescEntry* de = nullptr;
  st = desc_upload(ctx, s, 3 * n1 * sizeof(int64_t), L.clip_off, 0, &de, [&](void* mem) {
    int64_t* h = static_cast<int64_t*>(mem);
    for (size_t i = 0; i < n1; ++i) {
      h[i] = hd.clip_off[i];
      h[n1 + i] = hd.frame_off[i];
      h[2 * n1 + i] = hd.row_off[i] - row_origin;
    }
  });
  if (st != NSF_OK || (st = desc_commit(de, s)) != NSF_OK) return st;
  NSF_CUDA(cudaMemsetAsync(wbase + L.zero_begin, 0, L.zero_bytes, s));

  BatchView b;
  b.clip_off = L.clip_off; b.frame_off = L.frame_off; b.row_off = L.row_off;
  b.n_clips = n_clips; b.total_samples = hd.total_samples; b.total_frames = hd.total_frames;
  b.total_rows = hd.total_rows;
  float* out = out_dev + row_origin * out_ld;
  const DeviceTables& t = ctx->tables;
  StageTimer timer{ctx, s};

  // stage 0: decode / peak normalise
  timer.mark(0);
  const float* y = static_cast<const float*>(pcm_dev);
  if (need_y) {
    float* ydst = y_norm_dev ? y_norm_dev : L.y;
    if (normalize) NSF_LAUNCH(ctx, launch_absmax(s, pcm_dev, pcm_format, b, L.peak_bits, absmax_blocks));
    NSF_LAUNCH(ctx, launch_normalize(s, pcm_dev, pcm_format, b, L.peak_bits, normalize, ydst, normalize_blocks));
    y = ydst;
  } else if (y_norm_dev) {
    NSF_CUDA(cudaMemcpyAsync(y_norm_dev, pcm_dev, hd.total_samples * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }

  // the smoothing pass needs the un-smoothed rows in a scratch buffer
  float* stage_out = (flags & NSF_SMOOTH) ? L.tmp_out : out;
  const int64_t stage_ld = (flags & NSF_SMOOTH) ? cols : out_ld;
  const bool reduce = !(flags & NSF_NO_REDUCE);
  const bool deltas = !(flags & NSF_NO_DELTAS);
  const bool do_mfcc = !(flags & NSF_NO_MFCC);
  const int mfcc_cols = do_mfcc ? p.n_mfcc * (deltas ? 3 : 1) : 0;
  DeviceTables t_ac = t;
  if (flags & NSF_AC_NO_PAD) t_ac.pad = 0;    // autocorrelation only (build_desc)

  // stages 1-3: STFT power -> mel -> dB (+ per-clip max)
  bool fused_mel = false;
  if (!do_mfcc) {
    // autocorrelation block only
  } else if (flags & NSF_DEBUG_SIMT_DFT) {
    timer.mark(1);
    NSF_LAUNCH(ctx, launch_fold32(s, t, b, y, L.a32));
    timer.mark(2);
    NSF_LAUNCH(ctx, launch_dft_simt(s, t, b, L.a32, L.power));
  } else {
    timer.mark(1);
    NSF_LAUNCH(ctx, launch_stft_tc_fold(s, ctx->tc, t, b, y, L.tc_a));
    timer.mark(2);
    if (t.mel_col_ok && !(flags & NSF_DEBUG_UNFUSED_MEL)) {
      // product path: STFT GEMM with the power -> mel -> dB epilogue fused (no power round trip)
      NSF_LAUNCH(ctx, launch_stft_tc_mel(s, ctx->tc, t, b, L.tc_a, L.db, L.dbmax_key));
      fused_mel = true;
    } else {
      NSF_LAUNCH(ctx, launch_stft_tc_gemm(s, ctx->tc, t, b, L.tc_a, L.power));
    }
  }
  timer.mark(3);
  if (do_mfcc && !fused_mel) NSF_LAUNCH(ctx, launch_mel_db(s, t, b, L.power, L.db, L.dbmax_key));
  // stage 4: floor + DCT + CMVN statistics
  timer.mark(4);
  if (do_mfcc) {
    NSF_LAUNCH(ctx, launch_dct_sum(s, t, b, L.db, L.dbmax_key, L.mfcc_raw, L.sum, L.sumsq));
  }
  // stage 5: CMVN + deltas + pair reduce -> columns [0, mfcc_cols)
  timer.mark(5);
  if (do_mfcc)
    NSF_LAUNCH(ctx, launch_delta_reduce(s, b, L.mfcc_raw, p.n_mfcc, p.n_mfcc, L.sum, L.sumsq,
                                        !(flags & NSF_NO_CMVN), deltas, reduce, stage_out, stage_ld, 0));
  // stage 6: autocorrelation -> columns [mfcc_cols, ...)
  timer.mark(6);
  if (!(flags & NSF_NO_AUTOCORR)) {
    if (flags & NSF_AC_DELTAS) {
      BatchView bf = b;  // un-reduced: one row per hop-frame
      bf.row_off = L.frame_off; bf.total_rows = hd.total_frames;
      if (flags & NSF_DEBUG_FMA_AUTOCORR) NSF_LAUNCH(ctx, launch_autocorr(s, t_ac, bf, y, false, L.ac_raw, p.n_lags, 0));
      else NSF_LAUNCH(ctx, launch_autocorr_mma(s, t_ac, bf, y, false, L.ac_raw, p.n_lags, 0));
      NSF_LAUNCH(ctx, launch_delta_reduce(s, b, L.ac_raw, p.n_lags, p.n_lags, nullptr, nullptr, false, true,
                                          reduce, stage_out, stage_ld, mfcc_cols));
    } else {
      if (flags & NSF_DEBUG_FMA_AUTOCORR) NSF_LAUNCH(ctx, launch_autocorr(s, t_ac, b, y, reduce, stage_out, stage_ld, mfcc_cols));
      else NSF_LAUNCH(ctx, launch_autocorr_mma(s, t_ac, b, y, reduce, stage_out, stage_ld, mfcc_cols));
    }
  }
  // stage 7: optional smoothing
  timer.mark(7);
  if (flags & NSF_SMOOTH) NSF_LAUNCH(ctx, launch_smooth(s, b, L.tmp_out, cols, cols, out, out_ld));
  timer.finish();
  return NSF_OK;
}

// extract_enqueue of one group of a pipelined host pass, from the slot's in[0] into its out[0].
nsf_status extract_group(nsf_ctx* ctx, Slot* sl, int32_t pcm_format, const int64_t* clip_offsets, int32_t n,
                         uint32_t flags, int cols, float* y_norm_dev) {
  return extract_enqueue(ctx, sl->stream, sl->in[0].ptr, pcm_format, clip_offsets, n, flags,
                         static_cast<float*>(sl->out[0].ptr), cols, nullptr, y_norm_dev, sl->work.ptr,
                         static_cast<int64_t>(sl->work.bytes), kPipelinedAbsmaxBlocks, kPipelinedNormalizeBlocks);
}

// Enqueues k_collect_rows over n clips whose rows start at `audio` / `facial` and whose results start at `out_a` /
// `out_f`.  a_off / f_off / o_off (n + 1 entries each, rebased here to their first entry) place the clips in each.  The
// three arrays travel through the descriptor ring into the entry's device copy, which is reused only after the kernel.
nsf_status collect_enqueue(nsf_ctx* ctx, cudaStream_t s, int32_t dtype, const void* audio, int32_t a_cols,
                           const int64_t* a_off, const void* facial, int32_t f_cols, const int64_t* f_off,
                           const int64_t* o_off, int32_t n, uint32_t flags, int32_t blend_frames, void* out_a,
                           void* out_f) {
  const size_t n1 = static_cast<size_t>(n) + 1, bytes = 3 * n1 * sizeof(int64_t);
  DescEntry* de = nullptr;
  const nsf_status st = desc_upload(ctx, s, bytes, nullptr, bytes, &de, [&](void* mem) {
    int64_t* h = static_cast<int64_t*>(mem);
    for (size_t i = 0; i < n1; ++i) {
      h[i] = a_off[i] - a_off[0];
      h[n1 + i] = f_off[i] - f_off[0];
      h[2 * n1 + i] = o_off[i] - o_off[0];
    }
  });
  if (st != NSF_OK) return st;
  const int64_t* d = static_cast<const int64_t*>(de->dev.ptr);
  CollectView v;
  v.a_off = d; v.f_off = d + n1; v.o_off = d + 2 * n1;
  v.n_clips = n; v.total_out_rows = o_off[n] - o_off[0]; v.flags = flags; v.blend_frames = blend_frames;
  NSF_LAUNCH(ctx, launch_collect(s, dtype, v, audio, a_cols, facial, f_cols, out_a, out_f));
  return desc_commit(de, s);     // recorded after the kernel: the entry (host and device) is reused only after it
}

}  // namespace
}  // namespace nsf

using namespace nsf;

extern "C" {

int32_t nsf_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ++ok;
  }
  return ok;
}

nsf_status nsf_host_alloc(void** out_ptr, int64_t bytes) {
  if (!out_ptr || bytes <= 0) { set_error("nsf_host_alloc: bad argument"); return NSF_ERR_BAD_ARG; }
  // portable: page-locked for every device of the process (one host array filled by several GPUs)
  NSF_CUDA(cudaHostAlloc(out_ptr, static_cast<size_t>(bytes), cudaHostAllocPortable));
  return NSF_OK;
}

void nsf_host_free(void* ptr) { if (ptr) cudaFreeHost(ptr); }

nsf_status nsf_host_register(void* ptr, int64_t bytes) {
  if (!ptr || bytes <= 0) { set_error("nsf_host_register: bad argument"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaHostRegister(ptr, static_cast<size_t>(bytes), cudaHostRegisterPortable));
  return NSF_OK;
}

nsf_status nsf_host_unregister(void* ptr) {
  if (!ptr) { set_error("nsf_host_unregister: NULL"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaHostUnregister(ptr));
  return NSF_OK;
}

nsf_status nsf_ctx_set_option(nsf_ctx* ctx, int32_t option, double value) {
  if (!ctx) { set_error("nsf_ctx_set_option: NULL context"); return NSF_ERR_BAD_ARG; }
  switch (option) {
    case NSF_OPT_EDGE_ZERO_THRESHOLD:
      if (!(value >= 0.0)) { set_error("zero_threshold must be >= 0"); return NSF_ERR_BAD_ARG; }
      ctx->edge_zero_threshold = static_cast<float>(value);
      ctx->tables.edge_thr = ctx->edge_zero_threshold;
      return NSF_OK;
    case NSF_OPT_RESAMPLE_QUALITY:
      if (value != NSF_RESAMPLE_POLY && value != NSF_RESAMPLE_HQ) { set_error("unknown resample quality"); return NSF_ERR_BAD_ARG; }
      ctx->resample_quality = static_cast<int>(value);
      return NSF_OK;
    default:
      set_error("nsf_ctx_set_option: unknown option");
      return NSF_ERR_BAD_ARG;
  }
}

nsf_status nsf_ctx_create(const nsf_plan* plan, int32_t device, nsf_ctx** out_ctx) {
  if (!plan || !out_ctx) { set_error("nsf_ctx_create: NULL argument"); return NSF_ERR_BAD_ARG; }
  *out_ctx = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_error("no CUDA device is visible; this library has no CPU path");
    return NSF_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) { set_error("nsf_ctx_create: device index out of range"); return NSF_ERR_BAD_ARG; }
  int major = 0;
  NSF_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) {
    set_error("device is not sm_100 (Blackwell B200); the kernels are compiled for sm_100a only");
    return NSF_ERR_NO_DEVICE;
  }
  NSF_CUDA(cudaSetDevice(device));
  nsf_ctx* ctx = new nsf_ctx();
  ctx->plan = plan;
  ctx->device = device;
  nsf_status st = upload_tables(ctx);
  if (st != NSF_OK) { nsf_ctx_destroy(ctx); return st; }
  for (auto& d : ctx->desc) {
    if (cudaEventCreateWithFlags(&d.copied, cudaEventDisableTiming) != cudaSuccess ||
        d.mem.reserve(size_t(48) << 10) != NSF_OK) {      // room for ~2000 clips per call before the ring grows
      set_error("descriptor ring setup failed"); nsf_ctx_destroy(ctx); return NSF_ERR_CUDA;
    }
  }
  // opt-in shared-memory limits of every kernel, once per device: no launch path touches function attributes
  if (!init_kernel_attributes() || !init_autocorr_mma_attributes() || !init_stft_tc_attributes() ||
      !init_convert_attributes()) {
    set_error(cuda_msg("cudaFuncSetAttribute", cudaGetLastError())); nsf_ctx_destroy(ctx); return NSF_ERR_CUDA;
  }
  for (int i = 0; i <= kStages; ++i) {
    if (cudaEventCreate(&ctx->stage_ev[i]) != cudaSuccess) {
      set_error("cudaEventCreate failed"); nsf_ctx_destroy(ctx); return NSF_ERR_CUDA;
    }
  }
  *out_ctx = ctx;
  return NSF_OK;
}

void nsf_ctx_destroy(nsf_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto& s : ctx->slot) {
    if (s.stream) cudaStreamDestroy(s.stream);
    for (auto& a : s.in) a.release();
    for (auto& a : s.out) a.release();
    s.work.release();
    for (auto& a : s.stage_in) a.release();
    for (auto& a : s.stage_out) a.release();
  }
  for (auto& e : ctx->stage_ev) if (e) cudaEventDestroy(e);
  for (auto& d : ctx->desc) {
    if (d.copied) cudaEventDestroy(d.copied);
    d.mem.release();
    d.dev.release();
  }
  for (TapTable* t : ctx->tap_tables) { t->mem.release(); delete t; }
  ctx->table_mem.release();
  delete ctx;
}

int64_t nsf_launch_count(const nsf_ctx* ctx) { return ctx ? ctx->launches : -1; }

void nsf_set_profiling(nsf_ctx* ctx, int32_t enabled) { if (ctx) { ctx->profiling = enabled != 0; ctx->stage_valid = false; } }

int32_t nsf_stage_times_ms(nsf_ctx* ctx, float* ms, int32_t capacity) {
  if (!ctx || !ms || !ctx->stage_valid) return 0;
  if (cudaEventSynchronize(ctx->stage_ev[kStages]) != cudaSuccess) return 0;
  const int n = capacity < kStages ? capacity : kStages;
  for (int i = 0; i < n; ++i) {
    float t = 0.0f;
    if (cudaEventElapsedTime(&t, ctx->stage_ev[i], ctx->stage_ev[i + 1]) != cudaSuccess) t = -1.0f;
    ms[i] = t;
  }
  return n;
}

int64_t nsf_workspace_bytes(const nsf_plan* plan, int64_t total_samples, int32_t n_clips, uint32_t flags) {
  if (!plan || total_samples < 0 || n_clips <= 0) return -1;
  const Plan& p = plan->p;
  Sizes z;
  z.total_samples = total_samples;
  z.n_clips = n_clips;
  z.frames_ub = n_clips + total_samples / p.H;  // T_i <= 1 + L_i / H
  z.rows_ub = (flags & NSF_NO_REDUCE) ? z.frames_ub : (z.frames_ub + n_clips + 1) / 2 + n_clips;
  Layout L;
  return static_cast<int64_t>(plan_layout(p, z, flags, true, nullptr, 0, &L, nullptr)) + 256;
}

nsf_status nsf_extract_batch(nsf_ctx* ctx, void* cuda_stream, const void* pcm_dev, int32_t pcm_format,
                             const int64_t* clip_offsets_host, int32_t n_clips, uint32_t flags,
                             float* out_dev, int64_t out_ld, const int64_t* out_row_offsets_host,
                             float* y_norm_dev, void* workspace_dev, int64_t workspace_bytes) {
  return extract_enqueue(ctx, static_cast<cudaStream_t>(cuda_stream), pcm_dev, pcm_format, clip_offsets_host, n_clips,
                         flags, out_dev, out_ld, out_row_offsets_host, y_norm_dev, workspace_dev, workspace_bytes, 0, 0);
}

// ---- host-buffer pipeline ------------------------------------------------------------------------
nsf_status nsf_extract_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                            const int64_t* clip_offsets, int32_t n_clips, uint32_t flags,
                            float* out_host, int64_t out_ld, float* y_norm_host) {
  if (!ctx || !pcm_host || !out_host || !clip_offsets || n_clips <= 0) {
    set_error("nsf_extract_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  nsf_status st = check_pcm_format(pcm_format);
  if (st != NSF_OK) return st;
  const Plan& p = ctx->plan->p;
  const int cols = nsf_feature_cols(ctx->plan, flags);
  if (out_ld < cols) { set_error("out_ld smaller than the feature width"); return NSF_ERR_BAD_ARG; }
  // validate everything up front so nothing is queued for a bad batch
  HostDesc& all = ctx->hd_all;
  if ((st = build_desc(p, clip_offsets, n_clips, flags, nullptr, &all)) != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4, row_bytes = static_cast<size_t>(cols) * sizeof(float);
  // pageable caller buffers go through the slot's pinned staging arenas: the host copies group g + 1 in (and
  // group g - 2 out) while the copy engines and kernels work on the groups in between
  const bool in_dma = dma_reachable(pcm_host), out_dma = dma_reachable(out_host);
  const bool y_dma = y_norm_host ? dma_reachable(y_norm_host) : true;
  return run_groups(ctx, clip_offsets, n_clips, [&](int first, int last, Slot* sl) -> nsf_status {
    const int64_t samples = clip_offsets[last] - clip_offsets[first];
    const int64_t rows = all.row_off[last] - all.row_off[first];
    nsf_status st;
    if ((st = sl->in[0].reserve(samples * esz)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(rows * row_bytes)) != NSF_OK) return st;
    if ((st = sl->work.reserve(nsf_workspace_bytes(ctx->plan, samples, last - first, flags))) != NSF_OK) return st;
    if (y_norm_host && (st = sl->out[1].reserve(samples * sizeof(float))) != NSF_OK) return st;
    if ((st = upload(sl, 0, static_cast<const char*>(pcm_host) + clip_offsets[first] * esz, samples * esz, in_dma)) != NSF_OK)
      return st;
    if ((st = extract_group(ctx, sl, pcm_format, clip_offsets + first, last - first, flags, cols,
                            y_norm_host ? static_cast<float*>(sl->out[1].ptr) : nullptr)) != NSF_OK) return st;
    if ((st = download(sl, 0, out_host + all.row_off[first] * out_ld, static_cast<size_t>(out_ld) * sizeof(float),
                       row_bytes, rows, out_dma)) != NSF_OK) return st;
    if (!y_norm_host) return NSF_OK;
    const size_t y_bytes = samples * sizeof(float);
    return download(sl, 1, y_norm_host + (clip_offsets[first] - clip_offsets[0]), y_bytes, y_bytes, 1, y_dma);
  });
}

nsf_status nsf_normalize_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                              const int64_t* clip_offsets, int32_t n_clips, float* y_host, float* peaks_host) {
  if (!ctx || !pcm_host || !clip_offsets || !y_host || n_clips <= 0) {
    set_error("nsf_normalize_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  nsf_status st = check_pcm_format(pcm_format);
  if (st == NSF_OK) st = check_nondecreasing("clip_offsets", clip_offsets, n_clips);
  if (st != NSF_OK) return st;
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4;
  const int64_t samples = clip_offsets[n_clips] - clip_offsets[0];
  NSF_CUDA(cudaSetDevice(ctx->device));
  if (samples == 0) return NSF_OK;
  const size_t n1 = static_cast<size_t>(n_clips) + 1;
  // in[0] = PCM, out[0] = y, out[1] = per-clip peaks, work = clip offsets
  return run_once(ctx, [&](Slot* sl) -> nsf_status {
    nsf_status st;
    if ((st = sl->in[0].reserve(samples * esz)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(samples * sizeof(float))) != NSF_OK) return st;
    if ((st = sl->out[1].reserve(n_clips * sizeof(uint32_t))) != NSF_OK) return st;
    if ((st = sl->work.reserve(n1 * sizeof(int64_t))) != NSF_OK) return st;
    int64_t* d_off = static_cast<int64_t*>(sl->work.ptr);
    uint32_t* d_peak = static_cast<uint32_t*>(sl->out[1].ptr);
    DescEntry* de = nullptr;
    st = desc_upload(ctx, sl->stream, n1 * sizeof(int64_t), d_off, 0, &de, [&](void* mem) {
      int64_t* h = static_cast<int64_t*>(mem);
      for (size_t i = 0; i < n1; ++i) h[i] = clip_offsets[i] - clip_offsets[0];
    });
    if (st != NSF_OK || (st = desc_commit(de, sl->stream)) != NSF_OK) return st;
    NSF_CUDA(cudaMemsetAsync(d_peak, 0, n_clips * sizeof(uint32_t), sl->stream));
    if ((st = upload(sl, 0, static_cast<const char*>(pcm_host) + clip_offsets[0] * esz, samples * esz, true)) != NSF_OK)
      return st;
    BatchView b{};
    b.clip_off = d_off; b.frame_off = d_off; b.row_off = d_off;
    b.n_clips = n_clips; b.total_samples = samples;
    NSF_LAUNCH(ctx, launch_absmax(sl->stream, sl->in[0].ptr, pcm_format, b, d_peak));
    NSF_LAUNCH(ctx, launch_normalize(sl->stream, sl->in[0].ptr, pcm_format, b, d_peak, true, static_cast<float*>(sl->out[0].ptr)));
    const size_t y_bytes = samples * sizeof(float), p_bytes = n_clips * sizeof(uint32_t);
    if ((st = download(sl, 0, y_host, y_bytes, y_bytes, 1, true)) != NSF_OK) return st;
    // float bits of a non-negative float: copied as-is
    return peaks_host ? download(sl, 1, peaks_host, p_bytes, p_bytes, 1, true) : NSF_OK;
  });
}

// ---- sample-rate conversion + WAV conversion -----------------------------------------------------------
namespace {
int enc_bytes(int enc) {
  switch (enc) {
    case NSF_ENC_U8: return 1;
    case NSF_ENC_I16: return 2;
    case NSF_ENC_I24: return 3;
    case NSF_ENC_I32: case NSF_ENC_F32: return 4;
    case NSF_ENC_F64: return 8;
    default: return 0;
  }
}
int enc_align(int enc) { const int b = enc_bytes(enc); return b == 3 ? 1 : b; }

// Validates every descriptor (nothing is launched for a bad batch) and writes the output prefix sum.  `base` is the
// address the byte offsets are relative to (0 when only the offsets' own alignment matters).
nsf_status convert_offsets(const nsf_pcm_source* src, int32_t n, int32_t target_sr, int64_t payload_bytes,
                           uintptr_t base, int64_t* out_off) {
  if (!src || !out_off || n <= 0) { set_error("nsf_convert: NULL sources / offsets or n <= 0"); return NSF_ERR_BAD_ARG; }
  if (target_sr <= 0) { set_error("nsf_convert: target_sr must be positive"); return NSF_ERR_BAD_ARG; }
  if (payload_bytes < 0) { set_error("nsf_convert: negative payload_bytes"); return NSF_ERR_BAD_ARG; }
  out_off[0] = 0;
  for (int i = 0; i < n; ++i) {
    const nsf_pcm_source& c = src[i];
    char buf[200];
    auto fail = [&](const char* what) {
      std::snprintf(buf, sizeof buf, "nsf_convert: source %d: %s", i, what);
      set_error(buf);
      return NSF_ERR_BAD_ARG;
    };
    const int bps = enc_bytes(c.encoding);
    if (bps == 0) return fail("unknown encoding");
    if (c.channels < 1 || c.channels > 65535) return fail("channels must be in [1, 65535]");
    if (c.frames < 0) return fail("negative frame count");
    if (c.sample_rate <= 0) return fail("sample_rate must be positive");
    if (c.byte_offset < 0 || c.byte_offset > payload_bytes) return fail("byte_offset outside the payload");
    const int64_t frame_bytes = static_cast<int64_t>(c.channels) * bps;
    if (c.frames > (payload_bytes - c.byte_offset) / frame_bytes) return fail("byte range past payload_bytes");
    if ((base + static_cast<uintptr_t>(c.byte_offset)) % static_cast<uintptr_t>(enc_align(c.encoding)) != 0)
      return fail("samples are not aligned to their container size");
    const int64_t len = c.sample_rate == target_sr ? c.frames : nsf_resample_len(c.frames, c.sample_rate, target_sr);
    out_off[i + 1] = out_off[i] + len;
  }
  return NSF_OK;
}

// The context's filter table for (orig, target, its current quality); built and uploaded on first use (synchronous).
nsf_status get_taps(nsf_ctx* ctx, int orig, int target, const TapTable** out) {
  const int q = ctx->resample_quality;
  for (const TapTable* t : ctx->tap_tables)
    if (t->orig == orig && t->target == target && t->quality == q) { *out = t; return NSF_OK; }
  ResampleDesign d;
  if (!(q == NSF_RESAMPLE_HQ ? design_resampler_hq(orig, target, &d) : design_resampler(orig, target, &d))) {
    set_error("nsf_convert: rates must be positive"); return NSF_ERR_BAD_ARG;
  }
  // k-major table [kmax][up]: entry (k, p) = h[p + k up] (zero beyond the last tap).  Neighbouring threads of
  // k_convert_resample hold different phases at the same k, so their loads fall into one short row
  const int n_taps = static_cast<int>(d.h.size());
  const int kmax = (n_taps + d.up - 1) / d.up;
  std::vector<double> pm(static_cast<size_t>(d.up) * kmax, 0.0);
  for (int i = 0; i < n_taps; ++i) pm[static_cast<size_t>(i / d.up) * d.up + i % d.up] = d.h[i];
  TapTable* t = new TapTable();
  t->orig = orig; t->target = target; t->quality = q;
  t->up = d.up; t->down = d.down; t->n_pre_pad = d.n_pre_pad; t->n_pre_remove = d.n_pre_remove; t->kmax = kmax;
  nsf_status st = t->mem.reserve(pm.size() * sizeof(double));
  if (st == NSF_OK && cudaMemcpy(t->mem.ptr, pm.data(), pm.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) {
    set_error(cuda_msg("nsf_convert: filter upload", cudaGetLastError()));
    st = NSF_ERR_CUDA;
  }
  if (st != NSF_OK) { t->mem.release(); delete t; return st; }
  ctx->tap_tables.push_back(t);
  *out = t;
  return NSF_OK;
}

// Input frames of the window a k_convert_resample block of `span` outputs reads (upper bound over every tile).
int64_t window_frames(const TapTable& t, int64_t span) { return ((span - 1) * t.down + t.up - 1) / t.up + 1 + t.kmax; }

// Enqueues the conversion of n validated clips: clip i reads payload_dev + src[i].byte_offset and writes
// out_dev[out_off[i], out_off[i + 1]).  Same-rate clips are decode-only unless always_resample (nsf_resample_host
// filters at every rate pair, 1:1 included).  At most two launches (decode, resample); the descriptors travel through
// the ring, whose entry is released only after the kernels that read it.
nsf_status convert_enqueue(nsf_ctx* ctx, cudaStream_t s, const void* payload_dev, const nsf_pcm_source* src, int n,
                           int32_t target_sr, const int64_t* out_off, float* out_dev, bool always_resample) {
  std::vector<ConvClip>& cl = ctx->conv_clips;
  cl.clear();
  int64_t tiles[2] = {0, 0};
  int n_kind[2] = {0, 0};
  int64_t max_window = 0;
  for (int pass = 0; pass < 2; ++pass) {            // decode-only clips first, then the resampled ones
    for (int i = 0; i < n; ++i) {
      const nsf_pcm_source& c = src[i];
      const bool resample = always_resample || c.sample_rate != target_sr;
      if (resample != (pass == 1)) continue;
      const int64_t n_out = out_off[i + 1] - out_off[i];
      if (n_out <= 0) continue;
      ConvClip v{};
      v.byte_off = c.byte_offset; v.frames = c.frames; v.out_off = out_off[i]; v.n_out = n_out;
      v.enc = c.encoding; v.channels = c.channels; v.bps = enc_bytes(c.encoding);
      int64_t nt;
      if (!resample) {
        nt = (c.frames + kConvDecodeTile - 1) / kConvDecodeTile;
      } else {
        const TapTable* t = nullptr;
        const nsf_status st = get_taps(ctx, c.sample_rate, target_sr, &t);
        if (st != NSF_OK) return st;
        v.taps = static_cast<const double*>(t->mem.ptr);
        v.up = t->up; v.down = t->down; v.n_pre_pad = t->n_pre_pad; v.n_pre_remove = t->n_pre_remove; v.kmax = t->kmax;
        // tile: `slots` outputs (a multiple of up, >= 256 when up allows it) x `reps` outputs per slot, as large as
        // the float64 input window in shared memory allows
        // the slot count keeps the 256 threads busy: the multiple of up (up to 32 up) whose passes over the
        // block waste the fewest threads, preferring more outputs per slot
        const int64_t budget = static_cast<int64_t>(kConvMaxSmem / sizeof(double));
        int64_t slots = 0;
        int reps = 0;
        double best = -1.0;
        for (int r = kConvMaxReps; r >= 1 && best < 0.9; r /= 2)
          for (int64_t m = 1; m <= 32; ++m) {
            const int64_t sl = m * t->up;
            if (window_frames(*t, sl * r) > budget) break;
            const double eff = static_cast<double>(sl) / (256.0 * ((sl + 255) / 256));
            if (eff > best + 1e-9) { best = eff; slots = sl; reps = r; }
          }
        if (slots == 0) { set_error("nsf_convert: rate pair needs a larger filter window than one block holds"); return NSF_ERR_UNSUPPORTED; }
        if (slots > (int64_t(1) << 30)) { set_error("nsf_convert: rate pair too large"); return NSF_ERR_UNSUPPORTED; }
        v.slots = static_cast<int32_t>(slots); v.reps = reps;
        max_window = std::max(max_window, window_frames(*t, slots * reps));
        nt = (n_out + slots * reps - 1) / (slots * reps);
      }
      if (nt <= 0) continue;
      v.tile0 = tiles[pass];
      tiles[pass] += nt;
      ++n_kind[pass];
      cl.push_back(v);
    }
  }
  if (cl.empty()) return NSF_OK;
  if (tiles[0] > INT32_MAX || tiles[1] > INT32_MAX) { set_error("nsf_convert: batch too large for one launch"); return NSF_ERR_UNSUPPORTED; }
  const size_t bytes = cl.size() * sizeof(ConvClip);
  DescEntry* de = nullptr;
  const nsf_status st =
      desc_upload(ctx, s, bytes, nullptr, bytes, &de, [&](void* mem) { std::memcpy(mem, cl.data(), bytes); });
  if (st != NSF_OK) return st;
  const ConvClip* d = static_cast<const ConvClip*>(de->dev.ptr);
  for (int kind = 0; kind < 2; ++kind) {
    const ConvClip* first = d + (kind == 0 ? 0 : n_kind[0]);
    NSF_LAUNCH(ctx, launch_convert(s, kind == 1, first, n_kind[kind], tiles[kind],
                                   kind == 1 ? static_cast<size_t>(max_window) * sizeof(double) : 0, payload_dev, out_dev));
  }
  return desc_commit(de, s);     // recorded after the kernels: the entry (host and device) is reused only after them
}
}  // namespace

nsf_status nsf_resample_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format, int64_t n_in, int32_t orig_sr,
                             int32_t target_sr, float* out_host, int64_t out_capacity) {
  if (!ctx || !pcm_host || !out_host || n_in <= 0) { set_error("nsf_resample_host: NULL argument or empty input"); return NSF_ERR_BAD_ARG; }
  const nsf_status st = check_pcm_format(pcm_format);
  if (st != NSF_OK) return st;
  if (orig_sr <= 0 || target_sr <= 0) { set_error("nsf_resample_host: rates must be positive"); return NSF_ERR_BAD_ARG; }
  const int64_t n_out = nsf_resample_len(n_in, orig_sr, target_sr);
  if (out_capacity < n_out) { set_error("nsf_resample_host: out_capacity < nsf_resample_len()"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  // one mono clip of the conversion kernel (float32 samples are its f32 encoding, int16 its i16 encoding)
  const nsf_pcm_source src{0, n_in, pcm_format == NSF_PCM_I16 ? NSF_ENC_I16 : NSF_ENC_F32, 1, orig_sr, 0};
  const size_t in_bytes = static_cast<size_t>(n_in) * (pcm_format == NSF_PCM_I16 ? 2 : 4);
  const size_t out_bytes = static_cast<size_t>(n_out) * sizeof(float);
  const int64_t off[2] = {0, n_out};
  return run_once(ctx, [&](Slot* sl) -> nsf_status {
    nsf_status st;
    if ((st = sl->in[0].reserve(in_bytes)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(out_bytes)) != NSF_OK) return st;
    if ((st = upload(sl, 0, pcm_host, in_bytes, true)) != NSF_OK) return st;
    if ((st = convert_enqueue(ctx, sl->stream, sl->in[0].ptr, &src, 1, target_sr, off, static_cast<float*>(sl->out[0].ptr),
                              true)) != NSF_OK) return st;
    return download(sl, 0, out_host, out_bytes, out_bytes, 1, true);
  });
}

nsf_status nsf_convert_offsets(const nsf_pcm_source* sources, int32_t n, int32_t target_sr, int64_t payload_bytes,
                               int64_t* out_offsets) {
  return convert_offsets(sources, n, target_sr, payload_bytes, 0, out_offsets);
}

nsf_status nsf_convert_batch(nsf_ctx* ctx, void* cuda_stream, const void* payload_dev, int64_t payload_bytes,
                             const nsf_pcm_source* sources, int32_t n, int32_t target_sr, float* out_dev,
                             const int64_t* out_offsets_host) {
  if (!ctx || !payload_dev || !out_dev) { set_error("nsf_convert_batch: NULL argument"); return NSF_ERR_BAD_ARG; }
  std::vector<int64_t>& off = ctx->conv_off;
  off.resize(n > 0 ? n + 1 : 1);
  nsf_status st = convert_offsets(sources, n, target_sr, payload_bytes, reinterpret_cast<uintptr_t>(payload_dev), off.data());
  if (st != NSF_OK) return st;
  if (out_offsets_host) {
    for (int i = 0; i < n; ++i)
      if (out_offsets_host[i + 1] - out_offsets_host[i] != off[i + 1] - off[i]) {
        set_error("nsf_convert_batch: out_offsets is not a prefix sum of the output lengths"); return NSF_ERR_BAD_ARG;
      }
    for (int i = 0; i <= n; ++i) off[i] = out_offsets_host[i];
  }
  NSF_CUDA(cudaSetDevice(ctx->device));
  return convert_enqueue(ctx, static_cast<cudaStream_t>(cuda_stream), payload_dev, sources, n, target_sr, off.data(),
                         out_dev, false);
}

nsf_status nsf_convert_host(nsf_ctx* ctx, const void* payload_host, int64_t payload_bytes, const nsf_pcm_source* sources,
                            int32_t n, int32_t target_sr, float* out_host) {
  if (!ctx || !payload_host || !out_host) { set_error("nsf_convert_host: NULL argument"); return NSF_ERR_BAD_ARG; }
  std::vector<int64_t>& all = ctx->conv_group_off;
  all.resize(n > 0 ? n + 1 : 1);
  nsf_status st = convert_offsets(sources, n, target_sr, payload_bytes, 0, all.data());
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const bool in_dma = dma_reachable(payload_host), out_dma = dma_reachable(out_host);
  // clip groups by output samples
  return run_groups(ctx, all.data(), n, [&](int first, int last, Slot* sl) -> nsf_status {
    // the group's input bytes [b0, b1), b0 rounded down to 8 so every container keeps its alignment in the arena
    int64_t b0 = INT64_MAX, b1 = 0;
    for (int i = first; i < last; ++i) {
      const nsf_pcm_source& c = sources[i];
      const int64_t end = c.byte_offset + c.frames * c.channels * enc_bytes(c.encoding);
      if (c.frames > 0) { b0 = std::min(b0, c.byte_offset); b1 = std::max(b1, end); }
    }
    if (b0 > b1) b0 = b1 = 0;
    b0 &= ~int64_t(7);
    const int64_t in_bytes = b1 - b0, n_out = all[last] - all[first];
    std::vector<nsf_pcm_source>& g = ctx->conv_src;
    std::vector<int64_t>& goff = ctx->conv_off;
    g.assign(sources + first, sources + last);
    goff.resize(last - first + 1);
    for (int i = first; i < last; ++i) { g[i - first].byte_offset = sources[i].frames > 0 ? sources[i].byte_offset - b0 : 0; }
    for (int i = first; i <= last; ++i) goff[i - first] = all[i] - all[first];
    nsf_status st;
    if ((st = sl->in[0].reserve(std::max<int64_t>(in_bytes, 1))) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(std::max<int64_t>(n_out, 1) * sizeof(float))) != NSF_OK) return st;
    if (in_bytes > 0 && (st = upload(sl, 0, static_cast<const char*>(payload_host) + b0, in_bytes, in_dma)) != NSF_OK)
      return st;
    if ((st = convert_enqueue(ctx, sl->stream, sl->in[0].ptr, g.data(), last - first, target_sr, goff.data(),
                              static_cast<float*>(sl->out[0].ptr), false)) != NSF_OK) return st;
    const size_t bytes = static_cast<size_t>(n_out) * sizeof(float);
    return n_out > 0 ? download(sl, 0, out_host + all[first], bytes, bytes, 1, out_dma) : NSF_OK;
  });
}

// ---- FLAC decode -------------------------------------------------------------------------------------
namespace {
// Validates every descriptor; out_off[i] = first output byte of stream i, cost[i] = int32 samples before stream i.
nsf_status flac_offsets(const nsf_flac_source* src, int32_t n, int64_t payload_bytes, int64_t* out_off, int64_t* cost) {
  if (!src || n <= 0) { set_error("nsf_flac_decode_host: NULL sources or n <= 0"); return NSF_ERR_BAD_ARG; }
  if (payload_bytes < 0) { set_error("nsf_flac_decode_host: negative payload_bytes"); return NSF_ERR_BAD_ARG; }
  out_off[0] = cost[0] = 0;
  for (int i = 0; i < n; ++i) {
    const nsf_flac_source& c = src[i];
    char buf[200];
    auto fail = [&](const char* what) {
      std::snprintf(buf, sizeof buf, "nsf_flac_decode_host: source %d: %s", i, what);
      set_error(buf);
      return NSF_ERR_BAD_ARG;
    };
    if (c.bits != 8 && c.bits != 16 && c.bits != 24) return fail("bits must be 8, 16 or 24");
    if (c.channels < 1 || c.channels > 8) return fail("channels must be in [1, 8]");
    if (c.frames <= 0) return fail("frames must be positive");
    if (c.max_block < 1 || c.max_block > 65535) return fail("max_block must be in [1, 65535]");
    if (c.sample_rate <= 0) return fail("sample_rate must be positive");
    if (c.byte_offset < 0 || c.byte_length < 0 || c.byte_offset > payload_bytes ||
        c.byte_length > payload_bytes - c.byte_offset)
      return fail("byte range outside the payload");
    if (c.byte_length > INT32_MAX) return fail("byte_length must be below 2^31");
    if (c.frames > (int64_t(1) << 36)) return fail("frames above 2^36");
    out_off[i + 1] = out_off[i] + c.frames * c.channels * (c.bits / 8);
    cost[i + 1] = cost[i] + c.frames * c.channels;
  }
  return NSF_OK;
}

// Walks stream s's frame chain over the group's candidates cand[c0, c1) (those of stream s, in byte order): the first
// frame at the stream's first byte, each next one where the previous ended, numbers consecutive, samples tiling
// [0, frames).  Appends the kept frames; on a broken chain sets the error (payload offsets) and returns false.
bool flac_chain(const uint8_t* payload, int64_t b0, int s_index, const FlacStream& st, int64_t frames,
                const FlacCand* cand, int64_t c0, int64_t c1, int64_t g_base, int64_t scratch_base,
                std::vector<FlacKept>* kept) {
  int64_t at = st.begin, sample = 0, index = 0, c = c0;
  int variable = -1;
  char buf[256];
  auto fail = [&](const char* why) {
    std::snprintf(buf, sizeof buf, "FLAC stream %d: frame at byte %lld: %s", s_index, static_cast<long long>(b0 + at), why);
    set_error(buf);
    return false;
  };
  while (sample < frames) {
    if (at >= st.end) return fail("stream ends before its STREAMINFO total samples");
    while (c < c1 && cand[c].start < at) ++c;
    if (c == c1 || cand[c].start != at) {
      const int why = flac_header_status(payload, at, st.end);
      return fail(why == NSF_FLAC_OK ? "no frame header" : flac_status_text(why));
    }
    const FlacCand& f = cand[c];
    if (f.status != NSF_FLAC_OK) return fail(flac_status_text(f.status));
    const int var = f.assignment >> 4;
    if (variable < 0) variable = var;
    if (var != variable) return fail("blocking strategy changes within the stream");
    if (f.number != (variable ? sample : index))
      return fail(variable ? "first sample number out of sequence" : "frame number out of sequence");
    if (f.block > frames - sample) return fail("frame runs past the STREAMINFO total samples");
    kept->push_back(FlacKept{static_cast<int32_t>(c), 0, g_base + sample, sample, scratch_base + sample * st.channels});
    sample += f.block;
    ++index;
    at = f.end;
  }
  return true;
}
}  // namespace

nsf_status nsf_flac_decode_host(nsf_ctx* ctx, const void* payload_host, int64_t payload_bytes,
                                const nsf_flac_source* sources, int32_t n, void* pcm_host) {
  if (!ctx || !payload_host || !pcm_host) { set_error("nsf_flac_decode_host: NULL argument"); return NSF_ERR_BAD_ARG; }
  std::vector<int64_t> out_off(n > 0 ? n + 1 : 1), cost(n > 0 ? n + 1 : 1);
  nsf_status st = flac_offsets(sources, n, payload_bytes, out_off.data(), cost.data());
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const uint8_t* payload = static_cast<const uint8_t*>(payload_host);
  const bool in_dma = dma_reachable(payload_host), out_dma = dma_reachable(pcm_host);
  std::vector<FlacStream> gs;
  std::vector<FlacKept> kept;
  // stream groups by decoded samples
  return run_groups(ctx, cost.data(), n, [&](int first, int last, Slot* sl) -> nsf_status {
    int64_t b0 = INT64_MAX, b1 = 0, scan = 0, cap = 0, out_frames = 0;
    int max_ch = 1;
    for (int i = first; i < last; ++i) {
      b0 = std::min(b0, sources[i].byte_offset);
      b1 = std::max(b1, sources[i].byte_offset + sources[i].byte_length);
    }
    gs.clear();
    for (int i = first; i < last; ++i) {
      const nsf_flac_source& c = sources[i];
      gs.push_back(FlacStream{c.byte_offset - b0, c.byte_offset + c.byte_length - b0, scan, out_off[i] - out_off[first],
                              c.channels, c.bits, c.sample_rate, c.max_block});
      scan += c.byte_length;
      cap += 2 * ((c.frames + c.max_block - 1) / c.max_block) + 16;   // room for a few false syncs per stream
      out_frames += c.frames;
      max_ch = std::max(max_ch, c.channels);
    }
    const int ng = last - first;
    const int64_t in_bytes = b1 - b0, out_bytes = out_off[last] - out_off[first], samples = cost[last] - cost[first];
    if (scan == 0) return NSF_OK;   // unreachable: frames > 0 needs bytes, and the chain reports their absence
    nsf_status st;
    if ((st = sl->in[0].reserve(std::max<int64_t>(in_bytes, 1))) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(out_bytes)) != NSF_OK) return st;
    if ((st = upload(sl, 0, payload + b0, in_bytes, in_dma)) != NSF_OK) return st;
    const size_t streams_bytes = ng * sizeof(FlacStream);
    DescEntry* de_streams = nullptr;
    st = desc_upload(ctx, sl->stream, streams_bytes, nullptr, streams_bytes, &de_streams,
                     [&](void* mem) { std::memcpy(mem, gs.data(), streams_bytes); });
    if (st != NSF_OK) return st;
    const FlacStream* d_streams = static_cast<const FlacStream*>(de_streams->dev.ptr);
    const uint8_t* d_payload = static_cast<const uint8_t*>(sl->in[0].ptr);
    const int64_t n_blk = (scan + kFlacScanTile - 1) / kFlacScanTile;
    // work: [scratch | tile counts | tile offsets | total | positions | candidates]; the table comes back to the
    // pinned stage_out[1] as [total | candidates].  One wait, unless the candidates overflow `cap` (false syncs
    // beyond the allowance): then the scan runs again with room for all of them.
    FlacCand* d_cand = nullptr;
    int64_t* d_total = nullptr;
    int32_t* d_scratch = nullptr;
    const FlacCand* cand = nullptr;
    int64_t total = 0;
    for (;;) {
      Carver sizer(reinterpret_cast<void*>(0x1000), ~size_t(0) >> 1);
      auto carve = [&](Carver& c) {
        d_scratch = c.take<int32_t>(samples);
        int32_t* d_count = c.take<int32_t>(n_blk);
        int64_t* d_off = c.take<int64_t>(n_blk);
        d_total = c.take<int64_t>(1);
        int64_t* d_pos = c.take<int64_t>(cap);
        d_cand = c.take<FlacCand>(cap);
        return std::make_pair(d_count, std::make_pair(d_off, d_pos));
      };
      carve(sizer);
      if ((st = sl->work.reserve(sizer.used)) != NSF_OK) return st;
      Carver cv(sl->work.ptr, sl->work.bytes);
      const auto ptrs = carve(cv);
      const size_t table_bytes = sizeof(int64_t) + cap * sizeof(FlacCand);
      if ((st = sl->stage_out[1].reserve(table_bytes)) != NSF_OK) return st;
      NSF_LAUNCH(ctx, launch_flac_scan_parse(sl->stream, d_streams, ng, scan, d_payload, ptrs.first, ptrs.second.first,
                                             d_total, ptrs.second.second, d_cand, cap));
      char* table = static_cast<char*>(sl->stage_out[1].ptr);
      NSF_CUDA(cudaMemcpyAsync(table, d_total, sizeof(int64_t), cudaMemcpyDeviceToHost, sl->stream));
      NSF_CUDA(cudaMemcpyAsync(table + sizeof(int64_t), d_cand, cap * sizeof(FlacCand), cudaMemcpyDeviceToHost,
                               sl->stream));
      NSF_CUDA(cudaStreamSynchronize(sl->stream));
      std::memcpy(&total, table, sizeof total);
      cand = reinterpret_cast<const FlacCand*>(table + sizeof(int64_t));
      if (total <= cap) break;
      cap = total;
    }
    // each stream's chain; candidates are in scan order, so stream by stream
    kept.clear();
    int64_t c0 = 0, g_base = 0, scratch_base = 0;
    for (int s = 0; s < ng; ++s) {
      int64_t c1 = c0;
      while (c1 < total && cand[c1].stream == s) ++c1;
      const size_t k0 = kept.size();
      if (!flac_chain(payload + b0, b0, first + s, gs[s], sources[first + s].frames, cand, c0, c1, g_base, scratch_base,
                      &kept))
        return NSF_ERR_BAD_ARG;
      for (size_t k = k0; k < kept.size(); ++k) kept[k].stream = s;
      g_base += sources[first + s].frames;
      scratch_base += sources[first + s].frames * sources[first + s].channels;
      c0 = c1;
    }
    if (kept.size() > static_cast<size_t>(INT32_MAX)) { set_error("nsf_flac_decode_host: too many frames"); return NSF_ERR_UNSUPPORTED; }
    const size_t kept_bytes = kept.size() * sizeof(FlacKept);
    DescEntry* de_kept = nullptr;
    st = desc_upload(ctx, sl->stream, kept_bytes, nullptr, kept_bytes, &de_kept,
                     [&](void* mem) { std::memcpy(mem, kept.data(), kept_bytes); });
    if (st != NSF_OK) return st;
    NSF_LAUNCH(ctx, launch_flac_decode(sl->stream, d_streams, d_cand, static_cast<const FlacKept*>(de_kept->dev.ptr),
                                       static_cast<int>(kept.size()), max_ch, out_frames, d_payload, d_scratch,
                                       static_cast<uint8_t*>(sl->out[0].ptr)));
    if ((st = desc_commit(de_streams, sl->stream)) != NSF_OK || (st = desc_commit(de_kept, sl->stream)) != NSF_OK) return st;
    return download(sl, 0, static_cast<uint8_t*>(pcm_host) + out_off[first], out_bytes, out_bytes, 1, out_dma);
  });
}

// ---- collect ---------------------------------------------------------------------------------------
// Checks shared by the collect calls (element type, column counts, offsets) and their output packing: o_off is the
// prefix sum of nsf_collect_rows(), and must equal o_off_in when that is given.
static nsf_status collect_offsets(int32_t dtype, int32_t a_cols, int32_t f_cols, const int64_t* a_off,
                                  const int64_t* f_off, int32_t n, uint32_t flags, int32_t blend_frames,
                                  const int64_t* o_off_in, std::vector<int64_t>* o_off) {
  nsf_status st = check_dtype("nsf_collect", dtype);
  if (st != NSF_OK) return st;
  if (a_cols <= 0 || f_cols <= 0) { set_error("nsf_collect: column counts must be positive"); return NSF_ERR_BAD_ARG; }
  if (!a_off || !f_off || n <= 0) { set_error("nsf_collect: NULL offsets or n_clips <= 0"); return NSF_ERR_BAD_ARG; }
  if ((st = check_nondecreasing("nsf_collect: offsets", a_off, n)) != NSF_OK ||
      (st = check_nondecreasing("nsf_collect: offsets", f_off, n)) != NSF_OK) return st;
  o_off->resize(n + 1);
  (*o_off)[0] = 0;
  for (int i = 0; i < n; ++i) {
    const int64_t r = nsf_collect_rows(a_off[i + 1] - a_off[i], f_off[i + 1] - f_off[i], flags, blend_frames);
    if (o_off_in && o_off_in[i + 1] - o_off_in[i] != r) {
      set_error("nsf_collect: out_offsets is not the prefix sum of nsf_collect_rows()");
      return NSF_ERR_BAD_ARG;
    }
    (*o_off)[i + 1] = (*o_off)[i] + r;
  }
  return NSF_OK;
}

nsf_status nsf_collect_batch(nsf_ctx* ctx, void* cuda_stream, int32_t dtype, const void* audio_dev,
                             int32_t audio_cols, const int64_t* audio_offsets_host, const void* facial_dev,
                             int32_t facial_cols, const int64_t* facial_offsets_host, int32_t n_clips,
                             uint32_t collect_flags, int32_t blend_frames, void* out_audio_dev,
                             void* out_facial_dev, const int64_t* out_offsets_host) {
  if (!ctx || !audio_dev || !facial_dev || !out_audio_dev || !out_facial_dev) {
    set_error("nsf_collect_batch: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  std::vector<int64_t> o_off;
  nsf_status st = collect_offsets(dtype, audio_cols, facial_cols, audio_offsets_host, facial_offsets_host, n_clips,
                                  collect_flags, blend_frames, out_offsets_host, &o_off);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = dtype == NSF_F64 ? 8 : 4;
  const int64_t a0 = audio_offsets_host[0], f0 = facial_offsets_host[0], o0 = out_offsets_host ? out_offsets_host[0] : 0;
  return collect_enqueue(ctx, static_cast<cudaStream_t>(cuda_stream), dtype,
                         static_cast<const char*>(audio_dev) + a0 * audio_cols * esz, audio_cols, audio_offsets_host,
                         static_cast<const char*>(facial_dev) + f0 * facial_cols * esz, facial_cols, facial_offsets_host,
                         o_off.data(), n_clips, collect_flags, blend_frames,
                         static_cast<char*>(out_audio_dev) + o0 * audio_cols * esz,
                         static_cast<char*>(out_facial_dev) + o0 * facial_cols * esz);
}

nsf_status nsf_collect_host(nsf_ctx* ctx, int32_t dtype, const void* audio_host, int32_t audio_cols,
                            const int64_t* a_off, const void* facial_host, int32_t facial_cols,
                            const int64_t* f_off, int32_t n_clips, uint32_t collect_flags,
                            int32_t blend_frames, void* out_audio_host, void* out_facial_host) {
  if (!ctx || !audio_host || !facial_host || !out_audio_host || !out_facial_host) {
    set_error("nsf_collect_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  std::vector<int64_t> o_off;
  nsf_status st = collect_offsets(dtype, audio_cols, facial_cols, a_off, f_off, n_clips, collect_flags, blend_frames,
                                  nullptr, &o_off);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = dtype == NSF_F64 ? 8 : 4;
  const size_t a_bytes = (a_off[n_clips] - a_off[0]) * audio_cols * esz, f_bytes = (f_off[n_clips] - f_off[0]) * facial_cols * esz;
  const size_t oa_bytes = o_off[n_clips] * audio_cols * esz, of_bytes = o_off[n_clips] * facial_cols * esz;
  return run_once(ctx, [&](Slot* sl) -> nsf_status {
    nsf_status st;
    if ((st = sl->in[0].reserve(a_bytes)) != NSF_OK) return st;
    if ((st = sl->in[1].reserve(f_bytes)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(oa_bytes)) != NSF_OK) return st;
    if ((st = sl->out[1].reserve(of_bytes)) != NSF_OK) return st;
    if ((st = upload(sl, 0, static_cast<const char*>(audio_host) + a_off[0] * audio_cols * esz, a_bytes, true)) != NSF_OK ||
        (st = upload(sl, 1, static_cast<const char*>(facial_host) + f_off[0] * facial_cols * esz, f_bytes, true)) != NSF_OK)
      return st;
    if ((st = collect_enqueue(ctx, sl->stream, dtype, sl->in[0].ptr, audio_cols, a_off, sl->in[1].ptr, facial_cols, f_off,
                              o_off.data(), n_clips, collect_flags, blend_frames, sl->out[0].ptr, sl->out[1].ptr)) != NSF_OK)
      return st;
    if ((st = download(sl, 0, out_audio_host, oa_bytes, oa_bytes, 1, true)) != NSF_OK) return st;
    return download(sl, 1, out_facial_host, of_bytes, of_bytes, 1, true);
  });
}

// ---- fused extract + collect (dataset builders) -------------------------------------------------------
nsf_status nsf_extract_collect_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                                    const int64_t* clip_offsets, int32_t n_clips, uint32_t flags,
                                    const float* facial_host, int32_t facial_cols, const int64_t* f_off,
                                    uint32_t collect_flags, int32_t blend_frames, float* out_audio_host,
                                    float* out_facial_host, float* features_host) {
  if (!ctx || !pcm_host || !clip_offsets || !facial_host || !f_off || !out_audio_host || !out_facial_host ||
      n_clips <= 0 || facial_cols <= 0) {
    set_error("nsf_extract_collect_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  nsf_status st = check_pcm_format(pcm_format);
  if (st != NSF_OK) return st;
  const Plan& p = ctx->plan->p;
  const int cols = nsf_feature_cols(ctx->plan, flags);
  HostDesc& all = ctx->hd_all;
  if ((st = build_desc(p, clip_offsets, n_clips, flags, nullptr, &all)) != NSF_OK) return st;
  // output packing over the whole batch (validates the facial offsets)
  std::vector<int64_t> o_all;
  if ((st = collect_offsets(NSF_F32, cols, facial_cols, all.row_off.data(), f_off, n_clips, collect_flags, blend_frames,
                            nullptr, &o_all)) != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4;
  const size_t row_bytes = static_cast<size_t>(cols) * sizeof(float), fac_row_bytes = static_cast<size_t>(facial_cols) * sizeof(float);
  const bool pcm_dma = dma_reachable(pcm_host), fac_dma = dma_reachable(facial_host);
  const bool oa_dma = dma_reachable(out_audio_host), of_dma = dma_reachable(out_facial_host);
  const bool ft_dma = features_host ? dma_reachable(features_host) : true;
  // device: in = [PCM, facial rows], out = [feature rows, collected audio rows, collected facial rows]
  return run_groups(ctx, clip_offsets, n_clips, [&](int first, int last, Slot* sl) -> nsf_status {
    const int64_t samples = clip_offsets[last] - clip_offsets[first];
    const int64_t rows = all.row_off[last] - all.row_off[first];
    const int64_t frows = f_off[last] - f_off[first], orows = o_all[last] - o_all[first];
    nsf_status st;
    if ((st = sl->in[0].reserve(samples * esz)) != NSF_OK) return st;
    if ((st = sl->in[1].reserve(frows * fac_row_bytes)) != NSF_OK) return st;
    if ((st = sl->work.reserve(nsf_workspace_bytes(ctx->plan, samples, last - first, flags))) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(rows * row_bytes)) != NSF_OK) return st;
    if ((st = sl->out[1].reserve(orows * row_bytes)) != NSF_OK) return st;
    if ((st = sl->out[2].reserve(orows * fac_row_bytes)) != NSF_OK) return st;
    if ((st = upload(sl, 0, static_cast<const char*>(pcm_host) + clip_offsets[first] * esz, samples * esz, pcm_dma)) != NSF_OK)
      return st;
    if ((st = upload(sl, 1, facial_host + f_off[first] * facial_cols, frows * fac_row_bytes, fac_dma)) != NSF_OK) return st;
    if ((st = extract_group(ctx, sl, pcm_format, clip_offsets + first, last - first, flags, cols, nullptr)) != NSF_OK) return st;
    if ((st = collect_enqueue(ctx, sl->stream, NSF_F32, sl->out[0].ptr, cols, all.row_off.data() + first, sl->in[1].ptr,
                              facial_cols, f_off + first, o_all.data() + first, last - first, collect_flags, blend_frames,
                              sl->out[1].ptr, sl->out[2].ptr)) != NSF_OK) return st;
    if (features_host &&   // the un-augmented rows as well (what collect_features caches as audio_features.csv)
        (st = download(sl, 0, features_host + all.row_off[first] * cols, row_bytes, row_bytes, rows, ft_dma)) != NSF_OK)
      return st;
    if ((st = download(sl, 1, out_audio_host + o_all[first] * cols, row_bytes, row_bytes, orows, oa_dma)) != NSF_OK) return st;
    return download(sl, 2, out_facial_host + o_all[first] * facial_cols, fac_row_bytes, fac_row_bytes, orows, of_dma);
  });
}

// ---- audio_features.csv text ------------------------------------------------------------------------------
nsf_status nsf_format_csv_host(nsf_ctx* ctx, int32_t dtype, const void* rows_host, int32_t cols,
                               const int64_t* row_off, int32_t n_files, char* text_host, int64_t text_capacity,
                               int64_t* text_off) {
  if (!ctx || !rows_host || !row_off || !text_host || !text_off || cols < 1 || n_files < 0) {
    set_error("nsf_format_csv_host: NULL argument, cols < 1 or n_files < 0"); return NSF_ERR_BAD_ARG;
  }
  nsf_status st = check_dtype("nsf_format_csv_host", dtype);
  if (st == NSF_OK) st = check_nondecreasing("nsf_format_csv_host: offsets", row_off, n_files);
  if (st != NSF_OK) return st;
  const int64_t n_rows = row_off[n_files] - row_off[0];
  if (text_capacity < nsf_csv_bytes_bound(n_rows, cols, n_files)) {
    set_error("nsf_format_csv_host: text_capacity below nsf_csv_bytes_bound()"); return NSF_ERR_BAD_ARG;
  }
  text_off[0] = 0;
  if (n_files == 0) return NSF_OK;
  NSF_CUDA(cudaSetDevice(ctx->device));
  const size_t row_bytes = static_cast<size_t>(cols) * (dtype == NSF_F64 ? 8 : 4);
  const int64_t header = csv_header_bytes(cols);
  std::vector<int64_t> cost(n_files + 1);   // file groups by value count
  for (int i = 0; i <= n_files; ++i) cost[i] = (row_off[i] - row_off[0]) * cols;
  const bool in_dma = dma_reachable(rows_host), out_dma = dma_reachable(text_host);
  // device: in = [rows, row and header positions], out = [text, row lengths]
  return run_groups(ctx, cost.data(), n_files, [&](int first, int last, Slot* sl) -> nsf_status {
    const int64_t r0 = row_off[first] - row_off[0], nr = row_off[last] - row_off[first], nf = last - first;
    if (nr + nf > INT32_MAX) { set_error("nsf_format_csv_host: more than 2^31 rows in one file"); return NSF_ERR_UNSUPPORTED; }
    const size_t pos_bytes = static_cast<size_t>(nr + nf) * sizeof(int64_t), len_bytes = nr * sizeof(int64_t);
    nsf_status st;
    if ((st = sl->in[0].reserve(std::max<size_t>(nr * row_bytes, 1))) != NSF_OK) return st;
    if ((st = sl->in[1].reserve(pos_bytes)) != NSF_OK) return st;
    if ((st = sl->out[1].reserve(std::max<size_t>(len_bytes, 1))) != NSF_OK) return st;
    if ((st = sl->stage_in[1].reserve(pos_bytes)) != NSF_OK) return st;
    if ((st = sl->stage_out[1].reserve(std::max<size_t>(len_bytes, 1))) != NSF_OK) return st;
    if (nr > 0) {   // the group's row lengths, and with them its text size: the group's one wait
      if ((st = upload(sl, 0, static_cast<const char*>(rows_host) + r0 * row_bytes, nr * row_bytes, in_dma)) != NSF_OK) return st;
      NSF_LAUNCH(ctx, launch_csv_lengths(sl->stream, dtype, sl->in[0].ptr, nr, cols, static_cast<int64_t*>(sl->out[1].ptr)));
      if ((st = download(sl, 1, sl->stage_out[1].ptr, len_bytes, len_bytes, 1, true)) != NSF_OK) return st;
      NSF_CUDA(cudaStreamSynchronize(sl->stream));
    }
    // positions from the group's first byte: each file's header, then its rows
    const int64_t* len = static_cast<const int64_t*>(sl->stage_out[1].ptr);
    int64_t* pos = static_cast<int64_t*>(sl->stage_in[1].ptr);
    int64_t at = 0;
    for (int i = first; i < last; ++i) {
      pos[nr + i - first] = at;
      at += header;
      for (int64_t r = row_off[i] - row_off[first]; r < row_off[i + 1] - row_off[first]; ++r) { pos[r] = at; at += len[r]; }
      text_off[i + 1] = text_off[first] + at;
    }
    if ((st = upload(sl, 1, pos, pos_bytes, true)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(at)) != NSF_OK) return st;
    NSF_LAUNCH(ctx, launch_csv_write(sl->stream, dtype, sl->in[0].ptr, nr, cols, static_cast<int32_t>(nf),
                                     static_cast<const int64_t*>(sl->in[1].ptr), static_cast<char*>(sl->out[0].ptr)));
    return download(sl, 0, text_host + text_off[first], at, at, 1, out_dma);
  });
}

// ---- CSV text -> rows ----------------------------------------------------------------------------------------
namespace {
// Checks shared by the two CSV calls; tile_off[i] = tiles of the files before file i.
nsf_status csv_text_args(const char* fn, nsf_ctx* ctx, const char* text_dev, const int64_t* text_off, int32_t n_files,
                         std::vector<int64_t>* tile_off) {
  char buf[160];
  if (!ctx || !text_off || n_files < 0) {
    std::snprintf(buf, sizeof buf, "%s: NULL argument or n_files < 0", fn); set_error(buf); return NSF_ERR_BAD_ARG;
  }
  if (n_files == 0) return NSF_OK;
  if (text_off[0] < 0) { std::snprintf(buf, sizeof buf, "%s: negative text offset", fn); set_error(buf); return NSF_ERR_BAD_ARG; }
  const nsf_status st = check_nondecreasing(std::string(fn) + ": text offsets", text_off, n_files);
  if (st != NSF_OK) return st;
  tile_off->assign(n_files + 1, 0);
  for (int i = 0; i < n_files; ++i) (*tile_off)[i + 1] = (*tile_off)[i] + csv_tiles(text_off[i], text_off[i + 1]);
  if (text_off[n_files] > text_off[0] && (!text_dev || reinterpret_cast<uintptr_t>(text_dev) % 16 != 0)) {
    std::snprintf(buf, sizeof buf, "%s: text_dev is NULL or not 16-byte aligned", fn); set_error(buf); return NSF_ERR_BAD_ARG;
  }
  if ((*tile_off)[n_files] > INT32_MAX) {
    std::snprintf(buf, sizeof buf, "%s: text too long for one call", fn); set_error(buf); return NSF_ERR_UNSUPPORTED;
  }
  return NSF_OK;
}
}  // namespace

nsf_status nsf_csv_row_offsets(nsf_ctx* ctx, void* cuda_stream, const char* text_dev, const int64_t* text_off,
                               int32_t n_files, int64_t* row_off) {
  std::vector<int64_t> tile_off;
  nsf_status st = csv_text_args("nsf_csv_row_offsets", ctx, text_dev, text_off, n_files, &tile_off);
  if (st != NSF_OK) return st;
  if (!row_off) { set_error("nsf_csv_row_offsets: row_offsets_host is NULL"); return NSF_ERR_BAD_ARG; }
  row_off[0] = 0;
  if (n_files == 0) return NSF_OK;
  NSF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  const size_t n1 = static_cast<size_t>(n_files) + 1, n_tiles = static_cast<size_t>(tile_off[n_files]);
  // ring entry: host [text_off | tile_off], which the row counts overwrite on their way back (the download is queued
  // behind the upload); device [text_off | tile_off | row_off | tile_start | tile_rows]
  const size_t bytes = 2 * n1 * sizeof(int64_t);
  const size_t dev_bytes = bytes + (n1 + n_tiles + 1) * sizeof(int64_t) + std::max<size_t>(n_tiles, 1) * sizeof(int32_t);
  DescEntry* de = nullptr;
  st = desc_upload(ctx, s, bytes, nullptr, dev_bytes, &de, [&](void* mem) {
    std::memcpy(mem, text_off, n1 * sizeof(int64_t));
    std::memcpy(static_cast<int64_t*>(mem) + n1, tile_off.data(), n1 * sizeof(int64_t));
  });
  if (st != NSF_OK) return st;
  int64_t* d = static_cast<int64_t*>(de->dev.ptr);
  CsvView v{};
  v.text = text_dev; v.text_off = d; v.tile_off = d + n1; v.n_files = n_files; v.n_tiles = static_cast<int64_t>(n_tiles);
  int64_t* d_rows = d + 2 * n1;
  int64_t* d_tile_start = d + 3 * n1;
  int32_t* d_tile_rows = reinterpret_cast<int32_t*>(d_tile_start + n_tiles + 1);
  NSF_LAUNCH(ctx, launch_csv_row_offsets(s, v, d_tile_rows, d_tile_start, d_rows));
  NSF_CUDA(cudaMemcpyAsync(de->mem.ptr, d_rows, n1 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  if ((st = desc_commit(de, s)) != NSF_OK) return st;
  NSF_CUDA(cudaStreamSynchronize(s));   // the call's one host wait
  std::memcpy(row_off, de->mem.ptr, n1 * sizeof(int64_t));
  return NSF_OK;
}

nsf_status nsf_csv_parse(nsf_ctx* ctx, void* cuda_stream, int32_t dtype, const char* text_dev, const int64_t* text_off,
                         int32_t n_files, int32_t cols, const int32_t* out_col, int32_t out_cols, const int64_t* row_off,
                         void* out_dev, int64_t out_ld, uint32_t* status_dev) {
  std::vector<int64_t> tile_off;
  nsf_status st = csv_text_args("nsf_csv_parse", ctx, text_dev, text_off, n_files, &tile_off);
  if (st != NSF_OK) return st;
  if (!out_col || !row_off || !status_dev || cols < 1 || out_cols < 0) {
    set_error("nsf_csv_parse: NULL argument, cols < 1 or out_cols < 0"); return NSF_ERR_BAD_ARG;
  }
  if ((st = check_dtype("nsf_csv_parse", dtype)) != NSF_OK) return st;
  if (out_ld < out_cols) { set_error("nsf_csv_parse: out_ld < out_cols"); return NSF_ERR_BAD_ARG; }
  std::vector<char> used(out_cols, 0);
  for (int c = 0; c < cols; ++c) {
    const int oc = out_col[c];
    if (oc < -1 || oc >= out_cols || (oc >= 0 && used[oc]++)) {
      set_error("nsf_csv_parse: out_col entries must lie in [-1, out_cols) and name each output column at most once");
      return NSF_ERR_BAD_ARG;
    }
  }
  if (row_off[0] != 0) { set_error("nsf_csv_parse: row offsets must start at 0"); return NSF_ERR_BAD_ARG; }
  if ((st = check_nondecreasing("nsf_csv_parse: row offsets", row_off, n_files)) != NSF_OK) return st;
  const int64_t n_rows = row_off[n_files];
  if (n_rows > 0 && !out_dev) { set_error("nsf_csv_parse: out_dev is NULL"); return NSF_ERR_BAD_ARG; }
  if (n_rows > INT32_MAX) { set_error("nsf_csv_parse: more than 2^31 rows in one call"); return NSF_ERR_UNSUPPORTED; }
  if (n_files == 0) return NSF_OK;
  NSF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  const size_t n1 = static_cast<size_t>(n_files) + 1, n_tiles = static_cast<size_t>(tile_off[n_files]);
  // ring entry: [text_off | tile_off | row_off | out_col (int32)], then on the device only: tile_start, row_start,
  // col_flags, tile_rows
  const size_t desc = 3 * n1 * sizeof(int64_t) + align_up(static_cast<size_t>(cols) * sizeof(int32_t), 8);
  const size_t flags_bytes = n1 * static_cast<size_t>(cols) * sizeof(uint32_t);
  const size_t dev_bytes = desc + (n_tiles + 1 + static_cast<size_t>(n_rows)) * sizeof(int64_t) + flags_bytes +
                           std::max<size_t>(n_tiles, 1) * sizeof(int32_t);
  DescEntry* de = nullptr;
  st = desc_upload(ctx, s, desc, nullptr, dev_bytes, &de, [&](void* mem) {
    char* h = static_cast<char*>(mem);
    std::memcpy(h, text_off, n1 * sizeof(int64_t));
    std::memcpy(h + n1 * 8, tile_off.data(), n1 * sizeof(int64_t));
    std::memcpy(h + 2 * n1 * 8, row_off, n1 * sizeof(int64_t));
    std::memcpy(h + 3 * n1 * 8, out_col, static_cast<size_t>(cols) * sizeof(int32_t));
  });
  if (st != NSF_OK) return st;
  char* d = static_cast<char*>(de->dev.ptr);
  int64_t* d_tile_start = reinterpret_cast<int64_t*>(d + desc);
  int64_t* d_row_start = d_tile_start + n_tiles + 1;
  uint32_t* d_flags = reinterpret_cast<uint32_t*>(d_row_start + n_rows);
  int32_t* d_tile_rows = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(d_flags) + flags_bytes);
  NSF_CUDA(cudaMemsetAsync(d_flags, 0, flags_bytes, s));
  NSF_CUDA(cudaMemsetAsync(status_dev, 0, static_cast<size_t>(n_files) * sizeof(uint32_t), s));
  CsvView v{};
  v.text = text_dev;
  v.text_off = reinterpret_cast<const int64_t*>(d);
  v.tile_off = v.text_off + n1;
  v.row_off = v.text_off + 2 * n1;
  v.out_col = reinterpret_cast<const int32_t*>(d + 3 * n1 * 8);
  v.n_files = n_files; v.cols = cols; v.n_tiles = static_cast<int64_t>(n_tiles); v.n_rows = n_rows;
  NSF_LAUNCH(ctx, launch_csv_parse(s, v, dtype, d_tile_rows, d_tile_start, d_row_start, d_flags, out_dev, out_ld, status_dev));
  return desc_commit(de, s);
}

// ---- inference-side chunker ---------------------------------------------------------------------------
int64_t nsf_chunk_count(int64_t n_rows, int32_t frame, int32_t overlap) {
  if (n_rows <= 0 || frame <= 0 || overlap < 0 || overlap >= frame) return 0;
  const int64_t stride = frame - overlap;
  return (n_rows + stride - 1) / stride;            // starts 0, stride, 2 stride, ... while start < n_rows
}

// The reference blends every new chunk into the LAST `n` rows of what it has accumulated; the kernels assume those
// are the rows the chunk starts at, which holds whenever frame - overlap >= overlap (and in every other geometry
// this walk accepts).  Returns false for a geometry where the reference's own bookkeeping shifts rows.
static bool chunk_geometry_aligned(int64_t n_rows, int32_t frame, int32_t overlap) {
  const int64_t stride = frame - overlap, n_chunks = nsf_chunk_count(n_rows, frame, overlap);
  int64_t acc = std::min<int64_t>(frame, n_rows);
  for (int64_t k = 1; k < n_chunks; ++k) {
    const int64_t s = k * stride, len_k = std::min<int64_t>(frame, n_rows - s);
    const int64_t n = std::min<int64_t>(std::min<int64_t>(overlap, acc), len_k);
    if (acc - n != s) return false;
    if (k + 1 < n_chunks && (k + 1) * stride < s + n) return false;   // cross-fade zones must not overlap
    acc += len_k - n;
  }
  return acc == n_rows;
}

nsf_status nsf_chunk_gather(nsf_ctx* ctx, void* cuda_stream, const float* rows_dev, int64_t n_rows, int32_t cols,
                            int64_t ld, int32_t frame, int32_t overlap, float* chunks_dev) {
  if (!ctx || !rows_dev || !chunks_dev || cols <= 0 || ld < cols) { set_error("nsf_chunk_gather: bad argument"); return NSF_ERR_BAD_ARG; }
  const int64_t n_chunks = nsf_chunk_count(n_rows, frame, overlap);
  if (n_chunks <= 0) { set_error("nsf_chunk_gather: need n_rows > 0 and 0 <= overlap < frame"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  NSF_LAUNCH(ctx, launch_chunk_gather(static_cast<cudaStream_t>(cuda_stream), rows_dev, n_rows, cols, ld, frame, overlap,
                                      n_chunks, chunks_dev));
  return NSF_OK;
}

nsf_status nsf_chunk_blend(nsf_ctx* ctx, void* cuda_stream, const float* decoded_dev, int64_t n_rows, int32_t out_cols,
                           int32_t frame, int32_t overlap, int32_t scale_cols, float divisor, float* out_dev) {
  if (!ctx || !decoded_dev || !out_dev || out_cols <= 0 || scale_cols < 0) { set_error("nsf_chunk_blend: bad argument"); return NSF_ERR_BAD_ARG; }
  const int64_t n_chunks = nsf_chunk_count(n_rows, frame, overlap);
  if (n_chunks <= 0) { set_error("nsf_chunk_blend: need n_rows > 0 and 0 <= overlap < frame"); return NSF_ERR_BAD_ARG; }
  if (scale_cols > 0 && divisor == 0.0f) { set_error("nsf_chunk_blend: divisor is zero"); return NSF_ERR_BAD_ARG; }
  if (!chunk_geometry_aligned(n_rows, frame, overlap)) {
    set_error("nsf_chunk_blend: overlap larger than half a chunk shifts rows in the reference's bookkeeping; not implemented");
    return NSF_ERR_UNSUPPORTED;
  }
  NSF_CUDA(cudaSetDevice(ctx->device));
  NSF_LAUNCH(ctx, launch_chunk_blend(static_cast<cudaStream_t>(cuda_stream), decoded_dev, n_rows, out_cols, frame, overlap,
                                     n_chunks, scale_cols, divisor, out_dev));
  return NSF_OK;
}

// ---- training windows --------------------------------------------------------------------------------------
nsf_status nsf_window_offsets(const int64_t* a_off, const int64_t* f_off, int32_t n_clips, int32_t window,
                              int64_t* w_off) {
  if (!a_off || !f_off || !w_off || n_clips < 1) { set_error("nsf_window_offsets: NULL argument or n_clips < 1"); return NSF_ERR_BAD_ARG; }
  if (window < 1) { set_error("nsf_window_offsets: window must be >= 1"); return NSF_ERR_BAD_ARG; }
  if (a_off[0] < 0 || f_off[0] < 0) { set_error("nsf_window_offsets: negative offset"); return NSF_ERR_BAD_ARG; }
  nsf_status st = check_nondecreasing("nsf_window_offsets: offsets", a_off, n_clips);
  if (st != NSF_OK || (st = check_nondecreasing("nsf_window_offsets: offsets", f_off, n_clips)) != NSF_OK) return st;
  w_off[0] = 0;
  char buf[200];
  for (int i = 0; i < n_clips; ++i) {
    const int64_t na = a_off[i + 1] - a_off[i], nf = f_off[i + 1] - f_off[i];
    const int64_t top = std::max(na, nf);
    if (top < window) {   // dataset.py:77-91 fails on such a clip (broadcast error in the tail branch)
      std::snprintf(buf, sizeof buf, "clip %d has %lld rows, fewer than the window of %d", i, static_cast<long long>(top), window);
      set_error(buf);
      return NSF_ERR_BAD_ARG;
    }
    const bool tail = top % window != 0;
    if (tail) {
      // the tail window mirrors the last seg rows of each stream into the rest of the window: the host route fails
      // when a stream has fewer than window / 2 rows there, unless it has exactly one (which torch broadcasts)
      for (int64_t n : {na, nf}) {
        const int64_t seg = std::max<int64_t>(0, std::min(top, n) - (top - window));
        if (2 * seg < window && seg != 1) {
          std::snprintf(buf, sizeof buf, "clip %d: a stream of %lld rows leaves %lld rows for the tail window of %d (at least half are needed)",
                        i, static_cast<long long>(n), static_cast<long long>(seg), window);
          set_error(buf);
          return NSF_ERR_BAD_ARG;
        }
      }
    }
    w_off[i + 1] = w_off[i] + (top - window + 1) + (tail ? 1 : 0);
  }
  return NSF_OK;
}

nsf_status nsf_window_gather(nsf_ctx* ctx, void* cuda_stream, const float* audio_dev, int32_t audio_cols,
                             const int64_t* a_off, const float* facial_dev, int32_t facial_cols, const int64_t* f_off,
                             int32_t n_clips, int32_t window, const int64_t* indices, int64_t n, float* out_audio_dev,
                             float* out_facial_dev) {
  // an empty batch writes nothing: its outputs may be NULL (what a zero-size tensor's data pointer is)
  if (!ctx || !audio_dev || !facial_dev || audio_cols < 1 || facial_cols < 1 || n < 0 ||
      (n > 0 && (!indices || !out_audio_dev || !out_facial_dev))) {
    set_error("nsf_window_gather: bad argument"); return NSF_ERR_BAD_ARG;
  }
  if (n_clips < 1) { set_error("nsf_window_gather: n_clips < 1"); return NSF_ERR_BAD_ARG; }
  const size_t n1 = static_cast<size_t>(n_clips) + 1;
  std::vector<int64_t> w_off(n1);
  nsf_status st = nsf_window_offsets(a_off, f_off, n_clips, window, w_off.data());
  if (st != NSF_OK) return st;
  const int64_t total = w_off[n_clips];
  for (int64_t k = 0; k < n; ++k)
    if (indices[k] < 0 || indices[k] >= total) {
      char buf[120];
      std::snprintf(buf, sizeof buf, "nsf_window_gather: index %lld at position %lld is outside [0, %lld)",
                    static_cast<long long>(indices[k]), static_cast<long long>(k), static_cast<long long>(total));
      set_error(buf);
      return NSF_ERR_BAD_ARG;
    }
  if (n == 0) return NSF_OK;
  const int64_t tiles = (window + kWindowTileRows - 1) / kWindowTileRows;
  if (n > INT32_MAX / tiles) { set_error("nsf_window_gather: too many windows for one launch"); return NSF_ERR_UNSUPPORTED; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  // one descriptor block [a_off | f_off | w_off | indices] through the ring; its device copy lives in the ring entry,
  // which is reused only after this call's kernel has run
  const size_t bytes = (3 * n1 + static_cast<size_t>(n)) * sizeof(int64_t);
  DescEntry* de = nullptr;
  st = desc_upload(ctx, s, bytes, nullptr, bytes, &de, [&](void* mem) {
    int64_t* h = static_cast<int64_t*>(mem);
    std::memcpy(h, a_off, n1 * sizeof(int64_t));
    std::memcpy(h + n1, f_off, n1 * sizeof(int64_t));
    std::memcpy(h + 2 * n1, w_off.data(), n1 * sizeof(int64_t));
    std::memcpy(h + 3 * n1, indices, static_cast<size_t>(n) * sizeof(int64_t));
  });
  if (st != NSF_OK) return st;
  const int64_t* d = static_cast<const int64_t*>(de->dev.ptr);
  WindowView v;
  v.a_off = d; v.f_off = d + n1; v.w_off = d + 2 * n1; v.index = d + 3 * n1;
  v.n_clips = n_clips; v.window = window; v.n = n;
  NSF_LAUNCH(ctx, launch_window_gather(s, v, audio_dev, audio_cols, facial_dev, facial_cols, out_audio_dev, out_facial_dev));
  return desc_commit(de, s);
}

nsf_status nsf_rows_host(nsf_ctx* ctx, int32_t op, int32_t dtype, const void* a_host, int64_t na,
                         const void* b_host, int64_t nb, int32_t cols, int32_t blend_frames, void* out_host) {
  if (!ctx || !a_host || !out_host || na <= 0 || cols <= 0) { set_error("nsf_rows_host: bad argument"); return NSF_ERR_BAD_ARG; }
  nsf_status st = check_dtype("nsf_rows_host", dtype);
  if (st != NSF_OK) return st;
  int64_t out_rows = 0, k = 0;
  if (op == NSF_ROWS_INTERP_SLOWER) out_rows = 2 * na - 1;
  else if (op == NSF_ROWS_SMOOTH) out_rows = na;
  else if (op == NSF_ROWS_BLEND_STACK) {
    if (!b_host || nb <= 0) { set_error("nsf_rows_host: blend needs a second array"); return NSF_ERR_BAD_ARG; }
    k = std::max<int64_t>(0, std::min<int64_t>(std::min<int64_t>(blend_frames, na), nb));
    out_rows = na + nb - k;
  } else { set_error("nsf_rows_host: unknown op"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = dtype == NSF_F64 ? 8 : 4;
  const bool two = op == NSF_ROWS_BLEND_STACK;
  const size_t a_bytes = na * cols * esz, b_bytes = two ? nb * cols * esz : 0, out_bytes = out_rows * cols * esz;
  return run_once(ctx, [&](Slot* sl) -> nsf_status {
    nsf_status st;
    if ((st = sl->in[0].reserve(a_bytes)) != NSF_OK) return st;
    if (two && (st = sl->in[1].reserve(b_bytes)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(out_bytes)) != NSF_OK) return st;
    if ((st = upload(sl, 0, a_host, a_bytes, true)) != NSF_OK) return st;
    if (two && (st = upload(sl, 1, b_host, b_bytes, true)) != NSF_OK) return st;
    NSF_LAUNCH(ctx, launch_rows_op(sl->stream, op, dtype, sl->in[0].ptr, na, two ? sl->in[1].ptr : nullptr, nb, cols, k,
                                   sl->out[0].ptr, out_rows));
    return download(sl, 0, out_host, out_bytes, out_bytes, 1, true);
  });
}

nsf_status nsf_post_host(nsf_ctx* ctx, const float* in_host, int64_t T, int32_t Cc, uint32_t pf, float* out_host) {
  if (!ctx || !in_host || !out_host || T <= 0 || Cc <= 0) { set_error("nsf_post_host: bad argument"); return NSF_ERR_BAD_ARG; }
  if ((pf & NSF_POST_DELTAS) && T < 9) { set_error("nsf_post_host: delta needs at least 9 frames"); return NSF_ERR_TOO_SHORT; }
  if ((pf & NSF_POST_EDGEFIX) && T < 2) { set_error("nsf_post_host: edge fix needs 2 frames"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  const bool reduce = (pf & NSF_POST_REDUCE) != 0, deltas = (pf & NSF_POST_DELTAS) != 0, cmvn = (pf & NSF_POST_CMVN) != 0;
  const int64_t rows = reduce ? (T + 1) / 2 : T;
  const int out_c = Cc * (deltas ? 3 : 1);
  const size_t in_bytes = T * Cc * sizeof(float), out_bytes = rows * out_c * sizeof(float);
  // in[0] = frames, out[0] = rows, work = [desc 6 x int64][sum C][sumsq C]
  const size_t desc_b = align_up(6 * sizeof(int64_t)), st_b = align_up(Cc * sizeof(double));
  return run_once(ctx, [&](Slot* sl) -> nsf_status {
    nsf_status st;
    if ((st = sl->in[0].reserve(in_bytes)) != NSF_OK) return st;
    if ((st = sl->out[0].reserve(out_bytes)) != NSF_OK) return st;
    if ((st = sl->work.reserve(desc_b + 2 * st_b)) != NSF_OK) return st;
    char* base = static_cast<char*>(sl->work.ptr);
    float* d_in = static_cast<float*>(sl->in[0].ptr);
    int64_t* d_desc = reinterpret_cast<int64_t*>(base);
    double* d_sum = reinterpret_cast<double*>(base + desc_b);
    double* d_sq = reinterpret_cast<double*>(base + desc_b + st_b);
    DescEntry* de = nullptr;
    st = desc_upload(ctx, sl->stream, 6 * sizeof(int64_t), d_desc, 0, &de, [&](void* mem) {
      int64_t* h = static_cast<int64_t*>(mem);
      h[0] = 0; h[1] = 0;           // clip_off (unused by the post kernels)
      h[2] = 0; h[3] = T;           // frame_off
      h[4] = 0; h[5] = rows;        // row_off
    });
    if (st != NSF_OK || (st = desc_commit(de, sl->stream)) != NSF_OK) return st;
    if ((st = upload(sl, 0, in_host, in_bytes, true)) != NSF_OK) return st;
    if (pf & NSF_POST_EDGEFIX) NSF_LAUNCH(ctx, launch_edge_fix(sl->stream, d_in, T, Cc, ctx->edge_zero_threshold));
    if (cmvn) NSF_LAUNCH(ctx, launch_col_stats(sl->stream, d_in, T, Cc, d_sum, d_sq));
    BatchView b;
    b.clip_off = d_desc; b.frame_off = d_desc + 2; b.row_off = d_desc + 4;
    b.n_clips = 1; b.total_samples = 0; b.total_frames = T; b.total_rows = rows;
    NSF_LAUNCH(ctx, launch_delta_reduce(sl->stream, b, d_in, Cc, Cc, d_sum, d_sq, cmvn, deltas, reduce,
                                        static_cast<float*>(sl->out[0].ptr), out_c, 0));
    return download(sl, 0, out_host, out_bytes, out_bytes, 1, true);
  });
}

}  // extern "C"

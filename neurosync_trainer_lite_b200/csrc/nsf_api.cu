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
  Arena pcm, out, work, ynorm;
  Arena fac_in, col_a, col_f, col_desc;   // fused extract + collect path
  cudaEvent_t done = nullptr;
  // pageable callers: the group's PCM is gathered into `stage_in` (pinned) before its upload and its rows
  // come back through `stage_out` (pinned); `pending_*` describe the copy-out owed to the caller's buffers
  PinnedArena stage_in, stage_out, stage_aux, stage_fac, stage_feat;
  struct CopyOut { void* dst; const void* src; size_t bytes; size_t dst_pitch, src_pitch, width; int64_t rows; };
  CopyOut pending[4];
  int n_pending = 0;
};

// Ring of pinned descriptor staging buffers.  A stream-ordered call writes its (tiny) descriptor arrays into
// the next ring entry, enqueues the upload and records the entry's event; the entry is reused kDescRing calls
// later, so the host only ever waits when that many calls' descriptor uploads are still outstanding.
constexpr int kDescRing = 8;
struct DescEntry {
  PinnedArena mem;
  Arena dev;              // device copy of the entry, for calls whose descriptors have no other home (nsf_convert_batch)
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
  nsf::DctCoef dct_coef{};       // DCT matrix as a kernel parameter (default 128 -> 23 shape only)
  bool dct_coef_ok = false;
  nsf::Arena table_mem;
  nsf::DescEntry desc[nsf::kDescRing];
  int desc_next = 0;
  nsf::HostDesc hd_batch, hd_all;   // scratch of nsf_extract_batch / the host pipelines
  float edge_zero_threshold = 1e-7f;   // fix_edge_frames_autocorr(zero_threshold=1e-7)
  int resample_quality = NSF_RESAMPLE_HQ;
  nsf::Slot slot[nsf::kSlots];
  int64_t launches = 0;
  bool profiling = false;
  bool pipelined = false;     // set by the host passes around their nsf_extract_batch calls (front-end grid caps)
  cudaEvent_t stage_ev[nsf::kStages + 1] = {};
  bool stage_valid = false;
  nsf::Arena collect_in_a, collect_in_f, collect_out_a, collect_out_f, collect_desc;
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
  const bool dct_frag_ok = p.n_mels == kDctConstMels && p.n_mfcc == kDctConstMfcc;
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
  ctx->dct_coef_ok = p.n_mels == kDctConstMels && p.n_mfcc == kDctConstMfcc;
  if (ctx->dct_coef_ok)
    for (int m = 0; m < kDctConstMels; ++m)
      for (int k = 0; k < kDctConstMfcc; ++k)
        ctx->dct_coef.v[m * kDctConstLd + k] = p.dct[static_cast<size_t>(k) * p.n_mels + m];
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
nsf_status desc_commit(DescEntry* d, cudaStream_t s) {
  NSF_CUDA(cudaEventRecord(d->copied, s));
  d->pending = true;
  return NSF_OK;
}

// Host-side descriptor build + validation shared by the device and host entry points.
nsf_status build_desc(const Plan& p, const int64_t* clip_offsets, int32_t n_clips, uint32_t flags,
                      const int64_t* out_row_offsets, HostDesc* d) {
  if (!clip_offsets || n_clips <= 0) {
    set_error("clip_offsets is NULL or n_clips <= 0");
    return NSF_ERR_BAD_ARG;
  }
  d->clip_off.resize(n_clips + 1);
  d->frame_off.resize(n_clips + 1);
  d->row_off.resize(n_clips + 1);
  const int64_t origin = clip_offsets[0];
  d->frame_off[0] = 0;
  d->row_off[0] = out_row_offsets ? out_row_offsets[0] : 0;
  for (int i = 0; i < n_clips; ++i) {
    const int64_t len = clip_offsets[i + 1] - clip_offsets[i];
    if (len < 0) { set_error("clip_offsets must be non-decreasing"); return NSF_ERR_BAD_ARG; }
    // NSF_AC_NO_PAD (pad_signal=False): frames are y[t H : t H + F], as many as fit
    const bool no_pad = (flags & NSF_AC_NO_PAD) != 0;
    const int64_t T = no_pad ? (len >= p.F ? nsf_guard_frames(len, p.F, p.H) : 0) : nsf_hop_frames(len, p.F, p.H);
    // librosa.feature.delta(width=9) raises below 9 frames; the edge fix and reflect padding need
    // 2 frames and F/2 + 1 samples.  (The 9-frame *guard* of extract_features.py:16 counts
    // un-padded frames and belongs to the caller: see nsf_guard_frames.)
    const bool any_delta = (!(flags & NSF_NO_DELTAS) && !(flags & NSF_NO_MFCC)) ||
                           ((flags & NSF_AC_DELTAS) && !(flags & NSF_NO_AUTOCORR));
    const int64_t need = any_delta ? kMinGuardFrames : (no_pad ? 1 : 2);
    if (T < need || len <= p.F / 2) {
      char buf[160];
      std::snprintf(buf, sizeof buf, "clip %d is too short: %lld hop-frames, required: %lld", i,
                    static_cast<long long>(T), static_cast<long long>(need));
      set_error(buf);
      return NSF_ERR_TOO_SHORT;
    }
    const int64_t R = (flags & NSF_NO_REDUCE) ? T : (T + 1) / 2;
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
    if (s.done) cudaEventDestroy(s.done);
    s.pcm.release(); s.out.release(); s.work.release(); s.ynorm.release();
    s.fac_in.release(); s.col_a.release(); s.col_f.release(); s.col_desc.release();
    s.stage_in.release(); s.stage_out.release(); s.stage_aux.release(); s.stage_fac.release(); s.stage_feat.release();
  }
  for (auto& e : ctx->stage_ev) if (e) cudaEventDestroy(e);
  for (auto& d : ctx->desc) {
    if (d.copied) cudaEventDestroy(d.copied);
    d.mem.release();
    d.dev.release();
  }
  for (TapTable* t : ctx->tap_tables) { t->mem.release(); delete t; }
  ctx->table_mem.release();
  ctx->collect_in_a.release(); ctx->collect_in_f.release();
  ctx->collect_out_a.release(); ctx->collect_out_f.release(); ctx->collect_desc.release();
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
  if (!ctx || !pcm_dev || !out_dev || !workspace_dev) { set_error("nsf_extract_batch: NULL argument"); return NSF_ERR_BAD_ARG; }
  if (pcm_format != NSF_PCM_F32 && pcm_format != NSF_PCM_I16) { set_error("unknown pcm_format"); return NSF_ERR_BAD_ARG; }
  const Plan& p = ctx->plan->p;
  const int cols = nsf_feature_cols(ctx->plan, flags);
  if (out_ld < cols) { set_error("out_ld smaller than the feature width"); return NSF_ERR_BAD_ARG; }
  if (workspace_bytes <= 0) { set_error("workspace_bytes must be positive; size it with nsf_workspace_bytes()"); return NSF_ERR_WORKSPACE; }
  HostDesc& hd = ctx->hd_batch;
  nsf_status st = build_desc(p, clip_offsets_host, n_clips, flags, out_row_offsets_host, &hd);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);

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

  // descriptors: next entry of the pinned ring -> device, one stream-ordered upload, no host wait
  const size_t n1 = static_cast<size_t>(n_clips) + 1;
  DescEntry* de = nullptr;
  if ((st = desc_acquire(ctx, 3 * n1 * sizeof(int64_t), &de)) != NSF_OK) return st;
  int64_t* hstage = static_cast<int64_t*>(de->mem.ptr);
  const int64_t row_origin = hd.row_off[0];
  for (size_t i = 0; i < n1; ++i) {
    hstage[i] = hd.clip_off[i];
    hstage[n1 + i] = hd.frame_off[i];
    hstage[2 * n1 + i] = hd.row_off[i] - row_origin;
  }
  NSF_CUDA(cudaMemcpyAsync(L.clip_off, hstage, 3 * n1 * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  if ((st = desc_commit(de, s)) != NSF_OK) return st;
  NSF_CUDA(cudaMemsetAsync(wbase + L.zero_begin, 0, L.zero_bytes, s));

  BatchView b;
  b.clip_off = L.clip_off; b.frame_off = L.frame_off; b.row_off = L.row_off;
  b.n_clips = n_clips; b.total_samples = hd.total_samples; b.total_frames = hd.total_frames;
  b.total_rows = hd.total_rows;
  float* out = out_dev + row_origin * out_ld;
  const DeviceTables& t = ctx->tables;
  StageTimer timer{ctx, s};
  int launched = 0;
#define NSF_LAUNCH(expr)                                                   \
  do {                                                                     \
    const int n__ = (expr);                                                \
    if (n__ < 0) { set_error(cuda_msg(#expr, cudaGetLastError())); return NSF_ERR_CUDA; } \
    launched += n__;                                                       \
  } while (0)

  // stage 0: decode / peak normalise
  timer.mark(0);
  const float* y = static_cast<const float*>(pcm_dev);
  if (need_y) {
    float* ydst = y_norm_dev ? y_norm_dev : L.y;
    const bool capped = ctx->pipelined;           // inside a pipelined host pass: stay off the copy engine's HBM share
    if (normalize) NSF_LAUNCH(launch_absmax(s, pcm_dev, pcm_format, b, L.peak_bits, capped ? kPipelinedAbsmaxBlocks : 0));
    NSF_LAUNCH(launch_normalize(s, pcm_dev, pcm_format, b, L.peak_bits, normalize, ydst, capped ? kPipelinedNormalizeBlocks : 0));
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
  if (!do_mfcc && (flags & NSF_NO_AUTOCORR)) { set_error("NSF_NO_MFCC | NSF_NO_AUTOCORR leaves nothing to compute"); return NSF_ERR_BAD_ARG; }
  // pad_signal=False exists for the autocorrelation branch only (librosa's STFT always centre-pads)
  DeviceTables t_ac = t;
  if (flags & NSF_AC_NO_PAD) {
    if (do_mfcc) { set_error("NSF_AC_NO_PAD needs NSF_NO_MFCC: only the autocorrelation branch has a pad_signal switch"); return NSF_ERR_UNSUPPORTED; }
    t_ac.pad = 0;
  }

  // stages 1-3: STFT power -> mel -> dB (+ per-clip max)
  bool fused_mel = false;
  if (!do_mfcc) {
    // autocorrelation block only
  } else if (flags & NSF_DEBUG_SIMT_DFT) {
    timer.mark(1);
    NSF_LAUNCH(launch_fold32(s, t, b, y, L.a32));
    timer.mark(2);
    NSF_LAUNCH(launch_dft_simt(s, t, b, L.a32, L.power));
  } else {
    timer.mark(1);
    NSF_LAUNCH(launch_stft_tc_fold(s, ctx->tc, t, b, y, L.tc_a));
    timer.mark(2);
    if (t.mel_col_ok && !(flags & NSF_DEBUG_UNFUSED_MEL)) {
      // product path: STFT GEMM with the power -> mel -> dB epilogue fused (no power round trip)
      NSF_LAUNCH(launch_stft_tc_mel(s, ctx->tc, t, b, L.tc_a, L.db, L.dbmax_key));
      fused_mel = true;
    } else {
      NSF_LAUNCH(launch_stft_tc_gemm(s, ctx->tc, t, b, L.tc_a, L.power));
    }
  }
  timer.mark(3);
  if (do_mfcc && !fused_mel) NSF_LAUNCH(launch_mel_db(s, t, b, L.power, L.db, L.dbmax_key));
  // stage 4: floor + DCT + CMVN statistics
  timer.mark(4);
  if (do_mfcc) {
    NSF_LAUNCH(launch_dct_sum(s, t, b, L.db, L.dbmax_key, L.mfcc_raw, L.sum, L.sumsq,
                              ctx->dct_coef_ok ? &ctx->dct_coef : nullptr));
  }
  // stage 5: CMVN + deltas + pair reduce -> columns [0, mfcc_cols)
  timer.mark(5);
  if (do_mfcc)
    NSF_LAUNCH(launch_delta_reduce(s, b, L.mfcc_raw, p.n_mfcc, p.n_mfcc, L.sum, L.sumsq,
                                   !(flags & NSF_NO_CMVN), deltas, reduce, stage_out, stage_ld, 0));
  // stage 6: autocorrelation -> columns [mfcc_cols, ...)
  timer.mark(6);
  if (!(flags & NSF_NO_AUTOCORR)) {
    if (flags & NSF_AC_DELTAS) {
      BatchView bf = b;  // un-reduced: one row per hop-frame
      bf.row_off = L.frame_off; bf.total_rows = hd.total_frames;
      if (flags & NSF_DEBUG_FMA_AUTOCORR) NSF_LAUNCH(launch_autocorr(s, t_ac, bf, y, false, L.ac_raw, p.n_lags, 0));
      else NSF_LAUNCH(launch_autocorr_mma(s, t_ac, bf, y, false, L.ac_raw, p.n_lags, 0));
      NSF_LAUNCH(launch_delta_reduce(s, b, L.ac_raw, p.n_lags, p.n_lags, nullptr, nullptr, false, true,
                                     reduce, stage_out, stage_ld, mfcc_cols));
    } else {
      if (flags & NSF_DEBUG_FMA_AUTOCORR) NSF_LAUNCH(launch_autocorr(s, t_ac, b, y, reduce, stage_out, stage_ld, mfcc_cols));
      else NSF_LAUNCH(launch_autocorr_mma(s, t_ac, b, y, reduce, stage_out, stage_ld, mfcc_cols));
    }
  }
  // stage 7: optional smoothing
  timer.mark(7);
  if (flags & NSF_SMOOTH) NSF_LAUNCH(launch_smooth(s, b, L.tmp_out, cols, cols, out, out_ld));
  timer.finish();
  ctx->launches += launched;
#undef NSF_LAUNCH
  return NSF_OK;
}

// ---- host-buffer pipeline ------------------------------------------------------------------------
static nsf_status ensure_slot(Slot* sl) {
  if (!sl->stream) NSF_CUDA(cudaStreamCreateWithFlags(&sl->stream, cudaStreamNonBlocking));
  if (!sl->done) NSF_CUDA(cudaEventCreateWithFlags(&sl->done, cudaEventDisableTiming));
  return NSF_OK;
}

// Is `p` memory the copy engines can reach directly (cudaHostAlloc / cudaHostRegister / managed)?  Pageable
// buffers are staged through the slot's pinned arenas so that uploads and downloads stay asynchronous.
static bool dma_reachable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// memcpy split over a few threads once it is large enough to be bound by one core's copy bandwidth.
static void host_copy(void* dst, const void* src, size_t bytes) {
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

// Copy-outs a slot owes to pageable caller buffers; run once the slot's stream has drained.
static void flush_pending(Slot* sl) {
  for (int i = 0; i < sl->n_pending; ++i) {
    const Slot::CopyOut& c = sl->pending[i];
    if (c.rows <= 1 || (c.dst_pitch == c.width && c.src_pitch == c.width)) {
      host_copy(c.dst, c.src, c.rows <= 1 ? c.bytes : c.width * static_cast<size_t>(c.rows));
    } else {
      for (int64_t r = 0; r < c.rows; ++r)
        std::memcpy(static_cast<char*>(c.dst) + r * c.dst_pitch, static_cast<const char*>(c.src) + r * c.src_pitch, c.width);
    }
  }
  sl->n_pending = 0;
}
static nsf_status drain_slot(Slot* sl) {
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  flush_pending(sl);
  return NSF_OK;
}

nsf_status nsf_extract_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                            const int64_t* clip_offsets, int32_t n_clips, uint32_t flags,
                            float* out_host, int64_t out_ld, float* y_norm_host) {
  if (!ctx || !pcm_host || !out_host || !clip_offsets || n_clips <= 0) {
    set_error("nsf_extract_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  if (pcm_format != NSF_PCM_F32 && pcm_format != NSF_PCM_I16) { set_error("unknown pcm_format"); return NSF_ERR_BAD_ARG; }
  const Plan& p = ctx->plan->p;
  const int cols = nsf_feature_cols(ctx->plan, flags);
  if (out_ld < cols) { set_error("out_ld smaller than the feature width"); return NSF_ERR_BAD_ARG; }
  // validate everything up front so nothing is launched for a bad batch
  HostDesc& all = ctx->hd_all;
  nsf_status st = build_desc(p, clip_offsets, n_clips, flags, nullptr, &all);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  for (auto& sl : ctx->slot) sl.n_pending = 0;   // nothing is owed from an earlier call (errors drop their copy-outs)
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4;
  // pageable caller buffers go through the slot's pinned staging arenas: the host copies group g + 1 in (and
  // group g - 2 out) while the copy engines and kernels work on the groups in between
  const bool in_dma = dma_reachable(pcm_host), out_dma = dma_reachable(out_host);
  const bool y_dma = y_norm_host ? dma_reachable(y_norm_host) : true;
  int first = 0, turn = 0;
  while (first < n_clips) {
    int last = first;
    int64_t samples = 0;
    while (last < n_clips && (last == first || samples + (clip_offsets[last + 1] - clip_offsets[last]) <= group_budget(turn))) {
      samples += clip_offsets[last + 1] - clip_offsets[last];
      ++last;
    }
    const int gn = last - first;
    Slot* sl = &ctx->slot[turn % kSlots];
    st = ensure_slot(sl);
    if (st != NSF_OK) return st;
    // the slot's previous group must have fully drained before its buffers are reused
    if ((st = drain_slot(sl)) != NSF_OK) return st;
    const int64_t rows = all.row_off[last] - all.row_off[first];
    const int64_t wbytes = nsf_workspace_bytes(ctx->plan, samples, gn, flags);
    const size_t out_bytes = static_cast<size_t>(rows) * cols * sizeof(float);
    if ((st = sl->pcm.reserve(samples * esz)) != NSF_OK) return st;
    if ((st = sl->out.reserve(out_bytes)) != NSF_OK) return st;
    if ((st = sl->work.reserve(wbytes)) != NSF_OK) return st;
    if (y_norm_host && (st = sl->ynorm.reserve(samples * sizeof(float))) != NSF_OK) return st;
    const char* src = static_cast<const char*>(pcm_host) + clip_offsets[first] * esz;
    if (!in_dma) {
      if ((st = sl->stage_in.reserve(samples * esz)) != NSF_OK) return st;
      host_copy(sl->stage_in.ptr, src, samples * esz);
      src = static_cast<const char*>(sl->stage_in.ptr);
    }
    NSF_CUDA(cudaMemcpyAsync(sl->pcm.ptr, src, samples * esz, cudaMemcpyHostToDevice, sl->stream));
    ctx->pipelined = true;
    st = nsf_extract_batch(ctx, sl->stream, sl->pcm.ptr, pcm_format, clip_offsets + first, gn, flags,
                           static_cast<float*>(sl->out.ptr), cols, nullptr,
                           y_norm_host ? static_cast<float*>(sl->ynorm.ptr) : nullptr, sl->work.ptr,
                           static_cast<int64_t>(sl->work.bytes));
    ctx->pipelined = false;
    if (st != NSF_OK) return st;
    float* dst = out_host + all.row_off[first] * out_ld;
    if (!out_dma) {
      if ((st = sl->stage_out.reserve(out_bytes)) != NSF_OK) return st;
      NSF_CUDA(cudaMemcpyAsync(sl->stage_out.ptr, sl->out.ptr, out_bytes, cudaMemcpyDeviceToHost, sl->stream));
      sl->pending[sl->n_pending++] = Slot::CopyOut{dst, sl->stage_out.ptr, out_bytes, static_cast<size_t>(out_ld) * sizeof(float),
                                                   static_cast<size_t>(cols) * sizeof(float),
                                                   static_cast<size_t>(cols) * sizeof(float), rows};
    } else if (out_ld == cols) {
      NSF_CUDA(cudaMemcpyAsync(dst, sl->out.ptr, out_bytes, cudaMemcpyDeviceToHost, sl->stream));
    } else {
      NSF_CUDA(cudaMemcpy2DAsync(dst, out_ld * sizeof(float), sl->out.ptr, cols * sizeof(float),
                                 cols * sizeof(float), rows, cudaMemcpyDeviceToHost, sl->stream));
    }
    if (y_norm_host) {
      float* ydst = y_norm_host + (clip_offsets[first] - clip_offsets[0]);
      if (!y_dma) {
        if ((st = sl->stage_aux.reserve(samples * sizeof(float))) != NSF_OK) return st;
        NSF_CUDA(cudaMemcpyAsync(sl->stage_aux.ptr, sl->ynorm.ptr, samples * sizeof(float), cudaMemcpyDeviceToHost, sl->stream));
        sl->pending[sl->n_pending++] = Slot::CopyOut{ydst, sl->stage_aux.ptr, samples * sizeof(float), 0, 0, 0, 1};
      } else {
        NSF_CUDA(cudaMemcpyAsync(ydst, sl->ynorm.ptr, samples * sizeof(float), cudaMemcpyDeviceToHost, sl->stream));
      }
    }
    first = last;
    ++turn;
  }
  for (auto& sl : ctx->slot)
    if (sl.stream && (st = drain_slot(&sl)) != NSF_OK) return st;
  return NSF_OK;
}

nsf_status nsf_normalize_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                              const int64_t* clip_offsets, int32_t n_clips, float* y_host, float* peaks_host) {
  if (!ctx || !pcm_host || !clip_offsets || !y_host || n_clips <= 0) {
    set_error("nsf_normalize_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  if (pcm_format != NSF_PCM_F32 && pcm_format != NSF_PCM_I16) { set_error("unknown pcm_format"); return NSF_ERR_BAD_ARG; }
  for (int i = 0; i < n_clips; ++i)
    if (clip_offsets[i + 1] < clip_offsets[i]) { set_error("clip_offsets must be non-decreasing"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  Slot* sl = &ctx->slot[0];
  nsf_status st = ensure_slot(sl);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4;
  const int64_t samples = clip_offsets[n_clips] - clip_offsets[0];
  if (samples == 0) return NSF_OK;
  const size_t n1 = static_cast<size_t>(n_clips) + 1;
  // work arena: [clip_off n1 x int64][peak n x u32]
  const size_t off_b = align_up(n1 * sizeof(int64_t));
  if ((st = sl->pcm.reserve(samples * esz)) != NSF_OK) return st;
  if ((st = sl->ynorm.reserve(samples * sizeof(float))) != NSF_OK) return st;
  if ((st = sl->work.reserve(off_b + align_up(n_clips * sizeof(uint32_t)))) != NSF_OK) return st;
  DescEntry* de = nullptr;
  if ((st = desc_acquire(ctx, n1 * sizeof(int64_t), &de)) != NSF_OK) return st;
  int64_t* h = static_cast<int64_t*>(de->mem.ptr);
  for (size_t i = 0; i < n1; ++i) h[i] = clip_offsets[i] - clip_offsets[0];
  int64_t* d_off = static_cast<int64_t*>(sl->work.ptr);
  uint32_t* d_peak = reinterpret_cast<uint32_t*>(static_cast<char*>(sl->work.ptr) + off_b);
  NSF_CUDA(cudaMemcpyAsync(d_off, h, n1 * sizeof(int64_t), cudaMemcpyHostToDevice, sl->stream));
  if ((st = desc_commit(de, sl->stream)) != NSF_OK) return st;
  NSF_CUDA(cudaMemsetAsync(d_peak, 0, n_clips * sizeof(uint32_t), sl->stream));
  const char* src = static_cast<const char*>(pcm_host) + clip_offsets[0] * esz;
  NSF_CUDA(cudaMemcpyAsync(sl->pcm.ptr, src, samples * esz, cudaMemcpyHostToDevice, sl->stream));
  BatchView b{};
  b.clip_off = d_off; b.frame_off = d_off; b.row_off = d_off;
  b.n_clips = n_clips; b.total_samples = samples;
  int n = launch_absmax(sl->stream, sl->pcm.ptr, pcm_format, b, d_peak);
  if (n < 0) { set_error(cuda_msg("launch_absmax", cudaGetLastError())); return NSF_ERR_CUDA; }
  int m = launch_normalize(sl->stream, sl->pcm.ptr, pcm_format, b, d_peak, true, static_cast<float*>(sl->ynorm.ptr));
  if (m < 0) { set_error(cuda_msg("launch_normalize", cudaGetLastError())); return NSF_ERR_CUDA; }
  ctx->launches += n + m;
  NSF_CUDA(cudaMemcpyAsync(y_host, sl->ynorm.ptr, samples * sizeof(float), cudaMemcpyDeviceToHost, sl->stream));
  if (peaks_host)  // float bits of a non-negative float: copy as-is
    NSF_CUDA(cudaMemcpyAsync(peaks_host, d_peak, n_clips * sizeof(uint32_t), cudaMemcpyDeviceToHost, sl->stream));
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  return NSF_OK;
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
  nsf_status st = desc_acquire(ctx, bytes, &de);
  if (st != NSF_OK) return st;
  if ((st = de->dev.reserve(bytes)) != NSF_OK) return st;
  std::memcpy(de->mem.ptr, cl.data(), bytes);
  const ConvClip* d = static_cast<const ConvClip*>(de->dev.ptr);
  NSF_CUDA(cudaMemcpyAsync(de->dev.ptr, de->mem.ptr, bytes, cudaMemcpyHostToDevice, s));
  int launched = 0;
  for (int kind = 0; kind < 2; ++kind) {
    const ConvClip* first = d + (kind == 0 ? 0 : n_kind[0]);
    const int m = launch_convert(s, kind == 1, first, n_kind[kind], tiles[kind],
                                 kind == 1 ? static_cast<size_t>(max_window) * sizeof(double) : 0, payload_dev, out_dev);
    if (m < 0) { set_error(cuda_msg("launch_convert", cudaGetLastError())); return NSF_ERR_CUDA; }
    launched += m;
  }
  ctx->launches += launched;
  return desc_commit(de, s);     // recorded after the kernels: the entry (host and device) is reused only after them
}
}  // namespace

nsf_status nsf_resample_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format, int64_t n_in, int32_t orig_sr,
                             int32_t target_sr, float* out_host, int64_t out_capacity) {
  if (!ctx || !pcm_host || !out_host || n_in <= 0) { set_error("nsf_resample_host: NULL argument or empty input"); return NSF_ERR_BAD_ARG; }
  if (pcm_format != NSF_PCM_F32 && pcm_format != NSF_PCM_I16) { set_error("unknown pcm_format"); return NSF_ERR_BAD_ARG; }
  if (orig_sr <= 0 || target_sr <= 0) { set_error("nsf_resample_host: rates must be positive"); return NSF_ERR_BAD_ARG; }
  const int64_t n_out = nsf_resample_len(n_in, orig_sr, target_sr);
  if (out_capacity < n_out) { set_error("nsf_resample_host: out_capacity < nsf_resample_len()"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  Slot* sl = &ctx->slot[0];
  nsf_status st = ensure_slot(sl);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  // one mono clip of the conversion kernel (float32 samples are its f32 encoding, int16 its i16 encoding)
  const nsf_pcm_source src{0, n_in, pcm_format == NSF_PCM_I16 ? NSF_ENC_I16 : NSF_ENC_F32, 1, orig_sr, 0};
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4;
  const int64_t off[2] = {0, n_out};
  if ((st = sl->pcm.reserve(static_cast<size_t>(n_in) * esz)) != NSF_OK) return st;
  if ((st = sl->ynorm.reserve(static_cast<size_t>(n_out) * sizeof(float))) != NSF_OK) return st;
  NSF_CUDA(cudaMemcpyAsync(sl->pcm.ptr, pcm_host, static_cast<size_t>(n_in) * esz, cudaMemcpyHostToDevice, sl->stream));
  if ((st = convert_enqueue(ctx, sl->stream, sl->pcm.ptr, &src, 1, target_sr, off, static_cast<float*>(sl->ynorm.ptr),
                            true)) != NSF_OK) return st;
  NSF_CUDA(cudaMemcpyAsync(out_host, sl->ynorm.ptr, static_cast<size_t>(n_out) * sizeof(float), cudaMemcpyDeviceToHost, sl->stream));
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  return NSF_OK;
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
  for (auto& sl : ctx->slot) sl.n_pending = 0;
  const bool in_dma = dma_reachable(payload_host), out_dma = dma_reachable(out_host);
  // clip groups by output budget, rotating over the slots: the upload of group g + 1, the kernels of group g and the
  // download of group g - 1 overlap (see nsf_extract_host)
  int first = 0, turn = 0;
  while (first < n) {
    int last = first;
    while (last < n && (last == first || all[last + 1] - all[first] <= group_budget(turn))) ++last;
    Slot* sl = &ctx->slot[turn % kSlots];
    if ((st = ensure_slot(sl)) != NSF_OK) return st;
    if ((st = drain_slot(sl)) != NSF_OK) return st;
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
    if ((st = sl->pcm.reserve(std::max<int64_t>(in_bytes, 1))) != NSF_OK) return st;
    if ((st = sl->out.reserve(std::max<int64_t>(n_out, 1) * sizeof(float))) != NSF_OK) return st;
    if (in_bytes > 0) {
      const char* src = static_cast<const char*>(payload_host) + b0;
      if (!in_dma) {
        if ((st = sl->stage_in.reserve(in_bytes)) != NSF_OK) return st;
        host_copy(sl->stage_in.ptr, src, in_bytes);
        src = static_cast<const char*>(sl->stage_in.ptr);
      }
      NSF_CUDA(cudaMemcpyAsync(sl->pcm.ptr, src, in_bytes, cudaMemcpyHostToDevice, sl->stream));
    }
    if ((st = convert_enqueue(ctx, sl->stream, sl->pcm.ptr, g.data(), last - first, target_sr, goff.data(),
                              static_cast<float*>(sl->out.ptr), false)) != NSF_OK) return st;
    if (n_out > 0) {
      float* dst = out_host + all[first];
      const size_t bytes = static_cast<size_t>(n_out) * sizeof(float);
      if (!out_dma) {
        if ((st = sl->stage_out.reserve(bytes)) != NSF_OK) return st;
        NSF_CUDA(cudaMemcpyAsync(sl->stage_out.ptr, sl->out.ptr, bytes, cudaMemcpyDeviceToHost, sl->stream));
        sl->pending[sl->n_pending++] = Slot::CopyOut{dst, sl->stage_out.ptr, bytes, 0, 0, 0, 1};
      } else {
        NSF_CUDA(cudaMemcpyAsync(dst, sl->out.ptr, bytes, cudaMemcpyDeviceToHost, sl->stream));
      }
    }
    first = last;
    ++turn;
  }
  for (auto& sl : ctx->slot)
    if (sl.stream && (st = drain_slot(&sl)) != NSF_OK) return st;
  return NSF_OK;
}

// ---- collect ---------------------------------------------------------------------------------------
static nsf_status collect_offsets(const int64_t* a_off, const int64_t* f_off, int32_t n, uint32_t flags,
                                  int32_t blend_frames, const int64_t* o_off_in, std::vector<int64_t>* o_off) {
  if (!a_off || !f_off || n <= 0) { set_error("nsf_collect: NULL offsets or n_clips <= 0"); return NSF_ERR_BAD_ARG; }
  o_off->resize(n + 1);
  (*o_off)[0] = 0;
  for (int i = 0; i < n; ++i) {
    const int64_t na = a_off[i + 1] - a_off[i], nf = f_off[i + 1] - f_off[i];
    if (na < 0 || nf < 0) { set_error("nsf_collect: offsets must be non-decreasing"); return NSF_ERR_BAD_ARG; }
    const int64_t r = nsf_collect_rows(na, nf, flags, blend_frames);
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
  if ((dtype != NSF_F32 && dtype != NSF_F64) || audio_cols <= 0 || facial_cols <= 0) {
    set_error("nsf_collect_batch: bad dtype or column count"); return NSF_ERR_BAD_ARG;
  }
  std::vector<int64_t> o_off;
  nsf_status st = collect_offsets(audio_offsets_host, facial_offsets_host, n_clips, collect_flags,
                                  blend_frames, out_offsets_host, &o_off);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  const size_t n1 = static_cast<size_t>(n_clips) + 1;
  DescEntry* de = nullptr;
  if ((st = desc_acquire(ctx, 3 * n1 * sizeof(int64_t), &de)) != NSF_OK) return st;
  if ((st = ctx->collect_desc.reserve(3 * n1 * sizeof(int64_t))) != NSF_OK) return st;
  int64_t* h = static_cast<int64_t*>(de->mem.ptr);
  const int64_t a0 = audio_offsets_host[0], f0 = facial_offsets_host[0];
  const int64_t o0 = out_offsets_host ? out_offsets_host[0] : 0;
  for (size_t i = 0; i < n1; ++i) {
    h[i] = audio_offsets_host[i] - a0;
    h[n1 + i] = facial_offsets_host[i] - f0;
    h[2 * n1 + i] = o_off[i];
  }
  int64_t* d = static_cast<int64_t*>(ctx->collect_desc.ptr);
  NSF_CUDA(cudaMemcpyAsync(d, h, 3 * n1 * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  if ((st = desc_commit(de, s)) != NSF_OK) return st;
  CollectView v;
  v.a_off = d; v.f_off = d + n1; v.o_off = d + 2 * n1;
  v.n_clips = n_clips; v.total_out_rows = o_off[n_clips]; v.flags = collect_flags; v.blend_frames = blend_frames;
  const size_t esz = dtype == NSF_F64 ? 8 : 4;
  const char* a = static_cast<const char*>(audio_dev) + a0 * audio_cols * esz;
  const char* f = static_cast<const char*>(facial_dev) + f0 * facial_cols * esz;
  char* oa = static_cast<char*>(out_audio_dev) + o0 * audio_cols * esz;
  char* of = static_cast<char*>(out_facial_dev) + o0 * facial_cols * esz;
  const int n = launch_collect(s, dtype, v, a, audio_cols, f, facial_cols, oa, of);
  if (n < 0) { set_error(cuda_msg("launch_collect", cudaGetLastError())); return NSF_ERR_CUDA; }
  ctx->launches += n;
  return NSF_OK;
}

nsf_status nsf_collect_host(nsf_ctx* ctx, int32_t dtype, const void* audio_host, int32_t audio_cols,
                            const int64_t* a_off, const void* facial_host, int32_t facial_cols,
                            const int64_t* f_off, int32_t n_clips, uint32_t collect_flags,
                            int32_t blend_frames, void* out_audio_host, void* out_facial_host) {
  if (!ctx || !audio_host || !facial_host || !out_audio_host || !out_facial_host) {
    set_error("nsf_collect_host: NULL argument"); return NSF_ERR_BAD_ARG;
  }
  if (dtype != NSF_F32 && dtype != NSF_F64) { set_error("nsf_collect_host: bad dtype"); return NSF_ERR_BAD_ARG; }
  std::vector<int64_t> o_off;
  nsf_status st = collect_offsets(a_off, f_off, n_clips, collect_flags, blend_frames, nullptr, &o_off);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  Slot* sl = &ctx->slot[0];
  if ((st = ensure_slot(sl)) != NSF_OK) return st;
  const size_t esz = dtype == NSF_F64 ? 8 : 4;
  const size_t a_rows = a_off[n_clips] - a_off[0], f_rows = f_off[n_clips] - f_off[0];
  const size_t o_rows = o_off[n_clips];
  if ((st = ctx->collect_in_a.reserve(a_rows * audio_cols * esz)) != NSF_OK) return st;
  if ((st = ctx->collect_in_f.reserve(f_rows * facial_cols * esz)) != NSF_OK) return st;
  if ((st = ctx->collect_out_a.reserve(o_rows * audio_cols * esz)) != NSF_OK) return st;
  if ((st = ctx->collect_out_f.reserve(o_rows * facial_cols * esz)) != NSF_OK) return st;
  const char* ah = static_cast<const char*>(audio_host) + a_off[0] * audio_cols * esz;
  const char* fh = static_cast<const char*>(facial_host) + f_off[0] * facial_cols * esz;
  NSF_CUDA(cudaMemcpyAsync(ctx->collect_in_a.ptr, ah, a_rows * audio_cols * esz, cudaMemcpyHostToDevice, sl->stream));
  NSF_CUDA(cudaMemcpyAsync(ctx->collect_in_f.ptr, fh, f_rows * facial_cols * esz, cudaMemcpyHostToDevice, sl->stream));
  std::vector<int64_t> a_rel(n_clips + 1), f_rel(n_clips + 1);
  for (int i = 0; i <= n_clips; ++i) { a_rel[i] = a_off[i] - a_off[0]; f_rel[i] = f_off[i] - f_off[0]; }
  st = nsf_collect_batch(ctx, sl->stream, dtype, ctx->collect_in_a.ptr, audio_cols, a_rel.data(),
                         ctx->collect_in_f.ptr, facial_cols, f_rel.data(), n_clips, collect_flags,
                         blend_frames, ctx->collect_out_a.ptr, ctx->collect_out_f.ptr, nullptr);
  if (st != NSF_OK) return st;
  NSF_CUDA(cudaMemcpyAsync(out_audio_host, ctx->collect_out_a.ptr, o_rows * audio_cols * esz, cudaMemcpyDeviceToHost, sl->stream));
  NSF_CUDA(cudaMemcpyAsync(out_facial_host, ctx->collect_out_f.ptr, o_rows * facial_cols * esz, cudaMemcpyDeviceToHost, sl->stream));
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  return NSF_OK;
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
  if (pcm_format != NSF_PCM_F32 && pcm_format != NSF_PCM_I16) { set_error("unknown pcm_format"); return NSF_ERR_BAD_ARG; }
  const Plan& p = ctx->plan->p;
  const int cols = nsf_feature_cols(ctx->plan, flags);
  HostDesc& all = ctx->hd_all;
  nsf_status st = build_desc(p, clip_offsets, n_clips, flags, nullptr, &all);
  if (st != NSF_OK) return st;
  // output packing over the whole batch (validates the facial offsets)
  std::vector<int64_t> a_rows(n_clips + 1), o_all;
  for (int i = 0; i <= n_clips; ++i) a_rows[i] = all.row_off[i];
  if ((st = collect_offsets(a_rows.data(), f_off, n_clips, collect_flags, blend_frames, nullptr, &o_all)) != NSF_OK) return st;
  NSF_CUDA(cudaSetDevice(ctx->device));
  for (auto& sl : ctx->slot) sl.n_pending = 0;
  const size_t esz = pcm_format == NSF_PCM_I16 ? 2 : 4;
  // pageable caller buffers are staged through the slot's pinned arenas (see nsf_extract_host)
  const bool pcm_dma = dma_reachable(pcm_host), fac_dma = dma_reachable(facial_host);
  const bool oa_dma = dma_reachable(out_audio_host), of_dma = dma_reachable(out_facial_host);
  const bool ft_dma = features_host ? dma_reachable(features_host) : true;
  int first = 0, turn = 0;
  while (first < n_clips) {
    int last = first;
    int64_t samples = 0;
    while (last < n_clips && (last == first || samples + (clip_offsets[last + 1] - clip_offsets[last]) <= group_budget(turn))) {
      samples += clip_offsets[last + 1] - clip_offsets[last];
      ++last;
    }
    const int gn = last - first;
    Slot* sl = &ctx->slot[turn % kSlots];
    if ((st = ensure_slot(sl)) != NSF_OK) return st;
    if ((st = drain_slot(sl)) != NSF_OK) return st;   // the slot's previous group has fully drained
    const int64_t rows = all.row_off[last] - all.row_off[first];
    const int64_t frows = f_off[last] - f_off[first];
    const int64_t orows = o_all[last] - o_all[first];
    const int64_t wbytes = nsf_workspace_bytes(ctx->plan, samples, gn, flags);
    const size_t n1 = static_cast<size_t>(gn) + 1;
    if ((st = sl->pcm.reserve(samples * esz)) != NSF_OK) return st;
    if ((st = sl->out.reserve(static_cast<size_t>(rows) * cols * sizeof(float))) != NSF_OK) return st;
    if ((st = sl->work.reserve(wbytes)) != NSF_OK) return st;
    if ((st = sl->fac_in.reserve(static_cast<size_t>(frows) * facial_cols * sizeof(float))) != NSF_OK) return st;
    if ((st = sl->col_a.reserve(static_cast<size_t>(orows) * cols * sizeof(float))) != NSF_OK) return st;
    if ((st = sl->col_f.reserve(static_cast<size_t>(orows) * facial_cols * sizeof(float))) != NSF_OK) return st;
    if ((st = sl->col_desc.reserve(3 * n1 * sizeof(int64_t))) != NSF_OK) return st;
    const char* src = static_cast<const char*>(pcm_host) + clip_offsets[first] * esz;
    if (!pcm_dma) {
      if ((st = sl->stage_in.reserve(samples * esz)) != NSF_OK) return st;
      host_copy(sl->stage_in.ptr, src, samples * esz);
      src = static_cast<const char*>(sl->stage_in.ptr);
    }
    NSF_CUDA(cudaMemcpyAsync(sl->pcm.ptr, src, samples * esz, cudaMemcpyHostToDevice, sl->stream));
    const size_t fac_bytes = static_cast<size_t>(frows) * facial_cols * sizeof(float);
    const float* fsrc = facial_host + f_off[first] * facial_cols;
    if (!fac_dma) {
      if ((st = sl->stage_fac.reserve(fac_bytes)) != NSF_OK) return st;
      host_copy(sl->stage_fac.ptr, fsrc, fac_bytes);
      fsrc = static_cast<const float*>(sl->stage_fac.ptr);
    }
    NSF_CUDA(cudaMemcpyAsync(sl->fac_in.ptr, fsrc, fac_bytes, cudaMemcpyHostToDevice, sl->stream));
    // collect descriptors of this group (relative offsets) through the guarded pinned staging buffer.  Staged
    // BEFORE the extraction kernels are enqueued: the next wait on the staging buffer then ends as soon as this
    // group's uploads have run, so the host can start the next group's upload while these kernels execute
    DescEntry* de = nullptr;
    if ((st = desc_acquire(ctx, 3 * n1 * sizeof(int64_t), &de)) != NSF_OK) return st;
    int64_t* h = static_cast<int64_t*>(de->mem.ptr);
    for (size_t i = 0; i < n1; ++i) {
      h[i] = all.row_off[first + i] - all.row_off[first];
      h[n1 + i] = f_off[first + i] - f_off[first];
      h[2 * n1 + i] = o_all[first + i] - o_all[first];
    }
    int64_t* d = static_cast<int64_t*>(sl->col_desc.ptr);
    NSF_CUDA(cudaMemcpyAsync(d, h, 3 * n1 * sizeof(int64_t), cudaMemcpyHostToDevice, sl->stream));
    if ((st = desc_commit(de, sl->stream)) != NSF_OK) return st;
    ctx->pipelined = true;
    st = nsf_extract_batch(ctx, sl->stream, sl->pcm.ptr, pcm_format, clip_offsets + first, gn, flags,
                           static_cast<float*>(sl->out.ptr), cols, nullptr, nullptr, sl->work.ptr,
                           static_cast<int64_t>(sl->work.bytes));
    ctx->pipelined = false;
    if (st != NSF_OK) return st;
    CollectView v;
    v.a_off = d; v.f_off = d + n1; v.o_off = d + 2 * n1;
    v.n_clips = gn; v.total_out_rows = orows; v.flags = collect_flags; v.blend_frames = blend_frames;
    const int n = launch_collect(sl->stream, NSF_F32, v, sl->out.ptr, cols, sl->fac_in.ptr, facial_cols, sl->col_a.ptr,
                                 sl->col_f.ptr);
    if (n < 0) { set_error(cuda_msg("launch_collect", cudaGetLastError())); return NSF_ERR_CUDA; }
    ctx->launches += n;
    // downloads: straight into page-locked caller memory, else through a pinned stage + host copy at drain time
    auto download = [&](void* dst, const void* dev, size_t bytes, bool dma, PinnedArena* stage) -> nsf_status {
      if (dma) { NSF_CUDA(cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, sl->stream)); return NSF_OK; }
      const nsf_status r = stage->reserve(bytes);
      if (r != NSF_OK) return r;
      NSF_CUDA(cudaMemcpyAsync(stage->ptr, dev, bytes, cudaMemcpyDeviceToHost, sl->stream));
      sl->pending[sl->n_pending++] = Slot::CopyOut{dst, stage->ptr, bytes, 0, 0, 0, 1};
      return NSF_OK;
    };
    if (features_host &&   // the un-augmented rows as well (what collect_features caches as audio_features.csv)
        (st = download(features_host + all.row_off[first] * cols, sl->out.ptr,
                       static_cast<size_t>(rows) * cols * sizeof(float), ft_dma, &sl->stage_feat)) != NSF_OK) return st;
    if ((st = download(out_audio_host + o_all[first] * cols, sl->col_a.ptr,
                       static_cast<size_t>(orows) * cols * sizeof(float), oa_dma, &sl->stage_out)) != NSF_OK) return st;
    if ((st = download(out_facial_host + o_all[first] * facial_cols, sl->col_f.ptr,
                       static_cast<size_t>(orows) * facial_cols * sizeof(float), of_dma, &sl->stage_aux)) != NSF_OK) return st;
    first = last;
    ++turn;
  }
  for (auto& sl : ctx->slot)
    if (sl.stream && (st = drain_slot(&sl)) != NSF_OK) return st;
  return NSF_OK;
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
  const int n = launch_chunk_gather(static_cast<cudaStream_t>(cuda_stream), rows_dev, n_rows, cols, ld, frame, overlap, n_chunks, chunks_dev);
  if (n < 0) { set_error(cuda_msg("launch_chunk_gather", cudaGetLastError())); return NSF_ERR_CUDA; }
  ctx->launches += n;
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
  const int n = launch_chunk_blend(static_cast<cudaStream_t>(cuda_stream), decoded_dev, n_rows, out_cols, frame, overlap, n_chunks,
                                   scale_cols, divisor, out_dev);
  if (n < 0) { set_error(cuda_msg("launch_chunk_blend", cudaGetLastError())); return NSF_ERR_CUDA; }
  ctx->launches += n;
  return NSF_OK;
}

// ---- training windows --------------------------------------------------------------------------------------
nsf_status nsf_window_offsets(const int64_t* a_off, const int64_t* f_off, int32_t n_clips, int32_t window,
                              int64_t* w_off) {
  if (!a_off || !f_off || !w_off || n_clips < 1) { set_error("nsf_window_offsets: NULL argument or n_clips < 1"); return NSF_ERR_BAD_ARG; }
  if (window < 1) { set_error("nsf_window_offsets: window must be >= 1"); return NSF_ERR_BAD_ARG; }
  if (a_off[0] < 0 || f_off[0] < 0) { set_error("nsf_window_offsets: negative offset"); return NSF_ERR_BAD_ARG; }
  w_off[0] = 0;
  char buf[200];
  for (int i = 0; i < n_clips; ++i) {
    const int64_t na = a_off[i + 1] - a_off[i], nf = f_off[i + 1] - f_off[i];
    if (na < 0 || nf < 0) { set_error("nsf_window_offsets: offsets must be non-decreasing"); return NSF_ERR_BAD_ARG; }
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
  if ((st = desc_acquire(ctx, bytes, &de)) != NSF_OK) return st;
  if ((st = de->dev.reserve(bytes)) != NSF_OK) return st;
  int64_t* h = static_cast<int64_t*>(de->mem.ptr);
  std::memcpy(h, a_off, n1 * sizeof(int64_t));
  std::memcpy(h + n1, f_off, n1 * sizeof(int64_t));
  std::memcpy(h + 2 * n1, w_off.data(), n1 * sizeof(int64_t));
  std::memcpy(h + 3 * n1, indices, static_cast<size_t>(n) * sizeof(int64_t));
  int64_t* d = static_cast<int64_t*>(de->dev.ptr);
  NSF_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s));
  WindowView v;
  v.a_off = d; v.f_off = d + n1; v.w_off = d + 2 * n1; v.index = d + 3 * n1;
  v.n_clips = n_clips; v.window = window; v.n = n;
  const int m = launch_window_gather(s, v, audio_dev, audio_cols, facial_dev, facial_cols, out_audio_dev, out_facial_dev);
  if (m < 0) { set_error(cuda_msg("launch_window_gather", cudaGetLastError())); return NSF_ERR_CUDA; }
  ctx->launches += m;
  return desc_commit(de, s);
}

nsf_status nsf_rows_host(nsf_ctx* ctx, int32_t op, int32_t dtype, const void* a_host, int64_t na,
                         const void* b_host, int64_t nb, int32_t cols, int32_t blend_frames, void* out_host) {
  if (!ctx || !a_host || !out_host || na <= 0 || cols <= 0) { set_error("nsf_rows_host: bad argument"); return NSF_ERR_BAD_ARG; }
  if (dtype != NSF_F32 && dtype != NSF_F64) { set_error("nsf_rows_host: bad dtype"); return NSF_ERR_BAD_ARG; }
  int64_t out_rows = 0, k = 0;
  if (op == NSF_ROWS_INTERP_SLOWER) out_rows = 2 * na - 1;
  else if (op == NSF_ROWS_SMOOTH) out_rows = na;
  else if (op == NSF_ROWS_BLEND_STACK) {
    if (!b_host || nb <= 0) { set_error("nsf_rows_host: blend needs a second array"); return NSF_ERR_BAD_ARG; }
    k = std::max<int64_t>(0, std::min<int64_t>(std::min<int64_t>(blend_frames, na), nb));
    out_rows = na + nb - k;
  } else { set_error("nsf_rows_host: unknown op"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  Slot* sl = &ctx->slot[0];
  nsf_status st = ensure_slot(sl);
  if (st != NSF_OK) return st;
  const size_t esz = dtype == NSF_F64 ? 8 : 4;
  const bool two = op == NSF_ROWS_BLEND_STACK;
  if ((st = ctx->collect_in_a.reserve(na * cols * esz)) != NSF_OK) return st;
  if (two && (st = ctx->collect_in_f.reserve(nb * cols * esz)) != NSF_OK) return st;
  if ((st = ctx->collect_out_a.reserve(out_rows * cols * esz)) != NSF_OK) return st;
  NSF_CUDA(cudaMemcpyAsync(ctx->collect_in_a.ptr, a_host, na * cols * esz, cudaMemcpyHostToDevice, sl->stream));
  if (two) NSF_CUDA(cudaMemcpyAsync(ctx->collect_in_f.ptr, b_host, nb * cols * esz, cudaMemcpyHostToDevice, sl->stream));
  const int n = launch_rows_op(sl->stream, op, dtype, ctx->collect_in_a.ptr, na, two ? ctx->collect_in_f.ptr : nullptr,
                               nb, cols, k, ctx->collect_out_a.ptr, out_rows);
  if (n < 0) { set_error(cuda_msg("launch_rows_op", cudaGetLastError())); return NSF_ERR_CUDA; }
  ctx->launches += n;
  NSF_CUDA(cudaMemcpyAsync(out_host, ctx->collect_out_a.ptr, out_rows * cols * esz, cudaMemcpyDeviceToHost, sl->stream));
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  return NSF_OK;
}

nsf_status nsf_post_host(nsf_ctx* ctx, const float* in_host, int64_t T, int32_t Cc, uint32_t pf, float* out_host) {
  if (!ctx || !in_host || !out_host || T <= 0 || Cc <= 0) { set_error("nsf_post_host: bad argument"); return NSF_ERR_BAD_ARG; }
  if ((pf & NSF_POST_DELTAS) && T < 9) { set_error("nsf_post_host: delta needs at least 9 frames"); return NSF_ERR_TOO_SHORT; }
  if ((pf & NSF_POST_EDGEFIX) && T < 2) { set_error("nsf_post_host: edge fix needs 2 frames"); return NSF_ERR_BAD_ARG; }
  NSF_CUDA(cudaSetDevice(ctx->device));
  Slot* sl = &ctx->slot[0];
  nsf_status st = ensure_slot(sl);
  if (st != NSF_OK) return st;
  const bool reduce = (pf & NSF_POST_REDUCE) != 0, deltas = (pf & NSF_POST_DELTAS) != 0, cmvn = (pf & NSF_POST_CMVN) != 0;
  const int64_t rows = reduce ? (T + 1) / 2 : T;
  const int out_c = Cc * (deltas ? 3 : 1);
  // device layout: [in T*C floats][out rows*out_c floats][desc 6 x int64][sum C][sumsq C]
  const size_t in_b = align_up(T * Cc * sizeof(float)), out_b = align_up(rows * out_c * sizeof(float));
  const size_t desc_b = align_up(6 * sizeof(int64_t)), st_b = align_up(Cc * sizeof(double));
  if ((st = ctx->collect_in_a.reserve(in_b + out_b + desc_b + 2 * st_b)) != NSF_OK) return st;
  char* base = static_cast<char*>(ctx->collect_in_a.ptr);
  float* d_in = reinterpret_cast<float*>(base);
  float* d_out = reinterpret_cast<float*>(base + in_b);
  int64_t* d_desc = reinterpret_cast<int64_t*>(base + in_b + out_b);
  double* d_sum = reinterpret_cast<double*>(base + in_b + out_b + desc_b);
  double* d_sq = reinterpret_cast<double*>(base + in_b + out_b + desc_b + st_b);
  DescEntry* de = nullptr;
  if ((st = desc_acquire(ctx, 6 * sizeof(int64_t), &de)) != NSF_OK) return st;
  int64_t* h = static_cast<int64_t*>(de->mem.ptr);
  h[0] = 0; h[1] = 0;           // clip_off (unused by the post kernels)
  h[2] = 0; h[3] = T;           // frame_off
  h[4] = 0; h[5] = rows;        // row_off
  NSF_CUDA(cudaMemcpyAsync(d_desc, h, 6 * sizeof(int64_t), cudaMemcpyHostToDevice, sl->stream));
  if ((st = desc_commit(de, sl->stream)) != NSF_OK) return st;
  NSF_CUDA(cudaMemcpyAsync(d_in, in_host, T * Cc * sizeof(float), cudaMemcpyHostToDevice, sl->stream));
  int launched = 0, n;
  if (pf & NSF_POST_EDGEFIX) {
    if ((n = launch_edge_fix(sl->stream, d_in, T, Cc, ctx->edge_zero_threshold)) < 0) { set_error(cuda_msg("launch_edge_fix", cudaGetLastError())); return NSF_ERR_CUDA; }
    launched += n;
  }
  if (cmvn) {
    if ((n = launch_col_stats(sl->stream, d_in, T, Cc, d_sum, d_sq)) < 0) { set_error(cuda_msg("launch_col_stats", cudaGetLastError())); return NSF_ERR_CUDA; }
    launched += n;
  }
  BatchView b;
  b.clip_off = d_desc; b.frame_off = d_desc + 2; b.row_off = d_desc + 4;
  b.n_clips = 1; b.total_samples = 0; b.total_frames = T; b.total_rows = rows;
  if ((n = launch_delta_reduce(sl->stream, b, d_in, Cc, Cc, d_sum, d_sq, cmvn, deltas, reduce, d_out, out_c, 0)) < 0) {
    set_error(cuda_msg("launch_delta_reduce", cudaGetLastError())); return NSF_ERR_CUDA;
  }
  launched += n;
  ctx->launches += launched;
  NSF_CUDA(cudaMemcpyAsync(out_host, d_out, rows * out_c * sizeof(float), cudaMemcpyDeviceToHost, sl->stream));
  NSF_CUDA(cudaStreamSynchronize(sl->stream));
  return NSF_OK;
}

}  // extern "C"

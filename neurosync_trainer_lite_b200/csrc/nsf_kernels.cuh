// Device-side views and kernel launchers (sm_100a).  See DESIGN.md for the per-kernel rooflines.
#ifndef NSF_KERNELS_CUH_
#define NSF_KERNELS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

// Launchers return the number of kernels they launched, or -1 when a launch failed.
#define NSF_CHECK_LAUNCH() \
  do { if (cudaGetLastError() != cudaSuccess) return -1; } while (0)

namespace nsf {

// SMs of the one target, the B200 (sm_100a): grids sized in waves of resident blocks are multiples of it.
constexpr int kSmCount = 148;

// Segment descriptors of one batch of clips, all in device memory.
struct BatchView {
  const int64_t* clip_off;   // [n+1] first sample of each clip in the packed signal
  const int64_t* frame_off;  // [n+1] first hop-frame of each clip
  const int64_t* row_off;    // [n+1] first output row of each clip
  int32_t n_clips;
  int64_t total_samples;
  int64_t total_frames;
  int64_t total_rows;
};

// Constant tables of a plan, uploaded once per context.
struct DeviceTables {
  int F, H, pad, bins, bins_ld, n_mfcc, n_mels, n_lags, chains;
  float edge_thr;             // zero_threshold of fix_edge_frames_autocorr (1e-7 unless nsf_ctx_set_option changed it)
  int kp[2], np[2], nbins[2];
  int col_off[2];             // power rows are chain-major: column = col_off[chain] + m
  const int32_t* tap_idx[2];  // [part][tap][kp]
  const float* tap_coef[2];
  const float* mat32[2][2];   // [chain][part] row-major [kp][np] float32 (validation GEMM)
  const float* hann_sym;      // [F] np.hanning (autocorr branch)
  const float* hann_per;      // [F] periodic Hann (STFT branch)
  // sparse mel basis re-indexed to the chain-major power layout: per (chain, mel) one run of
  // consecutive power columns; arrays are [chains][n_mels]
  const int32_t* mel_start;   // first power column of the run
  const int32_t* mel_len;
  const int32_t* mel_ptr;     // offset of the run's weights in mel_w
  const float* mel_w;
  const float* dct_t;         // [n_mels][32] transposed, zero padded
  const uint2* dct_frag;      // DCT matrix x 2^10 as fp16 hi / lo MMA B fragments (k_dct_mma; default shape only, else NULL)
  // per power column of chain c (padded to whole 128-column tiles): {bits(m0), w[m0], w[m0+1], 0}.
  // A bin lies under at most two (adjacent) triangular mel filters; mel_col_ok == 0 if that ever fails.
  const float4* mel_col[2];
  int mel_col_ok;
};

struct ExtractBuffers {
  const float* y;          // packed (normalised) float32 signal
  float* a32;              // [chains*2][total_frames][kp] folded inputs (validation GEMM)
  float* power;            // [total_frames][bins_ld]
  float* db;               // [total_frames][n_mels]
  float* mfcc_raw;         // [total_frames][n_mfcc]
  uint32_t* peak_bits;     // [n] max|y| as float bits
  uint32_t* dbmax_key;     // [n] order-preserving key of the per-clip dB maximum
  double* sum;             // [n][n_mfcc]
  double* sumsq;           // [n][n_mfcc] sum of squares
  float* ac_raw;           // [total_frames][n_lags] (only with autocorr deltas)
};

// max_blocks: 0 = as many blocks as there are 16 K-sample chunks; > 0 caps the grid (pipelined host paths, see
// nsf_kernels.cu: an HBM-saturating kernel stalls the copy engine's upload of the next clip group)
int launch_absmax(cudaStream_t s, const void* pcm, int pcm_format, const BatchView& b,
                  uint32_t* peak_bits, int max_blocks = 0);
int launch_normalize(cudaStream_t s, const void* pcm, int pcm_format, const BatchView& b,
                     const uint32_t* peak_bits, bool use_peak, float* y_out, int max_blocks = 0);
int launch_fold32(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* y,
                  float* a32);
int launch_dft_simt(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* a32,
                    float* power);
int launch_mel_db(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* power,
                  float* db, uint32_t* dbmax_key);
// Shape of the tensor-pipe DCT kernel k_dct_mma: the reference's default 128 mels -> 23 MFCCs.  Other shapes run the
// shared-memory coefficient kernels.
constexpr int kDctMmaMels = 128, kDctMmaMfcc = 23;
int launch_dct_sum(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* db,
                   const uint32_t* dbmax_key, float* mfcc_raw, double* sum, double* sumsq);
// generic normalise + delta + pair-reduce over a [frames][C] matrix
int launch_delta_reduce(cudaStream_t s, const BatchView& b, const float* in, int C, int in_ld,
                        const double* sum, const double* sumsq, bool cmvn, bool deltas, bool reduce,
                        float* out, int64_t out_ld, int col0);
int launch_autocorr(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* y,
                    bool reduce, float* out, int64_t out_ld, int col0);
// tensor-pipe variant (mma.sync m16n8k16, Hankel fragments): the product path; launch_autocorr is
// the fp32-FMA validation variant (NSF_DEBUG_FMA_AUTOCORR)
int launch_autocorr_mma(cudaStream_t s, const DeviceTables& t, const BatchView& b, const float* y,
                        bool reduce, float* out, int64_t out_ld, int col0);
int launch_smooth(cudaStream_t s, const BatchView& b, const float* in, int64_t in_ld, int cols,
                  float* out, int64_t out_ld);

// collect_features augmentation (float or double rows)
struct CollectView {
  const int64_t* a_off;    // [n+1] audio rows in
  const int64_t* f_off;    // [n+1] facial rows in
  const int64_t* o_off;    // [n+1] rows out
  int32_t n_clips;
  int64_t total_out_rows;
  uint32_t flags;
  int32_t blend_frames;
};
int launch_collect(cudaStream_t s, int dtype, const CollectView& v, const void* audio, int a_cols,
                   const void* facial, int f_cols, void* out_audio, void* out_facial);

// stand-alone row helpers (interpolate_slower / smooth / one stack_with_blend step)
int launch_rows_op(cudaStream_t s, int op, int dtype, const void* a, int64_t na, const void* b,
                   int64_t nb, int cols, int64_t k_blend, void* out, int64_t out_rows);
// WAV conversion (nsf_convert.cu): one descriptor per clip.  `taps` is the clip's polyphase filter in k-major
// float64 layout [kmax][up] (zero beyond the last tap of a phase); decode-only clips leave the resampling fields 0.
struct ConvClip {
  int64_t byte_off;   // clip's first byte in the payload
  int64_t frames;     // input frames
  int64_t out_off;    // first output sample
  int64_t n_out;      // output samples
  int64_t tile0;      // first block of the clip in its launch
  const double* taps;
  int32_t enc, channels, bps;
  int32_t up, down, n_pre_pad, n_pre_remove, kmax;
  int32_t slots, reps;   // resampling tile: `slots` (a multiple of up) x `reps` outputs per block
};
constexpr int kConvDecodeTile = 4096;          // frames per block of k_convert_decode
constexpr int kConvMaxReps = 8;                // outputs per thread slot of k_convert_resample
constexpr size_t kConvMaxSmem = 96 * 1024;     // input window of one k_convert_resample block (float64)
// resample = false: k_convert_decode, else k_convert_resample with `smem_bytes` of dynamic shared memory
int launch_convert(cudaStream_t s, bool resample, const ConvClip* clips_dev, int n_clips, int64_t tiles,
                   size_t smem_bytes, const void* payload, float* out);
// generic per-channel statistics of one [T][C] matrix and the edge fix
int launch_col_stats(cudaStream_t s, const float* in, int64_t T, int C, double* sum, double* sumsq);
int launch_edge_fix(cudaStream_t s, float* data, int64_t T, int C, float zero_threshold);

// inference-side chunker: chunks [n_chunks][frame][cols] out of feature rows (reflect-completed tail), and the
// cross-faded reassembly of the decoded chunks [n_chunks][frame][cols] into [n_rows][cols]
int launch_chunk_gather(cudaStream_t s, const float* rows, int64_t n_rows, int cols, int64_t ld, int frame, int overlap,
                        int64_t n_chunks, float* out);
int launch_chunk_blend(cudaStream_t s, const float* decoded, int64_t n_rows, int cols, int frame, int overlap,
                       int64_t n_chunks, int scale_cols, float divisor, float* out);

// training windows of a packed dataset (nsf_window_gather): every array in device memory, geometry validated on the
// host.  One block per kWindowTileRows output rows of a window.
struct WindowView {
  const int64_t* a_off;    // [n_clips+1] audio rows of each clip
  const int64_t* f_off;    // [n_clips+1] facial rows of each clip
  const int64_t* w_off;    // [n_clips+1] first window of each clip (nsf_window_offsets)
  const int64_t* index;    // [n] windows to gather
  int32_t n_clips, window;
  int64_t n;
};
constexpr int kWindowTileRows = 32;
int launch_window_gather(cudaStream_t s, const WindowView& v, const float* audio, int a_cols, const float* facial,
                         int f_cols, float* out_a, float* out_f);

// audio_features.csv text (nsf_csv.cu): row_len[r] = bytes of row r (k_csv_lengths, one block per row); then every
// row at text + start[r] and the header of file f at text + start[n_rows + f] (k_csv_write).
int64_t csv_header_bytes(int cols);
int launch_csv_lengths(cudaStream_t s, int dtype, const void* rows, int64_t n_rows, int cols, int64_t* row_len);
int launch_csv_write(cudaStream_t s, int dtype, const void* rows, int64_t n_rows, int cols, int32_t n_files,
                     const int64_t* start, char* text);

// CSV text -> rows (nsf_csv_parse.cu).  File i is text[text_off[i], text_off[i+1]) (header line included); its
// tiles [tile_off[i], tile_off[i+1]) are the kCsvTile-aligned blocks of the text clipped to the file (csv_tiles).
// Data row r (rows of file i: [row_off[i], row_off[i+1]), row_off[0] = 0) goes to out + r * out_ld, column c of the
// file to output column out_col[c] (-1: dropped).
constexpr int64_t kCsvTile = 16384;
struct CsvView {
  const char* text;
  const int64_t* text_off;   // [n_files + 1]
  const int64_t* tile_off;   // [n_files + 1]
  const int64_t* row_off;    // [n_files + 1], parse only
  const int32_t* out_col;    // [cols], parse only
  int32_t n_files, cols;
  int64_t n_tiles, n_rows;
};
int64_t csv_tiles(int64_t begin, int64_t end);
// tile_rows [n_tiles] int32, tile_start [n_tiles + 1]: workspace; row_off [n_files + 1] <- data rows before file i.
int launch_csv_row_offsets(cudaStream_t s, const CsvView& v, int32_t* tile_rows, int64_t* tile_start, int64_t* row_off);
// + row_start [n_rows], col_flags [n_files x cols] (zeroed by the caller), status [n_files] (zeroed by the caller).
int launch_csv_parse(cudaStream_t s, const CsvView& v, int dtype, int32_t* tile_rows, int64_t* tile_start,
                     int64_t* row_start, uint32_t* col_flags, void* out, int64_t out_ld, uint32_t* status);

// FLAC frames (nsf_flac.cu).  Byte positions are relative to the group's payload; a stream's scan positions are
// [scan0, scan0 + end - begin) of the group's scan space (the streams' frame bytes one after the other, so that
// streams sharing payload bytes are each scanned).
struct FlacStream {
  int64_t begin, end;   // frame bytes of the stream
  int64_t scan0;        // first scan position
  int64_t out0;         // first output byte
  int32_t channels, bits, sample_rate, max_block;
};
struct FlacCand {       // a sync candidate: header fields and the result of decoding the frame that starts there
  int64_t start, end;   // frame bytes [start, end)
  int64_t number;       // coded number
  int32_t stream, block, status, assignment;   // status NSF_FLAC_*; assignment | variable << 4
  uint32_t sub_bit[8];  // first bit of each subframe, from `start`
};
struct FlacKept {       // a frame on a stream's frame chain
  int32_t cand, stream;
  int64_t g0;           // first output frame of the frame in the group (sorted)
  int64_t first;        // first sample of the frame in its stream
  int64_t scratch0;     // its samples in the int32 scratch: channel c at scratch0 + c * block
};
constexpr int kFlacScanTile = 4096;   // scan positions per block of the sync scan
// k_flac_count + k_flac_scan + k_flac_write + k_flac_parse: candidates in scan order; cand_total <- their count,
// of which the first min(count, cap) are parsed into cand.  blk_count / blk_off: one entry per scan tile.
int launch_flac_scan_parse(cudaStream_t s, const FlacStream* streams, int n_streams, int64_t scan_total,
                           const uint8_t* payload, int32_t* blk_count, int64_t* blk_off, int64_t* cand_total,
                           int64_t* cand_pos, FlacCand* cand, int64_t cap);
// k_flac_decode (one thread per kept frame and channel) + k_flac_interleave (one thread per output frame)
int launch_flac_decode(cudaStream_t s, const FlacStream* streams, const FlacCand* cand, const FlacKept* kept,
                       int n_kept, int max_channels, int64_t out_frames, const uint8_t* payload, int32_t* scratch,
                       uint8_t* out);
// The header at payload[pos] of a stream ending at `end`: NSF_FLAC_OK or why no frame starts there (no sync,
// truncated, bad number, CRC-8).  Host-side diagnosis of a broken frame chain.
int flac_header_status(const uint8_t* payload, int64_t pos, int64_t end);
const char* flac_status_text(int status);

// One-time (per device) cudaFuncSetAttribute calls of each translation unit; nsf_ctx_create runs them so that no
// launch path touches function attributes.
bool init_kernel_attributes();        // nsf_kernels.cu
bool init_autocorr_mma_attributes();  // nsf_autocorr_mma.cu
bool init_stft_tc_attributes();       // nsf_stft_tc.cu
bool init_convert_attributes();       // nsf_convert.cu

}  // namespace nsf
#endif  // NSF_KERNELS_CUH_

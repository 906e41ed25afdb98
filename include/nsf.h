/*
 * nsf.h -- C ABI of the B200-native NeuroSync audio feature front-end ("nsf").
 *
 * The reference (wolfi/NeuroSync_Trainer_Lite) has no FFI layer: its boundary for this path is the
 * Python call surface.  Each entry point below names the reference function(s) it replaces
 * (paths relative to the reference root).  INTEGRATION.md shows the ctypes binding a maintainer
 * would add to the reference's own modules.
 *
 * Conventions
 *   - plain C types only; every buffer is caller-owned unless stated otherwise;
 *   - "dev" pointers are CUDA device pointers on the context's device, "host" pointers are CPU
 *     memory (pinned memory makes the *_host calls faster but is not required);
 *   - device-level calls (nsf_extract_batch, nsf_collect_batch) are stream-ordered and do not wait for
 *     the device: their descriptor arrays travel through a ring of 8 pinned staging buffers, so the
 *     host blocks only if the descriptor uploads of the 8 previous calls have not run yet;
 *   - every call returns an nsf_status; nsf_last_error() gives a thread-local message;
 *   - one nsf_ctx per device and per host thread; plans are immutable and may be shared.
 *   - there is NO CPU fallback: compute calls fail with NSF_ERR_NO_DEVICE / NSF_ERR_CUDA when no
 *     sm_100 device is usable.  Only the integer helpers and plan/table queries run without a GPU.
 */
#ifndef NSF_H_
#define NSF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NSF_ABI_VERSION 2

#if defined(__GNUC__)
#define NSF_API __attribute__((visibility("default")))
#else
#define NSF_API
#endif

typedef enum nsf_status {
  NSF_OK = 0,
  NSF_ERR_BAD_ARG = 1,    /* null pointer, negative size, inconsistent offsets ...            */
  NSF_ERR_TOO_SHORT = 2,  /* a clip has fewer hop-frames than delta(width=9) / the edge fix need */
  NSF_ERR_CUDA = 3,       /* a CUDA runtime/driver call failed (see nsf_last_error)            */
  NSF_ERR_WORKSPACE = 4,  /* caller workspace smaller than nsf_workspace_bytes()               */
  NSF_ERR_NO_DEVICE = 5,  /* no CUDA device / not an sm_100 part                               */
  NSF_ERR_UNSUPPORTED = 6 /* parameter combination outside what the kernels implement          */
} nsf_status;

/* PCM sample formats accepted by the extract calls. */
#define NSF_PCM_F32 0 /* float32 samples (what librosa.load returns)                            */
#define NSF_PCM_I16 1 /* int16 PCM as stored in WAV; decoded as v / 32768 (soundfile semantics)  */

/* Behaviour flags (bit-or).  Defaults (flags == 0) reproduce
 * extract_and_combine_features(y, sr, F, H) of utils/audio/extraction/extract_features.py:26-46. */
#define NSF_PEAK_NORMALIZE 0x001u /* y /= max|y| per clip first   (utils/audio/load_audio.py:12-14)  */
#define NSF_NO_AUTOCORR 0x002u    /* include_autocorr=False       (extract_features.py:26,35)        */
#define NSF_SMOOTH 0x004u         /* apply_smoothing=True         (extract_features_utils.py:47-51)  */
#define NSF_NO_CMVN 0x008u        /* include_cepstral=False       (extract_features_utils.py:21-22)  */
#define NSF_NO_DELTAS 0x010u      /* include_deltas=False (MFCC)  (extract_features_utils.py:24-30)  */
#define NSF_AC_DELTAS 0x020u      /* compute_autocorr_with_deltas (extract_features_utils.py:131-135)*/
#define NSF_NO_REDUCE 0x040u      /* skip reduce_features: one row per hop-frame (utils API parity)  */
#define NSF_NO_MFCC 0x080u        /* autocorrelation block only (extract_autocorrelation_features)   */
#define NSF_AC_NO_PAD 0x800u      /* pad_signal=False of extract_overlapping_autocorr (extract_features_utils.py:54-61):
                                     frame t = y[t H : t H + F], T = (L - F) // H + 1; needs NSF_NO_MFCC.
                                     Other padding_mode values / trim_padded are host-side index work around
                                     this flag (np.pad before the call, column selection after it). */
#define NSF_DEBUG_SIMT_DFT 0x100u /* validation aid: run the STFT GEMM on CUDA cores in fp32 instead
                                     of tcgen05 (never selected automatically)                      */

#define NSF_DEBUG_FMA_AUTOCORR 0x200u /* validation aid: autocorrelation with fp32 CUDA-core FMAs instead
                                         of the mma.sync Hankel kernel (never selected automatically) */

#define NSF_DEBUG_UNFUSED_MEL 0x400u   /* validation aid: separate tcgen05 GEMM (power to HBM) + mel/dB kernel
                                         instead of the fused persistent kernel */

/* collect flags */
#define NSF_COLLECT_FAST 0x1u  /* include_fast      (dataset/data_processing.py:152-158) */
#define NSF_COLLECT_SLOW 0x2u  /* include_slow      (dataset/data_processing.py:161-167) */
#define NSF_COLLECT_BLEND 0x4u /* blend_boundaries  (dataset/data_processing.py:170-175) */

/* element types of nsf_collect_batch */
#define NSF_F32 0
#define NSF_F64 1

typedef struct nsf_plan nsf_plan; /* host-side constant tables for one (sr, F, H, ...) */
typedef struct nsf_ctx nsf_ctx;   /* per-device state: uploaded tables, arenas, streams */

/* ---- library ---------------------------------------------------------------------------- */
NSF_API int32_t nsf_abi_version(void);
NSF_API const char* nsf_last_error(void);
/* Number of visible CUDA devices that are sm_100 (0 when there is no GPU; never fails). */
NSF_API int32_t nsf_device_count(void);

/* ---- integer frame arithmetic: bit-exact, host only -------------------------------------- */
/* frame_length = int(0.01667 * sr)                        extract_features.py:12 */
NSF_API int32_t nsf_frame_length(int32_t sr);
/* hop_length = frame_length // 2                          extract_features.py:13 */
NSF_API int32_t nsf_hop_length(int32_t frame_length);
/* num_frames = (len(y) - F) // H + 1 (floor division)     extract_features.py:16 */
NSF_API int64_t nsf_guard_frames(int64_t n_samples, int32_t frame_length, int32_t hop_length);
/* T: hop-frames both branches produce (pad F//2 each side) extract_features_utils.py:19,57-64 */
NSF_API int64_t nsf_hop_frames(int64_t n_samples, int32_t frame_length, int32_t hop_length);
/* R = ceil(T / 2): rows after reduce_features              extract_features_utils.py:33-44 */
NSF_API int64_t nsf_feature_rows(int64_t n_samples, int32_t frame_length, int32_t hop_length);
/* Prefix sum of the per-clip row counts of a packed batch: row_offsets[0] = 0, row_offsets[i + 1] =
 * row_offsets[i] + rows of clip i under `flags` (nsf_feature_rows; nsf_hop_frames with NSF_NO_REDUCE;
 * whole un-padded frames with NSF_AC_NO_PAD).  The packing nsf_extract_batch uses when its
 * out_row_offsets is NULL; one call for the batch instead of one nsf_feature_rows call per clip (a
 * binding's per-clip loop costs more than the kernels for batches of thousands of short clips).
 * row_offsets has n_clips + 1 entries.                      extract_features_utils.py:33-44 */
NSF_API nsf_status nsf_row_offsets(int32_t frame_length, int32_t hop_length, const int64_t* clip_offsets,
                                   int32_t n_clips, uint32_t flags, int64_t* row_offsets);
/* Output columns for a flag set (256 by default, 69 without autocorr, ...). */
NSF_API int32_t nsf_feature_cols(const nsf_plan* plan, uint32_t flags);
/* Rows collect_features yields for given stream lengths    data_processing.py:126-197 */
NSF_API int64_t nsf_collect_rows(int64_t n_audio_rows, int64_t n_facial_rows, uint32_t collect_flags,
                         int32_t blend_frames);

/* ---- plan: constant tables (window, folded DFT, mel, DCT), host only ---------------------- */
/* Replaces the implicit constants of librosa.feature.mfcc(n_mfcc=23, n_fft=F, hop_length=H) and
 * np.hanning(F) used at extract_features_utils.py:19,79.  Defaults of the reference:
 * n_mfcc=23, n_mels=128, n_lags=187. */
NSF_API nsf_status nsf_plan_create(int32_t sr, int32_t frame_length, int32_t hop_length, int32_t n_mfcc,
                           int32_t n_mels, int32_t n_lags, nsf_plan** out_plan);
NSF_API void nsf_plan_destroy(nsf_plan* plan);

/* Table export (tests pin these against the oracle without a GPU).  Returns the element count of
 * the table; copies min(count, capacity) floats into dst when dst != NULL. */
#define NSF_TABLE_MEL 0        /* [n_mels x bins] dense float32 mel basis                      */
#define NSF_TABLE_DCT 1        /* [n_mfcc x n_mels] DCT-II ortho                               */
#define NSF_TABLE_HANN_SYM 2   /* [F] np.hanning(F) (autocorr branch)                          */
#define NSF_TABLE_HANN_PER 3   /* [F] periodic Hann (STFT branch)                              */
NSF_API int64_t nsf_plan_table(const nsf_plan* plan, int32_t which, float* dst, int64_t capacity);
/* Plan geometry: bins, fold chains (1 or 2), folded K, padded K. */
NSF_API int32_t nsf_plan_info(const nsf_plan* plan, int32_t* bins, int32_t* chains, int32_t* fold_k,
                      int32_t* fold_k_padded);
/* Host emulation of the folded-DFT index/sign tables on ONE frame (F float32 samples in, `bins`
 * complex values out as re[bins], im[bins], computed in float64).  Exists so the fold tables can
 * be verified against an FFT without a GPU; it is not a compute path. */
NSF_API nsf_status nsf_plan_fold_check(const nsf_plan* plan, const float* frame, double* re, double* im);

/* ---- context ------------------------------------------------------------------------------ */
NSF_API nsf_status nsf_ctx_create(const nsf_plan* plan, int32_t device, nsf_ctx** out_ctx);
NSF_API void nsf_ctx_destroy(nsf_ctx* ctx);
/* Pinned host memory helpers for callers without their own allocator. */
NSF_API nsf_status nsf_host_alloc(void** out_ptr, int64_t bytes);
NSF_API void nsf_host_free(void* ptr);
/* Page-lock caller memory (cudaHostRegister, portable) so that the *_host calls can DMA into / out of it
 * directly - e.g. ONE host array shared by the ranks of a box (a /dev/shm mapping every process registers and
 * fills at its own row offsets: the "gathered to host" array of the multi-GPU dataset builders). */
NSF_API nsf_status nsf_host_register(void* ptr, int64_t bytes);
NSF_API nsf_status nsf_host_unregister(void* ptr);
/* Per-context options.  NSF_OPT_EDGE_ZERO_THRESHOLD: zero_threshold of fix_edge_frames_autocorr
 * (utils/audio/extraction/extract_features_utils.py:105; default 1e-7). */
#define NSF_OPT_EDGE_ZERO_THRESHOLD 0
NSF_API nsf_status nsf_ctx_set_option(nsf_ctx* ctx, int32_t option, double value);

/* ---- feature extraction --------------------------------------------------------------------
 * Replaces, for a BATCH of clips, extract_and_combine_features (extract_features.py:26-46) and,
 * with NSF_PEAK_NORMALIZE, the arithmetic half of extract_audio_features (extract_features.py:6-24
 * + load_audio.py:12-14).  Clip i owns samples [clip_offsets[i], clip_offsets[i+1]) of `pcm` and
 * rows [row_offsets[i], row_offsets[i+1]) of `out`, row_offsets being the prefix sum of
 * nsf_feature_rows() (or nsf_hop_frames() under NSF_NO_REDUCE); pass out_row_offsets = NULL to get
 * exactly that packing.  `out` is row-major float32 with `out_ld` floats between rows
 * (>= nsf_feature_cols()).  Every clip must have >= 9 hop-frames when deltas are computed (what
 * librosa.feature.delta requires; 2 otherwise) and more than F/2 samples (reflect padding), else
 * NSF_ERR_TOO_SHORT and nothing is launched.  The reference's 9-frame guard on UN-padded frames
 * (extract_features.py:16-20) is the caller's policy: test it with nsf_guard_frames(). */
NSF_API int64_t nsf_workspace_bytes(const nsf_plan* plan, int64_t total_samples, int32_t n_clips,
                            uint32_t flags);

NSF_API nsf_status nsf_extract_batch(nsf_ctx* ctx, void* cuda_stream, const void* pcm_dev,
                             int32_t pcm_format, const int64_t* clip_offsets_host, int32_t n_clips,
                             uint32_t flags, float* out_dev, int64_t out_ld,
                             const int64_t* out_row_offsets_host,
                             float* y_norm_dev, /* optional: normalised float32 signal out */
                             void* workspace_dev, int64_t workspace_bytes);

/* Same contract with HOST buffers: uploads, extracts and downloads using context-owned device
 * arenas and streams, overlapping H2D / kernels / D2H across clip groups.  Synchronous.  Pinned (or
 * registered) buffers are read and written by the copy engines directly; pageable buffers are staged
 * group by group through context-owned pinned arenas, so the pipeline stays asynchronous either way. */
NSF_API nsf_status nsf_extract_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                            const int64_t* clip_offsets_host, int32_t n_clips, uint32_t flags,
                            float* out_host, int64_t out_ld, float* y_norm_host /* optional */);

/* Peak normalisation alone, HOST buffers: y = decode(pcm) / max|decode(pcm)| per clip when the peak
 * is > 0 (utils/audio/load_audio.py:12-14, applied by all four loaders).  y_host is float32 with the
 * packing of clip_offsets_host (rebased to 0).  peaks_host (optional) receives max|y| per clip. */
NSF_API nsf_status nsf_normalize_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                              const int64_t* clip_offsets_host, int32_t n_clips, float* y_host,
                              float* peaks_host /* optional */);

/* ---- collect_features augmentation ----------------------------------------------------------
 * Replaces the arithmetic of collect_features (data_processing.py:126-177): centre-trim to equal
 * length, fast = rows[::2], slow = interpolate_slower (+ smooth_facial_data on the facial copy),
 * stack_with_blend / vstack.  For clip i the audio rows are [audio_offsets[i], audio_offsets[i+1])
 * of `audio` (row-major, audio_cols wide), facial rows likewise; outputs are packed at
 * out_offsets (prefix sum of nsf_collect_rows; NULL = that packing).  dtype NSF_F64 reproduces the
 * reference's float64 arithmetic bit-for-bit; NSF_F32 is the device-resident training format. */
NSF_API nsf_status nsf_collect_batch(nsf_ctx* ctx, void* cuda_stream, int32_t dtype, const void* audio_dev,
                             int32_t audio_cols, const int64_t* audio_offsets_host,
                             const void* facial_dev, int32_t facial_cols,
                             const int64_t* facial_offsets_host, int32_t n_clips,
                             uint32_t collect_flags, int32_t blend_frames, void* out_audio_dev,
                             void* out_facial_dev, const int64_t* out_offsets_host);

NSF_API nsf_status nsf_collect_host(nsf_ctx* ctx, int32_t dtype, const void* audio_host, int32_t audio_cols,
                            const int64_t* audio_offsets_host, const void* facial_host,
                            int32_t facial_cols, const int64_t* facial_offsets_host,
                            int32_t n_clips, uint32_t collect_flags, int32_t blend_frames,
                            void* out_audio_host, void* out_facial_host);

/* Fused host entry point for the dataset builders (dataset/data_processing.py:44-78 process_folder ->
 * :108-177 collect_features): features of a batch of clips AND their collect_features augmentation in one
 * pipelined pass.  The feature rows never leave the device between the two steps - only PCM and facial rows go
 * up, only augmented rows come back.  float32 throughout (the training format, dataset/dataset.py:75); the
 * float64 bit-exact arithmetic of the reference remains available through nsf_collect_host.  Clip i owns
 * samples [clip_offsets[i], clip_offsets[i+1]) of pcm and rows [facial_offsets[i], facial_offsets[i+1]) of
 * facial; outputs are packed at the prefix sum of nsf_collect_rows(nsf_feature_rows(..), facial rows, ..).
 * features_host (optional, [sum R_i x cols] float32) also receives the un-augmented feature rows - what
 * collect_features writes to its audio_features.csv cache (data_processing.py:115-120). */
NSF_API nsf_status nsf_extract_collect_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format,
                                            const int64_t* clip_offsets_host, int32_t n_clips, uint32_t flags,
                                            const float* facial_host, int32_t facial_cols,
                                            const int64_t* facial_offsets_host, uint32_t collect_flags,
                                            int32_t blend_frames, float* out_audio_host, float* out_facial_host,
                                            float* features_host /* optional */);

/* ---- stand-alone array helpers of the reference API, on HOST arrays --------------------------
 * Row-wise helpers of dataset/data_processing.py (float32 or float64, the reference's exact
 * rounding order), computed on the device:
 *   NSF_ROWS_INTERP_SLOWER  a[na x cols]               -> out[(2 na - 1) x cols]  interpolate_slower :84-106
 *   NSF_ROWS_SMOOTH         a[na x cols]               -> out[na x cols]          smooth_facial_data :201-204,
 *                                                                                 smooth_features (utils :47-51)
 *   NSF_ROWS_BLEND_STACK    a[na x cols], b[nb x cols] -> out[(na + nb - k) x cols], k = min(blend_frames, na, nb)
 *                                                       one step of stack_with_blend :179-197 */
#define NSF_ROWS_INTERP_SLOWER 0
#define NSF_ROWS_SMOOTH 1
#define NSF_ROWS_BLEND_STACK 2
NSF_API nsf_status nsf_rows_host(nsf_ctx* ctx, int32_t op, int32_t dtype, const void* a_host, int64_t na,
                                 const void* b_host, int64_t nb, int32_t cols, int32_t blend_frames,
                                 void* out_host);

/* Per-clip post-processing helpers of extract_features_utils.py on ONE frame-major float32 matrix
 * in[T x C] (the Python wrappers transpose from the reference's channel-major [C x T]):
 *   NSF_POST_EDGEFIX  fix_edge_frames_autocorr             :105-113
 *   NSF_POST_CMVN     cepstral_mean_variance_normalization :5-8
 *   NSF_POST_DELTAS   vstack(x, delta(x), delta(x, 2))     :25-27, :131-135
 *   NSF_POST_REDUCE   reduce_features                      :33-44
 * applied in that order.  out is [rows x C * (3 if DELTAS else 1)], rows = ceil(T/2) with REDUCE. */
#define NSF_POST_EDGEFIX 0x1u
#define NSF_POST_CMVN 0x2u
#define NSF_POST_DELTAS 0x4u
#define NSF_POST_REDUCE 0x8u
NSF_API nsf_status nsf_post_host(nsf_ctx* ctx, const float* in_host, int64_t n_frames, int32_t channels,
                                 uint32_t post_flags, float* out_host);

/* ---- inference-side chunker --------------------------------------------------------------------------
 * The consumer of the feature rows at inference / validation time, process_audio_features
 * (utils/audio/processing/audio_processing.py:50-112): `frame`-row chunks every frame - overlap rows, the last
 * ones completed by reflection (pad_audio_chunk :14-23), decoded by the caller's model, cross-faded over `overlap`
 * rows (blend_chunks :33-48), trimmed to n_rows and `[:, :61] /= 100` (:103).  Device-resident and stream-ordered:
 * feature rows from nsf_extract_batch never leave the GPU between extraction and the model.
 *   nsf_chunk_count   number of chunks the reference's while loop produces (0 for an invalid geometry)
 *   nsf_chunk_gather  rows_dev [n_rows x cols] (row pitch ld) -> chunks_dev [n_chunks x frame x cols]
 *   nsf_chunk_blend   decoded_dev [n_chunks x frame x out_cols] -> out_dev [n_rows x out_cols]; the first
 *                     scale_cols columns are divided by `divisor`.  float32 arithmetic in NumPy's order (bit-identical
 *                     to the reference given the same decoded chunks).  NSF_ERR_UNSUPPORTED when 2 * overlap > frame. */
NSF_API int64_t nsf_chunk_count(int64_t n_rows, int32_t frame, int32_t overlap);
NSF_API nsf_status nsf_chunk_gather(nsf_ctx* ctx, void* cuda_stream, const float* rows_dev, int64_t n_rows, int32_t cols,
                                    int64_t ld, int32_t frame, int32_t overlap, float* chunks_dev);
NSF_API nsf_status nsf_chunk_blend(nsf_ctx* ctx, void* cuda_stream, const float* decoded_dev, int64_t n_rows,
                                   int32_t out_cols, int32_t frame, int32_t overlap, int32_t scale_cols, float divisor,
                                   float* out_dev);

/* ---- sample-rate conversion ------------------------------------------------------------------------
 * The resampling half of the loaders: `librosa.resample(y, orig_sr=sr, target_sr=88200)` of
 * load_and_preprocess_audio (utils/audio/load_audio.py:8-10) and the `sr=` conversion inside
 * `librosa.load` (:19, :25, :36).  The reference resolves both to soxr_hq, a closed-form description of
 * which is not available here (SURVEY.md section 8(f)-2: "parity unpinned"); this entry point is the
 * rational polyphase resampler  up/down = target_sr/orig_sr (reduced):  a Kaiser(beta = 5) windowed-sinc
 * low-pass of 20 * max(up, down) + 1 taps, cut-off 1 / max(up, down), unit DC gain, zero-extended
 * input, centred output of ceil(n_in * up / down) samples - the arithmetic of
 * scipy.signal.resample_poly, evaluated per output sample in float64 on the device and rounded once
 * to float32.  Synthetic benchmark configurations never resample.
 *   nsf_resample_len    output length (0 when a rate is not positive)
 *   nsf_resample_design filter of the conversion: returns the tap count 20 max(up,down)+1 and copies
 *                       min(count, capacity) float64 taps (already scaled by `up`) when taps != NULL;
 *                       up / down / n_pre_pad / n_pre_remove (all optional) describe the polyphase
 *                       indexing  out[j] = sum_n h[(j + n_pre_remove) down - n_pre_pad - n up] x[n].
 *                       Runs without a GPU.
 *   nsf_resample_host   host PCM (float32 or int16) -> host float32 at target_sr, through the device.
 *
 * Two filter designs share the polyphase kernel (same indexing, different taps); the context option
 * NSF_OPT_RESAMPLE_QUALITY picks the one nsf_resample_host applies (default NSF_RESAMPLE_HQ):
 *   NSF_RESAMPLE_POLY  the scipy.signal.resample_poly design above (Kaiser beta 5, ~60 dB; pinned to scipy);
 *   NSF_RESAMPLE_HQ    band-limited windowed sinc, 64 zero crossings, roll-off 0.9476, Kaiser beta 14.77 (> 140 dB):
 *                      out[m] = sum_n x[n] g((n/down - m/up) f), f = min(up, down) rolloff, the arithmetic of
 *                      torchaudio.functional.resample(resampling_method="sinc_interp_kaiser") with those
 *                      parameters (pinned to torchaudio).  Same class as the reference's soxr_hq: what lies above
 *                      the input band ends below the 80 dB floor of the dB stage, so the features agree with any
 *                      high-quality resampler up to the transition band (profiles/parity_r02.md). */
#define NSF_RESAMPLE_POLY 0
#define NSF_RESAMPLE_HQ 1
#define NSF_OPT_RESAMPLE_QUALITY 1
NSF_API int64_t nsf_resample_len(int64_t n_in, int32_t orig_sr, int32_t target_sr);
NSF_API int64_t nsf_resample_design_q(int32_t orig_sr, int32_t target_sr, int32_t quality, double* taps, int64_t capacity,
                                      int32_t* up, int32_t* down, int32_t* n_pre_pad, int32_t* n_pre_remove);
NSF_API int64_t nsf_resample_design(int32_t orig_sr, int32_t target_sr, double* taps, int64_t capacity,
                                    int32_t* up, int32_t* down, int32_t* n_pre_pad, int32_t* n_pre_remove);
NSF_API nsf_status nsf_resample_host(nsf_ctx* ctx, const void* pcm_host, int32_t pcm_format, int64_t n_in,
                                     int32_t orig_sr, int32_t target_sr, float* out_host, int64_t out_capacity);

/* ---- WAV conversion: decode + downmix + resample for a ragged batch ---------------------------------
 * Raw WAV data-chunk bytes in (any encoding decode_wav of utils/audio/load_audio.py accepts, any channel count,
 * any rate), mono float32 at target_sr out.  Clip i is described by sources[i]: `frames` interleaved frames of
 * `channels` samples of `encoding` starting `byte_offset` bytes into the payload.  Per clip the output is, bit for
 * bit, what decode_wav followed by nsf_resample_host (at the context's NSF_OPT_RESAMPLE_QUALITY) produces:
 *   decode   u8 (v - 128) / 128, i16 v / 32768, i24 v / 2^23, i32 v / 2^31 (rounded once to float32), f32 as is,
 *            f64 rounded to nearest float32;
 *   downmix  the channel mean in NumPy's order (mean(axis=1, dtype=float32): pairwise summation, then one
 *            division by the channel count); mono clips are not touched;
 *   resample the polyphase filter of nsf_resample_host when sample_rate != target_sr (same float64 FMA chain per
 *            output); a clip already at target_sr is decode-only.
 * Every descriptor is validated on the host before anything is launched (NSF_ERR_BAD_ARG): a known encoding,
 * 1 <= channels <= 65535, frames >= 0, sample_rate > 0, the byte range inside payload_bytes, and 2-, 4- and 8-byte
 * containers at addresses that are multiples of their size (a misaligned device load would fault).
 *   nsf_convert_offsets  out_offsets[0] = 0, out_offsets[i + 1] = out_offsets[i] + output length of clip i
 *                        (frames at target_sr, else nsf_resample_len(frames, sample_rate, target_sr)); runs without
 *                        a GPU; out_offsets has n + 1 entries.
 *   nsf_convert_batch    device payload -> device float32, stream-ordered; clip i writes
 *                        out_dev[out_offsets[i], out_offsets[i + 1]) (out_offsets_host NULL = the prefix sum).
 *                        Descriptors go through the descriptor ring.  Filter tables are cached in the context per
 *                        (rate pair, quality): the FIRST use of a pair uploads its table synchronously and may wait.
 *   nsf_convert_host     host payload -> host float32 at the prefix-sum packing; pipelined over clip groups like
 *                        nsf_extract_host (pageable buffers staged through pinned arenas).  Synchronous. */
#define NSF_ENC_U8 0
#define NSF_ENC_I16 1
#define NSF_ENC_I24 2
#define NSF_ENC_I32 3
#define NSF_ENC_F32 4
#define NSF_ENC_F64 5
typedef struct nsf_pcm_source {
  int64_t byte_offset;  /* first byte of the clip's frames in the payload                */
  int64_t frames;       /* interleaved frames (data bytes // (bytes per sample * channels)) */
  int32_t encoding;     /* NSF_ENC_*                                                     */
  int32_t channels;
  int32_t sample_rate;
  int32_t reserved;     /* 0 */
} nsf_pcm_source;
NSF_API nsf_status nsf_convert_offsets(const nsf_pcm_source* sources, int32_t n, int32_t target_sr,
                                       int64_t payload_bytes, int64_t* out_offsets);
NSF_API nsf_status nsf_convert_batch(nsf_ctx* ctx, void* cuda_stream, const void* payload_dev, int64_t payload_bytes,
                                     const nsf_pcm_source* sources_host, int32_t n, int32_t target_sr, float* out_dev,
                                     const int64_t* out_offsets_host);
NSF_API nsf_status nsf_convert_host(nsf_ctx* ctx, const void* payload_host, int64_t payload_bytes,
                                    const nsf_pcm_source* sources, int32_t n, int32_t target_sr, float* out_host);

/* ---- training windows ------------------------------------------------------------------------------
 * The consumer of the augmented rows at training time, AudioFacialDataset (dataset/dataset.py:58-98): every stride-1
 * window of `window` rows of each clip, plus one reflected tail window when the clip's length is not a multiple of
 * `window`.  Clip i owns audio rows [audio_offsets[i], audio_offsets[i+1]) and facial rows [facial_offsets[i],
 * facial_offsets[i+1]); top = max(n_audio, n_facial).  Regular window j < top - window + 1 starts at row j; a stream
 * shorter than j + window is zero-padded.  The tail window starts at row top - window: with seg = min(top, n_rows) -
 * (top - window) valid rows, row r >= seg is the reflection rows[start + 2 seg - 1 - r] (torch.flip of the segment;
 * a one-row segment is repeated, which is what torch's broadcast makes of it).  A clip with top < window, or with a
 * stream whose tail segment is shorter than half a window and not one row (the host route raises for both), is
 * rejected with NSF_ERR_BAD_ARG, as are decreasing or negative offsets and window < 1.
 *   nsf_window_offsets  window_offsets[0] = 0, window_offsets[i+1] = window_offsets[i] + (top - window + 1) +
 *                       (top % window != 0); validates the geometry; host only, no GPU.  n_clips + 1 entries.
 *   nsf_window_gather   out_audio [n][window][audio_cols], out_facial [n][window][facial_cols] float32, contiguous:
 *                       windows indices[k] of the dataset (global numbering of nsf_window_offsets), what
 *                       collate_fn(stack of __getitem__) yields, bit for bit.  Stream-ordered; geometry and every
 *                       index (in [0, total)) are validated on the host before anything is launched; the offsets and
 *                       indices go through the descriptor ring.  n == 0 launches nothing (the outputs and indices
 *                       may then be NULL). */
NSF_API nsf_status nsf_window_offsets(const int64_t* audio_offsets, const int64_t* facial_offsets, int32_t n_clips,
                                      int32_t window, int64_t* window_offsets);
NSF_API nsf_status nsf_window_gather(nsf_ctx* ctx, void* cuda_stream,
                                     const float* audio_dev, int32_t audio_cols, const int64_t* audio_offsets_host,
                                     const float* facial_dev, int32_t facial_cols, const int64_t* facial_offsets_host,
                                     int32_t n_clips, int32_t window, const int64_t* indices_host, int64_t n,
                                     float* out_audio_dev, float* out_facial_dev);

/* ---- instrumentation -------------------------------------------------------------------------
 * Kernel launches issued by this context since creation (bench.py reports it as gpu_launches). */
NSF_API int64_t nsf_launch_count(const nsf_ctx* ctx);
/* Per-stage device times of the most recent nsf_extract_batch on this context when profiling was
 * enabled with nsf_set_profiling(ctx, 1): CUDA events on the call's stream, milliseconds.
 * Stage ids: 0 peak/normalise, 1 fold, 2 stft-gemm, 3 mel/log, 4 dct/stats, 5 cmvn/delta/reduce,
 * 6 autocorr, 7 post (smoothing / ac-deltas).  Returns the number of stages written. */
NSF_API void nsf_set_profiling(nsf_ctx* ctx, int32_t enabled);
NSF_API int32_t nsf_stage_times_ms(nsf_ctx* ctx, float* ms, int32_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* NSF_H_ */

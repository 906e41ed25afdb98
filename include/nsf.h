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

/* ---- FLAC decode -------------------------------------------------------------------------------------
 * The decode half of librosa.load for FLAC files (utils/audio/load_audio.py:19, :25, :36; libsndfile reads FLAC
 * natively).  The metadata blocks are container parsing and stay with the caller (load_audio.flac_layout); the
 * frames are decoded on the device.  Stream i is described by sources[i]: its frame data is payload bytes
 * [byte_offset, byte_offset + byte_length) and decodes to `frames` interleaved frames of `channels` samples of
 * `bits` bits (STREAMINFO).  The output of stream i is the WAV data chunk holding those samples: u8 v + 128 for 8
 * bits, little-endian i16 for 16, packed little-endian i24 for 24, at the prefix sum of frames * channels * (bits / 8).
 * Decoded (RFC 9639): fixed and variable blocking, block sizes 1..65535, CONSTANT / VERBATIM / FIXED 0-4 / LPC 1-32
 * subframes, wasted bits, both Rice methods with escaped partitions, the four channel assignments.  Every frame's
 * header CRC-8 and frame CRC-16 are checked; the STREAMINFO MD5 is not.  Frames must follow each other from
 * byte_offset, with consecutive frame numbers (fixed blocking) or first samples (variable blocking), tiling
 * [0, frames) exactly; bytes after the last frame are ignored.  A frame whose channel count, bits per sample or
 * explicit sample rate disagrees with the descriptor, or whose block is larger than max_block, is corrupt.
 *   nsf_flac_decode_host  host payload -> host PCM bytes; synchronous, pipelined over stream groups like
 *                         nsf_convert_host (pageable or page-locked buffers).  Descriptors are validated before
 *                         anything is launched: the byte range inside payload_bytes and below 2^31 bytes,
 *                         bits 8 / 16 / 24, channels 1..8, frames > 0, max_block 1..65535, sample_rate > 0
 *                         (NSF_ERR_BAD_ARG).  A corrupt stream returns NSF_ERR_BAD_ARG, and nsf_last_error names the
 *                         stream, the frame's byte offset in the payload and the reason.
 *   nsf_flac_check        verification aid, like nsf_parse_check: the device's frame-header parser and frame decoder
 *                         run on the host over the ONE frame that starts at source->byte_offset (and ends before
 *                         byte_offset + byte_length).  Fills *frame (status NSF_FLAC_*: the call itself returns
 *                         NSF_OK once its arguments are valid) and, when samples != NULL and the frame decodes, its
 *                         samples channel by channel after the inter-channel decorrelation: samples[c * block + i],
 *                         NSF_ERR_BAD_ARG when capacity < channels * block.  Not a compute path. */
typedef struct nsf_flac_source {
  int64_t byte_offset;  /* first byte of the first frame (after the metadata blocks)      */
  int64_t byte_length;  /* bytes of frame data                                           */
  int64_t frames;       /* STREAMINFO total samples per channel, > 0                      */
  int32_t channels;     /* 1..8                                                           */
  int32_t bits;         /* 8, 16 or 24                                                    */
  int32_t sample_rate;  /* STREAMINFO                                                     */
  int32_t max_block;    /* STREAMINFO maximum block size, 1..65535                         */
} nsf_flac_source;
/* status of one frame (nsf_flac_frame.status) */
#define NSF_FLAC_OK 0
#define NSF_FLAC_NO_SYNC 1       /* no frame sync code 0xFFF8 / 0xFFF9                                 */
#define NSF_FLAC_TRUNCATED 2     /* the frame runs past the end of the stream                          */
#define NSF_FLAC_BAD_NUMBER 3    /* malformed coded frame / sample number                              */
#define NSF_FLAC_BAD_CRC8 4      /* header CRC-8 mismatch                                              */
#define NSF_FLAC_RESERVED 5      /* a reserved or invalid code in the header or a subframe             */
#define NSF_FLAC_CHANNELS 6      /* channel count disagrees with STREAMINFO                            */
#define NSF_FLAC_BITS 7          /* bits per sample disagree with STREAMINFO                           */
#define NSF_FLAC_RATE 8          /* sample rate disagrees with STREAMINFO                              */
#define NSF_FLAC_BLOCK 9         /* block size above the STREAMINFO maximum                            */
#define NSF_FLAC_WASTED 10       /* wasted bits leave no sample bits                                   */
#define NSF_FLAC_LPC_SHIFT 11    /* negative LPC shift                                                 */
#define NSF_FLAC_PARTITION 12    /* partition order does not divide the block, or a first partition
                                    shorter than the predictor order                                 */
#define NSF_FLAC_RANGE 13        /* a Rice-coded residual outside 32 bits                              */
#define NSF_FLAC_BAD_CRC16 14    /* frame CRC-16 mismatch                                              */
typedef struct nsf_flac_frame {
  int64_t end;          /* first byte after the frame's CRC-16 (payload offset)                         */
  int64_t number;       /* coded number: frame number (fixed blocking) or first sample (variable)      */
  int32_t block;        /* block size                                                                   */
  int32_t sample_rate;  /* from the header, the descriptor's when the header defers to STREAMINFO       */
  int32_t bits;         /* likewise                                                                     */
  int32_t assignment;   /* channel assignment code: 0-7 independent, 8 left/side, 9 side/right, 10 mid/side */
  int32_t channels;
  int32_t variable;     /* blocking strategy bit                                                        */
  int32_t crc8_ok;      /* header CRC-8 matches                                                         */
  int32_t crc16_ok;     /* frame CRC-16 matches (0 when the decode stopped before the CRC-16)           */
  int32_t status;       /* NSF_FLAC_*                                                                   */
  int32_t reserved;
} nsf_flac_frame;
NSF_API nsf_status nsf_flac_decode_host(nsf_ctx* ctx, const void* payload_host, int64_t payload_bytes,
                                        const nsf_flac_source* sources, int32_t n, void* pcm_host);
NSF_API nsf_status nsf_flac_check(const void* payload, const nsf_flac_source* source, nsf_flac_frame* frame,
                                  int32_t* samples, int64_t capacity);

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

/* ---- feature cache as CSV text ----------------------------------------------------------------------
 * The reference's audio_features.csv cache (dataset/data_processing.py:115-120): pd.DataFrame(rows.astype(float64))
 * .to_csv(path, index=False), formatted on the device byte for byte.  Each file is the header line "0,1,...,cols-1\n"
 * followed by one line per row, fields separated by ',' and each line ended by '\n' (a file without rows is the
 * header alone).  A finite field is Python's repr(float(v)): the shortest digits that round back to the double (the
 * nearest such string when several have that length), positional for 1e-4 <= |v| < 1e16 with ".0" on integers
 * (0.00015, 123.0, -0.0), scientific otherwise with a signed exponent of at least two digits (1e-05, 1e+16,
 * 5e-324).  float32 rows are widened to double first (0.1f -> 0.10000000149011612).  inf / -inf are written as
 * such, NaN as an empty field, or as "" when it is the row's only field. */
/* Upper bound of the text nsf_format_csv_host writes for n_files files, n_rows rows in total, cols columns
 * (24 characters per field + separator, plus one header per file); -1 for negative counts or cols < 1.  Host only.
 * (data_processing.py:115-120) */
NSF_API int64_t nsf_csv_bytes_bound(int64_t n_rows, int32_t cols, int32_t n_files);
/* rows_host: [row_offsets[n_files] - row_offsets[0]] x cols, row-major, NSF_F32 or NSF_F64.  File i = header +
 * rows [row_offsets[i], row_offsets[i+1]) -> text_host[text_offsets[i], text_offsets[i+1]), text_offsets[0] = 0
 * (n_files + 1 entries).  Synchronous, pipelined over file groups (one wait per group for its text size); pageable
 * or page-locked buffers.  NSF_ERR_BAD_ARG for NULLs, cols < 1, a bad dtype, decreasing offsets or text_capacity
 * below nsf_csv_bytes_bound, before anything is launched.  (data_processing.py:115-120) */
NSF_API nsf_status nsf_format_csv_host(nsf_ctx* ctx, int32_t dtype, const void* rows_host, int32_t cols,
                                       const int64_t* row_offsets_host, int32_t n_files,
                                       char* text_host, int64_t text_capacity, int64_t* text_offsets_host);
/* Verification aid, like nsf_plan_fold_check: the device's digit routine run on the host, value i -> out[32 i ..],
 * lengths[i] characters (0 for NaN).  Exists so the formatting can be checked against repr without a GPU; not a
 * compute path.  (data_processing.py:115-120) */
NSF_API nsf_status nsf_format_check(const double* values, int64_t n, char* out, int32_t* lengths);

/* ---- CSV text -> rows ------------------------------------------------------------------------------
 * The reference's reads of the facial CSVs and of the audio_features.csv cache (dataset/data_processing.py:112-123):
 * pd.read_csv(path).drop(columns=DROP).values, parsed on the device value for value.  A file is its header line
 * (the first line, skipped here: names, duplicates and DROP are the caller's business) and data rows.  A row ends at
 * '\n'; a '\r' directly before it is dropped; a line that is empty after that is skipped; the last line may lack its
 * '\n'.  A field is empty (-> NaN), "inf" / "-inf", or [+-]? digits* ( . digits* )? ( [eE] [+-]? digits+ )? with
 * at least one mantissa digit and at most 40 characters, valued by pandas' precise_xstrtod with the same IEEE double
 * operations in the same order (not correctly rounded: up to 17 mantissa digits as number * 10 + d, then one
 * multiplication or division by the double literal 1e<k>).  A column whose every field is an integer literal is
 * int64 in pandas, so its -0 is +0.  float32 output is the double rounded to nearest (NumPy's astype).
 * Anything else makes the file unaccepted and sets bits of its status word:
 *   NSF_CSV_BAD_FIELD  a field outside the grammar (spaces, NaN spellings, non-ASCII or control bytes, a decimal
 *                      exponent above 308, an overflow to inf) or longer than 40 characters;
 *   NSF_CSV_BAD_SHAPE  a row with more or fewer fields than `cols`;
 *   NSF_CSV_BAD_LINE   a quote character or a bare '\r' (pandas quotes / ends the line there);
 *   NSF_CSV_BAD_INT    an integer literal of more than 15 digits, or a -0 literal in a column that also holds other
 *                      fields (pandas' chunked reader types each chunk of rows on its own, so that zero's sign depends
 *                      on where the chunk boundaries fall);
 *   NSF_CSV_BAD_ROWS   row_offsets_host does not match the text.
 * The rows of an unaccepted file are unspecified; read it with pandas instead. */
#define NSF_CSV_BAD_FIELD 0x1u
#define NSF_CSV_BAD_SHAPE 0x2u
#define NSF_CSV_BAD_LINE 0x4u
#define NSF_CSV_BAD_INT 0x8u
#define NSF_CSV_BAD_ROWS 0x10u
/* kinds of nsf_parse_check */
#define NSF_CSV_KIND_NUMBER 0
#define NSF_CSV_KIND_INTEGER 1 /* [+-]? digits: pandas' int64 when the whole column is such literals */
#define NSF_CSV_KIND_EMPTY 2   /* NaN */
#define NSF_CSV_KIND_INF 3
#define NSF_CSV_KIND_BAD 4     /* unaccepted */
/* Data rows per file: row_offsets_host[i] = data rows of the files before file i (n_files + 1 entries), file i being
 * bytes [text_offsets_host[i], text_offsets_host[i+1]) of text_dev (header included; text_dev 16-byte aligned).
 * The call's one host wait is the download of those n_files + 1 counts.  NSF_ERR_BAD_ARG for NULLs,
 * n_files < 0, a negative first offset, decreasing offsets or an unaligned text_dev, before anything is launched;
 * n_files == 0 launches nothing.  (data_processing.py:112-123) */
NSF_API nsf_status nsf_csv_row_offsets(nsf_ctx* ctx, void* cuda_stream, const char* text_dev,
                                       const int64_t* text_offsets_host, int32_t n_files, int64_t* row_offsets_host);
/* The rows: file i's data rows go to out_dev rows [row_offsets_host[i], row_offsets_host[i+1]) (row_offsets_host as
 * nsf_csv_row_offsets returned it, starting at 0), row r at out_dev + r * out_ld, of dtype NSF_F32 or NSF_F64; the
 * file's column c goes to output column out_col_host[c] (cols entries, each in [-1, out_cols), -1 = dropped: not
 * parsed, only checked for quotes and bare '\r', each output column used at most once).  file_status_dev[i]
 * (uint32) == 0: file i's rows are final; else the NSF_CSV_BAD_* bits say why not.  Stream-ordered, no host wait:
 * offsets, column map and row offsets travel through the descriptor ring.  NSF_ERR_BAD_ARG for NULLs, n_files < 0,
 * cols < 1, bad offsets or alignment (as above), row offsets not starting at 0 or decreasing, a bad column map, a bad
 * dtype or out_ld < out_cols; NSF_ERR_UNSUPPORTED above 2^31 rows; all before anything is launched.  n_files == 0
 * launches nothing.  (data_processing.py:112-123) */
NSF_API nsf_status nsf_csv_parse(nsf_ctx* ctx, void* cuda_stream, int32_t dtype, const char* text_dev,
                                 const int64_t* text_offsets_host, int32_t n_files, int32_t cols,
                                 const int32_t* out_col_host, int32_t out_cols, const int64_t* row_offsets_host,
                                 void* out_dev, int64_t out_ld, uint32_t* file_status_dev);
/* Verification aid, like nsf_format_check: the device's field routine run on the host.  Field i is
 * text[field_offsets[i], field_offsets[i+1]) -> values[i], kinds[i] (NSF_CSV_KIND_*; values[i] is unspecified for
 * NSF_CSV_KIND_BAD).  Not a compute path.  (data_processing.py:112-123) */
NSF_API nsf_status nsf_parse_check(const char* text, const int64_t* field_offsets, int64_t n, double* values,
                                   int32_t* kinds);

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

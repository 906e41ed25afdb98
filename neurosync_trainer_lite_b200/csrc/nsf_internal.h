// Internal declarations shared by the host plan builder, the kernels and the C ABI.
#ifndef NSF_INTERNAL_H_
#define NSF_INTERNAL_H_

#include <stdint.h>

#include <string>
#include <vector>

#include "nsf.h"

namespace nsf {

constexpr int kMaxChains = 2;
constexpr int kFoldTaps = 4;      // every folded input is a signed sum of <= 4 windowed samples
constexpr int kMinGuardFrames = 9;  // extract_features.py:14

// One fold chain = the set of rFFT bins reached by one (Re, Im) pair of small GEMMs.
//   even F : chain 0 -> even bins, chain 1 -> odd bins   (two symmetry levels, K = F/4 + 1)
//   odd  F : chain 0 -> all bins                         (one symmetry level,  K = (F + 1) / 2)
struct FoldChain {
  int k = 0;         // folded inputs actually used
  int kp = 0;        // padded to a multiple of 16 (one fp16 UMMA k-step); extra inputs are zero
  int nbins = 0;     // output bins of this chain
  int np = 0;        // padded to a multiple of 16
  std::vector<int32_t> bin;  // [nbins] natural rFFT bin of output column m
  // taps, laid out [part(re=0, im=1)][tap][kp]
  std::vector<int32_t> tap_idx;
  std::vector<float> tap_coef;
  // DFT matrices in float64, row-major [kp][np]; part 0 = cos, part 1 = -sin
  std::vector<double> mat[2];
};

struct Plan {
  int sr = 0, F = 0, H = 0, pad = 0;
  int n_mfcc = 23, n_mels = 128, n_lags = 187;
  int bins = 0;
  int chains = 0;
  FoldChain chain[kMaxChains];
  std::vector<float> hann_per;   // [F] periodic (STFT)
  std::vector<float> hann_sym;   // [F] np.hanning (autocorr)
  std::vector<float> mel_dense;  // [n_mels][bins]
  std::vector<float> dct;        // [n_mfcc][n_mels]
  // sparse mel: per filter a contiguous bin range
  std::vector<int32_t> mel_start, mel_len, mel_ptr;  // mel_ptr[m] = offset into mel_w
  std::vector<float> mel_w;
  int mel_max_len = 0;
};

void set_error(const std::string& msg);

// Polyphase resampler design (scipy.signal.resample_poly arithmetic); see nsf_resample_design in nsf.h.
struct ResampleDesign {
  int up = 1, down = 1, half_len = 0, n_pre_pad = 0, n_pre_remove = 0;
  std::vector<double> h;   // 2 half_len + 1 taps, scaled by `up`
};
bool design_resampler(int orig_sr, int target_sr, ResampleDesign* d);      // NSF_RESAMPLE_POLY
bool design_resampler_hq(int orig_sr, int target_sr, ResampleDesign* d);   // NSF_RESAMPLE_HQ
nsf_status build_plan(int sr, int F, int H, int n_mfcc, int n_mels, int n_lags, Plan* plan);

// Python-style floor division for the guard (extract_features.py:16)
inline int64_t floordiv(int64_t a, int64_t b) {
  int64_t q = a / b, r = a % b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}

// Hop-frames of a clip of `len` samples under `flags`, and in *rows its feature rows.  Frames are centre-padded
// unless NSF_AC_NO_PAD (pad_signal=False: y[t H : t H + F], as many as fit); rows are frame pairs unless NSF_NO_REDUCE.
inline int64_t clip_frames(int64_t len, int32_t F, int32_t H, uint32_t flags, int64_t* rows) {
  const int64_t T = (flags & NSF_AC_NO_PAD) ? (len >= F ? nsf_guard_frames(len, F, H) : 0) : nsf_hop_frames(len, F, H);
  *rows = (flags & NSF_NO_REDUCE) ? T : (T + 1) / 2;
  return T;
}

}  // namespace nsf

struct nsf_plan {
  nsf::Plan p;
};

#endif  // NSF_INTERNAL_H_

// Host-side constant tables ("plan") and the bit-exact integer frame arithmetic.
//
// Everything here restates published definitions in float64 and rounds to float32 exactly where
// librosa / numpy do, so the GPU kernels consume the same constants the reference path uses:
//   - periodic Hann (scipy.signal.get_window('hann', F, fftbins=True))   -> STFT branch
//   - np.hanning(F)                                                      -> autocorr branch
//   - librosa.filters.mel(sr, n_fft=F, n_mels, norm='slaney', htk=False) -> dense + sparse form
//   - DCT-II 'ortho' matrix (scipy.fftpack.dct(type=2, norm='ortho'))
//   - the folded real-DFT tables described in DESIGN.md ("STFT as four small GEMMs")
// Reference call sites: utils/audio/extraction/extract_features_utils.py:19,79.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "nsf_internal.h"

namespace nsf {

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }
const std::string& last_error() { return g_error; }

namespace {

constexpr double kPi = 3.14159265358979323846264338327950288;

// librosa.core.convert.hz_to_mel / mel_to_hz, Slaney variant (htk=False)
double hz_to_mel(double f) {
  const double f_sp = 200.0 / 3;
  const double min_log_hz = 1000.0;
  const double min_log_mel = min_log_hz / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  if (f >= min_log_hz) return min_log_mel + std::log(f / min_log_hz) / logstep;
  return f / f_sp;
}
double mel_to_hz(double m) {
  const double f_sp = 200.0 / 3;
  const double min_log_hz = 1000.0;
  const double min_log_mel = min_log_hz / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  if (m >= min_log_mel) return min_log_hz * std::exp(logstep * (m - min_log_mel));
  return f_sp * m;
}

void build_mel(Plan* p) {
  const int bins = p->bins, nm = p->n_mels;
  // np.fft.rfftfreq(n=F, d=1/sr): val = 1/(n*d); k * val
  const double d = 1.0 / static_cast<double>(p->sr);
  const double val = 1.0 / (static_cast<double>(p->F) * d);
  std::vector<double> fftfreqs(bins);
  for (int k = 0; k < bins; ++k) fftfreqs[k] = static_cast<double>(k) * val;
  // mel_frequencies(n_mels + 2, fmin=0, fmax=sr/2): np.linspace in mel space, endpoint exact
  const int npts = nm + 2;
  const double lo = hz_to_mel(0.0), hi = hz_to_mel(static_cast<double>(p->sr) / 2);
  const double step = (hi - lo) / static_cast<double>(npts - 1);
  std::vector<double> mel_f(npts);
  for (int i = 0; i < npts; ++i) mel_f[i] = mel_to_hz(static_cast<double>(i) * step + lo);
  mel_f[npts - 1] = mel_to_hz(hi);
  p->mel_dense.assign(static_cast<size_t>(nm) * bins, 0.0f);
  for (int i = 0; i < nm; ++i) {
    const double fd0 = mel_f[i + 1] - mel_f[i], fd1 = mel_f[i + 2] - mel_f[i + 1];
    const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
    for (int k = 0; k < bins; ++k) {
      const double lower = -(mel_f[i] - fftfreqs[k]) / fd0;
      const double upper = (mel_f[i + 2] - fftfreqs[k]) / fd1;
      const float w32 = static_cast<float>(std::max(0.0, std::min(lower, upper)));
      // weights (float32) *= enorm (float64): computed in float64, stored float32
      p->mel_dense[static_cast<size_t>(i) * bins + k] =
          static_cast<float>(static_cast<double>(w32) * enorm);
    }
  }
  // sparse form: each triangular filter is one contiguous run of bins (possibly empty)
  p->mel_start.assign(nm, 0);
  p->mel_len.assign(nm, 0);
  p->mel_ptr.assign(nm + 1, 0);
  p->mel_w.clear();
  p->mel_max_len = 0;
  for (int i = 0; i < nm; ++i) {
    int first = -1, last = -1;
    for (int k = 0; k < bins; ++k)
      if (p->mel_dense[static_cast<size_t>(i) * bins + k] != 0.0f) {
        if (first < 0) first = k;
        last = k;
      }
    p->mel_ptr[i] = static_cast<int32_t>(p->mel_w.size());
    if (first >= 0) {
      p->mel_start[i] = first;
      p->mel_len[i] = last - first + 1;
      for (int k = first; k <= last; ++k)
        p->mel_w.push_back(p->mel_dense[static_cast<size_t>(i) * bins + k]);
      p->mel_max_len = std::max(p->mel_max_len, last - first + 1);
    }
  }
  p->mel_ptr[nm] = static_cast<int32_t>(p->mel_w.size());
}

void build_dct(Plan* p) {
  const int nm = p->n_mels, nc = p->n_mfcc;
  p->dct.resize(static_cast<size_t>(nc) * nm);
  const double s = std::sqrt(2.0 / nm);
  for (int k = 0; k < nc; ++k)
    for (int m = 0; m < nm; ++m) {
      double v = s * std::cos(kPi * k * (2 * m + 1) / (2.0 * nm));
      if (k == 0) v *= 1.0 / std::sqrt(2.0);
      p->dct[static_cast<size_t>(k) * nm + m] = static_cast<float>(v);
    }
}

void build_windows(Plan* p) {
  const int F = p->F;
  p->hann_per.resize(F);
  p->hann_sym.resize(F);
  for (int n = 0; n < F; ++n) {
    p->hann_per[n] = static_cast<float>(0.5 - 0.5 * std::cos(2.0 * kPi * n / F));
    // np.hanning(M): 0.5 + 0.5 * cos(pi * (2n + 1 - M) / (M - 1))
    p->hann_sym[n] =
        F > 1 ? static_cast<float>(0.5 + 0.5 * std::cos(kPi * (2.0 * n + 1 - F) / (F - 1))) : 1.0f;
  }
}

struct Tap {
  int idx;
  double sign;
};

void alloc_chain(FoldChain* c, int k, int nbins) {
  c->k = k;
  c->kp = (k + 15) / 16 * 16;
  // Rows of the operand planes are kp fp16 values apart and are fetched as 64-column (128-byte) TMA boxes:
  // with kp a multiple of 64 every box row is ONE aligned 128-byte line instead of straddling two.
  // Taken when it costs at most 1/8 extra operand bytes (F = 1470: 368 -> 384).
  const int kp64 = (k + 63) / 64 * 64;
  if (kp64 * 8 <= c->kp * 9) c->kp = kp64;
  c->nbins = nbins;
  c->np = (nbins + 15) / 16 * 16;
  c->bin.assign(nbins, 0);
  c->tap_idx.assign(static_cast<size_t>(2) * kFoldTaps * c->kp, 0);
  c->tap_coef.assign(static_cast<size_t>(2) * kFoldTaps * c->kp, 0.0f);
  for (int part = 0; part < 2; ++part) c->mat[part].assign(static_cast<size_t>(c->kp) * c->np, 0.0);
}

void set_taps(FoldChain* c, const Plan& p, int part, int j, const Tap* taps, int ntaps) {
  for (int t = 0; t < ntaps; ++t) {
    const size_t o = (static_cast<size_t>(part) * kFoldTaps + t) * c->kp + j;
    c->tap_idx[o] = taps[t].idx;
    // window in float64, rounded once to float32 together with the sign
    const double w = 0.5 - 0.5 * std::cos(2.0 * kPi * taps[t].idx / p.F);
    c->tap_coef[o] = static_cast<float>(taps[t].sign * w);
  }
}

// X_k = sum_n u[n] exp(-2 pi i k n / F), u = periodic-Hann * frame.  Two exact symmetries of the
// DFT kernel shrink the GEMM 4x for even F (2x for odd F); see DESIGN.md for the derivation.
void build_fold(Plan* p) {
  const int F = p->F;
  if (F % 2 == 0) {
    const int Nh = F / 2;
    const int K = Nh / 2 + 1;
    const int n_even = Nh / 2 + 1;     // k = 0, 2, ..., <= Nh
    const int n_odd = (Nh + 1) / 2;    // k = 1, 3, ..., <= Nh
    p->chains = 2;
    alloc_chain(&p->chain[0], K, n_even);
    alloc_chain(&p->chain[1], K, n_odd);
    for (int m = 0; m < n_even; ++m) p->chain[0].bin[m] = 2 * m;
    for (int m = 0; m < n_odd; ++m) p->chain[1].bin[m] = 2 * m + 1;
    for (int j = 0; j < K; ++j) {
      const bool single = (j == 0) || (2 * j == Nh);  // self-paired under n <-> Nh - n
      // a[n] = u[n] + u[n+Nh] (even bins), b[n] = u[n] - u[n+Nh] (odd bins)
      const int i0 = j, i1 = j + Nh, i2 = Nh - j, i3 = F - j;
      if (single) {
        const Tap e[2] = {{i0, 1.0}, {i1, 1.0}};
        const Tap o[2] = {{i0, 1.0}, {i1, -1.0}};
        set_taps(&p->chain[0], *p, 0, j, e, 2);
        set_taps(&p->chain[0], *p, 1, j, e, 2);  // multiplied by sin(...) == 0 for both cases
        set_taps(&p->chain[1], *p, 0, j, o, 2);  // j == Nh/2: cos(pi(2m+1)/2) == 0
        set_taps(&p->chain[1], *p, 1, j, o, 2);  // j == 0: sin(0) == 0
      } else {
        const Tap e_re[4] = {{i0, 1.0}, {i1, 1.0}, {i2, 1.0}, {i3, 1.0}};     // a[j] + a[Nh-j]
        const Tap e_im[4] = {{i0, 1.0}, {i1, 1.0}, {i2, -1.0}, {i3, -1.0}};   // a[j] - a[Nh-j]
        const Tap o_re[4] = {{i0, 1.0}, {i1, -1.0}, {i2, -1.0}, {i3, 1.0}};   // b[j] - b[Nh-j]
        const Tap o_im[4] = {{i0, 1.0}, {i1, -1.0}, {i2, 1.0}, {i3, -1.0}};   // b[j] + b[Nh-j]
        set_taps(&p->chain[0], *p, 0, j, e_re, 4);
        set_taps(&p->chain[0], *p, 1, j, e_im, 4);
        set_taps(&p->chain[1], *p, 0, j, o_re, 4);
        set_taps(&p->chain[1], *p, 1, j, o_im, 4);
      }
      for (int m = 0; m < n_even; ++m) {
        const double th = 2.0 * kPi * (static_cast<double>(m) * j) / Nh;
        p->chain[0].mat[0][static_cast<size_t>(j) * p->chain[0].np + m] = std::cos(th);
        p->chain[0].mat[1][static_cast<size_t>(j) * p->chain[0].np + m] = -std::sin(th);
      }
      for (int m = 0; m < n_odd; ++m) {
        const double th = 2.0 * kPi * (static_cast<double>(2 * m + 1) * j) / F;
        p->chain[1].mat[0][static_cast<size_t>(j) * p->chain[1].np + m] = std::cos(th);
        p->chain[1].mat[1][static_cast<size_t>(j) * p->chain[1].np + m] = -std::sin(th);
      }
    }
  } else {
    const int K = (F + 1) / 2;
    p->chains = 1;
    alloc_chain(&p->chain[0], K, p->bins);
    for (int m = 0; m < p->bins; ++m) p->chain[0].bin[m] = m;
    for (int j = 0; j < K; ++j) {
      if (j == 0) {
        const Tap s[1] = {{0, 1.0}};
        set_taps(&p->chain[0], *p, 0, j, s, 1);
        set_taps(&p->chain[0], *p, 1, j, s, 1);
      } else {
        const Tap re[2] = {{j, 1.0}, {F - j, 1.0}};
        const Tap im[2] = {{j, 1.0}, {F - j, -1.0}};
        set_taps(&p->chain[0], *p, 0, j, re, 2);
        set_taps(&p->chain[0], *p, 1, j, im, 2);
      }
      for (int m = 0; m < p->bins; ++m) {
        const double th = 2.0 * kPi * (static_cast<double>(m) * j) / F;
        p->chain[0].mat[0][static_cast<size_t>(j) * p->chain[0].np + m] = std::cos(th);
        p->chain[0].mat[1][static_cast<size_t>(j) * p->chain[0].np + m] = -std::sin(th);
      }
    }
  }
}

}  // namespace

nsf_status build_plan(int sr, int F, int H, int n_mfcc, int n_mels, int n_lags, Plan* p) {
  if (sr <= 0 || F < 4 || H < 1 || H > F || n_mfcc < 1 || n_mels < n_mfcc || n_lags < 1 ||
      n_lags >= F) {
    set_error("nsf_plan_create: invalid geometry");
    return NSF_ERR_BAD_ARG;
  }
  if (F > 4096 || n_mels > 128 || n_mfcc > 32 || n_lags > 191) {
    set_error("nsf_plan_create: geometry outside kernel limits (F<=4096, n_mels<=128, "
              "n_mfcc<=32, n_lags<=191)");
    return NSF_ERR_UNSUPPORTED;
  }
  p->sr = sr;
  p->F = F;
  p->H = H;
  p->pad = F / 2;
  p->n_mfcc = n_mfcc;
  p->n_mels = n_mels;
  p->n_lags = n_lags;
  p->bins = F / 2 + 1;
  build_windows(p);
  build_mel(p);
  build_dct(p);
  build_fold(p);
  return NSF_OK;
}


// ---- polyphase resampler design --------------------------------------------------------------------
namespace {
int gcd_int(int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; }
// modified Bessel function of the first kind, order 0 (power series; x <= 5 here)
double bessel_i0(double x) {
  const double q = 0.25 * x * x;
  double term = 1.0, sum = 1.0;
  for (int k = 1; k < 200; ++k) {
    term *= q / (static_cast<double>(k) * k);
    sum += term;
    if (term < 1e-18 * sum) break;
  }
  return sum;
}
}  // namespace

// scipy.signal.resample_poly(x, up, down): h = up * firwin(2 half_len + 1, 1/max(up,down), window=('kaiser', 5.0)),
// half_len = 10 max(up, down); h is front-padded with n_pre_pad = down - half_len % down zeros so that the
// output sample j is upfirdn output j + n_pre_remove, n_pre_remove = (half_len + n_pre_pad) / down.
//
// quality NSF_RESAMPLE_HQ (what the loaders use): the band-limited windowed-sinc interpolator with the "kaiser_best"
// parameters - 64 zero crossings, roll-off 0.9475937167399596, Kaiser beta 14.769656459379492 (stop band below
// -140 dB) - evaluated exactly like torchaudio.functional.resample(..., resampling_method="sinc_interp_kaiser"):
//     out[m] = sum_n x[n] g((n / down - m / up) f),  f = min(up, down) * rolloff,
//     g(t) = (f / down) sinc(t) I0(beta sqrt(1 - (t / 64)^2)) / I0(beta)   for |t| <= 64, else 0.
// The reference resamples with soxr_hq (not reproducible here); this design shares its class - linear phase, pass
// band to ~0.91-0.95 of the lower Nyquist, > 120 dB rejection - so what lies above the input's band ends far
// below the 80 dB floor of the dB stage, which the 60 dB Kaiser(5) design of scipy.signal.resample_poly does not.
bool design_resampler_hq(int orig_sr, int target_sr, ResampleDesign* d) {
  if (orig_sr <= 0 || target_sr <= 0) return false;
  const int g = gcd_int(target_sr, orig_sr);
  d->up = target_sr / g;
  d->down = orig_sr / g;
  const double width = 64.0, rolloff = 0.9475937167399596, beta = 14.769656459379492;
  const double pi = 3.14159265358979323846264338327950288;
  const double f = (d->up < d->down ? d->up : d->down) * rolloff;
  const double per_tap = f / (static_cast<double>(d->up) * d->down);     // |t| of the tap at distance 1
  d->half_len = static_cast<int>(std::floor(width / per_tap));
  const int n = 2 * d->half_len + 1;
  d->h.assign(n, 0.0);
  const double i0b = bessel_i0(beta), scale = f / d->down;
  for (int i = 0; i < n; ++i) {
    const double t = (i - d->half_len) * per_tap;
    const double r = t / width;
    const double win = bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
    const double arg = pi * t;
    d->h[i] = scale * (t == 0.0 ? 1.0 : std::sin(arg) / arg) * win;
  }
  d->n_pre_pad = d->down - d->half_len % d->down;
  d->n_pre_remove = (d->half_len + d->n_pre_pad) / d->down;
  return true;
}

bool design_resampler(int orig_sr, int target_sr, ResampleDesign* d) {
  if (orig_sr <= 0 || target_sr <= 0) return false;
  const int g = gcd_int(target_sr, orig_sr);
  d->up = target_sr / g;
  d->down = orig_sr / g;
  const int max_rate = d->up > d->down ? d->up : d->down;
  d->half_len = 10 * max_rate;
  const int n = 2 * d->half_len + 1;
  const double fc = 1.0 / max_rate, alpha = 0.5 * (n - 1), beta = 5.0;
  const double pi = 3.14159265358979323846264338327950288;
  d->h.assign(n, 0.0);
  const double i0b = bessel_i0(beta);
  double sum = 0.0;
  for (int i = 0; i < n; ++i) {
    const double m = i - alpha;
    const double arg = pi * fc * m;
    const double sinc = m == 0.0 ? 1.0 : std::sin(arg) / arg;                  // np.sinc(fc m)
    const double r = m / alpha;
    const double win = bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - r * r))) / i0b;   // np.kaiser(n, 5)
    d->h[i] = fc * sinc * win;
    sum += d->h[i];
  }
  for (double& v : d->h) v = v / sum * d->up;                                   // unit DC gain, then * up
  d->n_pre_pad = d->down - d->half_len % d->down;
  d->n_pre_remove = (d->half_len + d->n_pre_pad) / d->down;
  return true;
}

}  // namespace nsf

// ------------------------------------------------------------------------------------------------
// C ABI: host-only entry points
// ------------------------------------------------------------------------------------------------
namespace nsf {
const std::string& last_error();
}

extern "C" {

int32_t nsf_abi_version(void) { return NSF_ABI_VERSION; }

const char* nsf_last_error(void) { return nsf::last_error().c_str(); }

int32_t nsf_frame_length(int32_t sr) {
  // int(0.01667 * sr) with the product taken in IEEE double, as Python does
  volatile double prod = 0.01667 * static_cast<double>(sr);
  return static_cast<int32_t>(prod);
}

int32_t nsf_hop_length(int32_t frame_length) { return frame_length / 2; }

int64_t nsf_guard_frames(int64_t n, int32_t F, int32_t H) {
  if (H <= 0) return 0;
  return nsf::floordiv(n - F, H) + 1;
}

int64_t nsf_hop_frames(int64_t n, int32_t F, int32_t H) {
  if (H <= 0) return 0;
  const int64_t padded = n + 2 * static_cast<int64_t>(F / 2);
  if (padded < F) return 0;
  return 1 + (padded - F) / H;
}

int64_t nsf_feature_rows(int64_t n, int32_t F, int32_t H) {
  return (nsf_hop_frames(n, F, H) + 1) / 2;
}

nsf_status nsf_row_offsets(int32_t F, int32_t H, const int64_t* clip_offsets, int32_t n_clips, uint32_t flags,
                           int64_t* row_offsets) {
  if (!clip_offsets || !row_offsets || n_clips < 0 || F <= 0 || H <= 0) return NSF_ERR_BAD_ARG;
  row_offsets[0] = 0;
  for (int32_t i = 0; i < n_clips; ++i) {
    const int64_t len = clip_offsets[i + 1] - clip_offsets[i];
    if (len < 0) return NSF_ERR_BAD_ARG;
    int64_t rows;
    nsf::clip_frames(len, F, H, flags, &rows);
    row_offsets[i + 1] = row_offsets[i] + rows;
  }
  return NSF_OK;
}

int64_t nsf_collect_rows(int64_t n_audio, int64_t n_facial, uint32_t flags, int32_t blend_frames) {
  if (n_audio < 0 || n_facial < 0) return -1;
  const int64_t n = std::min(n_audio, n_facial);
  int64_t total = n;
  const bool blend = (flags & NSF_COLLECT_BLEND) != 0;
  int64_t extra[2];
  int ne = 0;
  if (flags & NSF_COLLECT_FAST) extra[ne++] = (n + 1) / 2;
  if (flags & NSF_COLLECT_SLOW) extra[ne++] = n > 0 ? 2 * n - 1 : 0;
  for (int i = 0; i < ne; ++i) {
    int64_t nb = blend ? std::min<int64_t>(std::min<int64_t>(blend_frames, total), extra[i]) : 0;
    if (nb < 0) nb = 0;
    total += extra[i] - nb;
  }
  return total;
}

nsf_status nsf_plan_create(int32_t sr, int32_t F, int32_t H, int32_t n_mfcc, int32_t n_mels,
                           int32_t n_lags, nsf_plan** out) {
  if (!out) {
    nsf::set_error("nsf_plan_create: out_plan is NULL");
    return NSF_ERR_BAD_ARG;
  }
  *out = nullptr;
  nsf_plan* pl = new nsf_plan();
  nsf_status st = nsf::build_plan(sr, F, H, n_mfcc, n_mels, n_lags, &pl->p);
  if (st != NSF_OK) {
    delete pl;
    return st;
  }
  *out = pl;
  return NSF_OK;
}

void nsf_plan_destroy(nsf_plan* plan) { delete plan; }

int32_t nsf_feature_cols(const nsf_plan* plan, uint32_t flags) {
  if (!plan) return -1;
  const nsf::Plan& p = plan->p;
  int cols = (flags & NSF_NO_MFCC) ? 0 : p.n_mfcc * ((flags & NSF_NO_DELTAS) ? 1 : 3);
  if (!(flags & NSF_NO_AUTOCORR)) cols += p.n_lags * ((flags & NSF_AC_DELTAS) ? 3 : 1);
  return cols;
}

int64_t nsf_plan_table(const nsf_plan* plan, int32_t which, float* dst, int64_t cap) {
  if (!plan) return -1;
  const std::vector<float>* v = nullptr;
  switch (which) {
    case NSF_TABLE_MEL: v = &plan->p.mel_dense; break;
    case NSF_TABLE_DCT: v = &plan->p.dct; break;
    case NSF_TABLE_HANN_SYM: v = &plan->p.hann_sym; break;
    case NSF_TABLE_HANN_PER: v = &plan->p.hann_per; break;
    default: return -1;
  }
  const int64_t n = static_cast<int64_t>(v->size());
  if (dst && cap > 0) std::memcpy(dst, v->data(), sizeof(float) * std::min(n, cap));
  return n;
}

int32_t nsf_plan_info(const nsf_plan* plan, int32_t* bins, int32_t* chains, int32_t* fold_k,
                      int32_t* fold_kp) {
  if (!plan) return -1;
  if (bins) *bins = plan->p.bins;
  if (chains) *chains = plan->p.chains;
  if (fold_k) *fold_k = plan->p.chain[0].k;
  if (fold_kp) *fold_kp = plan->p.chain[0].kp;
  return 0;
}

nsf_status nsf_plan_fold_check(const nsf_plan* plan, const float* frame, double* re, double* im) {
  if (!plan || !frame || !re || !im) {
    nsf::set_error("nsf_plan_fold_check: NULL argument");
    return NSF_ERR_BAD_ARG;
  }
  const nsf::Plan& p = plan->p;
  for (int c = 0; c < p.chains; ++c) {
    const nsf::FoldChain& ch = p.chain[c];
    std::vector<double> in[2];
    for (int part = 0; part < 2; ++part) {
      in[part].assign(ch.kp, 0.0);
      for (int j = 0; j < ch.kp; ++j) {
        double acc = 0.0;
        for (int t = 0; t < nsf::kFoldTaps; ++t) {
          const size_t o = (static_cast<size_t>(part) * nsf::kFoldTaps + t) * ch.kp + j;
          acc += static_cast<double>(ch.tap_coef[o]) * static_cast<double>(frame[ch.tap_idx[o]]);
        }
        in[part][j] = acc;
      }
    }
    for (int m = 0; m < ch.nbins; ++m) {
      double sr_ = 0.0, si_ = 0.0;
      for (int j = 0; j < ch.kp; ++j) {
        sr_ += in[0][j] * ch.mat[0][static_cast<size_t>(j) * ch.np + m];
        si_ += in[1][j] * ch.mat[1][static_cast<size_t>(j) * ch.np + m];
      }
      re[ch.bin[m]] = sr_;
      im[ch.bin[m]] = si_;
    }
  }
  return NSF_OK;
}


int64_t nsf_resample_len(int64_t n_in, int32_t orig_sr, int32_t target_sr) {
  nsf::ResampleDesign d;
  if (n_in <= 0 || !nsf::design_resampler(orig_sr, target_sr, &d)) return 0;
  const int64_t n_up = n_in * d.up;
  return n_up / d.down + (n_up % d.down != 0);
}

int64_t nsf_resample_design(int32_t orig_sr, int32_t target_sr, double* taps, int64_t capacity, int32_t* up,
                            int32_t* down, int32_t* n_pre_pad, int32_t* n_pre_remove) {
  return nsf_resample_design_q(orig_sr, target_sr, NSF_RESAMPLE_POLY, taps, capacity, up, down, n_pre_pad, n_pre_remove);
}

int64_t nsf_resample_design_q(int32_t orig_sr, int32_t target_sr, int32_t quality, double* taps, int64_t capacity,
                              int32_t* up, int32_t* down, int32_t* n_pre_pad, int32_t* n_pre_remove) {
  nsf::ResampleDesign d;
  if (quality != NSF_RESAMPLE_POLY && quality != NSF_RESAMPLE_HQ) { nsf::set_error("nsf_resample_design_q: unknown quality"); return 0; }
  const bool ok = quality == NSF_RESAMPLE_HQ ? nsf::design_resampler_hq(orig_sr, target_sr, &d)
                                             : nsf::design_resampler(orig_sr, target_sr, &d);
  if (!ok) { nsf::set_error("nsf_resample_design: rates must be positive"); return 0; }
  if (up) *up = d.up;
  if (down) *down = d.down;
  if (n_pre_pad) *n_pre_pad = d.n_pre_pad;
  if (n_pre_remove) *n_pre_remove = d.n_pre_remove;
  const int64_t n = static_cast<int64_t>(d.h.size());
  if (taps) for (int64_t i = 0; i < n && i < capacity; ++i) taps[i] = d.h[i];
  return n;
}

}  // extern "C"

// Per-thread phases of the fused waveform -> log-mel kernel (logmel.cu).
//
// A frame of n_fft = 1024 real samples is transformed by ONE group of 64
// threads: z[n] = x[2n] + i x[2n+1] (512 complex points), a 512-point complex
// FFT as three register-resident radix-8 passes (512 = 8*8*8) with two
// shared-memory exchanges, then the real-input split that yields the 513
// power bins, then the banded mel projection, log and normalisation.
//
// Every phase (logmel_fft.cuh) is a __host__ __device__ function of (thread index in group,
// group-private shared buffers), so the exact index arithmetic the kernel runs
// is also executed on the CPU by tests/emul/logmel_emul.cu (64 threads looped
// per phase).  Index derivation, with W_n = exp(-2 pi i / n):
//   n = j + 64 r,  k = q + 8 p:   Z[q + 8p] = sum_j W_64^{jp} ( W_512^{jq} sum_r z[j+64r] W_8^{rq} )
//   j = j0 + 8 j1, p = p0 + 8 p1: U_q[p0 + 8 p1] = sum_j0 W_8^{j0 p1} ( W_64^{j0 p0} sum_j1 u_q[j0+8j1] W_8^{j1 p0} )
//   phase A: thread j      holds r = 0..7   -> q;   twiddle W_512^{jq}
//   phase B: thread q+8*j0 holds j1 = 0..7  -> p0;  twiddle W_64^{j0 p0}
//   phase C: thread q+8*p0 holds j0 = 0..7  -> p1;  Z[t + 64 p1], natural order
//   phase D: X[k] = E + W_1024^k O,  X[512-k] = conj(E - W_1024^k O),
//            E = (Z[k] + conj Z[512-k])/2,  O = (Z[k] - conj Z[512-k])/(2i)
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define AFS_HD __host__ __device__ __forceinline__
#else
#define AFS_HD inline
#endif

namespace afs {
namespace logmel {

constexpr int kNfft = 1024;
constexpr int kHalf = 512;        // complex FFT length
constexpr int kBins = 513;        // n_fft/2 + 1
constexpr int kGroup = 64;        // threads per frame
constexpr int kMaxMels = 128;
constexpr int kBufA = 2 * 8 * 68;  // floats: re/im of exchange 1; reused (natural order) by exchange 3
constexpr int kBufB = 2 * kHalf;          // floats: re/im of exchange 2; reused by the 513 power bins
static_assert(kBufA >= 2 * kHalf, "exchange 3 must fit in buffer A");
static_assert(kBufB >= kBins, "power bins must fit in buffer B");

struct cpx {
  float re, im;
};

// Per-thread twiddle BASES, held in registers for the whole kernel; the powers each phase needs are rebuilt per
// frame with complex multiplications (the FMA pipe has headroom, the shared-memory pipe is the kernel's limiter):
//   a  = W_512^j          phase A uses a^q,  q = 1..7
//   b  = W_64^(t >> 3)    phase B uses b^p0, p0 = 1..7
//   d  = W_1024^t         phase D uses d * W_16^m, m = 0..3
struct ThreadTw {
  cpx a, b, d;
};

// tw1024[k] = (cos(2 pi k/1024), -sin(2 pi k/1024)), k in [0, 1024)
AFS_HD void load_thread_tw(ThreadTw& tw, int t, const float2* tw1024) {
  const float2 wa = tw1024[(2 * t) & 1023], wb = tw1024[(16 * (t >> 3)) & 1023], wd = tw1024[t];
  tw.a.re = wa.x; tw.a.im = wa.y;
  tw.b.re = wb.x; tw.b.im = wb.y;
  tw.d.re = wd.x; tw.d.im = wd.y;
}

// Reflect padding index (torch.stft center=True, pad_mode="reflect"); needs pad < L.
AFS_HD int64_t reflect_index(int64_t idx, int64_t L) {
  if (idx < 0) idx = -idx;
  if (idx >= L) idx = 2 * (L - 1) - idx;
  return idx;
}

// The mel projection runs for kMelBatch frames at once (their power spectra kPStride floats apart): one weight
// load feeds kMelBatch FMAs (mel_dot_batch_p in logmel_fft.cuh).
constexpr int kMelBatch = 4;
constexpr int kPStride = 516;  // 513 power bins, padded to a multiple of 4 floats

// log_mult * log10(e) = (log_mult * log10(2)) * log2(e); on the device log2 is the MUFU.LG2 approximation
// (abs error 2^-22 near 1, 2 ulp elsewhere: far inside the 1e-4 dB tolerance), on the host log2f.
AFS_HD float fast_log2(float x) {
#if defined(__CUDA_ARCH__)
  return __log2f(x);
#else
  return log2f(x);
#endif
}

// normalised log-mel value: (log_mult*log10(e + eps) - mean) / std, with scale = log_mult*log10(2)/std and
// shift = -mean/std precomputed per mel bin.
AFS_HD float norm_db(float e, float eps, float scale, float shift) {
  return fast_log2(e + eps) * scale + shift;
}

// Host-side packing of a dense [bins, n_mels] filterbank (bins = n_fft/2 + 1) into per-filter spans:
// band[m] = first non-zero bin, band[kMaxMels+m] = span length, band[2*kMaxMels+m] = offset
// into `weights`.  Returns the number of packed weights.
template <typename IntVec, typename FloatVec>
inline int pack_mel_bands(const float* fb, int n_mels, int bins, IntVec& band, FloatVec& weights) {
  band.assign(3 * kMaxMels, 0);
  weights.clear();
  for (int m = 0; m < n_mels; ++m) {
    int lo = -1, hi = -1;
    for (int k = 0; k < bins; ++k) {
      if (fb[static_cast<size_t>(k) * n_mels + m] != 0.f) {
        if (lo < 0) lo = k;
        hi = k;
      }
    }
    const int len = lo < 0 ? 0 : hi - lo + 1;
    band[m] = lo < 0 ? 0 : lo;
    band[kMaxMels + m] = len;
    band[2 * kMaxMels + m] = static_cast<int>(weights.size());
    for (int i = 0; i < len; ++i) weights.push_back(fb[static_cast<size_t>(lo + i) * n_mels + m]);
  }
  return static_cast<int>(weights.size());
}
template <typename IntVec, typename FloatVec>
inline int pack_mel_bands(const float* fb, int n_mels, IntVec& band, FloatVec& weights) {
  return pack_mel_bands(fb, n_mels, kBins, band, weights);
}

// Shared-memory wavefronts of one warp-pass of the mel projection for one frame: in iteration i lane l reads power
// bin start[l] + i when i < n[l] (all lanes execute iteration i in the same instruction).
//   kBanks32: one 32-bit word per bin (radix-8 engine) -- an instruction costs as many wavefronts as the largest
//             number of DISTINCT words that fall on one of the 32 banks;
//   kBanks64: one 64-bit word per bin, the powers of a frame PAIR side by side (pair engine) -- the access is served
//             per half-warp on 16 eight-byte banks, the cost is the sum over the two half-warps.
enum MelBankModel { kBanks32 = 0, kBanks64 = 1 };
inline int mel_read_wavefronts(const int (&start)[32], const int (&n)[32], MelBankModel model = kBanks32) {
  const int group = model == kBanks32 ? 32 : 16;
  int total = 0;
  for (int i = 0;; ++i) {
    bool any = false;
    for (int g0 = 0; g0 < 32; g0 += group) {
      int words[32][32], cnt[32] = {0}, worst = 0;
      for (int l = g0; l < g0 + group; ++l) {
        if (i >= n[l]) continue;
        any = true;
        const int a = start[l] + i, b = a & (group - 1);
        bool seen = false;
        for (int j = 0; j < cnt[b]; ++j) seen = seen || words[b][j] == a;
        if (!seen) words[b][cnt[b]++] = a;
        if (cnt[b] > worst) worst = cnt[b];
      }
      total += worst;
    }
    if (!any) break;
  }
  return total;
}

// The kernel's weight table (ELL layout): thread t of a 64-thread frame group owns filter t (pass 0) and filter
// n_mels-1-t when that is >= 64 (pass 1).  The 32 lanes of a warp read weight i of their filter in the same
// instruction, so the table is stored [warp-pass][i][lane] (zero padded to the longest filter of the warp-pass):
// every weight load is one conflict-free wavefront.
// The POWER reads of that instruction are bins start_l + i with a different start_l per lane; the upper slaney
// filters start 6-12 bins apart, which as it stands puts up to 4 lanes on one bank (102 wavefronts per frame for 43
// instructions).  A filter shorter than the longest one of its warp-pass has slack: it may begin r iterations
// late, i.e. read from bin lo - r with r leading zero weights, which moves its bank by -r in EVERY iteration
// without touching the summation order of its non-zero terms.  The shifts are chosen here, once per plan, by a
// deterministic local search on mel_read_wavefronts (47 wavefronts per frame for the 128-mel slaney bank).
//   band[m] = first bin READ (lo - r), band[kMaxMels+m] = iterations (r + span length),
//   band[2*kMaxMels+m] = index of the filter's table entry 0; consecutive entries are kEllStride apart.
constexpr int kEllStride = 32;
template <typename IntVec, typename FloatVec>
inline int pack_mel_ell(const float* fb, int n_mels, int bins, IntVec& band, FloatVec& weights,
                        MelBankModel model = kBanks32) {
  IntVec b0;
  FloatVec w0;
  pack_mel_bands(fb, n_mels, bins, b0, w0);
  band.assign(3 * kMaxMels, 0);
  weights.clear();
  for (int pass = 0; pass < 2; ++pass) {
    for (int warp = 0; warp < kGroup / 32; ++warp) {
      int filt[32], lo[32], len[32], maxlen = 0;
      for (int lane = 0; lane < 32; ++lane) {
        const int t = warp * 32 + lane;
        int m = pass == 0 ? (t < n_mels ? t : -1) : (n_mels - 1 - t >= kGroup ? n_mels - 1 - t : -1);
        filt[lane] = m;
        lo[lane] = m >= 0 ? b0[m] : 0;
        len[lane] = m >= 0 ? b0[kMaxMels + m] : 0;
        if (len[lane] > maxlen) maxlen = len[lane];
      }
      // start shifts: r <= maxlen - len (the table does not grow) and r <= lo (the first bin read exists)
      int shift[32] = {0}, start[32], n[32];
      for (int lane = 0; lane < 32; ++lane) { start[lane] = lo[lane]; n[lane] = len[lane]; }
      int best = mel_read_wavefronts(start, n, model);
      const int floor_cost = model == kBanks32 ? maxlen : 2 * maxlen;
      uint32_t rng = 0x9E3779B9u + static_cast<uint32_t>(pass * 2 + warp);
      for (int it = 0; it < 6000 && best > floor_cost; ++it) {
        rng = rng * 1664525u + 1013904223u;
        const int lane = static_cast<int>((rng >> 8) & 31u);
        if (len[lane] == 0) continue;
        int room = maxlen - len[lane];
        if (lo[lane] < room) room = lo[lane];
        if (room == 0) continue;
        rng = rng * 1664525u + 1013904223u;
        const int cand = static_cast<int>((rng >> 8) % static_cast<uint32_t>(room + 1));
        const int old = shift[lane];
        if (cand == old) continue;
        start[lane] = lo[lane] - cand; n[lane] = len[lane] + cand;
        const int c = mel_read_wavefronts(start, n, model);
        if (c <= best) {  // sideways moves are accepted: the landscape is full of plateaus
          best = c; shift[lane] = cand;
        } else {
          start[lane] = lo[lane] - old; n[lane] = len[lane] + old;
        }
      }
      const int base = static_cast<int>(weights.size());
      weights.resize(weights.size() + static_cast<size_t>(maxlen) * kEllStride, 0.f);
      for (int lane = 0; lane < 32; ++lane) {
        const int m = filt[lane];
        if (m < 0) continue;
        band[m] = lo[lane] - shift[lane];
        band[kMaxMels + m] = len[lane] + shift[lane];
        band[2 * kMaxMels + m] = base + lane;
        for (int i = 0; i < len[lane]; ++i)
          weights[base + (shift[lane] + i) * kEllStride + lane] = w0[b0[2 * kMaxMels + m] + i];
      }
    }
  }
  return static_cast<int>(weights.size());
}
template <typename IntVec, typename FloatVec>
inline int pack_mel_ell(const float* fb, int n_mels, IntVec& band, FloatVec& weights, MelBankModel model = kBanks32) {
  return pack_mel_ell(fb, n_mels, kBins, band, weights, model);
}

}  // namespace logmel
}  // namespace afs

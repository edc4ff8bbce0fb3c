// CPU emulation of the n_fft 512 / 2048 log-mel kernel's per-thread phases (host logic test).
//
// Runs the SAME __host__ __device__ phase functions the kernel runs (audio_fewshot_b200/csrc/logmel_nfft.cuh) with the
// 64 threads of a frame group looped sequentially per phase (the loop boundary plays the role of bar.sync), and the
// mel projection exactly as logmel_nfft.cu issues it.  Built by tests/test_logmel_nfft_emul.py with `nvcc -x cu`.
#include <math.h>
#include <stdint.h>

#include <vector>

#include "logmel_core.cuh"
#include "logmel_fft.cuh"
#include "logmel_nfft.cuh"

using namespace afs::logmel;

template <int N>
static int emul_impl(const float* wav, int64_t L, int hop, int center, const float* fb, const float* window, int n_mels,
                     const float* mean, const float* stdv, float log_mult, float log_eps, float* out /*[n_mels, T]*/,
                     float* power_out /*[T, N/2+1] nullable*/) {
  using C = Nfft<N>;
  constexpr int R = C::kR;
  std::vector<int> band;
  std::vector<float> weights;
  pack_mel_ell(fb, n_mels, C::kBins, band, weights);
  std::vector<float2> tw(N);
  for (int k = 0; k < N; ++k) {
    const double a = 6.283185307179586476925286766559 * k / N;
    tw[k] = make_float2(static_cast<float>(cos(a)), static_cast<float>(-sin(a)));
  }
  const int pad = center ? N / 2 : 0;
  const int T = center ? static_cast<int>(1 + L / hop) : static_cast<int>(1 + (L - N) / hop);
  std::vector<float> bufA(C::kBufA), bufB(C::kBufB), bufP(kMelBatch * C::kPStride, 0.f);
  std::vector<NfftTw<N>> tws(kGroup);
  for (int t = 0; t < kGroup; ++t) load_nfft_tw<N>(tws[t], t, tw.data());
  float2* a2 = reinterpret_cast<float2*>(bufA.data());
  float2* b2 = reinterpret_cast<float2*>(bufB.data());
  for (int f = 0; f < T; ++f) {
    const int64_t s0 = static_cast<int64_t>(f) * hop - pad;
    const bool interior = s0 >= 0 && s0 + N <= L;
    for (int t = 0; t < kGroup; ++t) {
      float2 zp[R];
      for (int r = 0; r < R; ++r) {
        const int n = t + 64 * r;
        int64_t i0 = s0 + 2 * n, i1 = i0 + 1;
        if (!interior) { i0 = reflect_index(i0, L); i1 = reflect_index(i1, L); }
        zp[r] = make_float2(wav[i0] * window[2 * n], wav[i1] * window[2 * n + 1]);
      }
      nfft_phase_a<N>(t, zp, tws[t], a2);
    }
    const int slot = f % kMelBatch;
    float* power = bufP.data() + slot * C::kPStride;
    for (int t = 0; t < kGroup; ++t) nfft_phase_b<N>(t, tws[t], a2, b2);
    for (int t = 0; t < kGroup; ++t) nfft_phase_c<N>(t, b2, a2);
    for (int t = 0; t < kGroup; ++t) nfft_phase_d<N>(t, tws[t], a2, power);
    if (power_out) for (int k = 0; k < C::kBins; ++k) power_out[static_cast<size_t>(f) * C::kBins + k] = power[k];
    if (slot != kMelBatch - 1 && f + 1 != T) continue;
    for (int t = 0; t < kGroup; ++t) {
      const int mel_id[2] = {t < n_mels ? t : -1, n_mels - 1 - t >= kGroup ? n_mels - 1 - t : -1};
      for (int i = 0; i < 2; ++i) {
        const int m = mel_id[i];
        if (m < 0) continue;
        float acc[kMelBatch];
        mel_dot_batch_p<C::kPStride>(bufP.data(), weights.data() + band[2 * kMaxMels + m], kEllStride, band[m],
                                     band[kMaxMels + m], acc);
        const float scale = log_mult * 0.30102999566398120f / stdv[m];
        const float shift = -mean[m] / stdv[m];
        for (int b = 0; b <= slot; ++b)
          out[static_cast<size_t>(m) * T + (f - slot) + b] = norm_db(acc[b], log_eps, scale, shift);
      }
    }
  }
  return T;
}

extern "C" int emul_logmel_nfft(int n_fft, const float* wav, int64_t L, int hop, int center, const float* fb,
                                const float* window, int n_mels, const float* mean, const float* stdv, float log_mult,
                                float log_eps, float* out, float* power_out) {
  if (n_fft == 512) return emul_impl<512>(wav, L, hop, center, fb, window, n_mels, mean, stdv, log_mult, log_eps, out, power_out);
  if (n_fft == 2048) return emul_impl<2048>(wav, L, hop, center, fb, window, n_mels, mean, stdv, log_mult, log_eps, out, power_out);
  return -1;
}

// Worst number of distinct words that one access group puts on one bank, over every shared-memory access pattern of the
// phases (1 = conflict-free): 64-bit accesses are served per half-warp on 16 eight-byte banks, 32-bit ones (the power
// stores of phase D) per warp on 32 four-byte banks.  Lanes a phase leaves idle do not count.  -1 unless the
// exchange-2 slot function is a bijection onto [0, M) and every slot fits its buffer.
template <int N>
static int bank_check() {
  using C = Nfft<N>;
  constexpr int R = C::kR, M = C::kM;
  std::vector<char> seen(M, 0);
  for (int q = 0; q < R; ++q)
    for (int j0 = 0; j0 < 8; ++j0)
      for (int p0 = 0; p0 < 8; ++p0) {
        const int s = e2n_slot<N>(q, j0, p0);
        if (s < 0 || s >= M || seen[s]) return -1;
        seen[s] = 1;
      }
  if (e1n_slot<N>(R - 1, 63) >= C::kBufA / 2) return -1;
  int worst = 0;
  // addr(t) < 0: thread t is idle in this access
  auto access = [&](int group, auto addr) {
    for (int g0 = 0; g0 < kGroup; g0 += group) {
      int words[32][32], cnt[32] = {0};
      for (int l = g0; l < g0 + group; ++l) {
        const int a = addr(l);
        if (a < 0) continue;
        const int b = a & (group - 1);
        bool dup = false;
        for (int i = 0; i < cnt[b]; ++i) dup = dup || words[b][i] == a;
        if (!dup) words[b][cnt[b]++] = a;
        if (cnt[b] > worst) worst = cnt[b];
      }
    }
  };
  for (int r = 0; r < R; ++r) access(16, [&](int t) { return e1n_slot<N>(r, t); });  // phase A writes (q = r)
  for (int i = 0; i < C::kBflyPerThread; ++i) {
    auto live = [&](int t) { return t + 64 * i < C::kBfly; };
    for (int r = 0; r < 8; ++r) {
      access(16, [&](int t) { const int b = t + 64 * i; return live(t) ? e1n_slot<N>(b % R, b / R + 8 * r) : -1; });  // B reads
      access(16, [&](int t) { const int b = t + 64 * i; return live(t) ? e2n_slot<N>(b % R, b / R, r) : -1; });        // B writes
      access(16, [&](int t) { const int b = t + 64 * i; return live(t) ? e2n_slot<N>(b % R, r, b / R) : -1; });        // C reads
      access(16, [&](int t) { const int b = t + 64 * i; return live(t) ? b + C::kBfly * r : -1; });                   // C writes
    }
  }
  for (int m = 0; m < C::kDSteps; ++m) {
    access(16, [&](int t) { return t + 64 * m; });                      // phase D reads Z[k]
    access(16, [&](int t) { return (M - (t + 64 * m)) & (M - 1); });   // phase D reads Z[M - k]
    access(32, [&](int t) { return t + 64 * m; });                      // phase D writes power[k]
    access(32, [&](int t) { return M - (t + 64 * m); });                // phase D writes power[M - k]
  }
  return worst;
}

extern "C" int emul_nfft_bank_check(int n_fft) {
  if (n_fft == 512) return bank_check<512>();
  if (n_fft == 2048) return bank_check<2048>();
  return -1;
}

// The ELL weight table packed over `bins` power bins, expanded back to a dense [bins, n_mels] matrix; owner_count[m] =
// number of (thread, pass) pairs that own filter m.  Returns the table size in floats, -1 on a misplaced entry or a
// power read outside [0, bins).
extern "C" int emul_mel_ell_dense_n(const float* fb, int n_mels, int bins, float* dense, int* owner_count) {
  std::vector<int> band;
  std::vector<float> weights;
  const int n = pack_mel_ell(fb, n_mels, bins, band, weights);
  for (int i = 0; i < bins * n_mels; ++i) dense[i] = 0.f;
  for (int m = 0; m < n_mels; ++m) owner_count[m] = 0;
  for (int t = 0; t < kGroup; ++t) {
    const int ids[2] = {t < n_mels ? t : -1, n_mels - 1 - t >= kGroup ? n_mels - 1 - t : -1};
    for (int i = 0; i < 2; ++i) {
      const int m = ids[i];
      if (m < 0) continue;
      owner_count[m] += 1;
      const int lo = band[m], len = band[kMaxMels + m], off = band[2 * kMaxMels + m];
      if (off % kEllStride != (t & 31) || lo < 0 || lo + len > bins) return -1;
      for (int j = 0; j < len; ++j) {
        const float w = weights[off + j * kEllStride];
        if (w != 0.f) dense[(lo + j) * n_mels + m] = w;
      }
    }
  }
  return n;
}

// Per-thread phases of the log-mel kernel for n_fft 512 and 2048 (logmel_nfft.cu).
//
// One group of 64 threads transforms a frame of N real samples: z[n] = x[2n] + i x[2n+1] (M = N/2 complex points),
// an M-point complex FFT split as M = R * 64 -- a radix-R pass in registers (R = 16 at 2048, 4 at 512), then the
// 64-point sub-transforms as the 8 x 8 cross-thread structure of logmel_fft.cuh -- then the real-input split that
// yields the M + 1 power bins.  With W_n = exp(-2 pi i / n):
//   n = j + 64 r,  k = q + R p:   Z[q + R p] = sum_j W_64^{jp} ( W_M^{jq} sum_r z[j+64r] W_R^{rq} )
//   j = j0 + 8 j1, p = p0 + 8 p1: U_q[p0 + 8 p1] = sum_j0 W_8^{j0 p1} ( W_64^{j0 p0} sum_j1 u_q[j0+8j1] W_8^{j1 p0} )
//   phase A: thread j holds r = 0..R-1 -> q;  twiddle W_M^{jq}
//   phase B: butterfly b = q + R j0 holds j1 = 0..7 -> p0;  twiddle W_64^{j0 p0}
//   phase C: butterfly b = q + R p0 holds j0 = 0..7 -> p1;  Z[b + 8 R p1], natural order
//   phase D: X[k] = E + W_N^k O,  X[M-k] = conj(E - W_N^k O)   (as logmel_fft.cuh phase D)
// Phases B and C run 8 R radix-8 butterflies on 64 threads: two per thread at 2048 (b = t, t + 64), one on threads
// 0..31 at 512 (threads 32..63 idle in those two phases).
//
// Layouts (float2 units; a 64-bit access is served per half-warp on 16 eight-byte banks -- checked for every access
// pattern by tests/emul/logmel_nfft_emul.cu):
//   exchange 1: element (q, j) at q * (64 + 16 / R) + j     (the read side b = q + R j0 lands on 16 banks)
//   exchange 2: R = 16: element (q, j0, p0) at q + 16 (j0 + 8 p0);
//               R = 4:  at q + 4 ((j0 + p0) & 3) + 16 (j0 + 8 (p0 >> 2))   (both dense bijections on [0, M))
//   exchange 3: Z[k] at k (natural order)
#pragma once
#include "logmel_core.cuh"
#include "logmel_fft.cuh"

namespace afs {
namespace logmel {

template <int N>
struct Nfft {
  static_assert(N == 512 || N == 2048, "built for n_fft 512 and 2048 (1024 has its own engines)");
  static constexpr int kM = N / 2;                 // complex FFT length
  static constexpr int kR = kM / kGroup;           // points per thread in phase A
  static constexpr int kBins = kM + 1;             // power bins
  static constexpr int kBfly = 8 * kR;             // radix-8 butterflies per pass of phases B and C
  static constexpr int kBflyPerThread = kBfly >= kGroup ? kBfly / kGroup : 1;
  static constexpr int kDSteps = kM / 128;         // phase D: k = u + 64 m, m < kDSteps covers [0, M/2)
  static constexpr int kE1Stride = kGroup + 16 / kR;
  static constexpr int kBufA = 2 * (kR * kE1Stride > kM ? kR * kE1Stride : kM);  // floats: exchanges 1 and 3
  static constexpr int kBufB = 2 * kM;             // floats: exchange 2
  static constexpr int kPStride = (kBins + 3) & ~3;  // floats per power spectrum
  static constexpr int kGroupFloats = kBufA + kBufB + kMelBatch * kPStride;
  // floats of the ELL weight table: at 2048 the filters span twice the bins of n_fft 1024, and 64 / 80 slaney mels at
  // 32-48 kHz need up to 4 928 (128 mels: 3 168)
  static constexpr int kMaxNnz = N == 2048 ? 8192 : 4096;
  static_assert(kBfly % kGroup == 0 || kBfly == kGroup / 2, "butterflies fill the group or half of it");
};

template <int N>
struct NfftTw {
  float2 a;                               // W_M^t: phase A uses a^q, q = 1..R-1
  float2 b[Nfft<N>::kBflyPerThread];      // W_64^{j0} of each butterfly: phase B uses b^p0
  float2 d[Nfft<N>::kDSteps];             // W_N^{t + 64 m}
};

// twN[k] = (cos(2 pi k/N), -sin(2 pi k/N)), k in [0, N)
template <int N>
AFS_HD void load_nfft_tw(NfftTw<N>& tw, int t, const float2* twN) {
  using C = Nfft<N>;
  tw.a = twN[2 * t];
#pragma unroll
  for (int i = 0; i < C::kBflyPerThread; ++i) tw.b[i] = twN[((N / 64) * ((t + 64 * i) / C::kR)) & (N - 1)];
#pragma unroll
  for (int m = 0; m < C::kDSteps; ++m) tw.d[m] = twN[t + 64 * m];
}

// In-place forward R-point DFT, natural order out.
AFS_HD void dft4_p(float2 (&a)[4]) {
  const float2 b0 = p_add(a[0], a[2]), b1 = p_sub(a[0], a[2]);
  const float2 b2 = p_add(a[1], a[3]), b3 = c_negi(p_sub(a[1], a[3]));
  a[0] = p_add(b0, b2); a[2] = p_sub(b0, b2); a[1] = p_add(b1, b3); a[3] = p_sub(b1, b3);
}

// 16 = 2 x 8: DFT8 of the even and of the odd points, W_16^q on the odd half, one radix-2 stage.
AFS_HD void dft16_p(float2 (&a)[16]) {
  const float c1 = 0.92387953251128673848f, s1 = 0.38268343236508978178f, h = 0.70710678118654752440f;
  const float2 w16[8] = {make_float2(1.f, 0.f), make_float2(c1, -s1), make_float2(h, -h), make_float2(s1, -c1),
                         make_float2(0.f, -1.f), make_float2(-s1, -c1), make_float2(-h, -h), make_float2(-c1, -s1)};
  float2 e[8], o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { e[i] = a[2 * i]; o[i] = a[2 * i + 1]; }
  dft8_p(e);
  dft8_p(o);
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float2 t = q == 0 ? o[0] : (q == 4 ? c_negi(o[4]) : c_mul(o[q], w16[q]));
    a[q] = p_add(e[q], t);
    a[q + 8] = p_sub(e[q], t);
  }
}

// p[q] = w^q, q = 1..R-1 (products of at most four factors of w)
template <int R>
AFS_HD void powers_p(float2 w, float2 (&p)[R]) {
  p[1] = w;
  p[2] = c_mul(w, w);
  p[3] = c_mul(p[2], w);
  if constexpr (R == 16) {
    p[4] = c_mul(p[2], p[2]);
    p[5] = c_mul(p[4], w);
    p[6] = c_mul(p[4], p[2]);
    p[7] = c_mul(p[4], p[3]);
    p[8] = c_mul(p[4], p[4]);
#pragma unroll
    for (int q = 9; q < 16; ++q) p[q] = c_mul(p[8], p[q - 8]);
  }
}

template <int N>
AFS_HD int e1n_slot(int q, int j) { return q * Nfft<N>::kE1Stride + j; }
template <int N>
AFS_HD int e2n_slot(int q, int j0, int p0) {
  if constexpr (Nfft<N>::kR == 16) return q + 16 * (j0 + 8 * p0);
  else return q + 4 * ((j0 + p0) & 3) + 16 * (j0 + 8 * (p0 >> 2));
}

// Phase A. in: z[r] = windowed (x[2n], x[2n+1]) as (re, im), n = j + 64 r.
template <int N>
AFS_HD void nfft_phase_a(int j, float2 (&z)[Nfft<N>::kR], const NfftTw<N>& tw, float2* bufA) {
  constexpr int R = Nfft<N>::kR;
  if constexpr (R == 16) dft16_p(z);
  else dft4_p(z);
  bufA[e1n_slot<N>(0, j)] = z[0];
  float2 pw[R];
  powers_p<R>(tw.a, pw);
#pragma unroll
  for (int q = 1; q < R; ++q) bufA[e1n_slot<N>(q, j)] = c_mul(z[q], pw[q]);
}

// Phase B. butterflies b = t + 64 i: q = b % R, j0 = b / R.
template <int N>
AFS_HD void nfft_phase_b(int t, const NfftTw<N>& tw, const float2* bufA, float2* bufB) {
  using C = Nfft<N>;
#pragma unroll
  for (int i = 0; i < C::kBflyPerThread; ++i) {
    const int b = t + 64 * i;
    if (b >= C::kBfly) break;
    const int q = b % C::kR, j0 = b / C::kR;
    float2 v[8];
#pragma unroll
    for (int j1 = 0; j1 < 8; ++j1) v[j1] = bufA[e1n_slot<N>(q, j0 + 8 * j1)];
    dft8_p(v);
    float2 pw[8];
    powers7_p(tw.b[i], pw);
    bufB[e2n_slot<N>(q, j0, 0)] = v[0];
#pragma unroll
    for (int p0 = 1; p0 < 8; ++p0) bufB[e2n_slot<N>(q, j0, p0)] = c_mul(v[p0], pw[p0]);
  }
}

// Phase C. butterflies b = t + 64 i: q = b % R, p0 = b / R; leaves Z[b + 8 R p1] in natural order in buffer A.
template <int N>
AFS_HD void nfft_phase_c(int t, const float2* bufB, float2* bufA) {
  using C = Nfft<N>;
#pragma unroll
  for (int i = 0; i < C::kBflyPerThread; ++i) {
    const int b = t + 64 * i;
    if (b >= C::kBfly) break;
    const int q = b % C::kR, p0 = b / C::kR;
    float2 v[8];
#pragma unroll
    for (int j0 = 0; j0 < 8; ++j0) v[j0] = bufB[e2n_slot<N>(q, j0, p0)];
    dft8_p(v);
#pragma unroll
    for (int p1 = 0; p1 < 8; ++p1) bufA[b + C::kBfly * p1] = v[p1];
  }
}

// Phase D. thread u handles k = u + 64 m and its mirror M - k; thread 0 also the self-paired bin M/2.
template <int N>
AFS_HD void nfft_phase_d(int u, const NfftTw<N>& tw, const float2* bufA, float* power) {
  constexpr int M = Nfft<N>::kM;
#pragma unroll
  for (int m = 0; m < Nfft<N>::kDSteps; ++m) {
    const int k = u + 64 * m;
    const int kb = (M - k) & (M - 1);
    const float2 a = bufA[k];
    const float2 cb = c_conj(bufA[kb]);
    const float2 e2 = p_add(a, cb);           // 2E = A + conj(B)
    const float2 o2 = c_negi(p_sub(a, cb));   // 2O = (A - conj(B)) / i
    const float2 t2 = c_mul(o2, tw.d[m]);
    const float2 x = p_add(e2, t2), y = p_sub(e2, t2);
    power[k] = 0.25f * (x.x * x.x + x.y * x.y);
    power[M - k] = 0.25f * (y.x * y.x + y.y * y.y);
  }
  if (u == 0) {
    const float2 a = bufA[M / 2];
    power[M / 2] = a.x * a.x + a.y * a.y;
  }
}

}  // namespace logmel
}  // namespace afs

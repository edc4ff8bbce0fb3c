// Fused waveform -> normalised log-mel front-end at n_fft 512 and 2048 (8 kHz and 32-48 kHz audio at its own rate),
// plain and augmented launches alike.  Same stage and contract as logmel.cu: Philox gain / time-shift / noise ->
// reflect padding -> framing -> periodic window -> N-point real FFT -> power -> banded mel projection ->
// log_mult*log10(. + eps) -> (. - mean)/std -> [B, 1, n_mels, T], no spectrum in HBM; algorithmic bytes per clip
// 4*L + 4*n_mels*T (2*L + ... for int16 PCM).
//
// The frame-group structure of logmel.cu carries over: 64 threads per frame (thread t owns mel filters t and
// n_mels-1-t, ELL table and mel_dot_batch_p unchanged), 4 groups per CTA, work item = 32 consecutive frames of one
// clip with the [n_mels x 32] output tile staged in shared memory, persistent grid.  The FFT is logmel_nfft.cuh's
// radix-R register pass plus the 8 x 8 cross-thread passes.  Shared memory per group: exchange buffers A and B and
// kMelBatch power spectra (2048: 8.1 + 8 + 16.1 KB; 512: 2.1 + 2 + 4.1 KB); per CTA add the ELL table (32 KB at
// 2048, 16 KB at 512), the band table and the 16.5 KB output tile.  That is 179 KB at 2048 (one CTA of 256 threads per
// SM, 235 registers) and 66 KB at 512 (two CTAs per SM, launch-bounded to 128 registers).
#include <stdint.h>

#include "common.cuh"
#include "logmel_core.cuh"
#include "logmel_fft.cuh"
#include "logmel_nfft.cuh"
#include "logmel_plan.cuh"
#include "philox.cuh"

namespace afs {
namespace {

using namespace logmel;

constexpr int kThreads = 256;
constexpr int kGroups = kThreads / kGroup;
constexpr int kFramesPerCta = 32;
constexpr int kFramesPerGroup = kFramesPerCta / kGroups;
constexpr int kTileStride = kFramesPerCta + 1;

template <int N>
struct NfftKernel {
  static constexpr int kCtasPerSm = N == 2048 ? 1 : 2;
  static constexpr size_t kSmemBytes =
      (Nfft<N>::kMaxNnz + 3 * kMaxMels + static_cast<size_t>(kGroups) * Nfft<N>::kGroupFloats +
       kMaxMels * kTileStride) * sizeof(float);
};
static_assert(NfftKernel<2048>::kSmemBytes <= 227 * 1024, "one CTA per SM at 2048");
static_assert(2 * (NfftKernel<512>::kSmemBytes + 1024) <= 228 * 1024, "two CTAs per SM at 512");

__device__ __forceinline__ void group_bar(int grp) {
  asm volatile("bar.sync %0, 64;" ::"r"(grp + 1) : "memory");
}

// Raw (augmented, reflect-padded, not yet windowed) samples 2n, 2n+1 for n = t + 64 r of the frame that starts at
// sample s0, r = R0..R-1; R0 = R/2 loads only the second half (hop == n_fft/2 reuse).
template <typename S, int N, int R0>
__device__ __forceinline__ void load_frame_n(const S* __restrict__ x, int64_t s0, int64_t L, int t, const AugState& aug,
                                             float2 (&raw)[Nfft<N>::kR]) {
  const bool interior = (s0 >= 0) && (s0 + N <= L);
#pragma unroll
  for (int r = R0; r < Nfft<N>::kR; ++r) {
    int64_t i0 = s0 + 2 * (t + 64 * r), i1 = i0 + 1;
    if (!interior) {
      i0 = reflect_index(i0, L);
      i1 = reflect_index(i1, L);
    }
    if (interior && (i0 & 1) == 0) {
      raw[r] = aug_pair(x, i0, L, aug);
    } else {
      raw[r].x = aug_sample(x, i0, L, aug);
      raw[r].y = aug_sample(x, i1, L, aug);
    }
  }
}

template <int N, typename S>
__global__ void __launch_bounds__(kThreads, NfftKernel<N>::kCtasPerSm) logmel_nfft_kernel(const Params p) {
  using C = Nfft<N>;
  constexpr int R = C::kR;
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;
  int* s_band = reinterpret_cast<int*>(s_w + C::kMaxNnz);
  float* s_grp = reinterpret_cast<float*>(s_band + 3 * kMaxMels);
  float* s_tile = s_grp + kGroups * C::kGroupFloats;

  const int tid = threadIdx.x;
  const int grp = tid >> 6;
  const int t = tid & 63;

  for (int i = tid; i < p.nnz; i += kThreads) s_w[i] = p.weights[i];
  for (int i = tid; i < 3 * kMaxMels; i += kThreads) s_band[i] = p.band[i];

  NfftTw<N> tw;
  load_nfft_tw<N>(tw, t, p.tw1024);  // the plan's twiddle table has n_fft entries

  int mel_id[2];
  float mel_scale[2], mel_shift[2];
  mel_id[0] = (t < p.n_mels) ? t : -1;
  mel_id[1] = (p.n_mels - 1 - t >= kGroup) ? p.n_mels - 1 - t : -1;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float sd = mel_id[i] >= 0 ? p.stdv[mel_id[i]] : 1.f;
    const float mu = mel_id[i] >= 0 ? p.mean[mel_id[i]] : 0.f;
    mel_scale[i] = p.log_mult * 0.30102999566398120f / sd;
    mel_shift[i] = -mu / sd;
  }

  float* bufA = s_grp + grp * C::kGroupFloats;
  float* bufB = bufA + C::kBufA;
  float* bufP = bufB + C::kBufB;
  float2 win[R];
  {
    const float2* w2 = reinterpret_cast<const float2*>(p.window);
#pragma unroll
    for (int r = 0; r < R; ++r) win[r] = __ldg(w2 + t + 64 * r);
  }
  const bool half_overlap = p.hop * 2 == N;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  __syncthreads();

  const int n_items = p.B * p.chunks;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int clip = item / p.chunks;
    const int chunk = item - clip * p.chunks;
    const S* __restrict__ x = static_cast<const S*>(p.wav) + static_cast<int64_t>(clip) * p.L;

    AugState aug;
    aug.pcm_scale = p.pcm_scale;
    init_clip_aug(aug, p, clip);

    const int t0 = chunk * kFramesPerCta;
    const int nfr = min(kFramesPerCta, p.T - t0);
    const int f_begin = grp * kFramesPerGroup;
    const int f_end = min(f_begin + kFramesPerGroup, nfr);

    float2 raw[R];
    if (f_begin < f_end)
      load_frame_n<S, N, 0>(x, static_cast<int64_t>(t0 + f_begin) * p.hop - p.pad, p.L, t, aug, raw);

    for (int fl = f_begin; fl < f_end; ++fl) {
      float2 zp[R];
#pragma unroll
      for (int r = 0; r < R; ++r) zp[r] = p_mul(raw[r], win[r]);
      if (fl + 1 < f_end) {  // prefetch the next frame while this one is transformed
        const int64_t s_next = static_cast<int64_t>(t0 + fl + 1) * p.hop - p.pad;
        if (half_overlap) {  // its first half is this frame's second half
#pragma unroll
          for (int r = 0; r < R / 2; ++r) raw[r] = raw[r + R / 2];
          load_frame_n<S, N, R / 2>(x, s_next, p.L, t, aug, raw);
        } else {
          load_frame_n<S, N, 0>(x, s_next, p.L, t, aug, raw);
        }
      }
      const int slot = (fl - f_begin) % kMelBatch;
      float2* a2 = reinterpret_cast<float2*>(bufA);
      float2* b2 = reinterpret_cast<float2*>(bufB);
      nfft_phase_a<N>(t, zp, tw, a2);
      group_bar(grp);
      nfft_phase_b<N>(t, tw, a2, b2);
      group_bar(grp);
      nfft_phase_c<N>(t, b2, a2);
      group_bar(grp);
      nfft_phase_d<N>(t, tw, a2, bufP + slot * C::kPStride);
      group_bar(grp);
      if (slot == kMelBatch - 1 || fl + 1 == f_end) {
        const int fl0 = fl - slot;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int m = mel_id[i];
          if (m >= 0) {
            float acc[kMelBatch];
            mel_dot_batch_p<C::kPStride>(bufP, s_w + s_band[2 * kMaxMels + m], kEllStride, s_band[m],
                                         s_band[kMaxMels + m], acc);
#pragma unroll
            for (int f = 0; f < kMelBatch; ++f)
              if (f <= slot) s_tile[m * kTileStride + fl0 + f] = norm_db(acc[f], p.log_eps, mel_scale[i], mel_shift[i]);
          }
        }
      }
    }
    __syncthreads();

    if (lane < nfr) {
      float* o = p.out + (static_cast<int64_t>(clip) * p.n_mels) * p.T + t0 + lane;
      for (int m = warp; m < p.n_mels; m += kThreads / 32) {
        o[static_cast<int64_t>(m) * p.T] = s_tile[m * kTileStride + lane];
      }
    }
    __syncthreads();
  }
}

template <int N, typename S>
int launch_n(const Params& p, int64_t items, cudaStream_t stream) {
  const int64_t cap = static_cast<int64_t>(NfftKernel<N>::kCtasPerSm) * kNumSMs;
  const unsigned grid = static_cast<unsigned>(items < cap ? items : cap);
  logmel_nfft_kernel<N, S><<<grid, kThreads, NfftKernel<N>::kSmemBytes, stream>>>(p);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

template <int N>
cudaError_t prepare_n() {
  const int smem = static_cast<int>(NfftKernel<N>::kSmemBytes);
  cudaError_t e = cudaFuncSetAttribute(logmel_nfft_kernel<N, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(logmel_nfft_kernel<N, int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  return e;
}

}  // namespace

namespace logmel {

int nfft_max_nnz(int n_fft) { return n_fft == 2048 ? Nfft<2048>::kMaxNnz : Nfft<512>::kMaxNnz; }

cudaError_t nfft_prepare(int n_fft) {
  return n_fft == 2048 ? prepare_n<2048>() : prepare_n<512>();
}

template <typename S>
int nfft_launch(const afs_logmel_plan* plan, const Params& p, cudaStream_t stream) {
  const int64_t items = static_cast<int64_t>(p.B) * p.chunks;
  return plan->cfg.n_fft == 2048 ? launch_n<2048, S>(p, items, stream) : launch_n<512, S>(p, items, stream);
}
template int nfft_launch<float>(const afs_logmel_plan*, const Params&, cudaStream_t);
template int nfft_launch<int16_t>(const afs_logmel_plan*, const Params&, cudaStream_t);

}  // namespace logmel
}  // namespace afs

// Fused waveform -> normalised log-mel front-end for sm_100a: the plan, the C ABI entry points, and the radix-8
// engine, which serves augmented launches at n_fft 1024 (plain launches at 1024 run the pair engine of
// logmel_pair.cu; n_fft 512 and 2048 run logmel_nfft.cu).
//
// One launch does: Philox gain / time-shift / additive-noise
// augmentation -> reflect padding -> framing -> window -> 1024-point real FFT
// (512-point complex radix-8 x3 in registers + shared-memory exchanges) ->
// power -> banded mel projection -> log_mult*log10(. + eps) -> (. - mean)/std
// -> [B, 1, n_mels, T].  Spectra never leave the SM; HBM sees the waveform once
// (frame overlap is served by L1/L2) and the output once.  Algorithmic bytes
// per clip: 4*L + 4*n_mels*T (SURVEY.md 8d).
//
// CTA = 256 threads = 4 frame groups of 64 threads; a work item is 32
// consecutive frames of one clip (8 per group), whose [n_mels x 32] output tile
// is staged in shared memory so the global store is coalesced along time.  The
// grid is persistent (2 CTAs per SM walk the items): the mel weight table, band
// table, twiddle bases and window coefficients are staged once per CTA.  The mel filters
// are triangular (<= 2 filters per bin), so the projection is a banded fp32 dot
// product (1 009 non-zeros for 128 slaney mels) rather than a dense 513x128
// GEMM: exact fp32, ~20x fewer flops than the dense contraction.
//
// There is no reference implementation of this stage (SURVEY.md F2); the
// canonical spec is oracle/frontend.py.
#include <math.h>
#include <stdlib.h>

#include <new>
#include <vector>

#include "common.cuh"
#include "logmel_core.cuh"
#include "logmel_fft.cuh"
#include "logmel_plan.cuh"
#include "philox.cuh"

namespace afs {
namespace {

using namespace logmel;

constexpr int kThreads = 256;
constexpr int kGroups = kThreads / kGroup;
constexpr int kFramesPerCta = 32;
constexpr int kFramesPerGroup = kFramesPerCta / kGroups;
constexpr int kMaxNnz = 4096;  // floats of the ELL weight table (128 slaney mels: 1 440; 40 mels: 3 584)
constexpr int kTileStride = kFramesPerCta + 1;
constexpr int kGroupFloats = kBufA + kBufB + kMelBatch * kPStride;

constexpr size_t kSmemFloats = kMaxNnz + 3 * kMaxMels + kGroups * kGroupFloats +
                               kMaxMels * kTileStride;
constexpr size_t kSmemBytes = kSmemFloats * sizeof(float);

__device__ __forceinline__ void group_bar(int grp) {
  asm volatile("bar.sync %0, 64;" ::"r"(grp + 1) : "memory");
}

// Raw (augmented, reflect-padded, NOT yet windowed) samples 2n, 2n+1 for n = t + 64 r of the frame that
// starts at sample s0.  Issued one frame ahead of their use so the global-load latency hides behind the
// previous frame's FFT.
// R0 = 0 loads the whole frame, R0 = 4 only its second half (see the hop == n_fft/2 reuse in the kernel).
template <typename S, int R0>
__device__ __forceinline__ void load_frame(const S* __restrict__ x, int64_t s0, int64_t L, int t,
                                           const AugState& aug, float2 (&raw)[8]) {
  const bool interior = (s0 >= 0) && (s0 + kNfft <= L);
#pragma unroll
  for (int r = R0; r < 8; ++r) {
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

template <typename S>
__global__ void __launch_bounds__(kThreads, 2) logmel_kernel(const Params p) {
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;
  int* s_band = reinterpret_cast<int*>(s_w + kMaxNnz);
  float* s_grp = reinterpret_cast<float*>(s_band + 3 * kMaxMels);
  float* s_tile = s_grp + kGroups * kGroupFloats;

  const int tid = threadIdx.x;
  const int grp = tid >> 6;
  const int t = tid & 63;

  for (int i = tid; i < p.nnz; i += kThreads) s_w[i] = p.weights[i];
  for (int i = tid; i < 3 * kMaxMels; i += kThreads) s_band[i] = p.band[i];

  ThreadTw tw;
  load_thread_tw(tw, t, p.tw1024);

  // this thread's (up to) two mel filters: t and, mirrored for balance, n_mels-1-t
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

  float* bufA = s_grp + grp * kGroupFloats;
  float* bufB = bufA + kBufA;
  float* bufP = bufB + kBufB;  // kMelBatch power spectra
  // this thread's 16 window coefficients stay in registers for every frame (the shared-memory pipe is the limiter)
  float2 win[8];
  {
    const float2* w2 = reinterpret_cast<const float2*>(p.window);
#pragma unroll
    for (int r = 0; r < 8; ++r) win[r] = __ldg(w2 + t + 64 * r);
  }
  const bool half_overlap = p.hop * 2 == kNfft;  // consecutive frames share half of their (padded, augmented) samples
  const int lane = tid & 31;
  const int warp = tid >> 5;
  __syncthreads();

  // Persistent over (clip, chunk) items: the tables above are staged once per CTA, not once per 32 frames.
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

    float2 raw[8];
    if (f_begin < f_end) load_frame<S, 0>(x, static_cast<int64_t>(t0 + f_begin) * p.hop - p.pad, p.L, t, aug, raw);

    for (int fl = f_begin; fl < f_end; ++fl) {
      float2 zp[8];  // complex numbers as (re, im) register pairs, 64-bit exchanges (logmel_fft.cuh)
#pragma unroll
      for (int r = 0; r < 8; ++r) zp[r] = p_mul(raw[r], win[r]);
      if (fl + 1 < f_end) {  // prefetch the next frame while this one is transformed
        const int64_t s_next = static_cast<int64_t>(t0 + fl + 1) * p.hop - p.pad;
        if (half_overlap) {  // its first half is this frame's second half: sample index s_next + 2(t+64r) = s0 + 2(t+64(r+4))
#pragma unroll
          for (int r = 0; r < 4; ++r) raw[r] = raw[r + 4];
          load_frame<S, 4>(x, s_next, p.L, t, aug, raw);
        } else {
          load_frame<S, 0>(x, s_next, p.L, t, aug, raw);
        }
      }
      const int slot = (fl - f_begin) % kMelBatch;
      float2* a2 = reinterpret_cast<float2*>(bufA);
      float2* b2 = reinterpret_cast<float2*>(bufB);
      phase_a_p(t, zp, tw, a2);
      group_bar(grp);
      phase_b_p(t, tw, a2, b2);
      group_bar(grp);
      phase_c_p(t, b2, a2);
      group_bar(grp);
      phase_d_p(t, tw, a2, bufP + slot * kPStride);
      group_bar(grp);
      if (slot == kMelBatch - 1 || fl + 1 == f_end) {
        const int fl0 = fl - slot;  // first frame of this batch
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int m = mel_id[i];
          if (m >= 0) {
            float acc[kMelBatch];
            mel_dot_batch_p(bufP, s_w + s_band[2 * kMaxMels + m], kEllStride, s_band[m], s_band[kMaxMels + m], acc);
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
    __syncthreads();  // the tile is free before the next item's first mel batch writes it
  }
}

}  // namespace
}  // namespace afs

extern "C" int afs_logmel_plan_create(const afs_logmel_cfg* cfg, const float* fb_host,
                                      const float* window_host, int device,
                                      afs_logmel_plan** plan_out) {
  using namespace afs;
  if (cfg == nullptr || fb_host == nullptr || window_host == nullptr || plan_out == nullptr)
    return AFS_ERR_INVALID_ARG;
  if (cfg->hop < 1 || cfg->n_mels < 1) return AFS_ERR_INVALID_ARG;
  const int n_fft = cfg->n_fft;
  if ((n_fft != 512 && n_fft != kNfft && n_fft != 2048) || cfg->n_mels > kMaxMels) return AFS_ERR_UNSUPPORTED;

  std::vector<int> band;
  std::vector<float> weights;
  pack_mel_ell(fb_host, cfg->n_mels, n_fft / 2 + 1, band, weights);
  const int max_nnz = n_fft == kNfft ? kMaxNnz : logmel::nfft_max_nnz(n_fft);
  if (weights.size() > static_cast<size_t>(max_nnz)) return AFS_ERR_UNSUPPORTED;
  if (weights.empty()) weights.push_back(0.f);
  std::vector<int> band64;
  std::vector<float> weights64;
  pack_mel_ell(fb_host, cfg->n_mels, n_fft / 2 + 1, band64, weights64, logmel::kBanks64);
  weights64.resize(weights.size(), 0.f);  // same rows per warp-pass, only the start shifts differ

  std::vector<float2> tw(n_fft);
  const double two_pi = 6.283185307179586476925286766559;
  for (int k = 0; k < n_fft; ++k) {
    const double a = two_pi * k / n_fft;
    tw[k] = make_float2(static_cast<float>(cos(a)), static_cast<float>(-sin(a)));
  }

  afs_logmel_plan* plan = new (std::nothrow) afs_logmel_plan();
  if (plan == nullptr) return AFS_ERR_INVALID_ARG;
  plan->cfg = *cfg;
  plan->device = device;
  plan->nnz = static_cast<int>(weights.size());
  plan->d_window = nullptr; plan->d_tw1024 = nullptr; plan->d_band = nullptr; plan->d_weights = nullptr;
  plan->d_band64 = nullptr; plan->d_weights64 = nullptr;

  int prev = 0;
  cudaError_t e = cudaGetDevice(&prev);
  if (e == cudaSuccess) e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaMalloc(&plan->d_window, n_fft * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&plan->d_tw1024, n_fft * sizeof(float2));
  if (e == cudaSuccess) e = cudaMalloc(&plan->d_band, band.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&plan->d_weights, weights.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(plan->d_window, window_host, n_fft * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(plan->d_tw1024, tw.data(), n_fft * sizeof(float2), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(plan->d_band, band.data(), band.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(plan->d_weights, weights.data(), weights.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&plan->d_band64, band64.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&plan->d_weights64, weights64.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(plan->d_band64, band64.data(), band64.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(plan->d_weights64, weights64.data(), weights64.size() * sizeof(float), cudaMemcpyHostToDevice);
  const int smem = static_cast<int>(kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(logmel_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(logmel_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess) e = n_fft == kNfft ? logmel::pair_prepare() : logmel::nfft_prepare(n_fft);
  cudaSetDevice(prev);
  if (e != cudaSuccess) {
    afs_logmel_plan_destroy(plan);
    return cuda_fail(e);
  }
  *plan_out = plan;
  return AFS_OK;
}

extern "C" int afs_logmel_plan_destroy(afs_logmel_plan* plan) {
  if (plan == nullptr) return AFS_OK;
  cudaFree(plan->d_window);
  cudaFree(plan->d_tw1024);
  cudaFree(plan->d_band);
  cudaFree(plan->d_weights);
  cudaFree(plan->d_band64);
  cudaFree(plan->d_weights64);
  delete plan;
  return AFS_OK;
}

extern "C" int afs_logmel_num_frames(const afs_logmel_plan* plan, int64_t L) {
  if (plan == nullptr || L < 0) return AFS_ERR_INVALID_ARG;
  return afs::num_frames(plan->cfg, L);
}

namespace afs {
namespace {

template <typename S>
int logmel_launch(const afs_logmel_plan* plan, const S* wav, float pcm_scale, int32_t B, int64_t L, const float* mean,
                  const float* std, const afs_aug_cfg* aug, uint64_t seed, uint64_t first_clip_index, float* out,
                  afs_stream_t stream_) {
  if (plan == nullptr || wav == nullptr || mean == nullptr || std == nullptr || out == nullptr ||
      B < 0 || L < 1)
    return AFS_ERR_INVALID_ARG;
  const afs_logmel_cfg& cfg = plan->cfg;
  const int pad = cfg.center ? cfg.n_fft / 2 : 0;
  if (cfg.center && L <= pad) return AFS_ERR_INVALID_ARG;  // reflect padding needs pad < L
  if (aug != nullptr && (aug->max_shift < 0 || aug->noise_std_lo < 0.f || aug->noise_std_hi < aug->noise_std_lo ||
                         aug->gain_db_hi < aug->gain_db_lo))
    return AFS_ERR_INVALID_ARG;
  const int T = num_frames(cfg, L);
  if (B == 0 || T <= 0) return AFS_OK;

  Params p{};
  p.wav = wav; p.pcm_scale = pcm_scale; p.out = out; p.mean = mean; p.stdv = std;
  p.window = plan->d_window; p.tw1024 = plan->d_tw1024; p.band = plan->d_band; p.weights = plan->d_weights;
  p.L = L; p.nnz = plan->nnz; p.B = B; p.T = T; p.hop = cfg.hop; p.n_mels = cfg.n_mels; p.pad = pad;
  p.chunks = (T + kFramesPerCta - 1) / kFramesPerCta;
  p.log_mult = cfg.log_mult; p.log_eps = cfg.log_eps;
  const int64_t items = static_cast<int64_t>(B) * p.chunks;
  if (items > 0x7fffffffLL) return AFS_ERR_UNSUPPORTED;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (aug == nullptr && cfg.n_fft == kNfft) return logmel::pair_launch<S>(plan, p, stream);

  if (aug != nullptr) {  // a plain launch of the n_fft 512 / 2048 kernel keeps the zero ranges: gain 1, no shift, no noise
    p.gain_lo = aug->gain_db_lo; p.gain_hi = aug->gain_db_hi;
    p.noise_lo = aug->noise_std_lo; p.noise_hi = aug->noise_std_hi;
    p.max_shift = aug->max_shift;
  }
  p.seed_lo = static_cast<uint32_t>(seed); p.seed_hi = static_cast<uint32_t>(seed >> 32);
  p.first_clip = first_clip_index;
  if (cfg.n_fft != kNfft) return logmel::nfft_launch<S>(plan, p, stream);
  // persistent: 2 resident CTAs per SM (128 registers x 256 threads, 100 KB of shared memory each) walk the items
  const unsigned grid = static_cast<unsigned>(items < 2 * kNumSMs ? items : 2 * kNumSMs);
  logmel_kernel<S><<<grid, kThreads, kSmemBytes, stream>>>(p);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

}  // namespace
}  // namespace afs

extern "C" int afs_logmel_fwd(const afs_logmel_plan* plan, const float* wav, int32_t B, int64_t L,
                              const float* mean, const float* std, const afs_aug_cfg* aug,
                              uint64_t seed, uint64_t first_clip_index, float* out,
                              afs_stream_t stream) {
  return afs::logmel_launch<float>(plan, wav, 1.f, B, L, mean, std, aug, seed, first_clip_index, out, stream);
}

extern "C" int afs_logmel_fwd_pcm16(const afs_logmel_plan* plan, const int16_t* wav, float pcm_scale, int32_t B,
                                    int64_t L, const float* mean, const float* std, const afs_aug_cfg* aug,
                                    uint64_t seed, uint64_t first_clip_index, float* out,
                                    afs_stream_t stream) {
  return afs::logmel_launch<int16_t>(plan, wav, pcm_scale, B, L, mean, std, aug, seed, first_clip_index, out, stream);
}

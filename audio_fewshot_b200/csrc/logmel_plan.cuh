// Shared by the two engines of the fused waveform -> log-mel front-end (logmel.cu: radix-8 FFT, one frame per 64
// threads; logmel_pair.cu: two frames per warp as one 1024-point FFT): the plan, the kernel parameters, and the sample
// fetch with the Philox waveform augmentation.
#pragma once
#include <stdint.h>

#include "common.cuh"
#include "logmel_core.cuh"
#include "philox.cuh"

struct afs_logmel_plan {
  afs_logmel_cfg cfg;
  int device;
  int nnz;
  float* d_window;   // [n_fft]
  float2* d_tw1024;  // [n_fft]: (cos, -sin)(2 pi k / n_fft)
  int* d_band;       // [3][128]: lo, len, off
  float* d_weights;  // [nnz]
  int* d_band64;     // the same table with start shifts chosen for 64-bit power reads (pair engine)
  float* d_weights64;
};

namespace afs {
namespace logmel {

struct Params {  // tw1024 carries the plan's n_fft-point table; the name is the 1024-point engines'.
  const void* wav;     // [B, L] fp32, or int16 PCM when launched with T = int16_t
  float pcm_scale;     // int16 PCM only: sample = (float)pcm * pcm_scale (1/32768 for full-scale [-1, 1))
  float* out;
  const float* mean;
  const float* stdv;
  const float* window;
  const float2* tw1024;
  const int* band;
  const float* weights;
  int64_t L;
  int nnz, B, T, hop, n_mels, pad, chunks;
  float log_mult, log_eps;
  // augmentation
  float gain_lo, gain_hi, noise_lo, noise_hi;
  int max_shift;
  uint32_t seed_lo, seed_hi;
  uint64_t first_clip;
};

struct AugState {
  float g, sigma, pcm_scale;
  int k;
  uint32_t c_lo, c_hi, seed_lo, seed_hi;
};

// Sample fetch: fp32 waveforms as they are, int16 PCM converted on the fly (exact in fp32 for a
// power-of-two scale), so 16-bit audio crosses PCIe and HBM at half the bytes.
__device__ __forceinline__ float ld_sample(const float* p, float) { return __ldg(p); }
__device__ __forceinline__ float ld_sample(const int16_t* p, float s) {
  return __fmul_rn(static_cast<float>(__ldg(p)), s);
}

// One augmented sample y[idx] = g * x[idx - k] + sigma * n[idx]; n[2i], n[2i+1]
// are the (cos, sin) Box-Muller pair of the first two words of
// Philox(counter = (i, 1, clip_lo, clip_hi), key = seed).
template <typename S>
__device__ __forceinline__ float aug_sample(const S* __restrict__ x, int64_t idx, int64_t L,
                                            const AugState& a) {
  const int64_t src = idx - a.k;
  float v = (src >= 0 && src < L) ? __fmul_rn(a.g, ld_sample(x + src, a.pcm_scale)) : 0.f;
  if (a.sigma > 0.f) {
    u32x4 c;
    c.x = static_cast<uint32_t>(idx >> 1); c.y = kStreamNoise; c.z = a.c_lo; c.w = a.c_hi;
    const u32x4 r = philox4x32_10(c, a.seed_lo, a.seed_hi);
    const float rad = sqrtf(-2.0f * logf(u01(r.x)));
    float sn, cs;
    sincospif(2.0f * u01(r.y), &sn, &cs);
    const float z = (idx & 1) ? rad * sn : rad * cs;
    v = __fadd_rn(v, __fmul_rn(a.sigma, z));
  }
  return v;
}

// Both samples of an aligned pair (idx even, idx + 1): they share one Philox block and one Box-Muller draw
// (cos for the even sample, sin for the odd one), so the pair costs one RNG evaluation instead of two.
template <typename S>
__device__ __forceinline__ float2 aug_pair(const S* __restrict__ x, int64_t idx, int64_t L, const AugState& a) {
  const int64_t s0 = idx - a.k, s1 = s0 + 1;
  float2 v;
  v.x = (s0 >= 0 && s0 < L) ? __fmul_rn(a.g, ld_sample(x + s0, a.pcm_scale)) : 0.f;
  v.y = (s1 >= 0 && s1 < L) ? __fmul_rn(a.g, ld_sample(x + s1, a.pcm_scale)) : 0.f;
  if (a.sigma > 0.f) {
    u32x4 c;
    c.x = static_cast<uint32_t>(idx >> 1); c.y = kStreamNoise; c.z = a.c_lo; c.w = a.c_hi;
    const u32x4 r = philox4x32_10(c, a.seed_lo, a.seed_hi);
    const float rad = sqrtf(-2.0f * logf(u01(r.x)));
    float sn, cs;
    sincospif(2.0f * u01(r.y), &sn, &cs);
    v.x = __fadd_rn(v.x, __fmul_rn(a.sigma, rad * cs));
    v.y = __fadd_rn(v.y, __fmul_rn(a.sigma, rad * sn));
  }
  return v;
}

// per-clip augmentation parameters: gain, shift, noise level from Philox(counter = (0, 0, clip), key = seed)
__device__ __forceinline__ void init_clip_aug(AugState& aug, const Params& p, int clip) {
  const uint64_t cg = p.first_clip + static_cast<uint64_t>(clip);
  aug.c_lo = static_cast<uint32_t>(cg);
  aug.c_hi = static_cast<uint32_t>(cg >> 32);
  aug.seed_lo = p.seed_lo;
  aug.seed_hi = p.seed_hi;
  u32x4 c;
  c.x = 0u; c.y = kStreamParams; c.z = aug.c_lo; c.w = aug.c_hi;
  const u32x4 r = philox4x32_10(c, p.seed_lo, p.seed_hi);
  const float gain_db = __fadd_rn(p.gain_lo, __fmul_rn(__fsub_rn(p.gain_hi, p.gain_lo), u01(r.x)));
  aug.g = exp10f(__fmul_rn(gain_db, 0.05f));
  const int span = 2 * p.max_shift + 1;
  int draw = static_cast<int>(floorf(__fmul_rn(u01(r.y), static_cast<float>(span))));
  if (draw > span - 1) draw = span - 1;
  aug.k = draw - p.max_shift;
  aug.sigma = __fadd_rn(p.noise_lo, __fmul_rn(__fsub_rn(p.noise_hi, p.noise_lo), u01(r.z)));
}

inline int num_frames(const afs_logmel_cfg& cfg, int64_t L) {
  if (cfg.center) return static_cast<int>(1 + L / cfg.hop);
  if (L < cfg.n_fft) return 0;
  return static_cast<int>(1 + (L - cfg.n_fft) / cfg.hop);
}

// logmel_pair.cu
cudaError_t pair_prepare();
template <typename S>
int pair_launch(const afs_logmel_plan* plan, const Params& p, cudaStream_t stream);

// logmel_nfft.cu: n_fft 512 and 2048, plain and augmented launches
cudaError_t nfft_prepare(int n_fft);
int nfft_max_nnz(int n_fft);  // floats of the ELL weight table the kernel stages
template <typename S>
int nfft_launch(const afs_logmel_plan* plan, const Params& p, cudaStream_t stream);

}  // namespace logmel
}  // namespace afs

// Fused waveform -> normalised log-mel, warp-per-frame-pair engine for sm_100a: runs every launch without waveform
// augmentation.
//
// Same stage and same contract as logmel.cu (reflect padding -> framing -> window -> 1024-point real
// DFT -> power -> banded mel projection -> log -> normalise -> [B, 1, n_mels, T]; algorithmic bytes per clip
// 4 L + 4 n_mels T), different decomposition: a WARP transforms two frames at a time as one 1024-point complex FFT
// (logmel_pair.cuh) -- one shared-memory exchange per frame PAIR and an in-warp shuffle split instead of three
// exchanges per frame.  Everything a warp touches is private to it (exchange buffer, power planes, output tile), so
// after the tables are staged there is no CTA-wide or group barrier at all.
//
// One persistent CTA of 12 warps per SM (168 registers per thread: the register file is split per SM sub-partition,
// three warps of 168 x 32 registers fill one).  The frame pairs of the whole batch form one sequence (clip-major);
// every warp owns a contiguous run of it, equal to within one pair, so there is no tail.  Within a clip the pairs are
// grouped in chunks of 8 frames: the mel projection runs once per 4 frames (one weight load feeds four frames) and the
// chunk's [n_mels x 8] tile is staged in shared memory so that every global store instruction writes four 32-byte row
// pieces.  The samples of the next pair are fetched half-way through the split loop, when half of the transform's 64
// registers have retired (fetching before the transform spills at 168 registers; fetching register by register as
// the split loop retires values was measured and is slower: 0.69 against 0.58 ms per 3 200 clips).
#include <math.h>

#include "common.cuh"
#include "logmel_core.cuh"
#include "logmel_pair.cuh"
#include "logmel_plan.cuh"

namespace afs {
namespace {

using namespace logmel;

constexpr int kPWarps = 12;
constexpr int kPThreads = 32 * kPWarps;
constexpr int kPFrames = 8;          // frames per chunk (output tile)
constexpr int kPTileStride = 132;    // floats per tile column (frame): 132 = 4 mod 32 -> conflict-free 4-row x 8-frame reads
constexpr int kPWinStride = 36;      // floats per lane of the staged window: 128-bit reads of 8 lanes hit 8 different 16-byte banks
constexpr int kPExchFloats = 2 * kPairExch;
constexpr int kPPlaneFloats = 2 * kPStride;  // one power plane: a 64-bit word (frame pair) per bin
constexpr int kPWarpFloats = kPExchFloats + kPPlaneFloats + kPFrames * kPTileStride;
static_assert(kPExchFloats >= kPPlaneFloats, "the second pair's power plane aliases the exchange buffer");
static_assert(kPExchFloats % 2 == 0 && kPWarpFloats % 2 == 0, "8-byte alignment of the per-warp buffers");

inline size_t pair_smem_bytes(int nnz) {
  const size_t nnz_pad = (static_cast<size_t>(nnz) + 3) & ~static_cast<size_t>(3);
  return (nnz_pad + 3 * kMaxMels + 2 * kMaxMels + 32 * kPWinStride + static_cast<size_t>(kPWarps) * kPWarpFloats) * sizeof(float);
}

template <bool HALF>
struct RawN {
  static constexpr int n = HALF ? 48 : 64;   // HALF (hop == n_fft/2): frame b = frame a shifted by 16 values per lane
  static constexpr int boff = HALF ? 16 : 32;
};

// Interior pair: value m of the fetch list straight from memory.
template <typename S, bool HALF>
__device__ __forceinline__ float ld_fast(const S* xa, int hop, int m, float pcm_scale) {
  if (HALF || m < 32) return ld_sample(xa + 32 * m, pcm_scale);
  return ld_sample(xa + hop + 32 * (m - 32), pcm_scale);
}

// Raw (reflect-padded, not yet windowed) samples of the frame pair (fa, fa + 1) of one clip: lane l holds sample
// l + 32 m of frame a in raw[m] and of frame b in raw[boff + m].  M0 = 16 (HALF only): raw[0..15] were carried over
// from the previous pair.  The general path: clip edges (reflection), missing second frame.
template <typename S, bool HALF, int M0>
__device__ __forceinline__ void load_pair(const S* __restrict__ x, int64_t L, int64_t s0, int hop, bool b_exists, int lane,
                                          float pcm_scale, float (&raw)[RawN<HALF>::n]) {
  constexpr int n = RawN<HALF>::n;
  if (s0 >= 0 && s0 + (HALF ? 1536 : static_cast<int64_t>(hop) + kNfft) <= L) {  // interior pair
    const S* xa = x + s0 + lane;
#pragma unroll
    for (int m = M0; m < n; ++m) raw[m] = ld_fast<S, HALF>(xa, hop, m, pcm_scale);
    return;
  }
#pragma unroll
  for (int m = M0; m < n; ++m) {
    const bool of_b_only = m >= 32;
    int64_t idx = s0 + lane + (HALF ? 32 * m : (of_b_only ? hop + 32 * (m - 32) : 32 * m));
    float v = 0.f;
    if (!of_b_only || b_exists) {
      idx = reflect_index(idx, L);
      v = ld_sample(x + idx, pcm_scale);
    }
    raw[m] = v;
  }
}

template <typename S, bool HALF>
__global__ void __launch_bounds__(kPThreads, 1) logmel_pair_kernel(const Params p) {
  extern __shared__ __align__(16) float smem[];
  const int nnz_pad = (p.nnz + 3) & ~3;
  float* s_w = smem;
  int* s_band = reinterpret_cast<int*>(s_w + nnz_pad);
  float* s_scale = reinterpret_cast<float*>(s_band + 3 * kMaxMels);
  float* s_shift = s_scale + kMaxMels;
  float* s_win = s_shift + kMaxMels;  // [lane][kPWinStride]: 0.5 * window[lane + 32 n2] at n2

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;

  for (int i = tid; i < p.nnz; i += kPThreads) s_w[i] = p.weights[i];
  for (int i = tid; i < 3 * kMaxMels; i += kPThreads) s_band[i] = p.band[i];
  for (int i = tid; i < kMaxMels; i += kPThreads) {
    const float sd = i < p.n_mels ? p.stdv[i] : 1.f;
    const float mu = i < p.n_mels ? p.mean[i] : 0.f;
    s_scale[i] = p.log_mult * 0.30102999566398120f / sd;
    s_shift[i] = -mu / sd;
  }
  for (int i = tid; i < kNfft; i += kPThreads) s_win[(i & 31) * kPWinStride + (i >> 5)] = 0.5f * p.window[i];

  float* s_warp = s_win + 32 * kPWinStride + warp * kPWarpFloats;
  float2* exch = reinterpret_cast<float2*>(s_warp);
  float2* planeB = reinterpret_cast<float2*>(s_warp);                 // power of the second pair of a batch (aliases the exchange buffer)
  float2* planeA = reinterpret_cast<float2*>(s_warp + kPExchFloats);  // power of the first pair of a batch
  float* tile = s_warp + kPExchFloats + kPPlaneFloats;                // [frame][mel], kPTileStride floats per frame
  const float4* win4 = reinterpret_cast<const float4*>(s_win + lane * kPWinStride);
  const float2 w = __ldg(p.tw1024 + lane);                            // W_1024^lane
  __syncthreads();

  constexpr int NR = RawN<HALF>::n;
  constexpr int BOFF = RawN<HALF>::boff;

  // this warp's run of the pair sequence: pair g = clip * ppc + q covers frames 2q, 2q + 1 of `clip`
  const int ppc = (p.T + 1) >> 1;
  const int64_t n_pairs = static_cast<int64_t>(p.B) * ppc;
  const int64_t n_warps = static_cast<int64_t>(gridDim.x) * kPWarps;
  const int64_t gw = static_cast<int64_t>(blockIdx.x) * kPWarps + warp;
  const int64_t g_begin = gw * n_pairs / n_warps;
  const int64_t g_end = (gw + 1) * n_pairs / n_warps;
  int left = static_cast<int>(g_end - g_begin);
  if (left <= 0) return;
  int clip = static_cast<int>(g_begin / ppc);
  int q = static_cast<int>(g_begin - static_cast<int64_t>(clip) * ppc);
  int col_lo = 2 * (q & 3);  // first tile column this warp owns in its current chunk

  const float pcm_scale = p.pcm_scale;  // a local: p.pcm_scale at every load spills in the int16 HALF kernel
  float raw[NR];
  {
    const S* x = static_cast<const S*>(p.wav) + static_cast<int64_t>(clip) * p.L;
    load_pair<S, HALF, 0>(x, p.L, static_cast<int64_t>(2 * q) * p.hop - p.pad, p.hop, 2 * q + 1 < p.T, lane, pcm_scale, raw);
  }

  while (left > 0) {
    const int j = q & 3;                   // pair within the 8-frame chunk
    const int t0 = (q & ~3) * 2;           // first frame of the chunk
    const bool clip_end = q + 1 >= ppc;
    const bool last = j == 3 || clip_end || left == 1;  // last pair this warp transforms in this chunk

    float2 z[32];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 wv = win4[i];
      z[4 * i + 0] = make_float2(raw[4 * i + 0] * wv.x, raw[BOFF + 4 * i + 0] * wv.x);
      z[4 * i + 1] = make_float2(raw[4 * i + 1] * wv.y, raw[BOFF + 4 * i + 1] * wv.y);
      z[4 * i + 2] = make_float2(raw[4 * i + 2] * wv.z, raw[BOFF + 4 * i + 2] * wv.z);
      z[4 * i + 3] = make_float2(raw[4 * i + 3] * wv.w, raw[BOFF + 4 * i + 3] * wv.w);
    }

    // the next pair of this warp's run
    const bool have_next = left > 1;
    const int nclip = clip_end ? clip + 1 : clip;
    const int nq = clip_end ? 0 : q + 1;
    const bool carry = HALF && !clip_end;  // its first 16 values per lane are this pair's last 16
    if (carry) {
#pragma unroll
      for (int m = 0; m < 16; ++m) raw[m] = raw[32 + m];
    }

    pair_pass1(lane, z, w, exch);
    __syncwarp();
    pair_pass2(lane, exch, z);
    __syncwarp();

    float2* plane = (j & 1) ? planeB : planeA;
    const int partner = pair_partner(lane);
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) {
      if (k2 == 8 && have_next) {  // z[0..7] and z[24..31] have retired: room for the next pair's samples
        const S* nx = static_cast<const S*>(p.wav) + static_cast<int64_t>(nclip) * p.L;
        const int64_t ns0 = static_cast<int64_t>(2 * nq) * p.hop - p.pad;
        if (carry) {
          load_pair<S, HALF, HALF ? 16 : 0>(nx, p.L, ns0, p.hop, 2 * nq + 1 < p.T, lane, pcm_scale, raw);
        } else {
          load_pair<S, HALF, 0>(nx, p.L, ns0, p.hop, 2 * nq + 1 < p.T, lane, pcm_scale, raw);
        }
      }
      const float2 src = pair_split_src(lane, z, k2);
      float2 b;
      b.x = __shfl_sync(0xffffffffu, src.x, partner);
      b.y = __shfl_sync(0xffffffffu, src.y, partner);
      plane[lane + 32 * k2] = pair_power(z[k2], b);
    }
    if (lane == 0) plane[512] = pair_power(z[16], z[16]);  // bin 512 is its own mirror
    __syncwarp();

    if ((j & 1) || last) {
      const int c0 = (j & ~1) * 2;  // first tile column of this batch of (up to) four frames
#pragma unroll
      for (int vp = 0; vp < 4; ++vp) {
        const int m = pair_mel_id(lane, vp & 1, vp >> 1, p.n_mels);
        if (m >= 0) {
          float acc[4];
          mel_dot_pairs(planeA, planeB, s_w + s_band[2 * kMaxMels + m], s_band[m], s_band[kMaxMels + m], acc);
          const float sc = s_scale[m], sh = s_shift[m];
#pragma unroll
          for (int f = 0; f < 4; ++f) tile[(c0 + f) * kPTileStride + m] = norm_db(acc[f], p.log_eps, sc, sh);
        }
      }
      __syncwarp();
    }

    if (last) {  // store the columns [col_lo, col_hi) of the chunk's tile: the frames this warp transformed
      const int col_hi = min(2 * j + 2, p.T - t0);
      const int col = lane & 7, r0 = lane >> 3;
      if (col >= col_lo && col < col_hi) {
        const float* tp = tile + col * kPTileStride + r0;
        float* o = p.out + (static_cast<int64_t>(clip) * p.n_mels + r0) * p.T + t0 + col;
        const int64_t step = 4 * static_cast<int64_t>(p.T);
        int m = r0;
        for (; m + 12 < p.n_mels; m += 16) {
          const float v0 = tp[0], v1 = tp[4], v2 = tp[8], v3 = tp[12];
          o[0] = v0; o[step] = v1; o[2 * step] = v2; o[3 * step] = v3;
          o += 4 * step;
          tp += 16;
        }
        for (; m < p.n_mels; m += 4) {
          *o = *tp;
          o += step;
          tp += 4;
        }
      }
      col_lo = 0;
      __syncwarp();
    }
    clip = nclip; q = nq; --left;
  }
}

}  // namespace

namespace logmel {

template <typename S>
int pair_launch(const afs_logmel_plan* plan, const Params& p_in, cudaStream_t stream) {
  Params p = p_in;
  p.band = plan->d_band64;
  p.weights = plan->d_weights64;
  const int64_t n_pairs = static_cast<int64_t>(p.B) * ((p.T + 1) / 2);
  if (n_pairs > 0x7fffffffLL) return AFS_ERR_UNSUPPORTED;
  const size_t smem = pair_smem_bytes(p.nnz);
  if (smem > 227 * 1024) return AFS_ERR_UNSUPPORTED;
  const int64_t ctas = (n_pairs + kPWarps - 1) / kPWarps;
  const unsigned grid = static_cast<unsigned>(ctas < kNumSMs ? ctas : kNumSMs);
  const bool half = p.hop * 2 == kNfft;
  if (half) logmel_pair_kernel<S, true><<<grid, kPThreads, smem, stream>>>(p);
  else logmel_pair_kernel<S, false><<<grid, kPThreads, smem, stream>>>(p);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

template <typename S>
static cudaError_t pair_prepare_t() {
  const int smem = 227 * 1024;
  cudaError_t e = cudaFuncSetAttribute(logmel_pair_kernel<S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(logmel_pair_kernel<S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  return e;
}

// Opt every instantiation into the large dynamic shared-memory carve-out (once per plan, on the plan's device).
cudaError_t pair_prepare() {
  cudaError_t e = pair_prepare_t<float>();
  if (e == cudaSuccess) e = pair_prepare_t<int16_t>();
  return e;
}

template int pair_launch<float>(const afs_logmel_plan*, const Params&, cudaStream_t);
template int pair_launch<int16_t>(const afs_logmel_plan*, const Params&, cudaStream_t);

}  // namespace logmel
}  // namespace afs

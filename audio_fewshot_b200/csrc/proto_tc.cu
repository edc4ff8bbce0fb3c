// Prototype head on the tensor cores (precision class "tf32", stated apart from the fp32 parity path of proto.cu):
//   logit[o, w] = -(||q_o||^2 - 2 <q_o, p_w> + ||p_w||^2)
// with the cross term <q, p> as a tcgen05 TF32 GEMM fed by TMA and the norms in exact fp32 -- the "prototype averaging
// plus squared-Euclidean logits as one tensor-core GEMM epilogue" of the north star (reference arithmetic:
// libfewshot_core/model/metric/proto_net.py:49-57, which subtracts before squaring).
//
// Why it is a separate precision class: the expansion cancels (two nearby vectors give a small difference of large
// terms) and the MMA truncates both operands to TF32 (10-bit mantissa), so logits carry an ABSOLUTE error of about
// 1e-3 |q| |p|; the fp32 kernel has none of either.  tests/test_gpu_heads.py reports the argmax flip rate on the
// reference goldens.  It is not faster than proto.cu either -- the head is HBM-bound (M = 75 query rows, N = 5
// prototypes, K = 1 600 per episode: 2 flops per byte) -- it exists because the north star names it.
//
// A tile is 128 CONSECUTIVE feature rows (support rows included: their logits are computed and dropped); the B
// operand is the 32 prototype rows starting at the first episode the tile touches, so a row finds its own episode's
// W columns at (e - e0) W.  Per K chunk of 32 features: one TMA box [128 x 32] of features and one [32 x 32] of
// prototypes (128-byte swizzle), 4 MMAs M128 N32 K8.  Warp 4 issues TMA, warp 5 the MMAs, warps 0-3 accumulate
// ||q||^2 from the SAME shared-memory tile while the MMAs run (conflict-free 128-bit reads of the swizzled rows) and
// then read the accumulator from tensor memory.
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace afs {
namespace {

using namespace tc;

constexpr int kPRows = 128, kPCols = 32, kPStages = 6;
constexpr uint32_t kABytes = kPRows * 128u, kBBytes = kPCols * 128u, kStageBytesP = kABytes + kBBytes;
constexpr int kPThreads = 192;

// [rows, D] fp32 (row stride ld floats), boxes of 32 features x box_rows rows, 128B swizzle, zero fill out of bounds
bool make_map_p(CUtensorMap* map, const float* base, uint64_t rows, uint32_t D, uint64_t ld, uint32_t box_rows) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr) return false;
  const cuuint64_t gdim[2] = {D, rows};
  const cuuint64_t gstride[1] = {ld * sizeof(float)};
  const cuuint32_t box[2] = {32, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// prototypes [E*W, D] and their squared norms
__global__ void __launch_bounds__(256) proto_tc_mean_kernel(const float* __restrict__ feat, int64_t ld,
                                                            const int32_t* __restrict__ cls_row, int EW, int S, int D4,
                                                            float4* __restrict__ protos, float* __restrict__ pp) {
  const int lane = threadIdx.x & 31;
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // one warp per prototype
  if (g >= EW) return;
  const float fS = static_cast<float>(S);
  const float* base = feat + static_cast<int64_t>(cls_row[g]) * ld;
  float ss = 0.f;
  for (int c = lane; c < D4; c += 32) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < S; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(base + s * ld + 4 * c);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    acc = make_float4(acc.x / fS, acc.y / fS, acc.z / fS, acc.w / fS);
    protos[static_cast<int64_t>(g) * D4 + c] = acc;
    ss = fmaf(acc.x, acc.x, ss); ss = fmaf(acc.y, acc.y, ss); ss = fmaf(acc.z, acc.z, ss); ss = fmaf(acc.w, acc.w, ss);
  }
  ss = warp_sum(ss);
  if (lane == 0) pp[g] = ss;
}

__device__ __forceinline__ int block_of_row(const int32_t* __restrict__ cls_row, int EW, int64_t row) {
  int lo = 0, hi = EW - 1;  // block g with cls_row[g] <= row < cls_row[g + 1]
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(cls_row + mid) <= row) lo = mid; else hi = mid - 1;
  }
  return lo;
}

struct PBars {
  uint64_t full[kPStages], empty[kPStages], acc_full[2], acc_empty[2];
};

__global__ void __launch_bounds__(kPThreads, 1)
proto_tc_kernel(const __grid_constant__ CUtensorMap map_f, const __grid_constant__ CUtensorMap map_p,
                const int32_t* __restrict__ cls_row, const float* __restrict__ pp, int N, int EW, int W, int S,
                int n_chunks, float* __restrict__ logits, int32_t* __restrict__ pred) {
  extern __shared__ __align__(1024) uint8_t p_smem_raw[];
  __shared__ PBars bars;
  __shared__ uint32_t s_tmem;
  uint8_t* sm = p_smem_raw + ((1024u - (smem_u32(p_smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = smem_u32(sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(&s_tmem, 64);
  if (tid == 32) {
    for (int s = 0; s < kPStages; ++s) {
      mbar_init(smem_u32(&bars.full[s]), 1);
      mbar_init(smem_u32(&bars.empty[s]), 1 + 128);  // tcgen05.commit + the 128 threads that read ||q||^2 from the tile
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&bars.acc_full[s]), 1);
      mbar_init(smem_u32(&bars.acc_empty[s]), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = s_tmem;
  const int n_tiles = (N + kPRows - 1) / kPRows;

  if (warp == 4) {
    // ===================================================== TMA producer
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row0 = tile * kPRows;
        const int e0 = block_of_row(cls_row, EW, row0) / W;
        for (int kc = 0; kc < n_chunks; ++kc, ++it) {
          const uint32_t st = it % kPStages, par = (it / kPStages) & 1u;
          mbar_wait_sleep(smem_u32(&bars.empty[st]), par ^ 1u);
          const uint32_t full = smem_u32(&bars.full[st]);
          mbar_expect_tx(full, kStageBytesP);
          tma_load_2d(sb + st * kStageBytesP, &map_f, 32 * kc, row0, full);
          tma_load_2d(sb + st * kStageBytesP + kABytes, &map_p, 32 * kc, e0 * W, full);
        }
      }
    }
  } else if (warp == 5) {
    // ===================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t kIdesc = idesc_tf32(kPRows, kPCols);
      uint32_t it = 0, t = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
        const uint32_t as = t & 1u;
        mbar_wait_sleep(smem_u32(&bars.acc_empty[as]), ((t >> 1) & 1u) ^ 1u);
        for (int kc = 0; kc < n_chunks; ++kc, ++it) {
          const uint32_t st = it % kPStages, par = (it / kPStages) & 1u;
          mbar_wait_sleep(smem_u32(&bars.full[st]), par);
          fence_after();
          const uint32_t a = sb + st * kStageBytesP, b = a + kABytes;
#pragma unroll
          for (int k = 0; k < 4; ++k) mma_tf32(tmem + as * kPCols, desc_sw128(a + 32 * k), desc_sw128(b + 32 * k), kIdesc, kc > 0 || k > 0);
          commit(smem_u32(&bars.empty[st]));
        }
        commit(smem_u32(&bars.acc_full[as]));
      }
    }
  } else {
    // ===================================================== warps 0-3: ||q||^2 from the staged tiles, then the epilogue
    const int r = warp * 32 + lane;  // row of the tile == TMEM lane
    uint32_t it = 0, t = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      float qq = 0.f;
      for (int kc = 0; kc < n_chunks; ++kc, ++it) {
        const uint32_t st = it % kPStages, par = (it / kPStages) & 1u;
        mbar_wait_warp_sleep(smem_u32(&bars.full[st]), par, lane);
        const uint8_t* rowp = sm + st * kStageBytesP + r * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 v = *reinterpret_cast<const float4*>(rowp + ((j ^ (r & 7)) << 4));  // 128-byte swizzle
          qq = fmaf(v.x, v.x, qq); qq = fmaf(v.y, v.y, qq); qq = fmaf(v.z, v.z, qq); qq = fmaf(v.w, v.w, qq);
        }
        mbar_arrive(smem_u32(&bars.empty[st]));
      }
      const uint32_t as = t & 1u;
      const int64_t gr = static_cast<int64_t>(tile) * kPRows + r;
      int g = 0, e0 = 0;
      if (gr < N) g = block_of_row(cls_row, EW, gr);
      e0 = block_of_row(cls_row, EW, static_cast<int64_t>(tile) * kPRows) / W;
      mbar_wait_warp_sleep(smem_u32(&bars.acc_full[as]), (t >> 1) & 1u, lane);
      fence_after();
      uint32_t v[32];
      tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16) + as * kPCols, v);
      fence_before();
      mbar_arrive(smem_u32(&bars.acc_empty[as]));
      if (gr < N) {
        const int e = g / W;
        const int pos = static_cast<int>(gr - __ldg(cls_row + g));
        if (pos >= S) {  // a query row (support rows were computed along and are dropped)
          const int64_t o = gr - static_cast<int64_t>(g + 1) * S;
          const int col0 = (e - e0) * W;
          float best = -INFINITY;
          int best_w = 0;
          for (int w = 0; w < W; ++w) {
            float val;
            if (col0 + w < kPCols) {
              float dot = 0.f;
#pragma unroll
              for (int c = 0; c < 32; ++c) dot = (c == col0 + w) ? __uint_as_float(v[c]) : dot;
              val = -(qq - 2.f * dot + __ldg(pp + e * W + w));
            } else {
              val = __int_as_float(0x7fc00000);  // the tile spans more episodes than 32 / W: caller's contract broken
            }
            logits[o * W + w] = val;
            if (val > best) { best = val; best_w = w; }
          }
          if (pred != nullptr) pred[o] = best_w;
        }
      }
    }
  }
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 64);
}

}  // namespace
}  // namespace afs

extern "C" size_t afs_proto_tc_workspace_bytes(int32_t E, int32_t W, int32_t D) {
  if (E <= 0 || W <= 0 || D <= 0) return 0;
  // the prototypes padded by 32 rows (the last tile's B box may start at the last episode), then their squared norms
  return (static_cast<size_t>(E) * W + 32) * D * sizeof(float) + ((static_cast<size_t>(E) * W * sizeof(float) + 15) & ~static_cast<size_t>(15));
}

extern "C" int afs_proto_fwd_tc(const float* feat, int64_t ld_feat, const int32_t* cls_row, int32_t N, int32_t E,
                                int32_t W, int32_t S, int32_t D, float* logits, int32_t* pred, void* ws, size_t ws_bytes,
                                afs_stream_t stream_) {
  using namespace afs;
  if (feat == nullptr || cls_row == nullptr || logits == nullptr || N < 0 || E < 0 || W < 1 || S < 1 || D < 1 || ld_feat < D)
    return AFS_ERR_INVALID_ARG;
  if (W > 8 || D % 32 != 0 || ld_feat % 4 != 0 || (reinterpret_cast<uintptr_t>(feat) & 15) != 0) return AFS_ERR_UNSUPPORTED;
  if (E == 0 || N == E * W * S) return AFS_OK;
  const size_t need = afs_proto_tc_workspace_bytes(E, W, D);
  if (ws == nullptr || ws_bytes < need) return AFS_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(ws) % 16 != 0) return AFS_ERR_INVALID_ARG;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  float* protos = static_cast<float*>(ws);
  float* pp = protos + (static_cast<size_t>(E) * W + 32) * D;
  proto_tc_mean_kernel<<<(E * W * 32 + 255) / 256, 256, 0, stream>>>(feat, ld_feat, cls_row, E * W, S, D / 4,
                                                                      reinterpret_cast<float4*>(protos), pp);
  AFS_LAUNCH_CHECK();
  CUtensorMap mf, mp;
  if (!make_map_p(&mf, feat, static_cast<uint64_t>(N), static_cast<uint32_t>(D), static_cast<uint64_t>(ld_feat), kPRows) ||
      !make_map_p(&mp, protos, static_cast<uint64_t>(E) * W, static_cast<uint32_t>(D), static_cast<uint64_t>(D), kPCols))
    return AFS_ERR_UNSUPPORTED;
  const int n_tiles = (N + kPRows - 1) / kPRows;
  const size_t smem = kPStages * kStageBytesP + 1024;
  AFS_CUDA_TRY(cudaFuncSetAttribute(proto_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int grid = n_tiles < kNumSMs ? n_tiles : kNumSMs;
  proto_tc_kernel<<<grid, kPThreads, smem, stream>>>(mf, mp, cls_row, pp, N, E * W, W, S, D / 32, logits, pred);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

// Brownian-distance-covariance pooling with the Gram matrix on the tensor cores (sm_100a): the same operator as
// bdc.cu (reference libfewshot_core/model/backbone/utils/bdc_pool.py:69-93) for C = 64 channels.
//
//   G = X X^T  (X in R^{64 x M}, both GEMM operands are the SAME K-major matrix: every channel row is contiguous
//   in memory) on tcgen05 with 3 x TF32 operand splitting: x = hi + lo, hi = the 19 bits the MMA keeps, lo = x - hi
//   (exact in fp32), G = hi hi^T + hi lo^T + lo hi^T accumulated in fp32 -- 21 mantissa bits per operand, which holds
//   the 1e-4 tolerance through the cancellation in G_ii + G_jj - 2 G_ij.
//
// A tile is TWO clips: 128 rows x 32 positions per K chunk arrive as one TMA box (128-byte swizzle); the accumulator
// is [128 x 256] -- columns 0-127 hold hi hi^T, columns 128-255 hi lo^T + lo hi^T (one N = 256 MMA against B = [hi; lo]
// and one N = 128 MMA per k step; the epilogue adds the halves) -- of which the two diagonal 64 x 64 blocks of each half
// are the clips' Gram matrices (the off-diagonal blocks cost
// nothing extra: an M128 N64 MMA takes as long as an M128 N128 one on this part).  bdc.cu keeps the Gram on the FMA
// pipe at 0.13 of HBM; here the FMA lanes only build the lo operand and run the epilogue.
//
// One persistent CTA per SM, 14 warps: TMA (warp 8), lo-operand builders (warps 4-7), MMA issuer (warp 9), and TWO
// epilogue groups (warps 0-3 and 10-13: thread = Gram row of one clip: distances, sqrt, row / column sums, double
// centring, upper triangle -- the arithmetic and summation orders of bdc.cu).  Operand ring of 4 stages, four
// accumulators (all 512 TMEM columns): even tiles go to group 0, odd tiles to group 1, each with two accumulators, its
// own A matrices and named barriers.  The epilogue of a tile is ~1 500 dependent instructions per thread (a chain of
// latencies, ~20 000 clk) against 7 800 clk of MMAs: with one group the tensor pipe idled 60 % of the time
// (profiles/r02_bdc_tc_ncu.csv).
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace afs {
namespace {

using namespace tc;

constexpr int kBC = 64;                       // channels
constexpr int kBStages = 4;
constexpr uint32_t kBTile = 128u * 128u;      // [128 rows][32 floats]
constexpr uint32_t kBStage = 2u * kBTile;     // hi | lo
constexpr int kBThreads = 448;
constexpr int kBAcc = 4;                      // accumulators: two per epilogue group
constexpr int kAStride = kBC + 1;

struct BBars {
  uint64_t full[kBStages], lo_ready[kBStages], empty[kBStages], acc_full[kBAcc], acc_empty[kBAcc];
};

__global__ void __launch_bounds__(kBThreads, 1)
bdc_tc_kernel(const __grid_constant__ CUtensorMap map_x, int B, int n_chunks, const float* __restrict__ log_temp,
              int triu, float* __restrict__ out) {
  extern __shared__ __align__(1024) uint8_t b_smem_raw[];
  __shared__ BBars bars;
  __shared__ uint32_t s_tmem;
  __shared__ __align__(16) float s_diag[4][kBC], s_rowsum[4][kBC], s_colsum[4][kBC];  // [2 * group + clip of the tile]
  uint8_t* sm = b_smem_raw + ((1024u - (smem_u32(b_smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = smem_u32(sm);
  float* sA = reinterpret_cast<float*>(sm + kBStages * kBStage);  // [2 groups][2 clips][64][65]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(&s_tmem, 512);
  if (tid == 32) {
    for (int s = 0; s < kBStages; ++s) {
      mbar_init(smem_u32(&bars.full[s]), 1);
      mbar_init(smem_u32(&bars.lo_ready[s]), 128);
      mbar_init(smem_u32(&bars.empty[s]), 1);
    }
    for (int s = 0; s < kBAcc; ++s) {
      mbar_init(smem_u32(&bars.acc_full[s]), 1);
      mbar_init(smem_u32(&bars.acc_empty[s]), 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = s_tmem;
  const int n_tiles = (B + 1) / 2;

  if (warp == 8) {
    // ===================================================== TMA producer
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int kc = 0; kc < n_chunks; ++kc, ++it) {
          const uint32_t st = it % kBStages, par = (it / kBStages) & 1u;
          mbar_wait_sleep(smem_u32(&bars.empty[st]), par ^ 1u);
          const uint32_t full = smem_u32(&bars.full[st]);
          mbar_expect_tx(full, kBTile);
          tma_load_2d(sb + st * kBStage, &map_x, 32 * kc, tile * 128, full);
        }
      }
    }
  } else if (warp == 9) {
    // ===================================================== MMA issuer
    if (lane == 0) {
      // hi hi^T and hi lo^T in ONE N = 256 MMA (B = [hi; lo]: the lo tile follows the hi tile in the stage, so the
      // 128-byte-swizzled operand simply has 256 rows), lo hi^T as an N = 128 MMA onto the second half: 20 KB of
      // operand reads per k step instead of 24 KB for three N = 128 MMAs; the epilogue adds the two halves
      constexpr uint32_t kIdesc256 = idesc_tf32(128, 256);
      constexpr uint32_t kIdesc = idesc_tf32(128, 128);
      uint32_t it = 0, t = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
        // local tile t belongs to epilogue group t & 1 and uses that group's 256-column accumulator
        const uint32_t as = t & 1u;
        mbar_wait_sleep(smem_u32(&bars.acc_empty[as]), ((t >> 1) & 1u) ^ 1u);
        for (int kc = 0; kc < n_chunks; ++kc, ++it) {
          const uint32_t st = it % kBStages, par = (it / kBStages) & 1u;
          mbar_wait_sleep(smem_u32(&bars.lo_ready[st]), par);
          fence_after();
          const uint32_t hi = sb + st * kBStage, lo = hi + kBTile;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t dh = desc_sw128(hi + 32 * k), dl = desc_sw128(lo + 32 * k);
            mma_tf32(tmem + as * 256u, dh, dh, kIdesc256, kc > 0 || k > 0);  // [hi hi^T | hi lo^T]
            mma_tf32(tmem + as * 256u + 128u, dl, dh, kIdesc, true);          // second half += lo hi^T
          }
          commit(smem_u32(&bars.empty[st]));
        }
        commit(smem_u32(&bars.acc_full[as]));
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================================================== lo operand: x - (the 19 bits the MMA keeps of x)
    const int s = tid - 128;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int kc = 0; kc < n_chunks; ++kc, ++it) {
        const uint32_t st = it % kBStages, par = (it / kBStages) & 1u;
        mbar_wait_warp_sleep(smem_u32(&bars.full[st]), par, lane);
        const float4* hi = reinterpret_cast<const float4*>(sm + st * kBStage);
        float4* lo = reinterpret_cast<float4*>(sm + st * kBStage + kBTile);
#pragma unroll
        for (int j = 0; j < 8; ++j) {  // elementwise: the swizzled position of a 16-byte chunk does not matter
          const float4 v = hi[s + 128 * j];
          float4 l;
          l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
          l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
          l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
          l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
          lo[s + 128 * j] = l;
        }
        fence_async_smem();
        mbar_arrive(smem_u32(&bars.lo_ready[st]));
      }
    }
  } else {
    // ===================================================== epilogue group (warps 0-3 / 10-13): thread = Gram row r of
    // clip (quarter >> 1), where quarter = warp % 4 is the TMEM lane quarter the warp may read
    const int group = warp >= 10 ? 1 : 0;
    const int quarter = warp & 3;
    const int clip_in_tile = quarter >> 1;
    const int slot = 2 * group + clip_in_tile;  // scratch row of this (group, clip)
    const int r = (quarter & 1) * 32 + lane;
    float* A = sA + slot * kBC * kAStride;
    const float et = expf(__ldg(log_temp));
    const float inv = 1.0f / static_cast<float>(kBC), inv2 = 1.0f / static_cast<float>(kBC * kBC);
    const int bar_id = 1 + slot;  // the two warps of a clip synchronise among themselves
    uint32_t t = static_cast<uint32_t>(group);
    for (int tile = blockIdx.x + group * gridDim.x; tile < n_tiles; tile += 2 * gridDim.x, t += 2) {
      const uint32_t as = t & 1u;
      mbar_wait_warp_sleep(smem_u32(&bars.acc_full[as]), (t >> 1) & 1u, lane);
      fence_after();
      uint32_t g0[32], g1[32];
      const uint32_t taddr = tmem + (static_cast<uint32_t>(quarter * 32) << 16) + as * 256u + 64u * clip_in_tile;
      {  // Gram row = first half (hi hi^T) + second half (hi lo^T + lo hi^T), 32 columns at a time
        uint32_t x[32];
        tmem_ld32_nowait(taddr, g0);
        tmem_ld32_nowait(taddr + 128u, x);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < 32; ++c) g0[c] = __float_as_uint(__uint_as_float(g0[c]) + __uint_as_float(x[c]));
        tmem_ld32_nowait(taddr + 32u, g1);
        tmem_ld32_nowait(taddr + 160u, x);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < 32; ++c) g1[c] = __float_as_uint(__uint_as_float(g1[c]) + __uint_as_float(x[c]));
      }
      fence_before();
      mbar_arrive(smem_u32(&bars.acc_empty[as]));
      const int b = 2 * tile + clip_in_tile;
      // diagonal of the Gram: element r of this thread's row
      float diag = 0.f;
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        diag = (c == r) ? __uint_as_float(g0[c]) : diag;
        diag = (c + 32 == r) ? __uint_as_float(g1[c]) : diag;
      }
      s_diag[slot][r] = diag;
      asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
      // distances in place of the Gram values (registers), the diagonal fetched as 128-bit loads: with the stores to A
      // inside this loop every load of s_diag waited for the previous store (the compiler must assume they alias)
#pragma unroll
      for (int c4 = 0; c4 < 16; ++c4) {
        const float4 dg = *reinterpret_cast<const float4*>(&s_diag[slot][4 * c4]);
        const float dgs[4] = {dg.x, dg.y, dg.z, dg.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c = 4 * c4 + k;
          const float g = __uint_as_float(c < 32 ? g0[c] : g1[c - 32]);
          float d = dgs[k] + diag - 2.f * g;
          d = fmaxf(d, 0.f);
          float a;
          asm("sqrt.approx.f32 %0, %1;" : "=f"(a) : "f"(fmaf(et, d, 1e-5f)));  // MUFU.SQRT: 1 ulp-class, tolerance is 1e-4
          if (c < 32) g0[c] = __float_as_uint(a);
          else g1[c - 32] = __float_as_uint(a);
        }
      }
      float rs = 0.f;  // row sum (dcov.bmm(I_M)): fixed order over j, as bdc.cu
#pragma unroll
      for (int c = 0; c < 64; ++c) {
        const float a = __uint_as_float(c < 32 ? g0[c] : g1[c - 32]);
        A[r * kAStride + c] = a;
        rs += a;
      }
      s_rowsum[slot][r] = rs;
      asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
      float cs = 0.f;  // column sum (I_M.bmm(dcov)): fixed order over i
#pragma unroll 8
      for (int i = 0; i < kBC; ++i) cs += A[i * kAStride + r];
      s_colsum[slot][r] = cs;
      asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
      float total = 0.f;
#pragma unroll
      for (int j4 = 0; j4 < kBC / 4; ++j4) {  // the same ascending order, four values per load
        const float4 v = *reinterpret_cast<const float4*>(&s_colsum[slot][4 * j4]);
        total += v.x; total += v.y; total += v.z; total += v.w;
      }
      if (b < B) {
        // thread = column c of the output; rows in order: for a fixed row the 64 threads write consecutive addresses
        const int c = r;
        const float colterm = inv2 * total - inv * cs;
        if (triu) {
          // row rr of the upper triangle starts at rr*64 - rr(rr-1)/2; element (rr, c) sits c - rr further.  Fully
          // unrolled: every offset is an immediate of the store, the row sums arrive four per load
          float* ob = out + static_cast<int64_t>(b) * (kBC * (kBC + 1) / 2) + c;
#pragma unroll
          for (int r4 = 0; r4 < kBC / 4; ++r4) {
            const float4 rs4 = *reinterpret_cast<const float4*>(&s_rowsum[slot][4 * r4]);
            const float rsv[4] = {rs4.x, rs4.y, rs4.z, rs4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int rr = 4 * r4 + k;
              if (c >= rr) ob[rr * kBC - rr * (rr - 1) / 2 - rr] = A[rr * kAStride + c] - inv * rsv[k] + colterm;
            }
          }
        } else {
          float* ob = out + static_cast<int64_t>(b) * kBC * kBC + c;
#pragma unroll 4
          for (int rr = 0; rr < kBC; ++rr) ob[rr * kBC] = A[rr * kAStride + c] - inv * s_rowsum[slot][rr] + colterm;
        }
      }
      asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");  // A, the sums and the diagonal are free for the next tile
    }
  }
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace

// Tensor-core path of afs_bdc_fwd: C == 64, M % 4 == 0, 16-byte aligned x.  Returns AFS_ERR_UNSUPPORTED otherwise.
int bdc_fwd_tc(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp, int32_t triu, float* out,
               cudaStream_t stream) {
  if (C != kBC || M % 4 != 0 || (reinterpret_cast<uintptr_t>(x) & 15) != 0) return AFS_ERR_UNSUPPORTED;
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr) return AFS_ERR_UNSUPPORTED;
  CUtensorMap map;
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(M), static_cast<cuuint64_t>(B) * kBC};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(M) * sizeof(float)};
  const cuuint32_t box[2] = {32, 128};
  const cuuint32_t estr[2] = {1, 1};
  if (fn(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x), gdim, gstride, box, estr,
         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return AFS_ERR_UNSUPPORTED;
  const int n_tiles = (B + 1) / 2;
  const size_t smem = kBStages * kBStage + 4 * kBC * kAStride * sizeof(float) + 1024;
  AFS_CUDA_TRY(cudaFuncSetAttribute(bdc_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int grid = n_tiles < kNumSMs ? n_tiles : kNumSMs;
  bdc_tc_kernel<<<grid, kBThreads, smem, stream>>>(map, B, (M + 31) / 32, log_temp, triu, out);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

}  // namespace afs

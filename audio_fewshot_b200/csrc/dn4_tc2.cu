// DN4 head, warp-specialised Blackwell pipeline: TMA -> shared memory (128B swizzle) -> tcgen05.mma (TF32)
// -> tensor memory -> tcgen05.ld -> top-k in registers.  sm_100a.
//
// Second generation of csrc/dn4_tc.cu (same arithmetic: DN4Layer.forward, reference
// libfewshot_core/model/metric/dn4.py:52-73).  dn4_tc.cu stages operands with ordinary loads and runs
// load -> MMA -> epilogue back to back; here the three stages overlap:
//   warp 4   TMA producer: one thread issues cp.async.bulk.tensor loads of [128 descriptors x 32 channels]
//            boxes (128-byte rows, hardware 128B swizzle) and arms the stage's mbarrier with expect_tx;
//   warp 5   MMA issuer: one thread waits for the operands, issues C/8 tcgen05.mma.kind::tf32 into one of
//            two 128-column TMEM accumulators and commits to the "operands free" / "accumulator full"
//            mbarriers; it also owns the TMEM allocation.  In the K-streaming schedule warps 5, 6, 7 each issue for
//            ONE of the three accumulators of a class: a single thread needs ~180 clk per tcgen05.mma (descriptor
//            arithmetic, predicate, issue latency) against 65 clk for the M128 N128 K8 MMA itself;
//   warps 0-3 epilogue: thread i owns accumulator row i (TMEM lane i): tcgen05.ld, running top-n_k,
//            then releases the accumulator stage.
// Operands come from a small pre-pass (dn4_tc_prep_kernel) that writes the L2-normalised, TF32-rounded
// descriptors K-major ([descriptor][C]) with queries compacted in output order and supports in class
// order, so every operand tile is a contiguous row range: a plain 2-D TMA box.
//
// Two operand schedules, one kernel (template flag KSTREAM):
//   C <= 128 (Conv64F maps): the 128 query rows of a tile stay resident for all C channels while the support
//            tiles stream through two whole-K stages;
//   C  > 128 (ResNet-12 maps, C = 640: an 8.3 GFLOP GEMM per 5w5s10q episode): a 3-stage ring of
//            [A slice | B slice x 3] groups of 32 channels (64 KB per stage) feeds the K loop: ONE query slice serves the
//            (up to) three column tiles of a class, which accumulate side by side in three of FOUR 128-column TMEM
//            accumulators (the fourth lets the next item start while the epilogue drains) -- 16 KB of operands per MMA
//            quartet instead of 32 KB: the round-1 schedule re-streamed both operands per 128 x 128 tile and sat at the
//            per-SM L2 bandwidth (157 clk per M128 N128 K8 MMA against 65 for the MMA itself).  Work items are
//            (row tile, class) pairs dealt over a persistent grid of ~148 CTAs.
// Built for C % 32 == 0 (one 128-byte swizzle atom per 32 channels); other widths use dn4_tc.cu (C % 8 == 0) or
// the fp32 path dn4.cu.
#include <cuda.h>
#include <limits.h>

#include "common.cuh"
#include "tc_common.cuh"
#include "topk.cuh"

namespace afs {
namespace {

using namespace tc;
using namespace topk;

constexpr int kThreads2 = 256;  // warps 0-3 epilogue, 4 TMA producer, 5-7 MMA issuers (6, 7: K-streaming schedule only)
constexpr int kRows2 = 128;   // UMMA M
constexpr int kCols2 = 128;   // UMMA N
constexpr int kMaxWay2 = 32;
constexpr uint32_t kAtomBytes = 128u * 128u;  // one [128 rows x 32 floats] swizzle-128B operand block

// [rows, C] fp32 row-major tensor, boxes of 32 channels x 128 rows, 128B swizzle, zero fill out of bounds
bool make_map(CUtensorMap* map, const float* base, uint64_t rows, uint32_t C) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr) return false;
  const cuuint64_t gdim[2] = {C, rows};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(C) * sizeof(float)};
  const cuuint32_t box[2] = {32, kRows2};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr uint32_t kIdesc2 = (1u << 4) | (2u << 7) | (2u << 10) | ((kCols2 >> 3) << 17) | ((kRows2 >> 4) << 24);

// ---- pre-pass: normalise, round to TF32, write K-major; queries compacted in output-row order.
// A transpose through shared memory: a CTA owns kPrepPos positions of one image, warp w reads channels w, w + 8, ...
// (a lane = a position: 128-byte coalesced reads of the NCHW map), keeps the tile [C][33] on chip while the per-position
// sums of squares are reduced, then writes each position's C channels as one contiguous run (the round-1 kernel had a
// thread per descriptor writing 16-byte pieces C floats apart: 169 us for 300 maps of [640, 8, 9]; this one ~25 us).
constexpr int kPrepPos = 32;
constexpr int kPrepThreads = 256;
constexpr int kPrepPitch = kPrepPos + 1;

__global__ void __launch_bounds__(kPrepThreads)
dn4_tc_prep_kernel(const float* __restrict__ feat, const int32_t* __restrict__ cls_row, int EW, int S, int C, int HW,
                   float* __restrict__ nfq, float* __restrict__ nfs) {
  extern __shared__ float s_tile[];            // [C][kPrepPitch]
  __shared__ float s_part[kPrepThreads / 32][kPrepPos];
  __shared__ float s_inv[kPrepPos];
  const int64_t row = blockIdx.x;
  const int per = (HW + gridDim.y - 1) / gridDim.y;  // positions per CTA (<= kPrepPos): HW = 72 -> 3 x 24
  const int m0 = blockIdx.y * per;
  const int np = min(per, HW - m0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kPrepThreads / 32;

  const float* src = feat + row * static_cast<int64_t>(C) * HW + m0;
  if ((np & 3) == 0 && (HW & 3) == 0 && (m0 & 3) == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0) {
    // 128-bit loads, all of a thread's loads in flight at once (a [640 x 24] slab is 15 per thread), then the sums of
    // squares from shared memory: 8 partial sums per position
    const int nq = np >> 2;
    const int total = C * nq;
    for (int i0 = tid; i0 < total; i0 += 8 * kPrepThreads) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * kPrepThreads;
        if (i < total) {
          const int c = i / nq, q = i - c * nq;
          v[u] = __ldg(reinterpret_cast<const float4*>(src + static_cast<int64_t>(c) * HW) + q);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * kPrepThreads;
        if (i < total) {
          const int c = i / nq, q = i - c * nq;
          float* d = s_tile + c * kPrepPitch + 4 * q;
          d[0] = v[u].x; d[1] = v[u].y; d[2] = v[u].z; d[3] = v[u].w;
        }
      }
    }
    __syncthreads();
    float ss = 0.f;
    if (lane < np)
      for (int c = warp; c < C; c += kWarps) {
        const float v = s_tile[c * kPrepPitch + lane];
        ss = fmaf(v, v, ss);
      }
    s_part[warp][lane] = ss;
  } else {
    float ss = 0.f;
#pragma unroll 8
    for (int c = warp; c < C; c += kWarps) {
      const float v = lane < np ? __ldg(src + static_cast<int64_t>(c) * HW + lane) : 0.f;
      s_tile[c * kPrepPitch + lane] = v;
      ss = fmaf(v, v, ss);
    }
    s_part[warp][lane] = ss;
  }
  __syncthreads();
  if (tid < kPrepPos) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) t += s_part[w][tid];
    s_inv[tid] = 1.0f / fmaxf(sqrtf(t), 1e-12f);  // F.normalize: x / max(||x||, eps)
  }
  __syncthreads();

  int lo = 0, hi = EW - 1;  // block g with cls_row[g] <= row < cls_row[g+1]
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (cls_row[mid] <= row) lo = mid; else hi = mid - 1;
  }
  const int g = lo;
  const int pos = static_cast<int>(row - cls_row[g]);
  float* dst = pos < S ? nfs + ((static_cast<int64_t>(g) * S + pos) * HW + m0) * C
                       : nfq + ((row - static_cast<int64_t>(g + 1) * S) * HW + m0) * C;
  for (int p = warp; p < np; p += kWarps) {
    const float inv = s_inv[p];
    float* d = dst + static_cast<int64_t>(p) * C;
    for (int c = lane; c < C; c += 32) {
      uint32_t r;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(s_tile[c * kPrepPitch + p] * inv));
      d[c] = __uint_as_float(r);
    }
  }
}

constexpr int kStgK = 3;   // ring stages of the K-streaming schedule
constexpr int kGrpK = 3;   // column tiles (accumulators) that share one query slice
constexpr uint32_t kStageK = (1u + kGrpK) * kAtomBytes;

struct Bars {
  uint64_t full_a, empty_a;
  uint64_t full_b[2], empty_b[2];
  uint64_t tmem_full[4], tmem_empty[4];
  uint64_t full_k[kStgK], empty_k[kStgK];
};

template <int NK, bool KSTREAM>
__global__ void __launch_bounds__(kThreads2)
dn4_tc2_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_s,
               const int32_t* __restrict__ cls_row, int W, int S, int C, int HW, float* __restrict__ rowsum,
               int32_t* __restrict__ topk_idx) {
  extern __shared__ uint8_t s_raw[];
  __shared__ __align__(8) Bars bars;
  __shared__ uint32_t s_tmem;
  __shared__ int s_qbase[kMaxWay2 + 1];

  const int e = blockIdx.z;
  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int KH = C / 32;  // 128-byte K blocks per descriptor
  const uint32_t blk_bytes = static_cast<uint32_t>(KH) * kAtomBytes;
  const uint32_t base = (smem_u32(s_raw) + 1023u) & ~1023u;  // swizzle atoms need 1024-byte alignment
  const uint32_t a_addr = base;
  const uint32_t b_addr0 = base + blk_bytes;

  if (tid <= W) {
    const int g = e * W + tid;
    s_qbase[tid] = cls_row[g] - g * S;
  }
  if (tid == 0) {
    mbar_init(smem_u32(&bars.full_a), 1);
    mbar_init(smem_u32(&bars.empty_a), 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&bars.full_b[s]), 1);
      mbar_init(smem_u32(&bars.empty_b[s]), 1);
    }
    for (int s = 0; s < 4; ++s) {
      mbar_init(smem_u32(&bars.tmem_full[s]), 1);
      mbar_init(smem_u32(&bars.tmem_empty[s]), 4);  // one arrival per epilogue warp
    }
    for (int s = 0; s < kStgK; ++s) {
      mbar_init(smem_u32(&bars.full_k[s]), 1);
      mbar_init(smem_u32(&bars.empty_k[s]), kGrpK);  // one arrival per MMA-issuing warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr uint32_t kTmemCols = KSTREAM ? 512u : 256u;  // four / two 128-column accumulators
  constexpr uint32_t kAccMask = KSTREAM ? 3u : 1u;
  constexpr uint32_t kAccShift = KSTREAM ? 2u : 1u;
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = s_tmem;

  const int out0 = s_qbase[0];
  const int out1 = s_qbase[W];
  const int NS = S * HW;
  const int n_rows = (out1 - out0) * HW;
  const int n_tiles = (n_rows + kRows2 - 1) / kRows2;
  const int n_ctiles = (NS + kCols2 - 1) / kCols2;
  const int n_items = n_tiles * W;  // K-streaming schedule: (row tile, class) work items

  if (warp == 4) {
    // ================= TMA producer (one thread) =================
    if (KSTREAM && lane == 0) {
      uint32_t ks = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int tile = item / W, w = item - tile * W;
        const int qrow0 = out0 * HW + tile * kRows2;
        const int srow_base = (e * W + w) * S * HW;
        for (int cg0 = 0; cg0 < n_ctiles; cg0 += kGrpK) {
          const int g = min(kGrpK, n_ctiles - cg0);
          for (int kh = 0; kh < KH; ++kh, ++ks) {
            const uint32_t st = ks % kStgK, ph = (ks / kStgK) & 1u;
            mbar_wait(smem_u32(&bars.empty_k[st]), ph ^ 1u);
            mbar_expect_tx(smem_u32(&bars.full_k[st]), (1u + static_cast<uint32_t>(g)) * kAtomBytes);
            const uint32_t sa = base + st * kStageK;
            tma_load_2d(sa, &map_q, kh * 32, qrow0, smem_u32(&bars.full_k[st]));
            for (int c = 0; c < g; ++c)
              tma_load_2d(sa + (1u + c) * kAtomBytes, &map_s, kh * 32, srow_base + (cg0 + c) * kCols2, smem_u32(&bars.full_k[st]));
          }
        }
      }
    } else if (lane == 0) {
      uint32_t it = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
        mbar_wait(smem_u32(&bars.empty_a), (tcount & 1u) ^ 1u);  // MMAs of the previous tile have read A
        mbar_expect_tx(smem_u32(&bars.full_a), blk_bytes);
        const int qrow0 = out0 * HW + tile * kRows2;
        for (int kh = 0; kh < KH; ++kh)
          tma_load_2d(a_addr + static_cast<uint32_t>(kh) * kAtomBytes, &map_q, kh * 32, qrow0, smem_u32(&bars.full_a));
        for (int w = 0; w < W; ++w) {
          const int srow_base = (e * W + w) * S * HW;
          for (int ct = 0; ct < n_ctiles; ++ct, ++it) {
            const uint32_t st = it & 1u, ph = (it >> 1) & 1u;
            mbar_wait(smem_u32(&bars.empty_b[st]), ph ^ 1u);
            mbar_expect_tx(smem_u32(&bars.full_b[st]), blk_bytes);
            for (int kh = 0; kh < KH; ++kh)
              tma_load_2d(b_addr0 + st * blk_bytes + static_cast<uint32_t>(kh) * kAtomBytes, &map_s, kh * 32,
                          srow_base + ct * kCols2, smem_u32(&bars.full_b[st]));
          }
        }
      }
    }
  } else if (warp >= 5) {
    // ================= MMA issuers (one thread per warp) =================
    if (KSTREAM && lane == 0) {
      const int c = warp - 5;  // this warp's accumulator within a group of column tiles
      uint32_t ks = 0, it = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        for (int cg0 = 0; cg0 < n_ctiles; cg0 += kGrpK) {
          const int g = min(kGrpK, n_ctiles - cg0);
          for (int kh = 0; kh < KH; ++kh, ++ks) {
            const uint32_t st = ks % kStgK, ph = (ks / kStgK) & 1u;
            mbar_wait(smem_u32(&bars.full_k[st]), ph);
            fence_after();
            if (c < g) {
              const uint32_t acc = (it + c) & 3u;
              if (kh == 0) {  // first touch of this accumulator: the epilogue must have drained its previous use
                mbar_wait(smem_u32(&bars.tmem_empty[acc]), (((it + c) >> 2) & 1u) ^ 1u);
                fence_after();
              }
              const uint32_t d_tmem = tmem_base + acc * kCols2;
              const uint32_t sa = base + st * kStageK;
              const uint64_t da = desc_sw128(sa), db = desc_sw128(sa + (1u + c) * kAtomBytes);
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4)  // +32 bytes inside the swizzle atom = +2 in the descriptor's address field
                mma_tf32(d_tmem, da + 2u * k4, db + 2u * k4, kIdesc2, (kh | k4) != 0);
              commit(smem_u32(&bars.empty_k[st]));  // slice group reusable once these MMAs have read it
            } else {
              mbar_arrive(smem_u32(&bars.empty_k[st]));
            }
          }
          if (c < g) commit(smem_u32(&bars.tmem_full[(it + c) & 3u]));  // all C channels accumulated
          it += g;
        }
      }
    } else if (warp == 5 && lane == 0) {
      uint32_t it = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
        mbar_wait(smem_u32(&bars.full_a), tcount & 1u);
        for (int w = 0; w < W; ++w) {
          for (int ct = 0; ct < n_ctiles; ++ct, ++it) {
            const uint32_t st = it & 1u, ph = (it >> 1) & 1u;
            mbar_wait(smem_u32(&bars.full_b[st]), ph);
            mbar_wait(smem_u32(&bars.tmem_empty[st]), ph ^ 1u);  // epilogue has drained this accumulator
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t d_tmem = tmem_base + st * kCols2;
            for (int kh = 0; kh < KH; ++kh) {
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                const uint64_t da = desc_sw128(a_addr + static_cast<uint32_t>(kh) * kAtomBytes + k4 * 32u);
                const uint64_t db = desc_sw128(b_addr0 + st * blk_bytes + static_cast<uint32_t>(kh) * kAtomBytes + k4 * 32u);
                const uint32_t acc = (kh | k4) ? 1u : 0u;
                asm volatile(
                    "{\n\t"
                    ".reg .pred p;\n\t"
                    "setp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
                    "}\n" ::"r"(d_tmem), "l"(da), "l"(db), "r"(kIdesc2), "r"(acc), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
                    : "memory");
              }
            }
            commit(smem_u32(&bars.empty_b[st]));    // operand stage reusable once these MMAs finish
            commit(smem_u32(&bars.tmem_full[st]));  // accumulator ready for the epilogue
          }
        }
        commit(smem_u32(&bars.empty_a));
      }
    }
  } else {
    // ================= epilogue warps 0..3: accumulator row == TMEM lane == tid =================
    uint32_t it = 0;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    // one (row tile, class): running top-n_k of this thread's accumulator row over the class's column tiles
    auto do_class = [&](int tile, int w) {
      const int dr = tile * kRows2 + tid;
      const bool live = dr < n_rows;
      const int o = out0 + dr / HW;
      const int m = dr - (dr / HW) * HW;
      float tv[NK];
      int ti[NK];
#pragma unroll
      for (int k = 0; k < NK; ++k) { tv[k] = -INFINITY; ti[k] = INT_MAX; }
      for (int ct = 0; ct < n_ctiles; ++ct, ++it) {
        const uint32_t st = it & kAccMask, ph = (it >> kAccShift) & 1u;
        mbar_wait(smem_u32(&bars.tmem_full[st]), ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint32_t tk[NK];
#pragma unroll
        for (int k = 0; k < NK; ++k) tk[k] = 0u;  // below every real key (keys of finite values are > 0)
        const int valid = NS - ct * kCols2;   // columns of this tile that exist (>= kCols2 for full tiles)
#pragma unroll 1
        for (int c0 = 0; c0 < kCols2; c0 += 32) {
          uint32_t v[32];
          if (c0 >= valid) break;  // tile-uniform: nothing left in this column tile
          tmem_ld32(t_row + st * kCols2 + static_cast<uint32_t>(c0), v);
          if (c0 + 32 <= valid) {
#pragma unroll
            for (int j = 0; j < 32; ++j) topk_push<NK>(tk, topk_key(v[j], c0 + j));
          } else {
#pragma unroll
            for (int g8 = 0; g8 < 4; ++g8) {  // boundary chunk: whole groups of 8 are skipped by a uniform branch
              if (c0 + 8 * g8 < valid) {
#pragma unroll
                for (int j = 8 * g8; j < 8 * g8 + 8; ++j)
                  if (c0 + j < valid) topk_push<NK>(tk, topk_key(v[j], c0 + j));
              }
            }
          }
        }
#pragma unroll
        for (int k = 0; k < NK; ++k)
          if (tk[k] != 0u) topk_merge<NK>(tv, ti, topk_key_value(tk[k]), ct * kCols2 + 127 - static_cast<int>(tk[k] & 127u));
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bars.tmem_empty[st]));
      }
      if (live) {
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < NK; ++k) sum += tv[k];
        const int64_t rb = (static_cast<int64_t>(o) * W + w) * HW + m;
        rowsum[rb] = sum;
        if (topk_idx != nullptr) {
#pragma unroll
          for (int k = 0; k < NK; ++k) topk_idx[rb * NK + k] = ti[k];
        }
      }
    };
    if (KSTREAM) {
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) do_class(item / W, item % W);
    } else {
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
        for (int w = 0; w < W; ++w) do_class(tile, w);
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 5) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
  }
}

// score[o, w] = sum over the HW descriptors of query o of their top-k sums: one warp per query, lanes stride the
// positions, fixed-order shuffle reduction (deterministic); lane 0 takes the argmax over the classes.
__global__ void __launch_bounds__(128)
dn4_tc2_reduce_kernel(const float* __restrict__ rowsum, int NQ, int W, int HW, float* __restrict__ score,
                      int32_t* __restrict__ pred) {
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (o >= NQ) return;
  float best = -INFINITY;
  int best_w = 0;
  for (int w = 0; w < W; ++w) {
    const float* p = rowsum + (static_cast<int64_t>(o) * W + w) * HW;
    float s = 0.f;
    for (int m = lane; m < HW; m += 32) s += p[m];
    s = warp_sum(s);
    if (lane == 0) score[static_cast<int64_t>(o) * W + w] = s;
    if (s > best) { best = s; best_w = w; }
  }
  if (pred != nullptr && lane == 0) pred[o] = best_w;
}

template <int NK, bool KSTREAM>
cudaError_t launch_tc2_impl(dim3 grid, size_t smem, cudaStream_t stream, const CUtensorMap& mq, const CUtensorMap& ms,
                            const int32_t* cls_row, int W, int S, int C, int HW, float* rowsum, int32_t* topk_idx) {
  cudaError_t e = cudaFuncSetAttribute(dn4_tc2_kernel<NK, KSTREAM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  dn4_tc2_kernel<NK, KSTREAM><<<grid, kThreads2, smem, stream>>>(mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx);
  return cudaSuccess;
}

template <int NK>
cudaError_t launch_tc2(dim3 grid, size_t smem, cudaStream_t stream, const CUtensorMap& mq, const CUtensorMap& ms,
                       const int32_t* cls_row, int W, int S, int C, int HW, float* rowsum, int32_t* topk_idx) {
  if (C > 128) return launch_tc2_impl<NK, true>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx);
  return launch_tc2_impl<NK, false>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx);
}

size_t align256b(size_t x) { return (x + 255) / 256 * 256; }

}  // namespace
}  // namespace afs

extern "C" size_t afs_dn4_tc2_workspace_bytes(int32_t N, int32_t E, int32_t W, int32_t S, int32_t C, int32_t HW) {
  if (N <= 0 || E <= 0 || W <= 0 || S <= 0 || C <= 0 || HW <= 0) return 0;
  const int64_t nq = static_cast<int64_t>(N) - static_cast<int64_t>(E) * W * S;
  if (nq <= 0) return 0;
  return afs::align256b(static_cast<size_t>(nq) * HW * C * sizeof(float)) +
         afs::align256b(static_cast<size_t>(E) * W * S * HW * C * sizeof(float)) +
         afs::align256b(static_cast<size_t>(nq) * W * HW * sizeof(float));
}

extern "C" int afs_dn4_fwd_tc2(const float* feat, const int32_t* cls_row, int32_t N, int32_t E, int32_t W,
                               int32_t S, int32_t C, int32_t HW, int32_t n_k, float* score, int32_t* topk_idx,
                               int32_t* pred, void* ws, size_t ws_bytes, afs_stream_t stream_) {
  using namespace afs;
  if (feat == nullptr || cls_row == nullptr || score == nullptr || E < 0 || W < 1 || W > kMaxWay2 || S < 1 ||
      C < 1 || HW < 1 || N < E * W * S || n_k < 1 || n_k > 8 || n_k > S * HW)
    return AFS_ERR_INVALID_ARG;
  if ((C & 31) != 0 || C > 4096) return AFS_ERR_UNSUPPORTED;
  const int NQ = N - E * W * S;
  if (E == 0 || NQ == 0) return AFS_OK;
  if (E > 65535) return AFS_ERR_UNSUPPORTED;
  if (ws == nullptr || ws_bytes < afs_dn4_tc2_workspace_bytes(N, E, W, S, C, HW) ||
      (reinterpret_cast<uintptr_t>(ws) & 255) != 0)
    return AFS_ERR_WORKSPACE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const uint64_t q_rows = static_cast<uint64_t>(NQ) * HW, s_rows = static_cast<uint64_t>(E) * W * S * HW;
  float* nfq = static_cast<float*>(ws);
  float* nfs = reinterpret_cast<float*>(static_cast<char*>(ws) + align256b(q_rows * C * sizeof(float)));
  float* rowsum = reinterpret_cast<float*>(reinterpret_cast<char*>(nfs) + align256b(s_rows * C * sizeof(float)));

  CUtensorMap mq, ms;
  if (!make_map(&mq, nfq, q_rows, C) || !make_map(&ms, nfs, s_rows, C)) return AFS_ERR_UNSUPPORTED;

  {
    const size_t prep_smem = static_cast<size_t>(C) * kPrepPitch * sizeof(float);
    if (prep_smem > 200 * 1024 || (HW + kPrepPos - 1) / kPrepPos > 65535) return AFS_ERR_UNSUPPORTED;
    if (prep_smem > 48 * 1024)
      AFS_CUDA_TRY(cudaFuncSetAttribute(dn4_tc_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(prep_smem)));
    const dim3 pgrid(N, (HW + kPrepPos - 1) / kPrepPos);
    dn4_tc_prep_kernel<<<pgrid, kPrepThreads, prep_smem, stream>>>(feat, cls_row, E * W, S, C, HW, nfq, nfs);
    AFS_LAUNCH_CHECK();
  }

  const int64_t avg_rows = static_cast<int64_t>(NQ) * HW / E;
  int tiles = static_cast<int>((avg_rows + kRows2 - 1) / kRows2);
  if (tiles < 1) tiles = 1;
  if (C > 128) {  // K-streaming: persistent CTAs over the (row tile, class) items of their episode, ~one CTA per SM in all
    int per_episode = kNumSMs / E;
    if (per_episode < 1) per_episode = 1;
    if (per_episode > tiles * W) per_episode = tiles * W;
    tiles = per_episode;
  }
  const dim3 grid(tiles, 1, E);
  const size_t smem = (C > 128 ? static_cast<size_t>(kStgK) * (1 + kGrpK) : 3 * static_cast<size_t>(C / 32)) * kAtomBytes + 1024;
  cudaError_t err = cudaSuccess;
  switch (n_k) {
    case 1: err = launch_tc2<1>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    case 2: err = launch_tc2<2>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    case 3: err = launch_tc2<3>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    case 4: err = launch_tc2<4>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    case 5: err = launch_tc2<5>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    case 6: err = launch_tc2<6>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    case 7: err = launch_tc2<7>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
    default: err = launch_tc2<8>(grid, smem, stream, mq, ms, cls_row, W, S, C, HW, rowsum, topk_idx); break;
  }
  if (err != cudaSuccess) return cuda_fail(err);
  AFS_LAUNCH_CHECK();
  dn4_tc2_reduce_kernel<<<(NQ + 3) / 4, 128, 0, stream>>>(rowsum, NQ, W, HW, score, pred);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

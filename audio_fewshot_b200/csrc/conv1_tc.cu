// First Conv64F block on the tensor cores: Conv2d(1->64, 3x3, pad 1) + BatchNorm(eval) + ReLU/LeakyReLU +
// MaxPool2d(3,3) as tcgen05 TF32 MMAs with the max-pool done on the accumulators in tensor memory.  sm_100a.
//
// Same operator as csrc/conv1.cu (reference libfewshot_core/model/backbone/conv_four.py:61-66,101-103);
// conv1.cu is the exact-fp32 SIMT kernel and is FMA-pipe bound (9 conv positions x 9 taps x 64 channels per
// pooled pixel: 0.37 ms per 800 clips, 69 % of the fp32 FMA peak).  The reference runs its convolutions in
// TF32 by default (torch.backends.cudnn.allow_tf32 = True), and under that setting this kernel is used.
//
// Formulation: a tile is 128 POOLED pixels = 128 accumulator rows = 128 TMEM lanes.  The conv output at each of the 9
// positions of the pooling window is an accumulator column block of the SAME lane, so the max-pool is an elementwise
// max over nine accumulators and needs no cross-thread traffic at all.  One operand row serves a whole window ROW g:
// A_g[128 x 16] holds patch rows g..g+2 x all five patch columns (K index 5 r + c, K 15 = 0) and ONE resident weight
// tile B[16 x 192] has column 64 dx + ch = tap (r, c - dx) of channel ch (zero where c - dx is outside 0..2):
//   D_g[128 x 192] = A_g . B   = the three window columns dx of row g, side by side  (2 MMAs M128 N192 K8 per row).
// (The first tensor-core version ran one [128 x 16].[16 x 64] GEMM per window position: 18 N = 64 MMAs and 72 KB of
// im2col stores per tile instead of 6 N = 192 MMAs and 24 KB; N <= 64 MMAs cost >= 50 clk whatever N is.)
//
// One persistent CTA per SM, 13 warps in three roles chained by mbarriers:
//   BUILD warps 0-3   thread = pooled pixel: 5x5 input patch (prefetched one tile ahead), TF32 rounding, the three
//                     operand rows of the tile (K-major no-swizzle UMMA layout, conflict-free 128-bit stores) into one
//                     of four 24 KB operand buffers
//   EPI   warps 4-11  thread = (pooled pixel, 32-channel half): the three windows of a row with three tcgen05.ld behind
//                     one wait, accumulators handed back, FMNMX3 folds into the running max, + folded shift,
//                     activation; each thread writes its pixel's 32 channels into the warp's staging box (32 pixels x
//                     32 channels, the TMA swizzle applied: 128-byte rows, 64-byte for the bf16 output) and one lane
//                     stores the box with a TMA tensor store.  Two boxes per warp, so a tile's store drains while the
//                     next tile is folded; TMA drops the rows of a tail tile past the last pixel.
//   MMA   warp 12     one thread: per window row 2 tcgen05.mma M128 N192 K8 (TF32) into one of two 192-column
//                     accumulator sets; tcgen05.commit hands accumulators to the epilogue and operand buffers back
//                     to BUILD
// Measured on B200, 3 200 clips (profiles/r02_conv1_tc_variants.txt): round-1 kernel 1.08 ms; warp-specialised with
// per-thread stores 0.95 ms, staged stores 0.77-0.83 ms, window-row operands 0.67-0.69 ms, trimmed epilogue 0.637 ms.
// TMA box stores (tools/time_stem.py, profiles/r03_stem_tma_store.txt; B200 at 1 000 W, alternating with the staged
// store in one process): 0.636-0.642 -> 0.539-0.542 ms (fp32 output), 0.631 -> 0.531 ms (bf16), bit-identical; the
// staged store's transposed shared-memory reads, 64-bit address arithmetic and predicated STG.E.128 are gone from the
// EPI chain.
// What bounds it (profiles/r02_stem_rows_ncu.txt, before the TMA store): the EPI warps' own latency chain -- TMEM-load
// data and fixed-latency dependencies at two EPI warps per scheduler; they never wait for the tensor core.  Tried and
// slower: 16 EPI warps of 16 channels (with and without a setmaxnreg register split), two BUILD groups, a
// software-pipelined epilogue over 8-channel groups (0.691 ms), spinning instead of suspended mbarrier waits (no change).
// Tried and not merged: rolling TMEM loads (row g+1's tcgen05.ld issued into each window's registers as soon as row g's
// maxima have consumed them, and the next tile's first row issued before this tile's store).  A row's three windows
// and the running maxima are 96 + 32 = 128 registers, so a load in flight before a row is fully folded needs registers
// 13 warps do not have: every arrangement spilled (188-748 B of spill stores per thread, -Xptxas -v) and ran 1.19-1.82 ms,
// and a 16-warp setmaxnreg split (EPI 144-160 registers) still spilled 56-360 B in the EPI code.
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace afs {
namespace {

using namespace tc;

constexpr int kPix1 = 128;                 // pooled pixels per tile
constexpr int kCh1 = 64;                   // output channels == UMMA N
constexpr int kThreads1 = 32 * 13;         // 4 BUILD + 8 EPI + 1 MMA warps
constexpr int kMmaWarp1 = 12;
constexpr int kNBuf1 = 4;                             // operand buffers (tiles BUILD may run ahead of the tensor core)
constexpr uint32_t kWinBytes = 4u * kPix1 * 16u;      // one window ROW's P_g: [4 chunks][128 rows][16 B] = 8 KB
constexpr uint32_t kTileBytes = 3u * kWinBytes;       // three window rows: 24 KB
constexpr uint32_t kAccCols = 3u * kCh1;              // one window row: three accumulators side by side = UMMA N
constexpr uint32_t kWBytes = 4u * kAccCols * 16u;     // Wf: [4 chunks][192 rows][16 B] = 12 KB
constexpr uint32_t kBoxBytes = 32u * 32u * 4u;        // one EPI warp's output box: 32 pixels x 32 channels (fp32)
constexpr uint32_t kStageOff = kNBuf1 * kTileBytes + kWBytes;  // two boxes per EPI warp from here (1024-aligned)
constexpr size_t kSmem1 = kStageOff + 8u * 2u * kBoxBytes + 1024u;  // + the base's alignment to 1024 B
constexpr uint32_t kTmemCols1 = 512;

struct Conv1TcParams {
  float w[kCh1 * 9];  // folded weights [c][ky][kx]
  float shift[kCh1];
};

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t bf162_bits(__nv_bfloat162 p) { return *reinterpret_cast<const uint32_t*>(&p); }

enum { kAFull = 0, kAEmpty = kNBuf1, kAccFull = 2 * kNBuf1, kAccEmpty = 2 * kNBuf1 + 2, kBars1 = 2 * kNBuf1 + 4 };

// OBF16: the channels-last output is written as bf16 (the input of the bf16 blocks of csrc/conv3_tc.cu) instead of fp32
template <bool LEAKY, bool OBF16>
__global__ void __launch_bounds__(kThreads1, 1)
conv1_tc_kernel(const float* __restrict__ x, int64_t total_pix, int H, int Wd, int PH, int PW, float slope,
                const __grid_constant__ CUtensorMap out_map,
                const __grid_constant__ Conv1TcParams prm) {
  // [kNBuf1][kTileBytes] patches | [kWBytes] weights | [8 EPI warps][2][kBoxBytes] output staging, from a 1024-byte
  // aligned base (the staging boxes are read by TMA with a 128-byte swizzle)
  extern __shared__ __align__(1024) uint8_t s_raw[];
  __shared__ __align__(8) uint64_t s_bars[kBars1];
  __shared__ uint32_t s_tmem;
  __shared__ __align__(16) float s_shift[kCh1];

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  uint8_t* s_buf = s_raw + ((1024u - (smem_u32(s_raw) & 1023u)) & 1023u);
  const uint32_t a_base = smem_u32(s_buf);
  const uint32_t stage_base = a_base + kStageOff;
  const uint32_t w_base = a_base + kNBuf1 * kTileBytes;
  if (tid < kCh1) s_shift[tid] = prm.shift[tid];
  const uint32_t bars = smem_u32(s_bars);
#define BAR1(id) (bars + 8u * static_cast<uint32_t>(id))

  // folded weights -> K-major operand [chunk][n = 64 dx + channel][4 K values], TF32-rounded.  K index 5 r + c is
  // patch row r (0..2, relative to the window row) and patch column c (0..4); window column dx sees tap (r, c - dx).
  for (int i = tid; i < 4 * static_cast<int>(kAccCols); i += kThreads1) {
    const int chunk = i / static_cast<int>(kAccCols), n = i - chunk * static_cast<int>(kAccCols);
    const int dx = n / kCh1, c = n - dx * kCh1;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = 4 * chunk + j, r = k / 5, kx = k - 5 * r - dx;
      v[j] = (k < 15 && kx >= 0 && kx < 3) ? to_tf32(prm.w[c * 9 + r * 3 + kx]) : 0.f;
    }
    reinterpret_cast<float4*>(s_buf + kNBuf1 * kTileBytes)[i] = make_float4(v[0], v[1], v[2], v[3]);
  }
  if (warp == 0) tmem_alloc(&s_tmem, kTmemCols1);
  if (tid == 32) {
    for (int s = 0; s < kNBuf1; ++s) {
      mbar_init(BAR1(kAFull + s), kPix1);
      mbar_init(BAR1(kAEmpty + s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(BAR1(kAccFull + s), 1);
      mbar_init(BAR1(kAccEmpty + s), 256);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = s_tmem;

  const int64_t n_tiles = (total_pix + kPix1 - 1) / kPix1;
  const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp < 4) {
    // =========================================================== BUILD
    float pn[5][5];  // patch of the NEXT tile: its global latency hides behind the current tile's stores
    const uint32_t per = static_cast<uint32_t>(PH * PW);
    auto load_patch = [&](int64_t it) {
      const int64_t tile = blockIdx.x + it * gridDim.x;
      int64_t pix = tile * kPix1 + tid;
      if (pix >= total_pix) pix = total_pix - 1;  // tail rows recompute the last pixel; never stored
      // 32-bit division: the host caps total_pix at 2^31 - 1 (TMA coordinates)
      const uint32_t n32 = static_cast<uint32_t>(pix) / per;
      const int64_t n = n32;
      const uint32_t r = static_cast<uint32_t>(pix) - n32 * per;
      const uint32_t ph = r / static_cast<uint32_t>(PW), pw = r - ph * static_cast<uint32_t>(PW);
      const int y0 = 3 * static_cast<int>(ph) - 1, x0 = 3 * static_cast<int>(pw) - 1;
      // validity of the five rows / columns as bit masks: only the first and the last can fall outside (H, Wd >= 3)
      const uint32_t ym = (y0 >= 0 ? 1u : 0u) | 14u | (y0 + 4 < H ? 16u : 0u);
      const uint32_t xm = (x0 >= 0 ? 1u : 0u) | 14u | (x0 + 4 < Wd ? 16u : 0u);
      const float* rowp = x + (n * H + y0) * static_cast<int64_t>(Wd) + x0;
#pragma unroll
      for (int i = 0; i < 5; ++i) {
#pragma unroll
        for (int j = 0; j < 5; ++j) pn[i][j] = ((ym >> i) & (xm >> j) & 1u) ? __ldg(rowp + j) : 0.f;
        rowp += Wd;
      }
    };
    if (my_tiles > 0) load_patch(0);
    for (int64_t it = 0; it < my_tiles; ++it) {
      const uint32_t st = static_cast<uint32_t>(it % kNBuf1), par = static_cast<uint32_t>((it / kNBuf1) & 1);
      float p[5][5];
#pragma unroll
      for (int i = 0; i < 5; ++i)
#pragma unroll
        for (int j = 0; j < 5; ++j) p[i][j] = to_tf32(pn[i][j]);
      if (it + 1 < my_tiles) load_patch(it + 1);  // in flight while this tile is written
      mbar_wait_warp_sleep(BAR1(kAEmpty + st), par ^ 1u, lane);  // the 6 MMAs that read this buffer have completed
      float4* dst = reinterpret_cast<float4*>(s_buf + st * kTileBytes) + tid;
#pragma unroll
      for (int g = 0; g < 3; ++g) {  // window row g: patch rows g..g+2, all five columns, K index 5 r + c, K 15 = 0
        float4* row = dst + g * (4 * kPix1);
        row[0 * kPix1] = make_float4(p[g][0], p[g][1], p[g][2], p[g][3]);
        row[1 * kPix1] = make_float4(p[g][4], p[g + 1][0], p[g + 1][1], p[g + 1][2]);
        row[2 * kPix1] = make_float4(p[g + 1][3], p[g + 1][4], p[g + 2][0], p[g + 2][1]);
        row[3 * kPix1] = make_float4(p[g + 2][2], p[g + 2][3], p[g + 2][4], 0.f);
      }
      fence_async_smem();
      mbar_arrive(BAR1(kAFull + st));
    }
  } else if (warp == kMmaWarp1) {
    // =========================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t kIdesc = idesc_tf32(kPix1, static_cast<int>(kAccCols));
      const uint64_t dA = desc_kmajor_noswizzle(a_base, 16u * kPix1, 128u);
      const uint64_t dB = desc_kmajor_noswizzle(w_base, 16u * kAccCols, 128u);
      uint32_t r = 0;  // running window-row counter: accumulator set r & 1
      for (int64_t it = 0; it < my_tiles; ++it) {
        const uint32_t st = static_cast<uint32_t>(it % kNBuf1), par = static_cast<uint32_t>((it / kNBuf1) & 1);
        mbar_wait_sleep(BAR1(kAFull + st), par);
#pragma unroll
        for (int g = 0; g < 3; ++g, ++r) {
          const uint32_t as = r & 1u;
          mbar_wait_sleep(BAR1(kAccEmpty + as), ((r >> 1) & 1u) ^ 1u);
          fence_after();
#pragma unroll
          for (int k8 = 0; k8 < 2; ++k8) {
            const uint64_t da = dA + ((st * kTileBytes + g * kWinBytes + k8 * 2u * (16u * kPix1)) >> 4);
            const uint64_t db = dB + ((k8 * 2u * (16u * kAccCols)) >> 4);
            mma_tf32(tmem_base + as * kAccCols, da, db, kIdesc, k8 > 0);
          }
          commit(BAR1(kAccFull + as));
        }
        commit(BAR1(kAEmpty + st));
      }
    }
  } else {
    // =========================================================== EPI: running max over nine windows, store
    const int e = warp - 4;
    const int half = e >> 2;  // channels 32 half .. 32 half + 31; TMEM lane quadrant = warp & 3 = e & 3
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) + 32u * half;
    uint32_t r = 0;
    for (int64_t it = 0; it < my_tiles; ++it) {
      float best[32];
#pragma unroll
      for (int g = 0; g < 3; ++g, ++r) {
        const uint32_t as = r & 1u;
        mbar_wait_warp_sleep(BAR1(kAccFull + as), (r >> 1) & 1u, lane);
        fence_after();
        uint32_t v0[32], v1[32], v2[32];
        tmem_ld32_nowait(t_row + as * kAccCols + 0 * kCh1, v0);
        tmem_ld32_nowait(t_row + as * kAccCols + 1 * kCh1, v1);
        tmem_ld32_nowait(t_row + as * kAccCols + 2 * kCh1, v2);
        tmem_wait_ld();
        fence_before();
        mbar_arrive(BAR1(kAccEmpty + as));  // this thread's part of the accumulator set is in registers
        if (g == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            best[j] = fmaxf(fmaxf(__uint_as_float(v0[j]), __uint_as_float(v1[j])), __uint_as_float(v2[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            best[j] = fmaxf(fmaxf(best[j], __uint_as_float(v0[j])), __uint_as_float(v1[j]));
            best[j] = fmaxf(best[j], __uint_as_float(v2[j]));
          }
        }
      }
      const int64_t tile = blockIdx.x + it * gridDim.x;
      // + folded shift, activation, and this thread's pixel row into the warp's staging box (16-byte chunks at their
      // swizzled positions; conflict-free: 8 consecutive lanes hit 8 different chunk columns); one lane stores the box
      const uint32_t box = stage_base + static_cast<uint32_t>(2 * e + (it & 1)) * kBoxBytes;
      if (lane == 0) bulk_wait_read<1>();  // the store issued from this box two tiles ago has read it
      __syncwarp();
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        // one 128-bit broadcast load of four shifts (a scalar load per channel was 12 % of the kernel's stall samples)
        const float4 sh4 = *reinterpret_cast<const float4*>(s_shift + 32 * half + 4 * c4);
        const float sh[4] = {sh4.x, sh4.y, sh4.z, sh4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float x = best[4 * c4 + k] + sh[k];
          best[4 * c4 + k] = LEAKY ? fmaxf(x, x * slope) : fmaxf(x, 0.f);  // 0 <= slope < 1: max(x, slope x)
        }
        if (OBF16) {
          if (c4 & 1) {  // 8 channels = one 16-byte chunk of the 64-byte row (SWIZZLE_64B: chunk ^= row bits 1-2)
            const float* q = best + 4 * (c4 - 1);
            const __nv_bfloat162 p0 = __floats2bfloat162_rn(q[0], q[1]), p1 = __floats2bfloat162_rn(q[2], q[3]);
            const __nv_bfloat162 p2 = __floats2bfloat162_rn(q[4], q[5]), p3 = __floats2bfloat162_rn(q[6], q[7]);
            const uint32_t c = static_cast<uint32_t>(c4 >> 1) ^ ((static_cast<uint32_t>(lane) >> 1) & 3u);
            st_shared_v4(box + 64u * lane + 16u * c, bf162_bits(p0), bf162_bits(p1), bf162_bits(p2), bf162_bits(p3));
          }
        } else {  // 4 channels = one 16-byte chunk of the 128-byte row (SWIZZLE_128B: chunk ^= row bits 0-2)
          const uint32_t c = static_cast<uint32_t>(c4) ^ (static_cast<uint32_t>(lane) & 7u);
          st_shared_v4(box + 128u * lane + 16u * c, __float_as_uint(best[4 * c4]), __float_as_uint(best[4 * c4 + 1]),
                       __float_as_uint(best[4 * c4 + 2]), __float_as_uint(best[4 * c4 + 3]));
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) {  // pixels past total_pix fall outside the tensor map and are not written
        const int64_t pix0 = tile * kPix1 + (warp & 3) * 32;
        if (pix0 < total_pix) tma_store_2d(&out_map, box, 32 * half, static_cast<int>(pix0));
        bulk_commit();
      }
    }
    if (lane == 0) bulk_wait<0>();  // the output is written and the staging boxes are no longer read
  }
#undef BAR1

  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, kTmemCols1);
}

}  // namespace
}  // namespace afs

namespace afs {
namespace {

template <bool LEAKY, bool OBF16>
int launch_conv1_tc(const float* x, int64_t total, int H, int Wd, int PH, int PW, float slope, const CUtensorMap& map,
                    const Conv1TcParams& prm, unsigned blocks, cudaStream_t stream) {
  AFS_CUDA_TRY(cudaFuncSetAttribute(conv1_tc_kernel<LEAKY, OBF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(kSmem1)));
  conv1_tc_kernel<LEAKY, OBF16><<<blocks, kThreads1, kSmem1, stream>>>(x, total, H, Wd, PH, PW, slope, map, prm);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

int conv1_tc_fwd(const float* x, int32_t N, int32_t H, int32_t Wd, const float* w_folded_host, const float* shift_host,
                 int32_t C, float negative_slope, void* out, bool out_bf16, afs_stream_t stream_) {
  if (x == nullptr || w_folded_host == nullptr || shift_host == nullptr || out == nullptr || N < 0 || H < 3 ||
      Wd < 3 || negative_slope < 0.f)
    return AFS_ERR_INVALID_ARG;
  if (C != kCh1) return AFS_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(out) & 15) != 0) return AFS_ERR_INVALID_ARG;  // TMA stores need 16-byte alignment
  if (negative_slope >= 1.f) return AFS_ERR_UNSUPPORTED;  // the activation is max(v, slope v)
  if (N == 0) return AFS_OK;
  const int PH = H / 3, PW = Wd / 3;
  const int64_t total = static_cast<int64_t>(N) * PH * PW;
  if (total > 0x7fffffffLL) return AFS_ERR_UNSUPPORTED;  // TMA coordinates are 32-bit signed
  const int64_t n_tiles = (total + kPix1 - 1) / kPix1;
  Conv1TcParams prm;
  for (int i = 0; i < kCh1 * 9; ++i) prm.w[i] = w_folded_host[i];
  for (int i = 0; i < kCh1; ++i) prm.shift[i] = shift_host[i];
  // the NHWC output as a [total pixels][64 channels] tensor; one box is one EPI warp's 32 pixels x 32 channels, rows
  // of 128 B (fp32) or 64 B (bf16) swizzled at their own width
  tc::EncodeTiledFn fn = tc::encode_tiled();
  if (fn == nullptr) return AFS_ERR_CUDA;
  CUtensorMap map;
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(kCh1), static_cast<cuuint64_t>(total)};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(kCh1) * (out_bf16 ? 2u : 4u)};
  const cuuint32_t box[2] = {32, 32};
  const cuuint32_t estr[2] = {1, 1};
  if (fn(&map, out_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, out, gdim, gstride,
         box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, out_bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
         CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return AFS_ERR_CUDA;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned blocks = static_cast<unsigned>(n_tiles < kNumSMs ? n_tiles : kNumSMs);  // persistent: one CTA per SM
  const bool leaky = negative_slope > 0.f;
  if (leaky && out_bf16) return launch_conv1_tc<true, true>(x, total, H, Wd, PH, PW, negative_slope, map, prm, blocks, stream);
  if (leaky) return launch_conv1_tc<true, false>(x, total, H, Wd, PH, PW, negative_slope, map, prm, blocks, stream);
  if (out_bf16) return launch_conv1_tc<false, true>(x, total, H, Wd, PH, PW, negative_slope, map, prm, blocks, stream);
  return launch_conv1_tc<false, false>(x, total, H, Wd, PH, PW, negative_slope, map, prm, blocks, stream);
}

}  // namespace
}  // namespace afs

extern "C" int afs_conv1_bn_act_pool3_fwd_tf32(const float* x, int32_t N, int32_t H, int32_t Wd,
                                               const float* w_folded_host, const float* shift_host, int32_t C,
                                               float negative_slope, float* out, afs_stream_t stream_) {
  return afs::conv1_tc_fwd(x, N, H, Wd, w_folded_host, shift_host, C, negative_slope, out, false, stream_);
}

extern "C" int afs_conv1_bn_act_pool3_fwd_tf32_bf16out(const float* x, int32_t N, int32_t H, int32_t Wd,
                                                       const float* w_folded_host, const float* shift_host, int32_t C,
                                                       float negative_slope, void* out_bf16, afs_stream_t stream_) {
  return afs::conv1_tc_fwd(x, N, H, Wd, w_folded_host, shift_host, C, negative_slope, out_bf16, true, stream_);
}

// 64 -> 64 channel 3x3 convolution block of Conv64F on the tensor cores, channels-last:
// Conv2d(64->64, 3x3, pad 1) + BatchNorm(eval, folded) + ReLU/LeakyReLU (+ MaxPool2d(3,3)) in ONE kernel.  sm_100a.
//
// Replaces blocks 2..4 of the reference's Conv64F in eval mode (libfewshot_core/model/backbone/conv_four.py:
// 67-86,104-113).  The reference runs them as cuDNN TF32 implicit GEMMs followed by separate BatchNorm, ReLU and
// MaxPool passes; block 2 alone is the largest kernel of an evaluation step on B200 (0.354 ms per 800 clips as a
// cuDNN conv+bias+ReLU, plus a 447 MB activation round trip to the max-pool).  Precision class: TF32 operands,
// fp32 accumulation -- what torch.backends.cudnn.allow_tf32 = True (PyTorch's and the reference's default) gives.
//
// Formulation ("shifted linear rows").  Think of one image, zero-padded to [H+2, HP = W+2], as a 1-D sequence of
// pixels.  The conv output at linear position q = y*HP + x needs, for tap (dy,dx), the padded pixel at linear
// position q + dy*HP + dx -- a CONSTANT offset.  So if a run of padded pixels sits in shared memory as the K-major
// UMMA operand [pixel][8 channels = 32 bytes] (32-byte swizzle, 8-pixel atoms of 256 bytes back to back), the A
// operand of tap (dy,dx) for 128 consecutive output positions is the same buffer with its start address advanced
// by (dy*HP + dx)*32 bytes: the nine taps need no im2col copies at all, and every A tile is one contiguous 4 KB
// span (33 instead of 32 shared-memory lines when the shift is odd).  The hardware applies the swizzle to absolute
// address bits (checked on B200: the descriptor's base-offset field must stay 0 for shifted starts).  Positions
// with x >= W are junk rows of the GEMM (2 of every HP) and are simply not stored.
//
// A tile is R image rows of one image = NM*128 accumulator rows (R*HP <= NM*128; block 2, HP = 54: R = 9, NM = 4 --
// tiles of 9, 9, 9, 9, 6 rows, 95 % of the accumulator rows useful; R = 6, NM = 3 is the alternative the host compares
// it with per shape, conv3_best_geometry).
// Roles (one persistent CTA per SM, 384 threads; 512 with the second epilogue group):
//   warps 4-7   producers: cp.async 16-byte copies of the tile's padded pixels, 8 channels (two chunks) per ring
//               stage, zero-filled outside the image; stages are released to the tensor core with
//               cp.async.wait_group + fence.proxy.async + mbarrier.arrive.  The ring is rolling: stage kc of the
//               NEXT tile is loaded as soon as the nine taps of the current tile have consumed stage kc.
//   warps 8-11  MMA issuers, one per accumulator: per stage 9 taps of tcgen05.mma.kind::tf32 (M = 128, N = 64,
//               K = 8) into its 64 TMEM columns, double-buffered across tiles (2 x NM x 64 = up to all 512 columns);
//               tcgen05.commit frees the stage.  A short last tile skips the accumulators it does not reach.
//   warps 0-3   epilogue: tcgen05.ld 8 channels at a time, + folded shift, activation, then either a direct
//               channels-last store or the 3x3/3 max-pool through a small shared staging tile.
//   warps 12-15 (bf16 kernel) a second epilogue group with its own staging tile: passes 4-7 while the first runs 0-3.
// All 64x64x9 folded weights stay resident in shared memory (144 KB, pre-packed and TF32-rounded on the host; 72 KB
// as bf16).  The bf16 instantiation (kind::f16, K = 16: half the MMAs) is the separately stated reduced-precision path.
#include <string.h>

#include <cuda_bf16.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace afs {
namespace {

using namespace tc;

constexpr int kC3 = 64;                       // channels in == channels out == UMMA N
constexpr int kThreads3 = 256 + 32 * 4;        // 4 epilogue + 4 producer warps + up to 4 MMA-issuing warps
constexpr int kThreads3E2 = kThreads3 + 128;   // + a second group of 4 epilogue warps (warps 12-15)
constexpr int kRing3 = 4;                     // operand ring stages (8 input channels each)
constexpr uint32_t kTapKcBytes = 2u * kC3 * 16u;          // weights of one (tap, 8-channel group): 2 KB
constexpr uint32_t kWBytes3 = 9u * 8u * kTapKcBytes;      // 147 456 B
// bf16 operands (kind::f16, K = 16 per MMA): a ring stage holds 16 input channels in the same 32 bytes per pixel, the
// weights of one (tap, 16-channel group) are the same 2 KB, there are 4 groups instead of 8 -> half the MMAs per tile,
// and the resident weights shrink to 72 KB, which pays for a 6-stage ring (one and a half tiles of look-ahead) and the
// second epilogue group's staging tile.
constexpr int kRing3B = 6;
constexpr uint32_t kWBytes3B = 9u * 4u * kTapKcBytes;     // 73 728 B
constexpr int kMaxPix3 = 10;                  // 16-byte copies per producer thread and stage (halo <= 640)
constexpr int kCg3 = 8;                       // channels per epilogue pass
constexpr int kStagePitch = 12;               // floats per staged position (8 channels + pad: conflict-free stores)

// Ring depth.  Four accumulators per tile (9 image rows of block 2 instead of 6: 95 % instead of 81 % of the accumulator
// rows are useful) need 20 KB stages and a 24 KB staging tile: next to the 144 KB of TF32 weights that leaves 3 stages.
__host__ __device__ constexpr int ring_stages(bool bf16, int nm) {
  return bf16 ? (nm == 4 ? 5 : kRing3B) : (nm == 4 ? 3 : kRing3);
}

template <int RING>
struct Bars3T {
  uint64_t full[RING], empty[RING];
  uint64_t acc_full[2], acc_empty[2];
};

// kind::f16 instruction descriptor with bf16 operands (a_format = b_format = 1), fp32 accumulate, both K-major
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

__device__ __forceinline__ void store4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void store4(__nv_bfloat16* p, float a, float b, float c, float d) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 v;
  v.x = *reinterpret_cast<const uint32_t*>(&lo);
  v.y = *reinterpret_cast<const uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = v;
}

__device__ __forceinline__ void epi_bar(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

struct Conv3Geom {
  int N, H, W, HP;        // HP = W + 2: padded row pitch
  int R;                  // image rows per tile
  int tiles_per_img;
  int rows;               // image rows the tiles cover (a multiple of 3 when pooling)
  int stage_pos;          // positions the pooling staging tile holds: R * HP rounded up to 8
  int halo;               // padded pixels held per stage: NM*128 + 2*HP + 2, rounded up to a multiple of 8
  int pool;               // 1: MaxPool2d(3,3) fused
  int PH, PW;             // pooled extent (pool == 1)
  float slope;
};

// ---- producer and epilogue building blocks of the kernel below -----------------------------------------------------

// One tile's copy plan of a producer thread: thread pair (2j, 2j+1) copies the two 16-byte halves of one pixel's
// 8-channel group, so a warp reads 16 whole 32-byte sectors and writes 512 contiguous shared-memory bytes per
// instruction.  dst already carries the 32-byte swizzle (16-byte chunk index ^= bit 2 of the pixel index).
struct ProducerPlan {
  const char* src[kMaxPix3];
  uint32_t dst[kMaxPix3], nbytes[kMaxPix3];

  // esz: bytes per activation element (4: fp32 / TF32 stages of 8 channels, 2: bf16 stages of 16 channels)
  __device__ __forceinline__ void setup(const char* x, int esz, const Conv3Geom& g, int ptid, int n, int y0) {
    const int half = ptid & 1;
#pragma unroll
    for (int i = 0; i < kMaxPix3; ++i) {
      const int h = (ptid >> 1) + 64 * i;  // padded pixel index inside the tile's run
      const int hr = h / g.HP, hc = h - hr * g.HP;
      const int y = y0 - 1 + hr, xx = hc - 1;
      const bool ok = h < g.halo && hr <= g.R + 1 && y >= 0 && y < g.H && xx >= 0 && xx < g.W;
      src[i] = (ok ? x + ((static_cast<int64_t>(n) * g.H + y) * g.W + xx) * (kC3 * esz) : x) + half * 16;
      nbytes[i] = ok ? 16u : 0u;   // 0 -> the 16 destination bytes are zero-filled (padding)
      dst[i] = static_cast<uint32_t>(h) * 32u + ((static_cast<uint32_t>(half) ^ ((static_cast<uint32_t>(h) >> 2) & 1u)) << 4);
    }
  }
  __device__ __forceinline__ void issue(uint32_t stage_addr, int kc, int ptid, int halo) const {
#pragma unroll
    for (int i = 0; i < kMaxPix3; ++i) {
      if ((ptid >> 1) + 64 * i < halo) cp_async16(stage_addr + dst[i], src[i] + kc * 32, nbytes[i]);
    }
    cp_async_commit();
  }
};

// Producer loop over this CTA's tiles.  RING stages, at most AHEAD of them in flight before the oldest is handed
// over; a thread that is about to block on a slot the tensor core still reads first hands over everything it has in
// flight.  next_tile(j) returns the j-th tile of this CTA or -1.
template <int RING, int AHEAD, int KC, class NextTile>
__device__ __forceinline__ void producer_loop(const char* x, int esz, const Conv3Geom& g, int ptid, int lane, uint32_t ring_base,
                                              uint32_t stage_bytes, uint64_t* full, uint64_t* empty, NextTile next_tile) {
  uint32_t gs = 0;       // stages issued so far (all tiles)
  uint32_t pending = 0;  // issued, not yet signalled: stages gs - pending .. gs - 1
  for (int j = 0;; ++j) {
    const int tile = next_tile(j);
    if (tile < 0) break;
    const int n = tile / g.tiles_per_img;
    const int y0 = (tile - n * g.tiles_per_img) * g.R;
    ProducerPlan plan;
    plan.setup(x, esz, g, ptid, n, y0);
#pragma unroll 1
    for (int kc = 0; kc < KC; ++kc, ++gs) {
      const uint32_t st = gs % RING, ph = (gs / RING) & 1u;
      uint32_t ready = lane == 0 ? (mbar_test(smem_u32(&empty[st]), ph ^ 1u) ? 1u : 0u) : 0u;
      ready = __shfl_sync(0xffffffffu, ready, 0);
      if (pending > 0 && !ready) {
        cp_async_wait<0>();
        fence_async_smem();
        for (; pending > 0; --pending) mbar_arrive(smem_u32(&full[(gs - pending) % RING]));
      }
      if (!ready) mbar_wait_warp(smem_u32(&empty[st]), ph ^ 1u, lane);
      plan.issue(ring_base + st * stage_bytes, kc, ptid, g.halo);
      ++pending;
      if (pending > static_cast<uint32_t>(AHEAD)) {
        cp_async_wait<AHEAD>();
        fence_async_smem();
        mbar_arrive(smem_u32(&full[(gs + 1 - pending) % RING]));
        --pending;
      }
    }
  }
  cp_async_wait<0>();
  fence_async_smem();
  for (; pending > 0; --pending) mbar_arrive(smem_u32(&full[(gs - pending) % RING]));
}

// Epilogue passes cg0 .. cg1-1 (8 channels each) of one tile by a group of four epilogue warps (accumulator row ==
// TMEM lane == tid): tcgen05.ld 8 channels at a time, + folded shift, activation, then a direct channels-last store or
// the 3x3/3 max-pool through the group's staging tile (synchronised on the group's named barrier `bar`).  A pass is a
// chain of latencies (TMEM load, staging store, barrier, staging reads, store, barrier: ~1 300 clk) rather than of
// work, so a second group running the other half of the passes on its own staging tile halves the epilogue time.
// release() is called once per warp as soon as the warp's share of the accumulator set has been read completely.
template <int NM, typename TOut, class Release>
__device__ __forceinline__ void epilogue_tile(const Conv3Geom& g, int n, int y0, bool store, uint32_t d0, float* s_stage,
                                              const float* s_shift, TOut* __restrict__ out, int tid, int cg0, int cg1,
                                              int bar, Release release) {
#pragma unroll 1
  for (int cg = cg0; cg < cg1; ++cg) {
    uint32_t v[NM][kCg3];
#pragma unroll
    for (int m = 0; m < NM; ++m) tmem_ld8(d0 + m * kC3 + cg * kCg3, v[m]);
    tmem_wait_ld();
    if (cg == cg1 - 1) {  // every value of this accumulator set this warp needs is in registers: hand it back
      fence_before();
      __syncwarp();
      release();
    }
#pragma unroll
    for (int m = 0; m < NM; ++m) {
      float r[kCg3];
#pragma unroll
      for (int j = 0; j < kCg3; ++j) {
        const float a = __uint_as_float(v[m][j]) + s_shift[cg * kCg3 + j];
        r[j] = a > 0.f ? a : a * g.slope;
      }
      const int q = m * 128 + tid;  // linear position inside the tile
      if (g.pool) {
        if (q < g.stage_pos) {  // positions past the tile's last row are junk rows of the last accumulator
          float4* d = reinterpret_cast<float4*>(s_stage + q * kStagePitch);
          d[0] = make_float4(r[0], r[1], r[2], r[3]);
          d[1] = make_float4(r[4], r[5], r[6], r[7]);
        }
      } else {
        const int yy = q / g.HP, xx = q - yy * g.HP;
        if (store && yy < g.R && y0 + yy < g.H && xx < g.W) {
          TOut* d = out + ((static_cast<int64_t>(n) * g.H + y0 + yy) * g.W + xx) * kC3 + cg * kCg3;
          store4(d, r[0], r[1], r[2], r[3]);
          store4(d + 4, r[4], r[5], r[6], r[7]);
        }
      }
    }
    if (g.pool) {
      epi_bar(bar);
      const int prt = g.R / 3;                 // pooled rows of this tile
      const int npp = prt * g.PW;
      const int items = npp * 2;               // (4-channel half of the group, pooled pixel): pixel fastest, so
      for (int it = tid; it < items; it += 128) {  // a quarter-warp reads 8 pixels 3*12 floats apart: no conflicts
        const int c4 = it >= npp ? 1 : 0, pp = it - c4 * npp;
        const int pyl = pp / g.PW, px = pp - pyl * g.PW;
        const int py = y0 / 3 + pyl;
        if (store && py < g.PH) {
          const float* s = s_stage + ((3 * pyl) * g.HP + 3 * px) * kStagePitch + c4 * 4;
          float4 best = *reinterpret_cast<const float4*>(s);
#pragma unroll
          for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              const float4 t = *reinterpret_cast<const float4*>(s + (i * g.HP + j) * kStagePitch);
              best.x = fmaxf(best.x, t.x); best.y = fmaxf(best.y, t.y);
              best.z = fmaxf(best.z, t.z); best.w = fmaxf(best.w, t.w);
            }
          }
          store4(out + ((static_cast<int64_t>(n) * g.PH + py) * g.PW + px) * kC3 + cg * kCg3 + c4 * 4, best.x, best.y, best.z,
                 best.w);
        }
      }
      epi_bar(bar);
    }
  }
}

// ---- one CTA per SM ------------------------------------------------------------------------------------------------
// BF16 = false: fp32 activations, TF32 MMAs (K = 8 channels per stage, 8 stages per tile).  BF16 = true: bf16
// activations and weights, kind::f16 MMAs (K = 16 channels per stage, 4 stages per tile) -- the separately stated
// reduced-precision path (Conv64F(precision="bf16")).  TOut: element type of the channels-last output.
// EPI2: a second group of four epilogue warps (warps 11-14) with its own staging tile runs passes 4-7 while the first
// runs passes 0-3 -- the bf16 kernel has half the MMAs per tile and would otherwise wait for the epilogue (the TF32
// kernel has no shared memory left for a second staging tile, and is MMA-bound).
template <int NM, bool BF16, typename TOut, bool EPI2>
__global__ void __launch_bounds__(EPI2 ? kThreads3E2 : kThreads3, 1)
conv3x3_c64_tc_kernel(const void* __restrict__ x, const void* __restrict__ wpk, const float* __restrict__ shift,
                      TOut* __restrict__ out, const Conv3Geom g) {
  constexpr int RING = ring_stages(BF16, NM);
  constexpr int AHEAD = RING - (BF16 ? 2 : 1);
  constexpr int KC = BF16 ? 4 : 8;                       // ring stages (K groups) per tile
  constexpr uint32_t kWB = BF16 ? kWBytes3B : kWBytes3;  // resident weights
  extern __shared__ __align__(16) uint8_t s_dyn_raw[];  // [weights][ring][staging][shift] after 256-byte alignment
  __shared__ __align__(8) Bars3T<RING> bars;
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const uint32_t stage_bytes = static_cast<uint32_t>(g.halo) * 32u;
  uint8_t* s_dyn = s_dyn_raw + ((256u - (smem_u32(s_dyn_raw) & 255u)) & 255u);  // swizzle atoms are 256 B
  const uint32_t w_base = smem_u32(s_dyn);
  const uint32_t ring_base = w_base + kWB;
  float* s_stage = reinterpret_cast<float*>(s_dyn + kWB + RING * stage_bytes);
  float* s_shift = s_stage + (EPI2 ? 2 : 1) * g.stage_pos * kStagePitch;
  constexpr uint32_t kTmemCols = NM == 1 ? 128u : (NM == 2 ? 256u : 512u);  // 2 x NM accumulators of 64 columns
  static_assert(NM >= 1 && NM <= 4, "two sets of NM 64-column accumulators must fit 512 TMEM columns");
  constexpr uint32_t kIdesc = BF16 ? idesc_bf16(128, kC3) : idesc_tf32(128, kC3);

  {  // resident weights (already in operand layout) and the folded shift
    const uint4* src = reinterpret_cast<const uint4*>(wpk);
    uint4* dst = reinterpret_cast<uint4*>(s_dyn);
    for (int i = tid; i < static_cast<int>(kWB / 16); i += (EPI2 ? kThreads3E2 : kThreads3)) dst[i] = __ldg(src + i);
    if (tid < kC3) s_shift[tid] = shift[tid];
  }
  if (tid == 0) {
    for (int s = 0; s < RING; ++s) {
      mbar_init(smem_u32(&bars.full[s]), 128);  // every producer thread arrives
      mbar_init(smem_u32(&bars.empty[s]), NM);  // one tcgen05.commit per MMA-issuing warp
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&bars.acc_full[s]), NM);
      mbar_init(smem_u32(&bars.acc_empty[s]), EPI2 ? 8 : 4);  // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) tmem_alloc(&s_tmem, kTmemCols);
  fence_async_smem();  // weights -> visible to the tensor core (async proxy)
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = s_tmem;
  const int total_tiles = g.N * g.tiles_per_img;
  auto next_tile = [&](int j) {
    const int64_t t = blockIdx.x + static_cast<int64_t>(j) * gridDim.x;
    return t < total_tiles ? static_cast<int>(t) : -1;
  };

  if (warp >= 4 && warp < 8) {
    // ======================= producers =======================
    producer_loop<RING, AHEAD, KC>(static_cast<const char*>(x), BF16 ? 2 : 4, g, tid - 128, lane, ring_base, stage_bytes,
                                   bars.full, bars.empty, next_tile);
  } else if (warp >= 8 && warp < 12) {
    // ======================= MMA issuers: warp 8 + m owns accumulator m of every tile =======================
    // (a single issuing thread spends ~80 cycles per tcgen05.mma on descriptor arithmetic and the election
    // wrapper, more than the 48 cycles the tensor core needs for M=128, N=64, K=8 from shared memory)
    const int m = warp - 8;
    if (m < NM && lane == 0) {
      uint32_t gs = 0, lt = 0;
      const uint64_t a_desc0 = desc_kmajor_sw32(ring_base + static_cast<uint32_t>(m) * 128u * 32u, 256u, 0u);
      const uint64_t b_desc0 = desc_kmajor_noswizzle(w_base, kC3 * 16u, 128u);
      uint32_t tap_off[9];  // start-address advance of tap (dy,dx) in 16-byte units
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) tap_off[tap] = static_cast<uint32_t>((tap / 3) * g.HP + tap % 3) * 2u;
      for (int j = 0;; ++j, ++lt) {
        const int tile = next_tile(j);
        if (tile < 0) break;
        // a short last tile of an image (fewer rows than R) may not reach this warp's accumulator: no MMAs then, but
        // the commits below still arrive so that every barrier keeps its count
        const int y0 = (tile % g.tiles_per_img) * g.R;
        const int rows_t = g.rows - y0 < g.R ? g.rows - y0 : g.R;
        const bool active = m * 128 < rows_t * g.HP;
        const uint32_t ab = lt & 1u, aph = (lt >> 1) & 1u;
        mbar_wait(smem_u32(&bars.acc_empty[ab]), aph ^ 1u);  // epilogue has drained this accumulator set
        fence_after();
        const uint32_t d_tmem = tmem_base + ab * (NM * kC3) + m * kC3;
#pragma unroll 1
        for (int kc = 0; kc < KC; ++kc, ++gs) {
          const uint32_t st = gs % RING, ph = (gs / RING) & 1u;
          mbar_wait(smem_u32(&bars.full[st]), ph);
          fence_after();
          const uint64_t da_st = a_desc0 + ((st * stage_bytes) >> 4);
          const uint64_t db_kc = b_desc0 + static_cast<uint32_t>(kc) * (kTapKcBytes >> 4);
          if (active) {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const uint64_t da = da_st + tap_off[tap];
              const uint64_t db = db_kc + static_cast<uint32_t>(tap) * (static_cast<uint32_t>(KC) * kTapKcBytes >> 4);
              if (BF16) mma_f16(d_tmem, da, db, kIdesc, (kc | tap) != 0);
              else mma_tf32(d_tmem, da, db, kIdesc, (kc | tap) != 0);
            }
          }
          commit(smem_u32(&bars.empty[st]));  // stage reusable once these MMAs have read it
        }
        commit(smem_u32(&bars.acc_full[ab]));
      }
    }
  } else {
    // ======================= epilogue (warps 0-3; with EPI2 also warps 11-14) =======================
    // a warp may only read the TMEM lanes 32 (warp % 4) .. + 31: that quarter is its share of the accumulator rows
    uint32_t lt = 0;
    const int part = warp >= 12 ? 1 : 0;
    const int etid = (warp & 3) * 32 + lane;
    const uint32_t t_lane = static_cast<uint32_t>((warp & 3) * 32) << 16;
    for (int j = 0;; ++j, ++lt) {
      const int tile = next_tile(j);
      if (tile < 0) break;
      const int n = tile / g.tiles_per_img;
      const int y0 = (tile - n * g.tiles_per_img) * g.R;
      const uint32_t ab = lt & 1u, aph = (lt >> 1) & 1u;
      mbar_wait_warp(smem_u32(&bars.acc_full[ab]), aph, lane);
      fence_after();
      epilogue_tile<NM, TOut>(g, n, y0, true, tmem_base + ab * (NM * kC3) + t_lane,
                              s_stage + part * (g.stage_pos * kStagePitch), s_shift, out, etid, EPI2 ? 4 * part : 0,
                              EPI2 ? 4 * part + 4 : 8, 1 + part, [&]() {
        if (lane == 0) mbar_arrive(smem_u32(&bars.acc_empty[ab]));
      });
    }
  }

  fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem_base, kTmemCols);
}

template <int NM, bool BF16, typename TOut, bool EPI2>
int launch_conv3(const void* x, const void* wpk, const float* shift, TOut* out, Conv3Geom g, cudaStream_t stream) {
  g.halo = (NM * 128 + 2 * g.HP + 2 + 7) & ~7;
  const size_t smem = (BF16 ? kWBytes3B : kWBytes3) + ring_stages(BF16, NM) * (g.halo * 32u) +
                      static_cast<size_t>(EPI2 ? 2 : 1) * g.stage_pos * kStagePitch * 4 + kC3 * 4 + 256;
  if (smem + 256u > 232448u) return AFS_ERR_UNSUPPORTED;  // 227 KB per CTA, static barriers included
  AFS_CUDA_TRY(cudaFuncSetAttribute(conv3x3_c64_tc_kernel<NM, BF16, TOut, EPI2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(smem)));
  const int total = g.N * g.tiles_per_img;
  const int blocks = total < kNumSMs ? total : kNumSMs;  // persistent: one CTA per SM
  conv3x3_c64_tc_kernel<NM, BF16, TOut, EPI2><<<blocks, EPI2 ? kThreads3E2 : kThreads3, smem, stream>>>(x, wpk, shift, out, g);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

// Epilogue groups: two for the bf16 kernel (its MMA phase is half as long), one for the TF32 kernel.  The TF32 kernel
// is MMA-bound at every tile size: measured, two groups do not help it even where they fit (block 3, two
// accumulators: 0.155 ms with, 0.144 ms without), and for the large tiles a second staging tile does not fit next to
// its 144 KB of weights.
template <bool BF16, typename TOut>
int dispatch_conv3(int NM, const void* x, const void* wpk, const float* shift, TOut* out, const Conv3Geom& g,
                   cudaStream_t stream) {
  if constexpr (BF16) {
    int rc;
    switch (NM) {
      case 1: rc = launch_conv3<1, BF16, TOut, true>(x, wpk, shift, out, g, stream); break;
      case 2: rc = launch_conv3<2, BF16, TOut, true>(x, wpk, shift, out, g, stream); break;
      case 3: rc = launch_conv3<3, BF16, TOut, true>(x, wpk, shift, out, g, stream); break;
      default: rc = launch_conv3<4, BF16, TOut, true>(x, wpk, shift, out, g, stream); break;
    }
    if (rc != AFS_ERR_UNSUPPORTED) return rc;  // else: no room for the second staging tile -> one group
  }
  switch (NM) {
    case 1: return launch_conv3<1, BF16, TOut, false>(x, wpk, shift, out, g, stream);
    case 2: return launch_conv3<2, BF16, TOut, false>(x, wpk, shift, out, g, stream);
    case 3: return launch_conv3<3, BF16, TOut, false>(x, wpk, shift, out, g, stream);
    default: return launch_conv3<4, BF16, TOut, false>(x, wpk, shift, out, g, stream);
  }
}

// Tile geometry shared by the TF32 and the bf16 entry point.  Returns NM (accumulators per tile) or an AFS_ERR_* code (< 0).
// max_nm: 3 or 4 accumulators of 128 rows per tile.  A tile is R image rows (a multiple of 3 when pooling); with 4
// accumulators block 2 (42 x 52, HP = 54) runs tiles of 9, 9, 9, 9, 6 rows = 19 accumulator-tiles per image (the short
// last tile skips its fourth accumulator) instead of 7 x 3 = 21.
int conv3_geometry(int32_t N, int32_t H, int32_t Wd, float negative_slope, int32_t pool3, int max_nm, Conv3Geom* gp) {
  Conv3Geom& g = *gp;
  g.N = N; g.H = H; g.W = Wd; g.HP = Wd + 2; g.pool = pool3 ? 1 : 0; g.slope = negative_slope;
  g.PH = H / 3; g.PW = Wd / 3;
  const int rows_needed = pool3 ? 3 * g.PH : H;  // rows below the last complete pooling window are never used
  int R = max_nm * 128 / g.HP;  // rows per tile: as many as fit the accumulator rows
  if (R > rows_needed) R = rows_needed;
  if (pool3) R -= R % 3;
  if (R < 1) return AFS_ERR_UNSUPPORTED;  // image rows wider than the tile (W > 126 when pooling)
  g.R = R;
  g.rows = rows_needed;
  g.stage_pos = (R * g.HP + 7) & ~7;
  g.tiles_per_img = (rows_needed + R - 1) / R;
  if (static_cast<int64_t>(N) * g.tiles_per_img > 0x7fffffffLL) return AFS_ERR_UNSUPPORTED;
  return (R * g.HP + 127) / 128;
}

// Accumulator-tiles (MMA work) per image of a geometry: what the choice between 3 and 4 accumulators minimises.
int conv3_acc_tiles(const Conv3Geom& g) {
  int total = 0;
  for (int y0 = 0; y0 < g.rows; y0 += g.R) {
    const int rows_t = g.rows - y0 < g.R ? g.rows - y0 : g.R;
    total += (rows_t * g.HP + 127) / 128;
  }
  return total;
}

// Geometry with the accumulator count (three or four) that needs the fewest MMAs.
int conv3_best_geometry(int32_t N, int32_t H, int32_t Wd, float negative_slope, int32_t pool3, Conv3Geom* gp) {
  Conv3Geom g3, g4;
  const int nm3 = conv3_geometry(N, H, Wd, negative_slope, pool3, 3, &g3);
  if (nm3 < 0) {
    *gp = g3;
    return nm3;
  }
  const int nm4 = conv3_geometry(N, H, Wd, negative_slope, pool3, 4, &g4);
  if (nm4 == 4 && conv3_acc_tiles(g4) < conv3_acc_tiles(g3)) {
    *gp = g4;
    return nm4;
  }
  *gp = g3;
  return nm3;
}

inline uint16_t round_bf16_host(float v) {  // round to nearest even (what __float2bfloat16_rn does); NaN kept quiet
  uint32_t b;
  memcpy(&b, &v, 4);
  if ((b & 0x7f800000u) == 0x7f800000u) return static_cast<uint16_t>((b >> 16) | ((b & 0xffffu) ? 0x40u : 0u));
  b += 0x7fffu + ((b >> 16) & 1u);
  return static_cast<uint16_t>(b >> 16);
}

inline float round_tf32_host(float v) {  // cvt.rna.tf32.f32: nearest, ties away from zero
  uint32_t b;
  memcpy(&b, &v, 4);
  if ((b & 0x7f800000u) != 0x7f800000u) b = (b + 0x1000u) & ~0x1fffu;
  float r;
  memcpy(&r, &b, 4);
  return r;
}

}  // namespace
}  // namespace afs

extern "C" size_t afs_conv3x3_c64_packed_floats(void) { return afs::kWBytes3 / 4; }

extern "C" int afs_conv3x3_c64_pack_weights(const float* w_folded_host, float* packed_host) {
  using namespace afs;
  if (w_folded_host == nullptr || packed_host == nullptr) return AFS_ERR_INVALID_ARG;
  // packed[tap][kc][chunk][cout][4] <- w[cout][cin = 8 kc + 4 chunk + i][ky][kx], tap = 3 ky + kx
  for (int tap = 0; tap < 9; ++tap)
    for (int kc = 0; kc < 8; ++kc)
      for (int ch = 0; ch < 2; ++ch)
        for (int co = 0; co < kC3; ++co)
          for (int i = 0; i < 4; ++i) {
            const int ci = 8 * kc + 4 * ch + i;
            const float v = round_tf32_host(w_folded_host[(co * kC3 + ci) * 9 + tap]);
            packed_host[(((tap * 8 + kc) * 2 + ch) * kC3 + co) * 4 + i] = v;
          }
  return AFS_OK;
}

extern "C" int afs_conv3x3_c64_bn_act_fwd_tf32(const float* x, int32_t N, int32_t H, int32_t Wd, const float* w_packed,
                                               const float* shift, float negative_slope, int32_t pool3, float* out,
                                               afs_stream_t stream_) {
  using namespace afs;
  if (x == nullptr || w_packed == nullptr || shift == nullptr || out == nullptr || N < 0 || H < 1 || Wd < 1 ||
      negative_slope < 0.f)
    return AFS_ERR_INVALID_ARG;
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(w_packed)) & 15) != 0)
    return AFS_ERR_INVALID_ARG;
  if (pool3 && (H < 3 || Wd < 3)) return AFS_ERR_INVALID_ARG;
  if (Wd > 61) return AFS_ERR_UNSUPPORTED;  // the operand ring of wider rows does not fit next to the weights
  if (N == 0) return AFS_OK;
  Conv3Geom g;
  int NM = conv3_best_geometry(N, H, Wd, negative_slope, pool3, &g);
  if (NM < 0) return NM;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = dispatch_conv3<false, float>(NM, x, w_packed, shift, out, g, stream);
  if (rc == AFS_ERR_UNSUPPORTED && NM == 4) {  // no shared memory for four accumulators' stages: three
    NM = conv3_geometry(N, H, Wd, negative_slope, pool3, 3, &g);
    rc = dispatch_conv3<false, float>(NM, x, w_packed, shift, out, g, stream);
  }
  return rc;
}

extern "C" size_t afs_conv3x3_c64_packed_bf16_elems(void) { return afs::kWBytes3B / 2; }

extern "C" int afs_conv3x3_c64_pack_weights_bf16(const float* w_folded_host, uint16_t* packed_host) {
  using namespace afs;
  if (w_folded_host == nullptr || packed_host == nullptr) return AFS_ERR_INVALID_ARG;
  // packed[tap][kc][chunk][cout][8] <- bf16(w[cout][cin = 16 kc + 8 chunk + i][ky][kx]), tap = 3 ky + kx
  for (int tap = 0; tap < 9; ++tap)
    for (int kc = 0; kc < 4; ++kc)
      for (int ch = 0; ch < 2; ++ch)
        for (int co = 0; co < kC3; ++co)
          for (int i = 0; i < 8; ++i) {
            const int ci = 16 * kc + 8 * ch + i;
            packed_host[(((tap * 4 + kc) * 2 + ch) * kC3 + co) * 8 + i] = round_bf16_host(w_folded_host[(co * kC3 + ci) * 9 + tap]);
          }
  return AFS_OK;
}

extern "C" int afs_conv3x3_c64_bn_act_fwd_bf16(const void* x, int32_t N, int32_t H, int32_t Wd, const void* w_packed,
                                               const float* shift, float negative_slope, int32_t pool3, void* out,
                                               int32_t out_bf16, afs_stream_t stream_) {
  using namespace afs;
  if (x == nullptr || w_packed == nullptr || shift == nullptr || out == nullptr || N < 0 || H < 1 || Wd < 1 ||
      negative_slope < 0.f)
    return AFS_ERR_INVALID_ARG;
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(w_packed)) & 15) != 0)
    return AFS_ERR_INVALID_ARG;
  if (pool3 && (H < 3 || Wd < 3)) return AFS_ERR_INVALID_ARG;
  if (Wd > 61) return AFS_ERR_UNSUPPORTED;
  if (N == 0) return AFS_OK;
  Conv3Geom g;
  int NM = conv3_best_geometry(N, H, Wd, negative_slope, pool3, &g);
  if (NM < 0) return NM;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  for (int attempt = 0; attempt < 2; ++attempt) {
    const int rc = out_bf16 ? dispatch_conv3<true, __nv_bfloat16>(NM, x, w_packed, shift, static_cast<__nv_bfloat16*>(out), g, stream)
                            : dispatch_conv3<true, float>(NM, x, w_packed, shift, static_cast<float*>(out), g, stream);
    if (rc != AFS_ERR_UNSUPPORTED || NM != 4) return rc;
    NM = conv3_geometry(N, H, Wd, negative_slope, pool3, 3, &g);  // no shared memory for four accumulators' stages
  }
  return AFS_ERR_UNSUPPORTED;
}

// Brownian-distance-covariance pooling at C = 128, 192, ..., 640 channels (whole 64-channel blocks), fp32 on the
// FMA pipe.  Same arithmetic as bdc.cu (BDCovpool + Triuvec, bdc_pool.py:69-93), cut into 64 x 64 tiles so that a
// clip's k = C / 64 channel blocks spread over k (k + 1) / 2 CTAs, one per unordered block pair I <= J:
//
//   bdc_wide_norms    n_i = sum_m x_im^2                       (warp per channel row; fixed shuffle tree)
//   bdc_wide_gram     G_IJ = X_I X_J^T in registers, D = max(n_i + n_j - 2 G_ij, 0), A = sqrt(e^t D + 1e-5) into
//                     `out`, and the tile's row sums (and, for I != J, its column sums) into fixed workspace slots
//   bdc_wide_center   r_i = the k slot values of row i in ascending block order, total = sum_i r_i in ascending i,
//                     out_ij = A_ij - r_lo / C - r_hi / C + total / C^2 with lo = min(i, j), hi = max(i, j)
//
// Tiles are independent because D_ii = 0 exactly: the reference's own fp32 D_ii is G_ii + G_ii - 2 G_ii = 0, so the
// norms can come from their own pass and no tile waits for a diagonal tile.  A pair (I, J) is computed once and
// stored at both (i, j) and (j, i), so A is exactly symmetric, its column sums equal its row sums, and the centred
// value is symmetric too (lo / hi ordering).  Every sum has a fixed order that depends on nothing but the clip's
// data: a clip's output is bit-identical whatever the batch size or its position in the batch.  The epilogue uses
// explicitly rounded intrinsics so that the backward's recompute of D and A has the forward's bits.
//
// Backward (same maths as bdc_bwd_kernel, bdc.cu):
//   bdc_wide_norms    as above
//   bdc_wide_dbstats  row sums R, column sums K and total T of dB (dB is zero below the diagonal when triu)
//   bdc_wide_bwd_tile recompute G, D, A of the pair with the forward's code; dA_ij = dB_ij - R_i/C - K_j/C + T/C^2;
//                     dD_ij = [raw >= 0] dA_ij e^t / (2 A_ij) for (i, j) and (j, i); S = dD + dD^T stored per pair
//                     (64 x 64, row-major, pairs I <= J only) with its row sums (and column sums) in fixed slots,
//                     and the pair's log-temperature partial sum_ij dA_ij e^t D_ij / (2 A_ij)
//   bdc_wide_dx       dX_i = -2 sum_j S_ij x_j + 2 sigma_i x_i, sigma_i = sum_j S_ij, tiled over (clip, row block,
//                     64 positions); grad_log_temp[b] = the clip's pair partials in ascending pair order
// The diagonal dD_ii is dropped: D_ii = n_i + n_i - 2 G_ii has zero derivative, so its terms cancel exactly.
#include "common.cuh"

namespace afs {
namespace {

constexpr int kThreads = 256;
constexpr int kBlk = 64;                 // channels per block: the tile unit
constexpr int kMaxBlocks = 10;           // C <= 640
constexpr int kMC = 32;                  // positions per shared-memory chunk of the Gram
constexpr int kXStride = kBlk + 4;       // sX[m][c]: 16-byte aligned rows, conflict-free 128-bit stores
constexpr int kAStride = kBlk + 1;       // sA[r][c]: conflict-free row and column walks
constexpr int kTile = kBlk * kBlk;
constexpr int kDxM = 64;                 // positions per dX tile
constexpr int kGramSmem = 2 * kMC * kXStride;
static_assert(kBlk * kAStride <= kGramSmem, "the A tile reuses the Gram's operand buffer");

// Workspace layout, in floats, every section 16-byte aligned.
struct WideWs {
  size_t norms, rowpart, dbr, dbk, dbt, s, dtpart, total;
};

__host__ __device__ inline size_t align4(size_t n) { return (n + 3) & ~static_cast<size_t>(3); }

__host__ __device__ inline WideWs wide_ws(int64_t B, int C, bool backward) {
  const int64_t k = C / kBlk, P = k * (k + 1) / 2;
  WideWs w{};
  size_t o = 0;
  w.norms = o;   o += align4(static_cast<size_t>(B) * C);
  w.rowpart = o; o += align4(static_cast<size_t>(B) * k * C);  // [b][row block][column block][64]
  if (backward) {
    w.dbr = o;    o += align4(static_cast<size_t>(B) * C);
    w.dbk = o;    o += align4(static_cast<size_t>(B) * C);
    w.dbt = o;    o += align4(static_cast<size_t>(B));
    w.s = o;      o += static_cast<size_t>(B) * P * kTile;     // [b][pair][64][64]
    w.dtpart = o; o += align4(static_cast<size_t>(B) * P);     // [b][pair]
  }
  w.total = o;
  return w;
}

bool wide_supported(int C) { return C % kBlk == 0 && C >= 2 * kBlk && C <= kMaxBlocks * kBlk; }

// Pair p (row-major over I <= J) -> (I, J), and back.
__device__ __forceinline__ void pair_of(int p, int k, int& I, int& J) {
  I = 0;
  int n = k;
  while (p >= n) {
    p -= n;
    --n;
    ++I;
  }
  J = I + p;
}
__device__ __forceinline__ int pair_index(int I, int J, int k) { return I * k - (I * (I - 1)) / 2 + (J - I); }

// Start of row r of the packed upper triangle of a C x C matrix.
__device__ __forceinline__ int64_t triu_row(int r, int C) {
  return static_cast<int64_t>(r) * C - (static_cast<int64_t>(r) * (r - 1)) / 2 - r;
}

// G_IJ for one clip: thread (ti, tj) = (tid >> 4, tid & 15) owns rows 64 I + 4 ti + i, columns 64 J + 4 tj + 2 h + e
// as g[i][h].{x, y}.  Every entry is one FMA chain over m = 0, 1, ..., M - 1 (the packed FMA rounds each lane as
// fmaf), so G_ij and G_ji have the same bits and the forward and the backward's recompute agree.
__device__ __forceinline__ void gram_tile(const float* __restrict__ xb, int M, int I, int J, float* sX,
                                          float2 (&g)[4][2]) {
  const int tid = threadIdx.x, ti = tid >> 4, tj = tid & 15;
  const float* sXI = sX;
  const float* sXJ = I == J ? sX : sX + kMC * kXStride;
#pragma unroll
  for (int i = 0; i < 4; ++i) g[i][0] = g[i][1] = make_float2(0.f, 0.f);
  for (int m0 = 0; m0 < M; m0 += kMC) {
    __syncthreads();
    // slots [block][quad][position]: 2 x 16 x 32; lanes run along m so the global loads are coalesced
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int blk = it >> 1;
      if (blk == 1 && I == J) continue;
      const int slot = tid + kThreads * (it & 1);
      const int lm = slot & (kMC - 1);
      const int c4 = slot >> 5;
      const int m = m0 + lm;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m < M) {
        const float* p = xb + static_cast<int64_t>(kBlk * (blk ? J : I) + 4 * c4) * M + m;
        v.x = __ldg(p);
        v.y = __ldg(p + M);
        v.z = __ldg(p + 2 * static_cast<int64_t>(M));
        v.w = __ldg(p + 3 * static_cast<int64_t>(M));
      }
      *reinterpret_cast<float4*>(&sX[blk * kMC * kXStride + lm * kXStride + 4 * c4]) = v;
    }
    __syncthreads();
#pragma unroll 8
    for (int lm = 0; lm < kMC; ++lm) {
      const float4 a = *reinterpret_cast<const float4*>(&sXI[lm * kXStride + 4 * ti]);
      const float4 c = *reinterpret_cast<const float4*>(&sXJ[lm * kXStride + 4 * tj]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 ai = make_float2(av[i], av[i]);
        g[i][0] = __ffma2_rn(ai, c01, g[i][0]);
        g[i][1] = __ffma2_rn(ai, c23, g[i][1]);
      }
    }
  }
  __syncthreads();  // the operand buffer is free for the epilogue
}

__device__ __forceinline__ float g_at(const float2 (&g)[4][2], int i, int j) {
  return (j & 1) ? g[i][j >> 1].y : g[i][j >> 1].x;
}

// raw = n_i + n_j - 2 G_ij (0 on the diagonal), ds = e^t max(raw, 0), A = sqrt(ds + 1e-5): no contraction, so every
// caller gets the same bits.
struct Dist {
  float raw, ds, a;
};
__device__ __forceinline__ Dist dist(float ni, float nj, float gij, float et, bool diag) {
  Dist d;
  d.raw = diag ? 0.f : __fsub_rn(__fadd_rn(ni, nj), __fmul_rn(2.f, gij));
  d.ds = __fmul_rn(et, fmaxf(d.raw, 0.f));
  d.a = sqrtf(__fadd_rn(d.ds, 1e-5f));
  return d;
}

// Row sums (and, when cols, column sums) of the 64 x 64 tile in sA, each in ascending order, into the slots
// part[row block][column block][64] of the clip.
__device__ __forceinline__ void tile_sums(const float* sA, float* part, int k, int I, int J, bool cols) {
  const int tid = threadIdx.x;
  if (tid < kBlk) {
    float s = 0.f;
    for (int c = 0; c < kBlk; ++c) s += sA[tid * kAStride + c];
    part[(static_cast<int64_t>(I) * k + J) * kBlk + tid] = s;
  } else if (cols && tid < 2 * kBlk) {
    const int c = tid - kBlk;
    float s = 0.f;
    for (int r = 0; r < kBlk; ++r) s += sA[r * kAStride + c];
    part[(static_cast<int64_t>(J) * k + I) * kBlk + c] = s;
  }
}

__global__ void __launch_bounds__(kThreads)
bdc_wide_norms(const float* __restrict__ x, int M, int64_t rows, float* __restrict__ norms) {
  const int lane = threadIdx.x & 31;
  for (int64_t row = static_cast<int64_t>(blockIdx.x) * (kThreads / 32) + (threadIdx.x >> 5); row < rows;
       row += static_cast<int64_t>(gridDim.x) * (kThreads / 32)) {
    const float* xr = x + row * M;
    float s = 0.f;
    for (int m = lane; m < M; m += 32) {
      const float v = __ldg(xr + m);
      s = fmaf(v, v, s);
    }
    s = warp_sum(s);
    if (lane == 0) norms[row] = s;
  }
}

__global__ void __launch_bounds__(kThreads)
bdc_wide_gram(const float* __restrict__ x, int C, int M, const float* __restrict__ log_temp, int triu,
              const float* __restrict__ norms, float* __restrict__ rowpart, float* __restrict__ out, int64_t tiles) {
  __shared__ __align__(16) float s_buf[kGramSmem];
  const int k = C / kBlk, P = k * (k + 1) / 2;
  const int tid = threadIdx.x, ti = tid >> 4, tj = tid & 15;
  const float et = expf(__ldg(log_temp));
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t b = t / P;
    int I, J;
    pair_of(static_cast<int>(t - b * P), k, I, J);
    float2 g[4][2];
    gram_tile(x + b * C * M, M, I, J, s_buf, g);

    const float* nb = norms + b * C;
    float* sA = s_buf;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = kBlk * I + 4 * ti + i;
      const float nr = nb[r];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = kBlk * J + 4 * tj + j;
        sA[(4 * ti + i) * kAStride + 4 * tj + j] = dist(nr, nb[c], g_at(g, i, j), et, r == c).a;
      }
    }
    __syncthreads();
    tile_sums(sA, rowpart + b * k * C, k, I, J, I != J);
    if (triu) {
      float* ob = out + b * (static_cast<int64_t>(C) * (C + 1) / 2);
      for (int idx = tid; idx < kTile; idx += kThreads) {
        const int rl = idx >> 6, cl = idx & (kBlk - 1);
        const int r = kBlk * I + rl, c = kBlk * J + cl;
        if (c >= r) ob[triu_row(r, C) + c] = sA[rl * kAStride + cl];
      }
    } else {
      float* ob = out + b * C * C;
      for (int idx = tid; idx < kTile; idx += kThreads) {
        const int rl = idx >> 6, cl = idx & (kBlk - 1);
        ob[static_cast<int64_t>(kBlk * I + rl) * C + kBlk * J + cl] = sA[rl * kAStride + cl];
        if (I != J) ob[static_cast<int64_t>(kBlk * J + rl) * C + kBlk * I + cl] = sA[cl * kAStride + rl];
      }
    }
    // the next tile's gram_tile synchronises before it overwrites s_buf
  }
}

// One CTA per (clip, row block): finishes r_i and total (every CTA of a clip computes them in the same order) and
// centres the block's 64 output rows in place, a warp per row.
__global__ void __launch_bounds__(kThreads)
bdc_wide_center(const float* __restrict__ rowpart, int C, int triu, float* __restrict__ out, int64_t units) {
  __shared__ float s_r[kMaxBlocks * kBlk];
  __shared__ float s_total;
  const int k = C / kBlk;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float inv = 1.0f / static_cast<float>(C);
  const float inv2 = 1.0f / static_cast<float>(C * C);
  for (int64_t t = blockIdx.x; t < units; t += gridDim.x) {
    const int64_t b = t / k;
    const int I = static_cast<int>(t - b * k);
    const float* rp = rowpart + b * k * C;
    __syncthreads();
    for (int i = tid; i < C; i += kThreads) {
      const float* p = rp + static_cast<int64_t>(i >> 6) * k * kBlk + (i & (kBlk - 1));
      float s = 0.f;
      for (int q = 0; q < k; ++q) s += p[q * kBlk];
      s_r[i] = s;
    }
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int i = 0; i < C; ++i) s += s_r[i];
      s_total = s;
    }
    __syncthreads();
    // explicitly rounded, so that the two layouts and the two halves of the full layout share their bits
    const float tot = __fmul_rn(inv2, s_total);
    for (int rl = warp; rl < kBlk; rl += kThreads / 32) {
      const int r = kBlk * I + rl;
      const float rr = __fmul_rn(inv, s_r[r]);
      float* orow = triu ? out + b * (static_cast<int64_t>(C) * (C + 1) / 2) + triu_row(r, C)
                         : out + b * C * C + static_cast<int64_t>(r) * C;
      for (int c = (triu ? r : 0) + lane; c < C; c += 32) {
        const float rc = __fmul_rn(inv, s_r[c]);
        const float lo = c >= r ? rr : rc, hi = c >= r ? rc : rr;
        orow[c] = __fadd_rn(__fsub_rn(__fsub_rn(orow[c], lo), hi), tot);
      }
    }
  }
}

// ---- backward
__device__ __forceinline__ float grad_at(const float* __restrict__ gb, int r, int c, int C, int triu) {
  if (triu) return c >= r ? __ldg(gb + triu_row(r, C) + c) : 0.f;
  return __ldg(gb + static_cast<int64_t>(r) * C + c);
}

// Per clip: R_i = sum_j dB_ij (a warp per row, fixed shuffle tree), K_j = sum_i dB_ij (a thread per column,
// ascending i; consecutive threads read consecutive addresses), T = sum_j K_j in ascending j.
__global__ void __launch_bounds__(kThreads)
bdc_wide_dbstats(const float* __restrict__ grad_out, int C, int triu, float* __restrict__ dbr,
                 float* __restrict__ dbk, float* __restrict__ dbt, int64_t B) {
  __shared__ float s_k[kMaxBlocks * kBlk];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t per = triu ? static_cast<int64_t>(C) * (C + 1) / 2 : static_cast<int64_t>(C) * C;
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    const float* gb = grad_out + b * per;
    __syncthreads();
    for (int r = warp; r < C; r += kThreads / 32) {
      float s = 0.f;
      for (int c = (triu ? r : 0) + lane; c < C; c += 32) s += grad_at(gb, r, c, C, triu);
      s = warp_sum(s);
      if (lane == 0) dbr[b * C + r] = s;
    }
    for (int c = tid; c < C; c += kThreads) {
      float s = 0.f;
      const int last = triu ? c : C - 1;
      for (int r = 0; r <= last; ++r) s += grad_at(gb, r, c, C, triu);
      dbk[b * C + c] = s;
      s_k[c] = s;
    }
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int c = 0; c < C; ++c) s += s_k[c];
      dbt[b] = s;
    }
  }
}

__global__ void __launch_bounds__(kThreads)
bdc_wide_bwd_tile(const float* __restrict__ x, int C, int M, const float* __restrict__ log_temp, int triu,
                  const float* __restrict__ grad_out, const float* __restrict__ norms, const float* __restrict__ dbr,
                  const float* __restrict__ dbk, const float* __restrict__ dbt, float* __restrict__ s_ws,
                  float* __restrict__ rowpart, float* __restrict__ dtpart, int64_t tiles) {
  __shared__ __align__(16) float s_buf[kGramSmem];
  __shared__ float s_dt[kThreads / 32];
  const int k = C / kBlk, P = k * (k + 1) / 2;
  const int tid = threadIdx.x, ti = tid >> 4, tj = tid & 15;
  const float et = expf(__ldg(log_temp));
  const float inv = 1.0f / static_cast<float>(C);
  const float inv2 = 1.0f / static_cast<float>(C * C);
  const int64_t per = triu ? static_cast<int64_t>(C) * (C + 1) / 2 : static_cast<int64_t>(C) * C;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t b = t / P;
    const int p = static_cast<int>(t - b * P);
    int I, J;
    pair_of(p, k, I, J);
    float2 g[4][2];
    gram_tile(x + b * C * M, M, I, J, s_buf, g);

    const float* nb = norms + b * C;
    const float* Rb = dbr + b * C;
    const float* Kb = dbk + b * C;
    const float* gb = grad_out + b * per;
    const float tot = __fmul_rn(inv2, dbt[b]);
    float* sS = s_buf;
    float* st = s_ws + (b * P + p) * kTile;
    float dt = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = kBlk * I + 4 * ti + i;
      const float nr = nb[r], rr = __fmul_rn(inv, Rb[r]), kr = __fmul_rn(inv, Kb[r]);
      float sv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = kBlk * J + 4 * tj + j;
        const bool diag = r == c;
        const Dist d = dist(nr, nb[c], g_at(g, i, j), et, diag);
        const float two_a = __fmul_rn(2.f, d.a);
        const bool pass = !diag && d.raw >= 0.f;  // torch.clamp's subgradient; dD_ii cancels (see the header)
        // (r, c)
        const float da = __fadd_rn(__fsub_rn(__fsub_rn(grad_at(gb, r, c, C, triu), rr), __fmul_rn(inv, Kb[c])), tot);
        const float h = __fdividef(da, two_a);  // 2 ulp; 2 A >= 2 sqrt(1e-5) is in its range
        const float e = pass ? __fmul_rn(h, et) : 0.f;
        // (c, r): below the diagonal, so dB_cr = 0, when triu and I < J
        const float dbcr = (triu && I != J) ? 0.f : grad_at(gb, c, r, C, triu);
        const float da2 = __fadd_rn(__fsub_rn(__fsub_rn(dbcr, __fmul_rn(inv, Rb[c])), kr), tot);
        const float h2 = __fdividef(da2, two_a);
        const float f = pass ? __fmul_rn(h2, et) : 0.f;
        dt = fmaf(h, d.ds, dt);
        if (I != J) dt = fmaf(h2, d.ds, dt);  // a diagonal tile holds (c, r) as its own element
        sv[j] = __fadd_rn(e, f);
        sS[(4 * ti + i) * kAStride + 4 * tj + j] = sv[j];
      }
      *reinterpret_cast<float4*>(st + (4 * ti + i) * kBlk + 4 * tj) = make_float4(sv[0], sv[1], sv[2], sv[3]);
    }
    dt = warp_sum(dt);
    if ((tid & 31) == 0) s_dt[tid >> 5] = dt;
    __syncthreads();
    tile_sums(sS, rowpart + b * k * C, k, I, J, I != J);
    if (tid == 0) {
      float s = 0.f;
      for (int w = 0; w < kThreads / 32; ++w) s += s_dt[w];
      dtpart[b * P + p] = s;
    }
  }
}

// dX tile (clip b, row block I, positions m0 .. m0 + 63): thread (ti, tm) = (tid >> 4, tid & 15) owns rows
// 64 I + 4 ti + i and positions m0 + 4 tm + e; the sum over j runs over blocks J = 0 .. k - 1, then j, ascending.
__global__ void __launch_bounds__(kThreads)
bdc_wide_dx(const float* __restrict__ x, int C, int M, const float* __restrict__ s_ws,
            const float* __restrict__ rowpart, const float* __restrict__ dtpart, float* __restrict__ grad_x,
            float* __restrict__ grad_t, int64_t units) {
  __shared__ __align__(16) float sST[kBlk * kXStride];  // sST[j][i] = S_ij
  __shared__ __align__(16) float sX[kBlk * kXStride];   // sX[j][m]
  __shared__ float s_sigma[kBlk];
  const int k = C / kBlk, P = k * (k + 1) / 2;
  const int nch = (M + kDxM - 1) / kDxM;
  const int tid = threadIdx.x, ti = tid >> 4, tm = tid & 15;
  for (int64_t t = blockIdx.x; t < units; t += gridDim.x) {
    const int64_t b = t / (static_cast<int64_t>(k) * nch);
    const int rem = static_cast<int>(t - b * k * nch);
    const int I = rem / nch, m0 = (rem - I * nch) * kDxM;
    const float* xb = x + b * C * M;
    __syncthreads();
    if (tid < kBlk) {
      const float* p = rowpart + (b * k + I) * k * kBlk + tid;
      float s = 0.f;
      for (int q = 0; q < k; ++q) s += p[q * kBlk];
      s_sigma[tid] = s;
    }
    if (tid == 0 && I == 0 && m0 == 0) {
      float s = 0.f;
      for (int q = 0; q < P; ++q) s += dtpart[b * P + q];
      grad_t[b] = s;
    }
    float2 acc[4][2];
    float xs[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
    for (int J = 0; J < k; ++J) {
      __syncthreads();
      const float* st = s_ws + (b * P + (J >= I ? pair_index(I, J, k) : pair_index(J, I, k))) * kTile;
      for (int idx = tid; idx < kTile; idx += kThreads) {
        const int j = idx >> 6, i = idx & (kBlk - 1);
        // S_IJ[i][j] is tile (I, J)[i][j] for J >= I and tile (J, I)[j][i] below
        sST[j * kXStride + i] = J >= I ? st[i * kBlk + j] : st[j * kBlk + i];
        const int m = m0 + i;
        sX[j * kXStride + i] = m < M ? __ldg(xb + static_cast<int64_t>(kBlk * J + j) * M + m) : 0.f;
      }
      __syncthreads();
#pragma unroll 8
      for (int j = 0; j < kBlk; ++j) {
        const float4 s = *reinterpret_cast<const float4*>(&sST[j * kXStride + 4 * ti]);
        const float4 v = *reinterpret_cast<const float4*>(&sX[j * kXStride + 4 * tm]);
        const float sv[4] = {s.x, s.y, s.z, s.w};
        const float2 v01 = make_float2(v.x, v.y), v23 = make_float2(v.z, v.w);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 si = make_float2(sv[i], sv[i]);
          acc[i][0] = __ffma2_rn(si, v01, acc[i][0]);
          acc[i][1] = __ffma2_rn(si, v23, acc[i][1]);
        }
      }
      if (J == I) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) xs[i][e] = sX[(4 * ti + i) * kXStride + 4 * tm + e];
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rl = 4 * ti + i;
      float* gxr = grad_x + b * C * M + static_cast<int64_t>(kBlk * I + rl) * M;
      const float two_sigma = 2.f * s_sigma[rl];
      const float a[4] = {acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int m = m0 + 4 * tm + e;
        if (m < M) gxr[m] = fmaf(two_sigma, xs[i][e], -2.f * a[e]);
      }
    }
  }
}

inline unsigned grid_of(int64_t units) {
  return static_cast<unsigned>(units < 0x7fffffffLL ? units : 0x7fffffffLL);
}

}  // namespace
}  // namespace afs

extern "C" size_t afs_bdc_wide_workspace_bytes(int32_t B, int32_t C, int32_t backward) {
  using namespace afs;
  if (B < 0 || !wide_supported(C)) return 0;
  return wide_ws(B, C, backward != 0).total * sizeof(float);
}

extern "C" int afs_bdc_wide_fwd(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp,
                                int32_t triu, float* out, void* ws, size_t ws_bytes, afs_stream_t stream_) {
  using namespace afs;
  if (B < 0 || C < 1 || M < 1) return AFS_ERR_INVALID_ARG;
  if (!wide_supported(C)) return AFS_ERR_UNSUPPORTED;
  if (B == 0) return AFS_OK;
  if (x == nullptr || log_temp == nullptr || out == nullptr) return AFS_ERR_INVALID_ARG;
  const WideWs w = wide_ws(B, C, false);
  if (ws == nullptr || ws_bytes < w.total * sizeof(float) || reinterpret_cast<uintptr_t>(ws) % 16 != 0)
    return AFS_ERR_WORKSPACE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  float* wf = static_cast<float*>(ws);
  const int64_t k = C / kBlk, P = k * (k + 1) / 2;
  const int64_t rows = static_cast<int64_t>(B) * C;
  bdc_wide_norms<<<grid_of((rows + 7) / 8), kThreads, 0, stream>>>(x, M, rows, wf + w.norms);
  AFS_LAUNCH_CHECK();
  bdc_wide_gram<<<grid_of(B * P), kThreads, 0, stream>>>(x, C, M, log_temp, triu, wf + w.norms, wf + w.rowpart,
                                                         out, B * P);
  AFS_LAUNCH_CHECK();
  bdc_wide_center<<<grid_of(B * k), kThreads, 0, stream>>>(wf + w.rowpart, C, triu, out, B * k);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

extern "C" int afs_bdc_wide_bwd(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp, int32_t triu,
                                const float* grad_out, float* grad_x, float* grad_log_temp, void* ws, size_t ws_bytes,
                                afs_stream_t stream_) {
  using namespace afs;
  if (B < 0 || C < 1 || M < 1) return AFS_ERR_INVALID_ARG;
  if (!wide_supported(C)) return AFS_ERR_UNSUPPORTED;
  if (B == 0) return AFS_OK;
  if (x == nullptr || log_temp == nullptr || grad_out == nullptr || grad_x == nullptr || grad_log_temp == nullptr)
    return AFS_ERR_INVALID_ARG;
  const WideWs w = wide_ws(B, C, true);
  if (ws == nullptr || ws_bytes < w.total * sizeof(float) || reinterpret_cast<uintptr_t>(ws) % 16 != 0)
    return AFS_ERR_WORKSPACE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  float* wf = static_cast<float*>(ws);
  const int64_t k = C / kBlk, P = k * (k + 1) / 2;
  const int64_t rows = static_cast<int64_t>(B) * C;
  const int64_t nch = (M + kDxM - 1) / kDxM;
  bdc_wide_norms<<<grid_of((rows + 7) / 8), kThreads, 0, stream>>>(x, M, rows, wf + w.norms);
  AFS_LAUNCH_CHECK();
  bdc_wide_dbstats<<<grid_of(B), kThreads, 0, stream>>>(grad_out, C, triu, wf + w.dbr, wf + w.dbk, wf + w.dbt, B);
  AFS_LAUNCH_CHECK();
  bdc_wide_bwd_tile<<<grid_of(B * P), kThreads, 0, stream>>>(x, C, M, log_temp, triu, grad_out, wf + w.norms,
                                                             wf + w.dbr, wf + w.dbk, wf + w.dbt, wf + w.s,
                                                             wf + w.rowpart, wf + w.dtpart, B * P);
  AFS_LAUNCH_CHECK();
  bdc_wide_dx<<<grid_of(B * k * nch), kThreads, 0, stream>>>(x, C, M, wf + w.s, wf + w.rowpart, wf + w.dtpart,
                                                             grad_x, grad_log_temp, B * k * nch);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

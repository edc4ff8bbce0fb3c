// First Conv64F block in TRAINING mode, forward and backward, without ever materialising the [N,64,H,W]
// activation: Conv2d(1->64, 3x3, pad 1, bias) + BatchNorm2d(batch statistics) + ReLU/LeakyReLU + MaxPool2d(3,3).
// sm_100a.
//
// Reference: layer1 of Conv64F (libfewshot_core/model/backbone/conv_four.py:61-66,101-103) under
// set_forward_loss (proto_net.py:122-154, dn4.py:122-155, deepbdc.py:354-378).  In the eager graph this block is
// ~15 passes over a [N,64,128,157] fp32 tensor (1 GB for a 2-episode batch): conv, batch-norm statistics,
// normalise, ReLU, max-pool forward, and their backward counterparts -- > 80 % of a ProtoNet training step on B200.
//
// Because the block has ONE input channel, everything BatchNorm needs is a function of tiny statistics of the input:
// with x_t the input shifted by tap t (zero padded), s[t] = sum_pos x_t and R[t,u] = sum_pos x_t x_u,
//     mean_c = w_c . s / P + b_c,     var_c = w_c^T (R/P - s s^T/P^2) w_c          (P = N*H*W positions)
// so the batch statistics come from a 9-vector and a 9x9 matrix (afs_conv1_autocorr), and the forward pass is the
// inference kernel with scale/shift derived from them.  In the backward pass the gradient that reaches a conv
// output is  dconv = scale_c (dy - mean(dy) - xhat mean(dy xhat)),  where dy is non-zero only at the arg-max of each
// pooling window; the two dense correction terms again reduce to s and R:
//     dW[c,t] = scale_c ( G[c,t] - A1_c/P s[t] - A2_c/P Q[c,t] ),   Q[c,t] = invstd_c ( (w_c R)[t] - mnob_c s[t] )
// with sparse sums over POOLED pixels only:  A1 = sum dy,  A2 = sum dy xhat,  G[c,t] = sum dy x_t(argmax).
// dbeta = A1, dgamma = A2, dbias = 0.  The backward kernel recomputes the nine conv values of every pooling
// window (cheaper than storing arg-max indices and reading them back) and produces per-CTA partial sums that the
// host side adds in a fixed order (deterministic).  The input needs no gradient (it is data).
#include "common.cuh"

namespace afs {
namespace {

constexpr int kCT = 64;            // output channels
constexpr int kAcStats = 54;       // 9 sums + 45 products (upper triangle of R, row-major)
constexpr int kAcCols = kAcStats + 1;  // a partial row: the 54 sums, then the pivot they were taken around
constexpr int kBwdStats = 11;      // per channel: A1, A2, G[9]

// ------------------------------------------------------------------------------------------------ autocorrelation
// The sums are taken of x_t - p for a pivot p near the mean of the input (zero-padded taps included, as -p): with a DC
// offset (normalised log-mel in silence sits near -5.4; an unnormalised input may sit anywhere) the sums of raw
// products are dominated by mean^2 and lose the variance to fp32 rounding, while the centred moments that BatchNorm
// needs are the same for x_t - p.  p is the mean of 32 inputs spread over the batch: every warp loads the same 32
// values and reduces them in the same butterfly, so every thread holds the same p.
__global__ void __launch_bounds__(256)
conv1_autocorr_kernel(const float* __restrict__ x, int64_t total, int H, int W, float* __restrict__ partials) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float pivot = total > 0 ? warp_sum(__ldg(x + total * lane / 32)) * (1.f / 32.f) : 0.f;
  float acc[kAcStats];
#pragma unroll
  for (int i = 0; i < kAcStats; ++i) acc[i] = 0.f;
  const int64_t hw = static_cast<int64_t>(H) * W;
  for (int64_t pos = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; pos < total;
       pos += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t n = pos / hw;
    const int r = static_cast<int>(pos - n * hw);
    const int y = r / W, xx = r - y * W;
    const float* img = x + n * hw;
    float v[9];
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int yy = y + dy - 1, xc = xx + dx - 1;
        v[dy * 3 + dx] = ((yy >= 0 && yy < H && xc >= 0 && xc < W) ? __ldg(img + static_cast<int64_t>(yy) * W + xc) : 0.f) - pivot;
      }
    }
    int k = 9;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      acc[t] += v[t];
#pragma unroll
      for (int u = t; u < 9; ++u) {
        acc[k] = fmaf(v[t], v[u], acc[k]);
        ++k;
      }
    }
  }
  __shared__ float s_red[8][kAcStats];
#pragma unroll
  for (int i = 0; i < kAcStats; ++i) {
    const float v = warp_sum(acc[i]);
    if (lane == 0) s_red[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < kAcStats) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += s_red[w][threadIdx.x];
    partials[static_cast<int64_t>(blockIdx.x) * kAcCols + threadIdx.x] = v;
  } else if (threadIdx.x == kAcStats) {
    partials[static_cast<int64_t>(blockIdx.x) * kAcCols + kAcStats] = pivot;
  }
}

// ------------------------------------------------------------------------------------------------ forward
// The inference kernel's layout (csrc/conv1.cu: a thread owns one pooled pixel and its 5x5 patch), with the folded
// weights scale_c * w_c and the shift read from shared memory (warp-uniform broadcasts) because they are device data
// that depend on the batch statistics.
constexpr int kPixT = 128;
constexpr int kTileStrideT = kCT + 1;

__global__ void __launch_bounds__(kPixT)
conv1_train_fwd_kernel(const float* __restrict__ x, int64_t total_pix, int H, int Wd, int PH, int PW, float slope,
                       const float* __restrict__ w, const float* __restrict__ scale, const float* __restrict__ shift,
                       float* __restrict__ out) {
  __shared__ float s_tile[kPixT * kTileStrideT];
  __shared__ float s_w[kCT * 9];
  __shared__ float s_shift[kCT];
  const int tid = threadIdx.x;
  for (int i = tid; i < kCT * 9; i += kPixT) s_w[i] = w[i] * scale[i / 9];
  if (tid < kCT) s_shift[tid] = shift[tid];
  const int64_t pix0 = static_cast<int64_t>(blockIdx.x) * kPixT;
  const int64_t pix = pix0 + tid;
  const bool live = pix < total_pix;
  float p[5][5];
  {
    const int64_t pp = live ? pix : total_pix - 1;
    const int per = PH * PW;
    const int64_t n = pp / per;
    const int r = static_cast<int>(pp - n * per);
    const int ph = r / PW;
    const int pw = r - ph * PW;
    const float* img = x + n * static_cast<int64_t>(H) * Wd;
    const int y0 = 3 * ph - 1, x0 = 3 * pw - 1;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int yy = y0 + i;
      const bool yin = (yy >= 0) && (yy < H);
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int xx = x0 + j;
        p[i][j] = (yin && xx >= 0 && xx < Wd) ? __ldg(img + static_cast<int64_t>(yy) * Wd + xx) : 0.f;
      }
    }
  }
  __syncthreads();
#pragma unroll 2
  for (int c = 0; c < kCT; ++c) {
    float wr[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) wr[k] = s_w[c * 9 + k];
    float best = -INFINITY;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        float acc = p[dy][dx] * wr[0];
        acc = fmaf(p[dy][dx + 1], wr[1], acc);
        acc = fmaf(p[dy][dx + 2], wr[2], acc);
        acc = fmaf(p[dy + 1][dx], wr[3], acc);
        acc = fmaf(p[dy + 1][dx + 1], wr[4], acc);
        acc = fmaf(p[dy + 1][dx + 2], wr[5], acc);
        acc = fmaf(p[dy + 2][dx], wr[6], acc);
        acc = fmaf(p[dy + 2][dx + 1], wr[7], acc);
        acc = fmaf(p[dy + 2][dx + 2], wr[8], acc);
        best = fmaxf(best, acc);
      }
    }
    float v = best + s_shift[c];
    v = v > 0.f ? v : v * slope;
    s_tile[tid * kTileStrideT + c] = v;
  }
  __syncthreads();
  const int64_t remain = total_pix - pix0;
  const int npix = remain < kPixT ? static_cast<int>(remain) : kPixT;
  float* dst = out + pix0 * kCT;
  for (int i = tid; i < npix * kCT; i += kPixT) {
    const int pxl = i >> 6;
    const int c = i & (kCT - 1);
    dst[i] = s_tile[pxl * kTileStrideT + c];
  }
}

// ------------------------------------------------------------------------------------------------ backward
// A warp walks strips of 4 horizontally adjacent pooled pixels; lane l owns channels l and l+32, so the 22 running
// sums per lane stay in registers for the whole kernel and need no cross-thread reduction until the end.  The
// strip's 5 x 14 input patch sits in warp-private shared memory (broadcast reads; the nine arg-max-relative taps are
// per-lane dynamic reads inside the same 80 floats).
constexpr int kWarpsB = 8;
constexpr int kStripPix = 4;
constexpr int kStripW = 3 * kStripPix + 2;  // 14 input columns
constexpr int kStripPitch = 16;

__global__ void __launch_bounds__(kWarpsB * 32)
conv1_train_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g, int N, int H, int Wd, int PH, int PW,
                       float slope, const float* __restrict__ w, const float* __restrict__ scale,
                       const float* __restrict__ shift, const float* __restrict__ mean_nob,
                       const float* __restrict__ invstd, float* __restrict__ partials) {
  __shared__ float s_strip[kWarpsB][5 * kStripPitch];
  __shared__ float s_part[kWarpsB][2 * 32 * kBwdStats];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float wr[2][9], sc[2], sh[2], mn[2], is[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int c = lane + 32 * h;
#pragma unroll
    for (int k = 0; k < 9; ++k) wr[h][k] = w[c * 9 + k];
    sc[h] = scale[c]; sh[h] = shift[c]; mn[h] = mean_nob[c]; is[h] = invstd[c];
  }
  float acc[2][kBwdStats];
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int i = 0; i < kBwdStats; ++i) acc[h][i] = 0.f;

  float* strip = s_strip[warp];
  const int strips_per_row = (PW + kStripPix - 1) / kStripPix;
  const int64_t total_strips = static_cast<int64_t>(N) * PH * strips_per_row;
  const int64_t warp_global = static_cast<int64_t>(blockIdx.x) * kWarpsB + warp;
  const int64_t warp_stride = static_cast<int64_t>(gridDim.x) * kWarpsB;
  for (int64_t s = warp_global; s < total_strips; s += warp_stride) {
    const int sx = static_cast<int>(s % strips_per_row);
    int64_t r = s / strips_per_row;
    const int py = static_cast<int>(r % PH);
    const int64_t n = r / PH;
    const float* img = x + n * static_cast<int64_t>(H) * Wd;
    const int y0 = 3 * py - 1, x0 = 3 * sx * kStripPix - 1;
    __syncwarp();
    for (int i = lane; i < 5 * kStripW; i += 32) {
      const int rr = i / kStripW, cc = i - rr * kStripW;
      const int yy = y0 + rr, xx = x0 + cc;
      strip[rr * kStripPitch + cc] = (yy >= 0 && yy < H && xx >= 0 && xx < Wd) ? __ldg(img + static_cast<int64_t>(yy) * Wd + xx) : 0.f;
    }
    __syncwarp();
    const int npx = min(kStripPix, PW - sx * kStripPix);
    for (int q = 0; q < npx; ++q) {
      float p[5][5];
#pragma unroll
      for (int i = 0; i < 5; ++i)
#pragma unroll
        for (int j = 0; j < 5; ++j) p[i][j] = strip[i * kStripPitch + 3 * q + j];
      const int64_t pix = (n * PH + py) * PW + sx * kStripPix + q;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float go = __ldg(g + pix * kCT + lane + 32 * h);
        float best_y = -INFINITY, best_conv = 0.f;
        int best_pos = 0;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            float cv = p[dy][dx] * wr[h][0];
            cv = fmaf(p[dy][dx + 1], wr[h][1], cv);
            cv = fmaf(p[dy][dx + 2], wr[h][2], cv);
            cv = fmaf(p[dy + 1][dx], wr[h][3], cv);
            cv = fmaf(p[dy + 1][dx + 1], wr[h][4], cv);
            cv = fmaf(p[dy + 1][dx + 2], wr[h][5], cv);
            cv = fmaf(p[dy + 2][dx], wr[h][6], cv);
            cv = fmaf(p[dy + 2][dx + 1], wr[h][7], cv);
            cv = fmaf(p[dy + 2][dx + 2], wr[h][8], cv);
            const float y = fmaf(cv, sc[h], sh[h]);
            if (y > best_y) { best_y = y; best_conv = cv; best_pos = dy * kStripPitch + dx; }  // first maximum wins
          }
        }
        const float dyv = best_y > 0.f ? go : go * slope;
        const float xhat = (best_conv - mn[h]) * is[h];
        acc[h][0] += dyv;
        acc[h][1] = fmaf(dyv, xhat, acc[h][1]);
        const float* tp = strip + best_pos + 3 * q;
#pragma unroll
        for (int ty = 0; ty < 3; ++ty)
#pragma unroll
          for (int tx = 0; tx < 3; ++tx) acc[h][2 + ty * 3 + tx] = fmaf(dyv, tp[ty * kStripPitch + tx], acc[h][2 + ty * 3 + tx]);
      }
    }
  }
  // CTA partial = sum over its warps in a fixed order
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int i = 0; i < kBwdStats; ++i) s_part[warp][(lane + 32 * h) * kBwdStats + i] = acc[h][i];
  __syncthreads();
  for (int i = threadIdx.x; i < kCT * kBwdStats; i += kWarpsB * 32) {
    float v = 0.f;
#pragma unroll
    for (int wv = 0; wv < kWarpsB; ++wv) v += s_part[wv][i];
    partials[static_cast<int64_t>(blockIdx.x) * (kCT * kBwdStats) + i] = v;
  }
}

// ------------------------------------------------------------------------------------------------ finalisers
// One CTA of 64 threads (thread = channel) turns the autocorrelation partials into everything the forward and the
// backward kernels need, in fp64: s[9], R[9][9] (kept for the backward), mean_nob, invstd, scale, shift, and the
// running-statistics update of nn.BatchNorm2d.  stats layout (doubles): [0,9) s, [9,90) R row-major.  The partials
// are sums of x_t - p; the variance is taken from their centred moments (which p does not change), s and R are
// shifted back in fp64: s[t] = s'[t] + p P, R[t,u] = R'[t,u] + p (s'[t] + s'[u]) + p^2 P.
__global__ void __launch_bounds__(64)
conv1_train_stats_kernel(const float* __restrict__ partials, int n_part, double P, const float* __restrict__ w,
                         const float* __restrict__ bias, const float* __restrict__ gamma,
                         const float* __restrict__ beta, double eps, double momentum, float* running_mean,
                         float* running_var, double* __restrict__ stats, float* __restrict__ mean_nob,
                         float* __restrict__ invstd, float* __restrict__ scale, float* __restrict__ shift) {
  __shared__ double s_st[kAcStats];
  __shared__ double s_R[81];
  __shared__ double s_cov[81];
  const int c = threadIdx.x;
  if (c < kAcStats) {
    double v = 0.0;
    for (int i = 0; i < n_part; ++i) v += static_cast<double>(partials[static_cast<int64_t>(i) * kAcCols + c]);
    s_st[c] = v;
  }
  __syncthreads();
  const double p = static_cast<double>(partials[kAcStats]);  // every row carries the same pivot
  if (c == 0) {
    int k = 9;
    for (int t = 0; t < 9; ++t)
      for (int u = t; u < 9; ++u) {
        const double r = s_st[k] + p * (s_st[t] + s_st[u]) + p * p * P;
        const double cv = s_st[k] / P - s_st[t] * s_st[u] / (P * P);
        s_R[t * 9 + u] = r;
        s_R[u * 9 + t] = r;
        s_cov[t * 9 + u] = cv;
        s_cov[u * 9 + t] = cv;
        ++k;
      }
  }
  __syncthreads();
  if (c < 9) stats[c] = s_st[c] + p * P;
  for (int i = c; i < 81; i += 64) stats[9 + i] = s_R[i];
  double wc[9], m = 0.0;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    wc[t] = static_cast<double>(w[c * 9 + t]);
    m += wc[t] * (s_st[t] + p * P);
  }
  m /= P;  // mean of the conv output without its bias
  double var = 0.0;
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int u = 0; u < 9; ++u) var += wc[t] * wc[u] * s_cov[t * 9 + u];
  if (var < 0.0) var = 0.0;
  const double is = 1.0 / sqrt(var + eps);
  const double sc = static_cast<double>(gamma[c]) * is;
  mean_nob[c] = static_cast<float>(m);
  invstd[c] = static_cast<float>(is);
  scale[c] = static_cast<float>(sc);
  shift[c] = static_cast<float>(static_cast<double>(beta[c]) - m * sc);
  if (running_mean != nullptr) {  // nn.BatchNorm2d in train(): unbiased running variance
    running_mean[c] = static_cast<float>((1.0 - momentum) * running_mean[c] + momentum * (m + static_cast<double>(bias[c])));
    running_var[c] = static_cast<float>((1.0 - momentum) * running_var[c] + momentum * var * (P / (P > 1.0 ? P - 1.0 : 1.0)));
  }
}

// Backward partials [n_part][64][11] -> dW [64][9], dgamma, dbeta (fp64 accumulation, fixed order).
__global__ void __launch_bounds__(64)
conv1_train_grads_kernel(const float* __restrict__ partials, int n_part, double P, const double* __restrict__ stats,
                         const float* __restrict__ w, const float* __restrict__ gamma, double eps,
                         float* __restrict__ dW, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = threadIdx.x;
  double t[kBwdStats];
#pragma unroll
  for (int i = 0; i < kBwdStats; ++i) t[i] = 0.0;
  for (int p = 0; p < n_part; ++p) {
    const float* row = partials + (static_cast<int64_t>(p) * kCT + c) * kBwdStats;
#pragma unroll
    for (int i = 0; i < kBwdStats; ++i) t[i] += static_cast<double>(row[i]);
  }
  const double* s = stats;
  const double* R = stats + 9;
  double wc[9], m = 0.0;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    wc[k] = static_cast<double>(w[c * 9 + k]);
    m += wc[k] * s[k];
  }
  m /= P;
  double var = 0.0;
#pragma unroll
  for (int a = 0; a < 9; ++a)
#pragma unroll
    for (int b = 0; b < 9; ++b) var += wc[a] * wc[b] * (R[a * 9 + b] / P - s[a] * s[b] / (P * P));
  if (var < 0.0) var = 0.0;
  const double is = 1.0 / sqrt(var + eps);
  const double sc = static_cast<double>(gamma[c]) * is;
  const double a1 = t[0], a2 = t[1];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    double wr = 0.0;
#pragma unroll
    for (int u = 0; u < 9; ++u) wr += wc[u] * R[u * 9 + k];
    const double q = is * (wr - m * s[k]);
    dW[c * 9 + k] = static_cast<float>(sc * (t[2 + k] - (a1 / P) * s[k] - (a2 / P) * q));
  }
  dgamma[c] = static_cast<float>(a2);
  dbeta[c] = static_cast<float>(a1);
}

}  // namespace
}  // namespace afs

extern "C" int32_t afs_conv1_train_num_partials(int32_t which) {
  // which 0: autocorrelation CTAs, 1: backward CTAs (fixed grids: partial buffers have a static size)
  return which == 0 ? afs::kNumSMs * 4 : afs::kNumSMs * 2;
}

extern "C" int afs_conv1_autocorr(const float* x, int32_t N, int32_t H, int32_t Wd, float* partials,
                                  afs_stream_t stream_) {
  using namespace afs;
  if (x == nullptr || partials == nullptr || N < 0 || H < 1 || Wd < 1) return AFS_ERR_INVALID_ARG;
  const int64_t total = static_cast<int64_t>(N) * H * Wd;
  const int blocks = afs_conv1_train_num_partials(0);
  conv1_autocorr_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream_)>>>(x, total, H, Wd, partials);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

extern "C" int afs_conv1_train_stats(const float* ac_partials, int32_t N, int32_t H, int32_t Wd, const float* w,
                                     const float* bias, const float* gamma, const float* beta, double eps,
                                     double momentum, float* running_mean, float* running_var, double* stats,
                                     float* mean_nob, float* invstd, float* scale, float* shift, afs_stream_t stream_) {
  using namespace afs;
  if (ac_partials == nullptr || w == nullptr || bias == nullptr || gamma == nullptr || beta == nullptr ||
      stats == nullptr || mean_nob == nullptr || invstd == nullptr || scale == nullptr || shift == nullptr || N < 1 ||
      H < 1 || Wd < 1 || (running_mean == nullptr) != (running_var == nullptr))
    return AFS_ERR_INVALID_ARG;
  const double P = static_cast<double>(N) * H * Wd;
  conv1_train_stats_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream_)>>>(
      ac_partials, afs_conv1_train_num_partials(0), P, w, bias, gamma, beta, eps, momentum, running_mean, running_var,
      stats, mean_nob, invstd, scale, shift);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

extern "C" int afs_conv1_train_grads(const float* bwd_partials, int32_t N, int32_t H, int32_t Wd, const double* stats,
                                     const float* w, const float* gamma, double eps, float* dW, float* dgamma,
                                     float* dbeta, afs_stream_t stream_) {
  using namespace afs;
  if (bwd_partials == nullptr || stats == nullptr || w == nullptr || gamma == nullptr || dW == nullptr ||
      dgamma == nullptr || dbeta == nullptr || N < 1 || H < 1 || Wd < 1)
    return AFS_ERR_INVALID_ARG;
  const double P = static_cast<double>(N) * H * Wd;
  conv1_train_grads_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream_)>>>(
      bwd_partials, afs_conv1_train_num_partials(1), P, stats, w, gamma, eps, dW, dgamma, dbeta);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

extern "C" int afs_conv1_train_fwd(const float* x, int32_t N, int32_t H, int32_t Wd, const float* w, const float* scale,
                                   const float* shift, float negative_slope, float* out, afs_stream_t stream_) {
  using namespace afs;
  if (x == nullptr || w == nullptr || scale == nullptr || shift == nullptr || out == nullptr || N < 0 || H < 3 ||
      Wd < 3 || negative_slope < 0.f)
    return AFS_ERR_INVALID_ARG;
  if (N == 0) return AFS_OK;
  const int PH = H / 3, PW = Wd / 3;
  const int64_t total = static_cast<int64_t>(N) * PH * PW;
  const int64_t blocks = (total + kPixT - 1) / kPixT;
  if (blocks > 0x7fffffffLL) return AFS_ERR_UNSUPPORTED;
  conv1_train_fwd_kernel<<<static_cast<unsigned>(blocks), kPixT, 0, static_cast<cudaStream_t>(stream_)>>>(
      x, total, H, Wd, PH, PW, negative_slope, w, scale, shift, out);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

extern "C" int afs_conv1_train_bwd(const float* x, const float* grad_out, int32_t N, int32_t H, int32_t Wd,
                                   const float* w, const float* scale, const float* shift, const float* mean_nob,
                                   const float* invstd, float negative_slope, float* partials, afs_stream_t stream_) {
  using namespace afs;
  if (x == nullptr || grad_out == nullptr || w == nullptr || scale == nullptr || shift == nullptr ||
      mean_nob == nullptr || invstd == nullptr || partials == nullptr || N < 0 || H < 3 || Wd < 3 ||
      negative_slope < 0.f)
    return AFS_ERR_INVALID_ARG;
  const int blocks = afs_conv1_train_num_partials(1);
  conv1_train_bwd_kernel<<<blocks, kWarpsB * 32, 0, static_cast<cudaStream_t>(stream_)>>>(
      x, grad_out, N, H, Wd, H / 3, Wd / 3, negative_slope, w, scale, shift, mean_nob, invstd, partials);
  AFS_LAUNCH_CHECK();
  return AFS_OK;
}

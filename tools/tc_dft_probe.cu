// Hardware probe for a tensor-core DFT log-mel kernel (development tool, B200 / sm_100a; DESIGN.md 3.1b, 9).
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -I audio_fewshot_b200/csrc \
//        tools/tc_dft_probe.cu -o tools/tc_dft_probe && ./tools/tc_dft_probe
//
// 1. step-1 GEMM of the 32x32 four-step real DFT with ZERO-COPY framing: the clip is stored once in shared memory
//    as fp16 (hi, lo) sample rows of 32 (64 B, SWIZZLE_64B pattern on absolute address bits) and the A operand of
//    four overlapping frames is the MN-major descriptor {start = first sample row, LBO = hop * 2 B, SBO = 512 B}.
//    Result against a float64 DFT: tells whether the layout is what the hardware reads and what the 3-term fp16
//    split (hi*hi + hi*lo + lo*hi, fp32 accumulate in TMEM) is worth.
// 2. tcgen05.ld throughput per SM with 4 / 8 / 16 warps.
// 3. tcgen05.mma issue-to-completion cost for M128 x N x K16 (kind::f16) shapes, SS operands.
#include <cuda_fp16.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "tc_common.cuh"

using namespace afs::tc;

#define CK(x)                                                                         \
  do {                                                                                \
    cudaError_t e_ = (x);                                                             \
    if (e_ != cudaSuccess) {                                                          \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      exit(1);                                                                        \
    }                                                                                 \
  } while (0)

__host__ __device__ constexpr uint32_t idesc_f16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// Generic shared-memory matrix descriptor: layout 0 = no swizzle, 6 = 32 B, 4 = 64 B, 2 = 128 B.
//   K-major,  no swizzle: LBO = distance between the 8-element K groups, SBO = between 8-row groups
//   MN-major, no swizzle: LBO = distance between the 8-row K groups,    SBO = between 8-element MN groups
//   MN-major, swizzled:   LBO = distance between MN groups of one swizzle row (32 elements for 64 B), SBO = between
//                         8-row K groups (both orders measured on B200 with this probe)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
  uint64_t d = static_cast<uint64_t>((saddr >> 4) & 0x3FFFu);
  d |= static_cast<uint64_t>((lbo >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout) << 61;
  return d;
}

constexpr int kHop = 512;
constexpr int kFrames = 4;
constexpr int kSamples = kHop * (kFrames - 1) + 1024;  // 2560

// ---------------------------------------------------------------- probe 1
// smem: [hi 5120 B | lo 5120 B] (1024-aligned), [B hi 2048 | B lo 2048]
__global__ void __launch_bounds__(128) probe_step1(const float* __restrict__ x, float scale, const __half* __restrict__ bimg,
                                                   float* __restrict__ out, int use_terms) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t bar;
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_hi = smem;
  uint8_t* s_lo = smem + 6144;
  uint8_t* s_bhi = smem + 12288;
  uint8_t* s_blo = s_bhi + 2048;
  const int tid = threadIdx.x;
  if (tid < 32) tmem_alloc(&tmem_slot, 32);
  if (tid == 0) {
    mbar_init(smem_u32(&bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // convert: chunks of 8 samples
  for (int c = tid; c < kSamples / 8; c += 128) {
    __half hi[8], lo[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float v = x[8 * c + i] * scale;
      hi[i] = __float2half_rn(v);
      lo[i] = __float2half_rn(v - __half2float(hi[i]));
    }
    uint32_t off = 16u * c;
    off ^= ((off >> 7) & 3u) << 4;  // SWIZZLE_64B on (1024-aligned base => absolute) address bits
    *reinterpret_cast<uint4*>(s_hi + off) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(s_lo + off) = *reinterpret_cast<const uint4*>(lo);
  }
  for (int i = tid; i < 2048 / 16; i += 128) {
    reinterpret_cast<uint4*>(s_bhi)[i] = reinterpret_cast<const uint4*>(bimg)[i];
    reinterpret_cast<uint4*>(s_blo)[i] = reinterpret_cast<const uint4*>(bimg)[128 + i];
  }
  fence_async_smem();
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = tmem_slot;
  if (tid == 0) {
    const uint32_t idesc = idesc_f16(128, 32, 1, 0);
    bool acc = false;
    for (int term = 0; term < use_terms; ++term) {
      const uint32_t a_base = smem_u32(term == 2 ? s_lo : s_hi);
      const uint32_t b_base = smem_u32(term == 1 ? s_blo : s_bhi);
      for (int ks = 0; ks < 2; ++ks) {
        const uint64_t da = make_desc(a_base + ks * 1024, /*LBO (MN groups of 32 = frames)*/ kHop * 2, /*SBO (K groups of 8 rows)*/ 512, 4);
        const uint64_t db = make_desc(b_base + ks * 1024, /*LBO (K groups)*/ 512, /*SBO (N groups of 8)*/ 128, 0);
        mma_f16(tmem, da, db, idesc, acc);
        acc = true;
      }
    }
    commit(smem_u32(&bar));
  }
  mbar_wait(smem_u32(&bar), 0);
  fence_after();
  uint32_t v[32];
  const int warp = tid >> 5;
  tmem_ld32(tmem + (static_cast<uint32_t>(warp * 32) << 16), v);
#pragma unroll
  for (int i = 0; i < 32; ++i) out[tid * 32 + i] = __uint_as_float(v[i]);
  fence_before();
  __syncthreads();
  if (tid < 32) tmem_dealloc(tmem, 32);
}

// ---------------------------------------------------------------- probe 2: tcgen05.ld throughput
__global__ void probe_tmem_ld(int iters, long long* cycles, uint32_t* sink) {
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == 0) tmem_alloc(&tmem_slot, 512);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = tmem_slot;
  const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
  uint32_t acc = 0;
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
    uint32_t a[32], b[32];
    const uint32_t col = static_cast<uint32_t>(((it + warp) * 64) & 511);
    tmem_ld32_nowait(tmem + lane_base + col, a);
    tmem_ld32_nowait(tmem + lane_base + ((col + 32) & 511), b);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; ++i) acc ^= a[i] + b[i];
  }
  __syncthreads();
  const long long t1 = clock64();
  if (tid == 0) cycles[blockIdx.x] = t1 - t0;
  if (acc == 0x12345678u) sink[0] = acc;
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------- probe 3: MMA cost
// A: MN-major SW64 (the zero-copy framing layout) or K-major no swizzle; B: K-major no swizzle; garbage data.
__global__ void __launch_bounds__(128) probe_mma(int N, int n_mma, int a_mn, long long* cycles) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t bar;
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int tid = threadIdx.x;
  for (int i = tid; i < 49152 / 4; i += 128) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;  // 1.0h
  if (tid < 32) tmem_alloc(&tmem_slot, 256);
  if (tid == 0) {
    mbar_init(smem_u32(&bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = tmem_slot;
  if (tid == 0) {
    const uint32_t idesc = idesc_f16(128, N, a_mn, 0);
    const uint32_t a_base = smem_u32(smem), b_base = smem_u32(smem + 16384);
    const long long t0 = clock64();
    for (int i = 0; i < n_mma; ++i) {
      const uint64_t da = a_mn ? make_desc(a_base + (i & 3) * 1024, 1024, 512, 4) : make_desc(a_base + (i & 3) * 4096, 2048, 128, 0);
      const uint64_t db = make_desc(b_base + (i & 1) * 8192, N * 16, 128, 0);
      mma_f16(tmem, da, db, idesc, i > 0);
    }
    commit(smem_u32(&bar));
    mbar_wait(smem_u32(&bar), 0);
    const long long t1 = clock64();
    cycles[0] = t1 - t0;
  }
  fence_before();
  __syncthreads();
  if (tid < 32) tmem_dealloc(tmem, 256);
}

int main() {
  // ---- probe 1
  std::vector<float> x(kSamples);
  srand(1);
  for (auto& v : x) v = 0.1f * (static_cast<float>(rand()) / RAND_MAX * 2.f - 1.f) + 0.05f * (static_cast<float>(rand()) / RAND_MAX - 0.5f);
  float mx = 0.f;
  for (auto v : x) mx = fmaxf(mx, fabsf(v));
  int e;
  frexpf(mx, &e);                       // mx = m * 2^e, m in [0.5, 1)
  const float scale = ldexpf(1.f, 14 - e);  // max |x * scale| in [2^13, 2^14)
  // B image: [kgroup 4][n 32][8] for hi, then lo
  std::vector<__half> bimg(2 * 1024);
  std::vector<double> F(32 * 32);
  const double two_pi = 6.283185307179586476925286766559;
  for (int n2 = 0; n2 < 32; ++n2)
    for (int c = 0; c < 32; ++c) {
      double v;
      if (c == 0) v = 1.0;
      else if (c == 1) v = (n2 & 1) ? -1.0 : 1.0;
      else {
        const int k1 = c >> 1;
        const double a = two_pi * ((n2 * k1) % 32) / 32.0;
        v = (c & 1) ? -sin(a) : cos(a);
      }
      F[n2 * 32 + c] = v;
      const __half h = __float2half_rn(static_cast<float>(v));
      const __half l = __float2half_rn(static_cast<float>(v - static_cast<double>(__half2float(h))));
      const int idx = (n2 / 8) * 256 + c * 8 + (n2 % 8);
      bimg[idx] = h;
      bimg[1024 + idx] = l;
    }
  float *d_x, *d_out;
  __half* d_b;
  CK(cudaMalloc(&d_x, x.size() * 4));
  CK(cudaMalloc(&d_out, 128 * 32 * 4));
  CK(cudaMalloc(&d_b, bimg.size() * 2));
  CK(cudaMemcpy(d_x, x.data(), x.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_b, bimg.data(), bimg.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaFuncSetAttribute(probe_step1, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 + 1024));
  std::vector<double> ref(128 * 32);
  double ref_max = 0;
  for (int f = 0; f < kFrames; ++f)
    for (int n1 = 0; n1 < 32; ++n1)
      for (int c = 0; c < 32; ++c) {
        double s = 0;
        for (int n2 = 0; n2 < 32; ++n2) s += static_cast<double>(x[f * kHop + n1 + 32 * n2]) * scale * F[n2 * 32 + c];
        ref[(f * 32 + n1) * 32 + c] = s;
        ref_max = fmax(ref_max, fabs(s));
      }
  for (int terms = 1; terms <= 3; ++terms) {
    CK(cudaMemset(d_out, 0, 128 * 32 * 4));
    probe_step1<<<1, 128, 16384 + 1024>>>(d_x, scale, d_b, d_out, terms);
    CK(cudaDeviceSynchronize());
    std::vector<float> out(128 * 32);
    CK(cudaMemcpy(out.data(), d_out, out.size() * 4, cudaMemcpyDeviceToHost));
    double err = 0, rms = 0;
    int worst = 0;
    for (int i = 0; i < 128 * 32; ++i) {
      const double d = fabs(out[i] - ref[i]);
      rms += d * d;
      if (d > err) { err = d; worst = i; }
    }
    printf("probe1 step-1 GEMM, %d split term(s): max err / max|Y| = %.3e, rms err / max|Y| = %.3e (worst row %d col %d: got %.6g want %.6g)\n",
           terms, err / ref_max, sqrt(rms / (128 * 32)) / ref_max, worst / 32, worst % 32, out[worst], ref[worst]);
  }

  // ---- probe 2
  long long* d_cyc;
  uint32_t* d_sink;
  CK(cudaMalloc(&d_cyc, 1024 * 8));
  CK(cudaMalloc(&d_sink, 4));
  for (int warps : {4, 8, 16}) {
    const int iters = 2000;
    probe_tmem_ld<<<1, warps * 32>>>(iters, d_cyc, d_sink);
    CK(cudaDeviceSynchronize());
    probe_tmem_ld<<<1, warps * 32>>>(iters, d_cyc, d_sink);
    CK(cudaDeviceSynchronize());
    long long cyc;
    CK(cudaMemcpy(&cyc, d_cyc, 8, cudaMemcpyDeviceToHost));
    const double bytes = static_cast<double>(iters) * warps * 2 * 32 * 32 * 4;
    printf("probe2 tcgen05.ld 32x32b.x32, %2d warps: %.1f B/clk/SM (%lld clk for %d x 2 loads per warp)\n", warps, bytes / cyc, cyc, iters);
  }

  // ---- probe 3
  CK(cudaFuncSetAttribute(probe_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, 49152 + 1024));
  for (int a_mn : {1, 0})
    for (int N : {32, 48, 64, 96, 128, 256}) {
      const int n_mma = 512;
      probe_mma<<<1, 128, 49152 + 1024>>>(N, n_mma, a_mn, d_cyc);
      CK(cudaDeviceSynchronize());
      probe_mma<<<1, 128, 49152 + 1024>>>(N, n_mma, a_mn, d_cyc);
      CK(cudaDeviceSynchronize());
      long long cyc;
      CK(cudaMemcpy(&cyc, d_cyc, 8, cudaMemcpyDeviceToHost));
      printf("probe3 tcgen05.mma kind::f16 M128 N%-3d K16, A %s: %.1f clk per MMA (math floor %.0f)\n", N,
             a_mn ? "MN-major SW64" : "K-major none ", static_cast<double>(cyc) / n_mma, 128.0 * N / 256.0);
    }
  printf("done\n");
  return 0;
}

/*
 * afs_b200.h -- C ABI of the B200-native episodic few-shot audio hot path.
 *
 * One shared library (libafs_b200.so, built by audio_fewshot_b200/build.py with
 * nvcc -gencode arch=compute_100a,code=sm_100a) exports exactly the entry points
 * below.  Plain pointers and sizes only: no torch types, no C++ types, no
 * exceptions across the boundary.  All data pointers are DEVICE pointers unless
 * the parameter name ends in `_host`.  Every call is asynchronous on `stream`
 * (a cudaStream_t passed as void*), allocates nothing (plans excepted), does
 * not synchronise, and is re-entrant.  The caller owns every buffer.
 *
 * Return value: AFS_OK (0) or a negative afs_status.  afs_status_string() maps
 * it to text; afs_last_cuda_error() returns the cudaError_t of the last failing
 * CUDA runtime call made by the calling thread inside this library.
 *
 * Each entry point cites the reference interface (Jerryaa98/Audio-Fewshot,
 * paths relative to the reference root) whose arithmetic it replaces.
 * There is no CPU fallback anywhere behind this ABI.
 */
#ifndef AFS_B200_H_
#define AFS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AFS_ABI_VERSION 1

typedef void* afs_stream_t; /* cudaStream_t */

typedef enum afs_status {
  AFS_OK = 0,
  AFS_ERR_INVALID_ARG = -1,  /* null pointer, negative size, unsupported shape */
  AFS_ERR_UNSUPPORTED = -2,  /* valid but not built (e.g. n_fft not 512/1024/2048) */
  AFS_ERR_CUDA = -3,         /* a CUDA runtime call failed; see afs_last_cuda_error */
  AFS_ERR_WORKSPACE = -4     /* workspace too small                              */
} afs_status;

int afs_abi_version(void);
const char* afs_status_string(int status);
int afs_last_cuda_error(void);
/* Kernels launched by this library in this process so far (every entry point below counts
 * its own launches; memsets and copies are not counted).  For benchmarks and tests that must
 * prove the CUDA path ran.                                                               */
uint64_t afs_launch_count(void);

/* ------------------------------------------------------------------------
 * (1) Fused waveform -> normalised log-mel front-end.
 *
 * Replaces the (absent, see SURVEY.md F2) offline feature extraction that
 * produced the reference's `<set>_spec` folders (config/headers/data.yaml:1) and
 * the `(x-mean)/std` step of libfewshot_core/audio_augmentations.py:36-53
 * with statistics from Auxiliary/<set>_Mean_Std.npy (libfewshot_core/test.py:398-399).
 * Canonical spec (oracle/frontend.py): reflect-pad n_fft/2, frame, window,
 * |rFFT|^2, mel projection, log_mult*log10(. + log_eps), (. - mean[m])/std[m].
 * Output layout [B, 1, n_mels, T] fp32 contiguous, T = 1 + L/hop (center) --
 * the `image` tensor every set_forward consumes (proto_net.py:86-90).
 * No spectrum is ever written to HBM.
 * ---------------------------------------------------------------------- */
typedef struct afs_logmel_cfg {
  int32_t n_fft;    /* 512, 1024 or 2048 (8 kHz / 16 kHz / 32-48 kHz)   */
  int32_t hop;      /* >= 1                                             */
  int32_t n_mels;   /* 1..128                                           */
  int32_t center;   /* 1: reflect padding of n_fft/2 on both sides      */
  float log_mult;   /* 10.0f for dB                                     */
  float log_eps;    /* added to the mel power before the log            */
} afs_logmel_cfg;

/* Waveform-domain augmentation (new functionality, SURVEY.md F3).  Randomness
 * is Philox4x32-10 keyed by (seed, global clip index); see oracle/philox.py.
 * A field pair with lo == hi disables the draw (fixed value).             */
typedef struct afs_aug_cfg {
  float gain_db_lo, gain_db_hi; /* gain g = 10^(U[lo,hi]/20)                      */
  int32_t max_shift;            /* time shift k ~ U{-max_shift..max_shift}, zero fill */
  float noise_std_lo, noise_std_hi; /* additive N(0, sigma^2), sigma ~ U[lo,hi]      */
} afs_aug_cfg;

typedef struct afs_logmel_plan afs_logmel_plan; /* opaque; owns device tables */

/* fb_host: dense mel filterbank [n_fft/2+1, n_mels] row-major (torchaudio
 * melscale_fbanks layout); window_host: [n_fft].  Both HOST pointers; the
 * plan packs each filter's contiguous non-zero band and uploads it together
 * with the window and the FFT twiddles.  device: CUDA device ordinal.
 * AFS_ERR_UNSUPPORTED for any other n_fft, n_mels > 128, or when the packed table exceeds the kernel's budget
 * (16 KB at n_fft 512 and 1024, 32 KB at 2048; very wide filters: fewer than about 30 slaney mels at 1024, fewer
 * than about 48 at 32-48 kHz and 2048). */
int afs_logmel_plan_create(const afs_logmel_cfg* cfg, const float* fb_host,
                           const float* window_host, int device, afs_logmel_plan** plan_out);
int afs_logmel_plan_destroy(afs_logmel_plan* plan);
/* number of output frames for clips of L samples */
int afs_logmel_num_frames(const afs_logmel_plan* plan, int64_t L);

/* wav [B, L] fp32; mean/std [n_mels] fp32 (per-bin; broadcast the scalar of
 * Auxiliary/<set>_Mean_Std.npy into it); aug nullable; out [B, 1, n_mels, T].
 * At n_fft 1024 both entry points run the pair engine (two frames per warp as one 1024-point FFT,
 * csrc/logmel_pair.cu) when aug is null and the radix-8 engine (one frame per 64 threads, csrc/logmel.cu) otherwise,
 * because the pair engine's lanes hold samples 32 apart and would evaluate each Philox block, shared by a sample pair,
 * twice.  At n_fft 512 and 2048 every launch runs csrc/logmel_nfft.cu (one frame per 64 threads, radix-4 / radix-16
 * register pass + two radix-8 cross-thread passes).  */
int afs_logmel_fwd(const afs_logmel_plan* plan, const float* wav, int32_t B, int64_t L,
                   const float* mean, const float* std, const afs_aug_cfg* aug,
                   uint64_t seed, uint64_t first_clip_index, float* out, afs_stream_t stream);

/* The same kernel fed with 16-bit PCM (the sample format of the wav files behind the reference's `<set>_spec`
 * folders): wav [B, L] int16, sample value = (float)pcm * pcm_scale (1/32768 for full scale in [-1, 1); the
 * product is exact in fp32 for a power-of-two scale, so the result is bit-identical to afs_logmel_fwd on the
 * converted fp32 waveform).  Halves the PCIe and HBM bytes of the waveform: 2*L + 4*n_mels*T per clip.   */
int afs_logmel_fwd_pcm16(const afs_logmel_plan* plan, const int16_t* wav, float pcm_scale, int32_t B, int64_t L,
                         const float* mean, const float* std, const afs_aug_cfg* aug,
                         uint64_t seed, uint64_t first_clip_index, float* out, afs_stream_t stream);

/* ------------------------------------------------------------------------
 * (1b) First Conv64F block, inference only: Conv2d(1->C,3x3,pad 1) + BatchNorm2d(eval) +
 * ReLU / LeakyReLU(negative_slope) + MaxPool2d(3,3), fused.  Replaces layer1 of Conv64F
 * (libfewshot_core/model/backbone/conv_four.py:61-66,101-103) in eval mode.
 * x [N,1,H,Wd] fp32 (device); w_folded_host [C*9] = conv weight * gamma/sqrt(var+eps) and
 * shift_host [C] = (bias - mean)*gamma/sqrt(var+eps) + beta are HOST pointers (they travel
 * as kernel parameters: constant-bank operands); out [N, H/3, Wd/3, C] fp32 channels-last
 * (the NHWC bytes of a torch channels_last [N,C,H/3,Wd/3] tensor).  C == 64 built.   */
int afs_conv1_bn_act_pool3_fwd(const float* x, int32_t N, int32_t H, int32_t Wd,
                               const float* w_folded_host, const float* shift_host, int32_t C,
                               float negative_slope, float* out, afs_stream_t stream);

/* (1b') The same block on the tensor cores: per tile of 128 pooled pixels three tcgen05 TF32 GEMMs
 * [128 x 16].[16 x 192] (one per pooling-window row: patch rows g..g+2 x five columns against a weight tile whose
 * columns hold the three window columns side by side), max over the nine accumulator blocks taken in tensor memory
 * lanes.  TF32 operands, fp32 accumulation -- the precision class of the reference's default convolutions
 * (torch.backends.cudnn.allow_tf32 = True); afs_conv1_bn_act_pool3_fwd stays the exact-fp32 kernel.        */
int afs_conv1_bn_act_pool3_fwd_tf32(const float* x, int32_t N, int32_t H, int32_t Wd,
                                    const float* w_folded_host, const float* shift_host, int32_t C,
                                    float negative_slope, float* out, afs_stream_t stream);

/* (1b-train) First Conv64F block in TRAINING mode (batch statistics), forward and backward, fused: replaces
 * layer1 of libfewshot_core/model/backbone/conv_four.py:61-66 under set_forward_loss.  The block has one input
 * channel, so the BatchNorm statistics and the dense BatchNorm-backward correction terms are functions of the 9-tap
 * sums s[t] and the 9x9 autocorrelation R[t,u] of the input (csrc/conv1_train.cu).  All pointers are device pointers.
 *   afs_conv1_autocorr: x [N,1,H,Wd] -> partials [afs_conv1_train_num_partials(0)][55]: 9 sums, then the upper
 *     triangle of R row-major, of the tap values minus a pivot p near the input's mean (so that a DC offset does not
 *     cancel the variance away in fp32), then p, the same in every row; afs_conv1_train_stats adds the rows in a
 *     fixed order (deterministic) and shifts s and R back in fp64.
 *   afs_conv1_train_fwd: out[N, H/3, Wd/3, 64] (NHWC) = MaxPool3(act(scale_c * (w_c * x) + shift_c)); w [64*9] raw
 *     conv weights, scale = gamma*invstd, shift = beta - mean_nob*scale (the conv bias cancels under batch statistics).
 *   afs_conv1_train_bwd: grad_out [N, H/3, Wd/3, 64] (NHWC) -> partials [afs_conv1_train_num_partials(1)][64][11]:
 *     per channel A1 = sum dy, A2 = sum dy*xhat, G[9] = sum dy * x_tap(argmax), dy = grad routed through the max-pool
 *     arg-max (first maximum) and the activation.  dgamma = A2, dbeta = A1, dbias = 0,
 *     dW[c,t] = scale_c (G[c,t] - A1_c/P s[t] - A2_c/P Q[c,t]), Q = invstd_c ((w_c R)[t] - mean_nob_c s[t]).        */
int32_t afs_conv1_train_num_partials(int32_t which);
int afs_conv1_autocorr(const float* x, int32_t N, int32_t H, int32_t Wd, float* partials, afs_stream_t stream);
/* afs_conv1_train_stats: autocorrelation partials -> stats (90 doubles: s[9], R[9][9], kept for the backward),
 * mean_nob / invstd / scale / shift [64] in fp64 arithmetic, and nn.BatchNorm2d's running-statistics update
 * (running_mean / running_var nullable together; bias only enters the running mean).
 * afs_conv1_train_grads: backward partials + stats -> dW [64*9], dgamma [64], dbeta [64] (fp64, fixed order).   */
int afs_conv1_train_stats(const float* ac_partials, int32_t N, int32_t H, int32_t Wd, const float* w,
                          const float* bias, const float* gamma, const float* beta, double eps, double momentum,
                          float* running_mean, float* running_var, double* stats, float* mean_nob, float* invstd,
                          float* scale, float* shift, afs_stream_t stream);
int afs_conv1_train_grads(const float* bwd_partials, int32_t N, int32_t H, int32_t Wd, const double* stats,
                          const float* w, const float* gamma, double eps, float* dW, float* dgamma, float* dbeta,
                          afs_stream_t stream);
int afs_conv1_train_fwd(const float* x, int32_t N, int32_t H, int32_t Wd, const float* w, const float* scale,
                        const float* shift, float negative_slope, float* out, afs_stream_t stream);
int afs_conv1_train_bwd(const float* x, const float* grad_out, int32_t N, int32_t H, int32_t Wd, const float* w,
                        const float* scale, const float* shift, const float* mean_nob, const float* invstd,
                        float negative_slope, float* partials, afs_stream_t stream);

/* (1b'') Conv64F blocks 2..4, inference only: Conv2d(64->64, 3x3, pad 1) + BatchNorm2d(eval) + ReLU / LeakyReLU
 * (+ MaxPool2d(3,3) when pool3 != 0), fused, channels-last, on the tensor cores (tcgen05 TF32, fp32 accumulate).
 * Replaces layer2..layer4 of libfewshot_core/model/backbone/conv_four.py:67-86,104-113 in eval mode.
 * x [N, H, Wd, 64] fp32 NHWC (device); out [N, H, Wd, 64] or, pooled, [N, H/3, Wd/3, 64] NHWC (device).
 * w_packed (device, afs_conv3x3_c64_packed_floats() floats, 16-byte aligned): the BatchNorm-folded weights in
 * operand order [tap][8-channel group][4-channel chunk][cout][4], produced on the host by afs_conv3x3_c64_pack_weights
 * from w_folded_host [64][64][3][3] (OIHW) with round-to-nearest TF32;
 * shift [64] (device) = (bias - mean)*gamma/sqrt(var+eps) + beta.
 * Built for Wd <= 61; AFS_ERR_UNSUPPORTED otherwise (the caller keeps cuDNN for such shapes).
 * Tiling is chosen per shape: three or four 128-row accumulators per tile, whichever needs fewer MMAs (three when
 * the operand ring of four does not fit in shared memory).                                                    */
size_t afs_conv3x3_c64_packed_floats(void);
int afs_conv3x3_c64_pack_weights(const float* w_folded_host, float* packed_host);
int afs_conv3x3_c64_bn_act_fwd_tf32(const float* x, int32_t N, int32_t H, int32_t Wd, const float* w_packed,
                                    const float* shift, float negative_slope, int32_t pool3, float* out,
                                    afs_stream_t stream);

/* (1b-bf16) The separately stated bf16 path of the same blocks (north star: "bf16 tensor-core path stated separately";
 * SURVEY 8f row 4 "channels-last/bf16 backbone"): bf16 activations and weights, tcgen05 kind::f16 MMAs with K = 16
 * (half the MMAs and half the activation bytes of the TF32 kernel), fp32 accumulation, fp32 BatchNorm shift and
 * activation.  NOT the parity path: logits move by ~1e-2 relative; the host side reports the argmax-flip rate.
 * x [N, H, Wd, 64] bf16 NHWC (device); w_packed (device, afs_conv3x3_c64_packed_bf16_elems() bf16 values, 16-byte
 * aligned) from afs_conv3x3_c64_pack_weights_bf16 (round to nearest even); out NHWC, bf16 when out_bf16 != 0 else
 * fp32.  The stem variant writes the first block's output as bf16 for it (TF32 arithmetic inside, as (1b')).    */
size_t afs_conv3x3_c64_packed_bf16_elems(void);
int afs_conv3x3_c64_pack_weights_bf16(const float* w_folded_host, uint16_t* packed_host);
int afs_conv3x3_c64_bn_act_fwd_bf16(const void* x, int32_t N, int32_t H, int32_t Wd, const void* w_packed,
                                    const float* shift, float negative_slope, int32_t pool3, void* out,
                                    int32_t out_bf16, afs_stream_t stream);
int afs_conv1_bn_act_pool3_fwd_tf32_bf16out(const float* x, int32_t N, int32_t H, int32_t Wd,
                                            const float* w_folded_host, const float* shift_host, int32_t C,
                                            float negative_slope, void* out_bf16, afs_stream_t stream);

/* (1c) MaxPool2d(3, 3) on channels-last activations: x [N, H, W, C] -> out [N, H/3, W/3, C], fp32,
 * C % 4 == 0, 16-byte aligned.  Replaces the nn.MaxPool2d(3, 3) after each Conv64F block
 * (libfewshot_core/model/backbone/conv_four.py:65,71,77,84) on the inference path.           */
int afs_maxpool3_nhwc_fwd(const float* x, int32_t N, int32_t H, int32_t W, int32_t C, float* out,
                          afs_stream_t stream);

/* (1c') The last max-pool of Conv64F fused with its linear head, inference path: x [N, H, W, C = 64] channels-last
 * (the output of block 4), 3 <= H, W < 6 so that MaxPool2d(3, 3) leaves one pixel; out[n, j] = bl[j] + sum_c
 * max_{3x3}(x[n, :, :, c]) * wl[j, c], wl [J, 64] row-major and bl [J] with BatchNorm1d already folded in, J % 8 == 0,
 * all pointers device, 16-byte aligned; fp32 FMA, channels summed in ascending order.  Replaces layer4_pool, the
 * flatten and `logits` (BatchNorm1d + Linear) of libfewshot_core/model/backbone/conv_four.py:84,89-92,120-123 in
 * eval mode.  AFS_ERR_UNSUPPORTED for other shapes (the caller keeps the pool + GEMM sequence).                  */
int afs_pool3_linear_fwd(const float* x, int32_t N, int32_t H, int32_t W, int32_t C, const float* wl, const float* bl,
                         int32_t J, float* out, afs_stream_t stream);

/* (1d) Tail of a ResNet-12 BasicBlock on the inference path, channels-last, BatchNorms folded into the
 * convolutions: out = MaxPool2d(k)( LeakyReLU_slope( a + b + bias[c] ) ), k in {1,2,3} (floor mode).
 * a, b [N, H, W, C] (b nullable), bias [C] (nullable), out [N, H/k, W/k, C]; fp32, C % 4 == 0, 16-byte aligned.
 * out may alias a when k == 1 (in-place bias + activation after a folded convolution).  Replaces
 * bn -> += residual -> relu -> maxpool of libfewshot_core/model/backbone/resnet_12.py:79-101 in eval mode. */
int afs_add_bias_act_pool_nhwc_fwd(const float* a, const float* b, const float* bias, int32_t N, int32_t H,
                                   int32_t W, int32_t C, float negative_slope, int32_t k, float* out,
                                   afs_stream_t stream);

/* (1d-bf16) The same tail for the separately stated bf16 trunk (ResNet.precision = "bf16"; SURVEY 8f row 4): a, b bf16
 * NHWC (b nullable), bias fp32 [C] (nullable), C % 8 == 0; sum, max, bias and activation in fp32; out bf16, or fp32 when
 * out_f32 != 0 (the last block feeds the fp32 heads).  out may alias a when k == 1 and out_f32 == 0.                  */
int afs_add_bias_act_pool_nhwc_bf16_fwd(const void* a, const void* b, const float* bias, int32_t N, int32_t H,
                                        int32_t W, int32_t C, float negative_slope, int32_t k, void* out,
                                        int32_t out_f32, afs_stream_t stream);

/* ------------------------------------------------------------------------
 * Episode row table shared by the heads (replaces the host slicing of
 * AbstractModel.split_by_episode, libfewshot_core/model/abstract_model.py:176-332).
 * Rows of `feat` are episode-major, class-major; block g = e*W + w holds S
 * support rows followed by that class's query window rows.
 *   cls_row[g]   = first row of block g, g in [0, E*W];  cls_row[E*W] = N.
 * Query window r of block g sits at feat row cls_row[g]+S+r and its logits
 * go to output row cls_row[g] - g*S + r (the order torch.cat gives at
 * proto_net.py:106-113).
 * ---------------------------------------------------------------------- */

/* (2a) ProtoNet head: prototype mean + logits, and per-row argmax.
 * Replaces ProtoLayer.forward (libfewshot_core/model/metric/proto_net.py:34-64)
 * and deepbdc.ProtoLayer.forward (libfewshot_core/model/metric/deepbdc.py:27-53).
 * mode: 0 = -sum_d (q-p)^2, 1 = cosine(q, p) with eps 1e-12, 2 = raw dot q.p.
 * feat [N, D] (row stride ld_feat floats), logits [NQ, W], pred [NQ] nullable
 * (argmax over W, lowest index on ties), NQ = N - E*W*S.  W <= 32.  D % 4 == 0
 * and 16-byte aligned rows.  ws: scratch of afs_proto_workspace_bytes() bytes,
 * 16-byte aligned: the E*W prototypes (written once by a pre-kernel, so that
 * support rows are read exactly once) and their inverse norms.               */
#define AFS_PROTO_EUCLIDEAN 0
#define AFS_PROTO_COSINE 1
#define AFS_PROTO_DOT 2
size_t afs_proto_workspace_bytes(int32_t E, int32_t W, int32_t S, int32_t D);
int afs_proto_fwd(const float* feat, int64_t ld_feat, const int32_t* cls_row, int32_t N,
                  int32_t E, int32_t W, int32_t S, int32_t D, int32_t mode, float* logits,
                  int32_t* pred, void* ws, size_t ws_bytes, afs_stream_t stream);

/* (2a') The same head in the "tf32" precision class, stated apart from the parity path above (north star: "one
 * tensor-core GEMM epilogue"): logit = -(|q|^2 - 2 q.p + |p|^2) with q.p as a tcgen05 TF32 GEMM fed by TMA and the
 * norms in fp32 (csrc/proto_tc.cu).  Euclidean mode only.  The expansion cancels and the MMA truncates its operands
 * to TF32: absolute logit error ~1e-3 |q| |p|, so near-tie predictions may differ from afs_proto_fwd.
 * Requirements: W <= 8, D % 32 == 0, ld_feat % 4 == 0, 16-byte aligned feat, and every run of 128 consecutive
 * feature rows must touch at most 32 / W episodes (logits of rows that break this come back as NaN).
 * ws: afs_proto_tc_workspace_bytes(E, W, D) bytes, 16-byte aligned.                                          */
size_t afs_proto_tc_workspace_bytes(int32_t E, int32_t W, int32_t D);
int afs_proto_fwd_tc(const float* feat, int64_t ld_feat, const int32_t* cls_row, int32_t N, int32_t E, int32_t W,
                     int32_t S, int32_t D, float* logits, int32_t* pred, void* ws, size_t ws_bytes, afs_stream_t stream);

/* Backward of (2a) for set_forward_loss (proto_net.py:148-154 under autograd):
 * grad_feat [N, D] (row stride ld_grad) is fully overwritten.  Modes 0 and 2. */
int afs_proto_bwd(const float* feat, int64_t ld_feat, const int32_t* cls_row, int32_t N,
                  int32_t E, int32_t W, int32_t S, int32_t D, int32_t mode,
                  const float* grad_logits, float* grad_feat, int64_t ld_grad,
                  afs_stream_t stream);

/* Backward of the cosine mode (MetaBaseline.set_forward_loss, libfewshot_core/model/metric/
 * meta_baseline.py:305-332 under autograd; the temperature factor stays outside, in the caller).
 * logits: the forward output (cosines) [NQ, W]; ws: afs_proto_bwd_cos_workspace_bytes() (row norms). */
size_t afs_proto_bwd_cos_workspace_bytes(int32_t N, int32_t E, int32_t W, int32_t S);
int afs_proto_bwd_cos(const float* feat, int64_t ld_feat, const int32_t* cls_row, int32_t N, int32_t E,
                      int32_t W, int32_t S, int32_t D, const float* logits, const float* grad_logits,
                      float* grad_feat, int64_t ld_grad, void* ws, size_t ws_bytes, afs_stream_t stream);

/* (2b) DN4 head: L2-normalised local descriptors, cosine relation, top-n_k
 * over each class's S*HW support descriptors, summed over the query's HW
 * descriptors.  Replaces DN4Layer.forward (libfewshot_core/model/metric/dn4.py:39-75).
 * feat [N, C, HW]; score [NQ, W]; topk_idx [NQ, W, HW, n_k] nullable (column
 * index in [0, S*HW), descending value, lowest index on ties); pred nullable.
 * 1 <= n_k <= min(8, S*HW); W <= 32.  ws/ws_bytes: scratch of
 * afs_dn4_workspace_bytes() (normalised descriptors + per-descriptor sums). */
size_t afs_dn4_workspace_bytes(int32_t N, int32_t E, int32_t W, int32_t S, int32_t C, int32_t HW);
int afs_dn4_fwd(const float* feat, const int32_t* cls_row, int32_t N, int32_t E, int32_t W,
                int32_t S, int32_t C, int32_t HW, int32_t n_k, float* score, int32_t* topk_idx,
                int32_t* pred, void* ws, size_t ws_bytes, afs_stream_t stream);

/* (2b') The same head with the cosine relation on the tensor cores: tcgen05 TF32 MMA into tensor
 * memory, top-n_k read straight out of TMEM, L2-normalisation fused into the operand staging (no
 * normalised copy in HBM).  Scores agree with afs_dn4_fwd to ~1e-4 relative; top-k indices may differ
 * at near-ties (TF32 operands), so afs_dn4_fwd remains the bit-stable parity path.  Built for
 * C % 8 == 0 and C <= 128 (AFS_ERR_UNSUPPORTED otherwise).  ws: afs_dn4_tc_workspace_bytes().   */
size_t afs_dn4_tc_workspace_bytes(int32_t N, int32_t E, int32_t W, int32_t S, int32_t HW);
int afs_dn4_fwd_tc(const float* feat, const int32_t* cls_row, int32_t N, int32_t E, int32_t W, int32_t S,
                   int32_t C, int32_t HW, int32_t n_k, float* score, int32_t* topk_idx, int32_t* pred,
                   void* ws, size_t ws_bytes, afs_stream_t stream);

/* (2b'') Warp-specialised version of (2b'): a pre-pass writes normalised TF32 descriptors K-major, the main
 * kernel feeds tcgen05.mma from TMA (cp.async.bulk.tensor, 128B swizzle) through a two-stage mbarrier
 * pipeline with two TMEM accumulators, so loads, MMAs and the top-k epilogue overlap.  C % 32 == 0 and
 * C <= 4096 (AFS_ERR_UNSUPPORTED otherwise); ws (256-byte aligned): afs_dn4_tc2_workspace_bytes().     */
size_t afs_dn4_tc2_workspace_bytes(int32_t N, int32_t E, int32_t W, int32_t S, int32_t C, int32_t HW);
int afs_dn4_fwd_tc2(const float* feat, const int32_t* cls_row, int32_t N, int32_t E, int32_t W, int32_t S,
                    int32_t C, int32_t HW, int32_t n_k, float* score, int32_t* topk_idx, int32_t* pred,
                    void* ws, size_t ws_bytes, afs_stream_t stream);

/* Backward of (2b) for DN4.set_forward_loss (dn4.py:122-155 under autograd): the top-k selection is
 * held fixed (topk_idx from afs_dn4_fwd), grad_feat [N, C, HW] is fully overwritten.  ws: scratch of
 * afs_dn4_bwd_workspace_bytes() (normalised descriptors + their gradient).                  */
size_t afs_dn4_bwd_workspace_bytes(int32_t N, int32_t C, int32_t HW);
int afs_dn4_bwd(const float* feat, const int32_t* cls_row, int32_t N, int32_t E, int32_t W, int32_t S,
                int32_t C, int32_t HW, int32_t n_k, const int32_t* topk_idx, const float* grad_score,
                float* grad_feat, void* ws, size_t ws_bytes, afs_stream_t stream);

/* (2c) BDC matrix: Gram, pairwise squared distance between channels, exp(t)
 * scale, sqrt, double centring, row-major upper triangle.  Replaces
 * BDCovpool + Triuvec (libfewshot_core/model/backbone/utils/bdc_pool.py:69-93).
 * x [B, C, M]; log_temp: device pointer to the scalar `temperature`;
 * out [B, C*(C+1)/2] if triu else [B, C*C].  afs_bdc_fwd / afs_bdc_bwd take C <= 64
 * (AFS_ERR_UNSUPPORTED above); C = 128, 192, ..., 640 go to afs_bdc_wide_fwd / _bwd below.
 * For C == 64 and M % 4 == 0 (16-byte aligned x) the Gram runs on the tcgen05 tensor cores
 * with 3 x TF32 operand splitting (csrc/bdc_tc.cu, within the same 1e-4 tolerance); other
 * shapes, or after afs_bdc_set_tensor_core(0), the fp32 FMA kernel of csrc/bdc.cu.  The
 * switch has no effect on the wide entries.                                        */
int afs_bdc_set_tensor_core(int32_t enable);
int afs_bdc_fwd(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp,
                int32_t triu, float* out, afs_stream_t stream);

/* Backward of (2c) for DeepBDC.set_forward_loss (deepbdc.py:354-378 under autograd through
 * BdcPool): grad_out as `out` of afs_bdc_fwd; grad_x [B, C, M]; grad_log_temp [B] = per-clip
 * contributions to d loss / d temperature (the caller sums them).                           */
int afs_bdc_bwd(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp, int32_t triu,
                const float* grad_out, float* grad_x, float* grad_log_temp, afs_stream_t stream);

/* (2c-wide) The same forward and backward for C = 128, 192, ..., 640 (whole 64-channel blocks; every other C returns
 * AFS_ERR_UNSUPPORTED), any M >= 1, any B >= 0 (B == 0 is a no-op), both layouts; csrc/bdc_wide.cu.  fp32 on the FMA
 * pipe, one CTA per clip and 64-channel block pair I <= J, no tensor cores whatever afs_bdc_set_tensor_core says.  A
 * clip's output has the same bits whatever the batch size and its position in the batch; the full output is exactly
 * symmetric.  ws: afs_bdc_wide_workspace_bytes(B, C, backward) bytes, 16-byte aligned (AFS_ERR_WORKSPACE if smaller
 * or misaligned); the size is 0 for an unsupported C.  Forward: norms and per-tile row sums, 4 C (k + 1) bytes per
 * clip (k = C / 64).  Backward: also dB's row and column sums and the k (k + 1) / 2 tiles of dD + dD^T, about
 * 8 C^2 bytes per clip.                                                                                          */
size_t afs_bdc_wide_workspace_bytes(int32_t B, int32_t C, int32_t backward);
int afs_bdc_wide_fwd(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp, int32_t triu,
                     float* out, void* ws, size_t ws_bytes, afs_stream_t stream);
int afs_bdc_wide_bwd(const float* x, int32_t B, int32_t C, int32_t M, const float* log_temp, int32_t triu,
                     const float* grad_out, float* grad_x, float* grad_log_temp, void* ws, size_t ws_bytes,
                     afs_stream_t stream);

/* (3) Window argmax -> per-query majority vote -> accuracy, all on device.
 * Replaces majority_vote + vote_catagorical_acc
 * (libfewshot_core/utils/utils.py:432-446) and the per-query D2H syncs.
 * logits [NQ, W]; q_start [nq+1] window offsets (exclusive cumsum of repeats);
 * q_target [nq]; q_pred [nq] out (mode of the window argmaxes); stats: int32[4]
 * scratch+out, stats[0] = #correct, stats[1] = nq (stats[2..3] internal);
 * acc_pct out = 100*correct/nq.  W <= 64.
 * tie_rule picks the label when several are equally frequent in a query:
 *   AFS_VOTE_TIE_SMALLEST   = what torch.mode returns for a CPU tensor;
 *   AFS_VOTE_TIE_TORCH_CUDA = what torch.mode returns for a CUDA tensor of <= 2048
 *     elements -- the reference's live rule, its set_forward being CUDA-only
 *     (proto_net.py:116-118).  See csrc/vote.cu for the rule.              */
#define AFS_VOTE_TIE_SMALLEST 0
#define AFS_VOTE_TIE_TORCH_CUDA 1
int afs_vote_acc(const float* logits, int32_t W, const int32_t* q_start, int32_t nq,
                 const int32_t* q_target, int32_t tie_rule, int32_t* q_pred, int32_t* stats,
                 float* acc_pct, afs_stream_t stream);

/* Energy score of DeepBDC (deepbdc.py:318-319 + utils.py:449-471):
 * u[q] = -logsumexp_w( mean over the query's windows of logits[., w] ).     */
int afs_energy_score(const float* logits, int32_t W, const int32_t* q_start, int32_t nq,
                     float* energy, afs_stream_t stream);

/* ------------------------------------------------------------------------
 * (4) Spectrogram-domain augmentation, fused with its de-/re-normalisation.
 * Replaces augment_spectrogram (libfewshot_core/audio_augmentations.py:531-604) and the eight
 * augmentations it dispatches to (:56-528) between denormalize_spectrogram (:16-33) and
 * normalize_spectrogram (:36-53).  in/out: `planes` contiguous [H, W] fp32 planes (every
 * (batch, channel) pair of the reference's [B,C,H,W] / [C,H,W] / [H,W] inputs); mean/std: the
 * scalar pair of Auxiliary/<set>_Mean_Std.npy.  The random parameters are drawn by the host (the
 * reference draws them with Python's `random`) and arrive in `cfg`:
 *   CUTOUT                 n_rect rectangles rect[k] = {top, left, height, width}, value `fill`
 *   LINEAR_FILTER          filter_curve [H] (device): per-frequency gain
 *   NOISE_SUPPRESSION      p0 = noise_percentile/100, p1 = suppression_strength
 *   NOISE_MATCHING         p0 = target_noise_level, i0 = smoothing_window
 *   BACKGROUND_SUBTRACTION p0 = percentile/100 (quantile along time, per frequency row)
 *   CONTRAST               p0 = contrast_factor, p1 = clip_percentile/100 (>= 1: no clipping)
 *   FOREGROUND_NORM        p0 = 1 - top_k_percent/100
 *   WIENER                 p0 = noise_floor_percentile/100, p1 = gain_factor
 * Quantiles are torch.quantile's (linear interpolation, fp32 rank arithmetic), found exactly. */
#define AFS_AUG_CUTOUT 0
#define AFS_AUG_LINEAR_FILTER 1
#define AFS_AUG_NOISE_SUPPRESSION 2
#define AFS_AUG_NOISE_MATCHING 3
#define AFS_AUG_BACKGROUND_SUBTRACTION 4
#define AFS_AUG_CONTRAST 5
#define AFS_AUG_FOREGROUND_NORM 6
#define AFS_AUG_WIENER 7
typedef struct afs_specaug_cfg {
  int32_t type;
  int32_t n_rect;
  int32_t rect[8][4];
  float fill;
  float p0, p1;
  int32_t i0;
} afs_specaug_cfg;
int afs_spec_augment(const float* in, int32_t planes, int32_t H, int32_t W, float mean, float std,
                     const afs_specaug_cfg* cfg, const float* filter_curve, float* out,
                     afs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AFS_B200_H_ */

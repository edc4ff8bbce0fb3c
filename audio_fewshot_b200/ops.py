"""Tensor-level wrappers over the C ABI (include/afs_b200.h).

Each function checks device / dtype / contiguity, allocates the outputs with
torch (device memory and streams are torch's job; the arithmetic is not) and
launches the sm_100a kernel on torch's current CUDA stream.  Nothing here
computes on the CPU and nothing falls back to PyTorch ops: a non-CUDA tensor or
a missing libafs_b200.so raises.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

PROTO_MODES = {"euclidean": 0, "cos_sim": 1, "dot": 2}


def launch_count():
    """Kernels launched through the C ABI by this process so far."""
    return int(_lib.lib().afs_launch_count())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _need_cuda(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.AfsError("%s must be a CUDA tensor (no CPU fallback exists)" % name)
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if t.device.index != torch.cuda.current_device():
        # kernels launch on the CURRENT device's current stream; a tensor of another GPU would fault in the kernel
        raise _lib.AfsError("%s lives on %s but the current CUDA device is cuda:%d; wrap the call in "
                            "`with torch.cuda.device(%r):`" % (name, t.device, torch.cuda.current_device(), str(t.device)))
    return t


# --------------------------------------------------------------------------- front-end
class LogMelPlan:
    """Owns an afs_logmel_plan (device tables: window, twiddles, packed mel bands).  n_fft is the window's length:
    512, 1024 or 2048 (AfsError otherwise); fb is [n_fft/2+1, n_mels], n_mels <= 128.  At n_fft 1024 plain launches
    run the pair engine and augmented ones the radix-8 engine; at 512 and 2048 every launch runs logmel_nfft_kernel
    (include/afs_b200.h)."""

    @property
    def engine(self):  # names that fixed rule; bench.py reads it to stamp logmel_engine
        return "auto"

    def __init__(self, fb, window, hop, n_mels, center=True, log_mult=10.0, log_eps=2.220446049250313e-16,
                 device=None):
        if device is None:
            device = torch.cuda.current_device()
        device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if device.index is None:  # "cuda" without an ordinal means the current device, not GPU 0
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        fb = np.ascontiguousarray(np.asarray(fb, dtype=np.float32))
        window = np.ascontiguousarray(np.asarray(window, dtype=np.float32))
        n_fft = window.shape[0]
        if fb.shape != (n_fft // 2 + 1, n_mels):
            raise ValueError("fb must be [n_fft/2+1, n_mels], got %s" % (fb.shape,))
        self.cfg = _lib.LogMelCfg(n_fft, int(hop), int(n_mels), 1 if center else 0, float(log_mult), float(log_eps))
        self.n_mels = int(n_mels)
        self._handle = C.c_void_p(0)
        h = _lib.lib()
        _lib.check(h.afs_logmel_plan_create(C.byref(self.cfg), fb.ctypes.data_as(C.c_void_p),
                                            window.ctypes.data_as(C.c_void_p), device.index,
                                            C.byref(self._handle)), "afs_logmel_plan_create")

    def num_frames(self, L):
        return int(_lib.lib().afs_logmel_num_frames(self._handle, int(L)))

    def forward(self, wav, mean, std, aug=None, seed=0, first_clip_index=0, out=None, pcm_scale=1.0 / 32768.0):
        """wav [B, L] CUDA, fp32 or int16 PCM (sample = pcm * pcm_scale) -> [B, 1, n_mels, T] fp32.
        mean/std: [n_mels] CUDA tensors."""
        _need_cuda(wav, "wav", torch.int16 if isinstance(wav, torch.Tensor) and wav.dtype == torch.int16
                   else torch.float32)
        _need_cuda(mean, "mean")
        _need_cuda(std, "std")
        if wav.dim() != 2:
            raise ValueError("wav must be [B, L]")
        if wav.device != self.device:
            raise _lib.AfsError("wav lives on %s but the plan's tables are on %s" % (wav.device, self.device))
        if mean.numel() != self.n_mels or std.numel() != self.n_mels:
            raise ValueError("mean/std must have n_mels entries")
        wav = wav.contiguous()
        B, L = wav.shape
        T = self.num_frames(L)
        if out is None:
            out = torch.empty((B, 1, self.n_mels, T), dtype=torch.float32, device=wav.device)
        elif tuple(out.shape) != (B, 1, self.n_mels, T) or not out.is_contiguous():
            raise ValueError("out has the wrong shape")
        aug_ref = None
        if aug is not None:
            aug_ref = C.byref(_lib.AugCfg(float(aug["gain_db"][0]), float(aug["gain_db"][1]),
                                          int(aug.get("max_shift", 0)),
                                          float(aug["noise_std"][0]), float(aug["noise_std"][1])))
        if wav.dtype == torch.int16:
            _lib.check(_lib.lib().afs_logmel_fwd_pcm16(self._handle, _ptr(wav), float(pcm_scale), B, L,
                                                       _ptr(mean.contiguous()), _ptr(std.contiguous()), aug_ref,
                                                       int(seed), int(first_clip_index), _ptr(out), _stream()),
                       "afs_logmel_fwd_pcm16")
            return out
        _lib.check(_lib.lib().afs_logmel_fwd(self._handle, _ptr(wav), B, L, _ptr(mean.contiguous()),
                                             _ptr(std.contiguous()), aug_ref, int(seed), int(first_clip_index),
                                             _ptr(out), _stream()), "afs_logmel_fwd")
        return out

    def __del__(self):
        try:
            if self._handle:
                _lib.lib().afs_logmel_plan_destroy(self._handle)
                self._handle = C.c_void_p(0)
        except Exception:
            pass


# --------------------------------------------------------------------------- backbone stem
def conv1_bn_act_pool3(x, w_folded, shift, negative_slope=0.0, tf32=False, out_dtype=torch.float32):
    """Fused eval-mode first block of Conv64F.  x [N,1,H,W] CUDA fp32; w_folded [C,9] / shift [C]:
    contiguous float32 numpy arrays (BatchNorm already folded).  Returns a channels_last
    [N, C, H//3, W//3] tensor.  tf32=True runs the tcgen05 tensor-core kernel (TF32 operands, the precision
    class of cuDNN's default convolutions); tf32=False the exact-fp32 SIMT kernel.  out_dtype=torch.bfloat16
    (tensor-core kernel only) writes the activation as bf16 for the bf16 blocks (conv3x3_c64_bn_act_bf16)."""
    _need_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 1:
        raise ValueError("x must be [N, 1, H, W]")
    x = x.contiguous()
    N, _, H, Wd = x.shape
    Cc = int(shift.shape[0])
    w_folded = np.ascontiguousarray(w_folded, dtype=np.float32).reshape(Cc, 9)
    shift = np.ascontiguousarray(shift, dtype=np.float32)
    if out_dtype not in (torch.float32, torch.bfloat16) or (out_dtype == torch.bfloat16 and not tf32):
        raise ValueError("out_dtype must be float32, or bfloat16 with tf32=True")
    out = torch.empty((N, Cc, H // 3, Wd // 3), dtype=out_dtype, device=x.device,
                      memory_format=torch.channels_last)
    if out_dtype == torch.bfloat16:
        fn = _lib.lib().afs_conv1_bn_act_pool3_fwd_tf32_bf16out
    else:
        fn = _lib.lib().afs_conv1_bn_act_pool3_fwd_tf32 if tf32 else _lib.lib().afs_conv1_bn_act_pool3_fwd
    _lib.check(fn(_ptr(x), N, H, Wd, w_folded.ctypes.data_as(C.c_void_p), shift.ctypes.data_as(C.c_void_p), Cc,
                  float(negative_slope), _ptr(out), _stream()), "afs_conv1_bn_act_pool3_fwd")
    return out


class _Conv1TrainFn(torch.autograd.Function):
    """Conv2d(1->64,3x3,pad 1,bias) + BatchNorm2d(batch statistics) + ReLU/LeakyReLU + MaxPool2d(3,3), training mode,
    as five sm_100a kernels (csrc/conv1_train.cu: autocorrelation, statistics, forward; backward, gradients); gradients
    for conv.weight, conv.bias (zero), bn.weight, bn.bias."""

    @staticmethod
    def forward(ctx, x, weight, bias, gamma, beta, running_mean, running_var, momentum, eps, slope):
        h = _lib.lib()
        N, _, H, Wd = x.shape
        x = x.contiguous()
        dev = x.device
        f32 = dict(dtype=torch.float32, device=dev)
        ac = torch.empty((int(h.afs_conv1_train_num_partials(0)), 55), **f32)
        _lib.check(h.afs_conv1_autocorr(_ptr(x), N, H, Wd, _ptr(ac), _stream()), "afs_conv1_autocorr")
        w32 = weight.detach().reshape(64, 9).contiguous()
        b32, g32, be32 = bias.detach().contiguous(), gamma.detach().contiguous(), beta.detach().contiguous()
        stats = torch.empty((90,), dtype=torch.float64, device=dev)
        vec = torch.empty((4, 64), **f32)  # mean_nob, invstd, scale, shift
        track = running_mean is not None and momentum is not None
        _lib.check(h.afs_conv1_train_stats(_ptr(ac), N, H, Wd, _ptr(w32), _ptr(b32), _ptr(g32), _ptr(be32), float(eps),
                                           float(momentum) if track else 0.0,
                                           _ptr(running_mean) if track else None, _ptr(running_var) if track else None,
                                           _ptr(stats), _ptr(vec[0]), _ptr(vec[1]), _ptr(vec[2]), _ptr(vec[3]),
                                           _stream()), "afs_conv1_train_stats")
        out = torch.empty((N, 64, H // 3, Wd // 3), memory_format=torch.channels_last, **f32)
        _lib.check(h.afs_conv1_train_fwd(_ptr(x), N, H, Wd, _ptr(w32), _ptr(vec[2]), _ptr(vec[3]), float(slope),
                                         _ptr(out), _stream()), "afs_conv1_train_fwd")
        ctx.save_for_backward(x, w32, g32, vec, stats)
        ctx.consts = (float(eps), float(slope))
        ctx.shapes = (weight.shape, bias.shape)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        x, w32, g32, vec, stats = ctx.saved_tensors
        eps, slope = ctx.consts
        h = _lib.lib()
        N, _, H, Wd = x.shape
        f32 = dict(dtype=torch.float32, device=x.device)
        g = grad_out.contiguous(memory_format=torch.channels_last)
        part = torch.empty((int(h.afs_conv1_train_num_partials(1)), 64, 11), **f32)
        _lib.check(h.afs_conv1_train_bwd(_ptr(x), _ptr(g), N, H, Wd, _ptr(w32), _ptr(vec[2]), _ptr(vec[3]),
                                         _ptr(vec[0]), _ptr(vec[1]), slope, _ptr(part), _stream()),
                   "afs_conv1_train_bwd")
        w_shape, b_shape = ctx.shapes
        dW = torch.empty((64, 9), **f32)
        dgb = torch.empty((2, 64), **f32)
        _lib.check(h.afs_conv1_train_grads(_ptr(part), N, H, Wd, _ptr(stats), _ptr(w32), _ptr(g32), eps, _ptr(dW),
                                           _ptr(dgb[0]), _ptr(dgb[1]), _stream()), "afs_conv1_train_grads")
        return (None, dW.reshape(w_shape), torch.zeros(b_shape, **f32), dgb[0], dgb[1], None, None, None, None, None)


def conv1_bn_act_pool3_train(x, conv, bn, negative_slope=0.0):
    """Training-mode first Conv64F block (batch statistics, running-stat update, autograd for the four parameter
    tensors) on CUDA.  x [N,1,H,W] fp32 without grad; conv: nn.Conv2d(1,64,3,padding=1); bn: nn.BatchNorm2d(64)."""
    _need_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 1 or conv.out_channels != 64 or x.requires_grad:
        raise ValueError("x must be [N, 1, H, W] data (no grad) and the block 1 -> 64 channels")
    track = bn.track_running_stats and bn.running_mean is not None
    if track:
        bn.num_batches_tracked += 1
    return _Conv1TrainFn.apply(x, conv.weight, conv.bias, bn.weight, bn.bias,
                               bn.running_mean if track else None, bn.running_var if track else None,
                               bn.momentum, bn.eps, float(negative_slope))


def conv3x3_c64_pack_weights(w_folded):
    """BatchNorm-folded [64, 64, 3, 3] weights (any device) -> the packed, TF32-rounded operand buffer of
    conv3x3_c64_bn_act (a float32 numpy array; upload it once and keep it)."""
    w = np.ascontiguousarray(w_folded.detach().float().cpu().numpy() if isinstance(w_folded, torch.Tensor)
                             else w_folded, dtype=np.float32)
    if w.shape != (64, 64, 3, 3):
        raise ValueError("weights must be [64, 64, 3, 3]")
    h = _lib.lib()
    packed = np.empty((int(h.afs_conv3x3_c64_packed_floats()),), dtype=np.float32)
    _lib.check(h.afs_conv3x3_c64_pack_weights(w.ctypes.data_as(C.c_void_p), packed.ctypes.data_as(C.c_void_p)),
               "afs_conv3x3_c64_pack_weights")
    return packed


def conv3x3_c64_supported(x):
    """Shapes the tensor-core block kernel is built for (others stay on cuDNN)."""
    return x.dim() == 4 and x.shape[1] == 64 and x.shape[3] <= 61


def conv3x3_c64_bn_act(x, w_packed, shift, negative_slope=0.0, pool=False):
    """Fused eval-mode Conv64F block (64 -> 64, 3x3, pad 1, folded BatchNorm, ReLU/LeakyReLU, optional 3x3/3
    max-pool) on the tensor cores.  x: channels_last [N, 64, H, W] CUDA fp32; w_packed: CUDA tensor from
    conv3x3_c64_pack_weights; shift: CUDA [64].  Returns a channels_last tensor."""
    _need_cuda(x, "x")
    _need_cuda(w_packed, "w_packed")
    _need_cuda(shift, "shift")
    if not conv3x3_c64_supported(x):
        raise ValueError("x must be [N, 64, H, W] with W <= 61")
    x = x.contiguous(memory_format=torch.channels_last)
    N, Cc, H, Wd = x.shape
    oh, ow = (H // 3, Wd // 3) if pool else (H, Wd)
    out = torch.empty((N, Cc, oh, ow), dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
    _lib.check(_lib.lib().afs_conv3x3_c64_bn_act_fwd_tf32(_ptr(x), N, H, Wd, _ptr(w_packed), _ptr(shift.contiguous()),
                                                          float(negative_slope), 1 if pool else 0, _ptr(out),
                                                          _stream()), "afs_conv3x3_c64_bn_act_fwd_tf32")
    return out


def conv3x3_c64_pack_weights_bf16(w_folded):
    """BatchNorm-folded [64, 64, 3, 3] weights -> the packed bf16 operand buffer of conv3x3_c64_bn_act_bf16 (a uint16
    numpy array of bf16 bit patterns, round to nearest even; upload with torch.from_numpy(p).view(torch.bfloat16))."""
    w = np.ascontiguousarray(w_folded.detach().float().cpu().numpy() if isinstance(w_folded, torch.Tensor)
                             else w_folded, dtype=np.float32)
    if w.shape != (64, 64, 3, 3):
        raise ValueError("weights must be [64, 64, 3, 3]")
    h = _lib.lib()
    packed = np.empty((int(h.afs_conv3x3_c64_packed_bf16_elems()),), dtype=np.uint16)
    _lib.check(h.afs_conv3x3_c64_pack_weights_bf16(w.ctypes.data_as(C.c_void_p), packed.ctypes.data_as(C.c_void_p)),
               "afs_conv3x3_c64_pack_weights_bf16")
    return packed


def conv3x3_c64_bn_act_bf16(x, w_packed, shift, negative_slope=0.0, pool=False, out_dtype=torch.bfloat16):
    """The bf16 variant of conv3x3_c64_bn_act (stated separately from the TF32 parity path): x channels_last
    [N, 64, H, W] CUDA bf16; w_packed: CUDA bf16 tensor from conv3x3_c64_pack_weights_bf16; shift: CUDA fp32 [64].
    fp32 accumulation, shift and activation; the channels_last result is bf16 or fp32 (out_dtype)."""
    _need_cuda(x, "x", torch.bfloat16)
    _need_cuda(w_packed, "w_packed", torch.bfloat16)
    _need_cuda(shift, "shift")
    if not conv3x3_c64_supported(x):
        raise ValueError("x must be [N, 64, H, W] with W <= 61")
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("out_dtype must be float32 or bfloat16")
    x = x.contiguous(memory_format=torch.channels_last)
    N, Cc, H, Wd = x.shape
    oh, ow = (H // 3, Wd // 3) if pool else (H, Wd)
    out = torch.empty((N, Cc, oh, ow), dtype=out_dtype, device=x.device, memory_format=torch.channels_last)
    _lib.check(_lib.lib().afs_conv3x3_c64_bn_act_fwd_bf16(_ptr(x), N, H, Wd, _ptr(w_packed), _ptr(shift.contiguous()),
                                                          float(negative_slope), 1 if pool else 0, _ptr(out),
                                                          1 if out_dtype == torch.bfloat16 else 0, _stream()),
               "afs_conv3x3_c64_bn_act_fwd_bf16")
    return out


def maxpool3_channels_last(x):
    """MaxPool2d(3, 3) of a channels_last [N, C, H, W] CUDA tensor -> channels_last [N, C, H//3, W//3]."""
    _need_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] % 4 != 0:
        raise ValueError("x must be [N, C, H, W] with C % 4 == 0")
    x = x.contiguous(memory_format=torch.channels_last)
    N, Cc, H, Wd = x.shape
    out = torch.empty((N, Cc, H // 3, Wd // 3), dtype=torch.float32, device=x.device,
                      memory_format=torch.channels_last)
    _lib.check(_lib.lib().afs_maxpool3_nhwc_fwd(_ptr(x), N, H, Wd, Cc, _ptr(out), _stream()),
               "afs_maxpool3_nhwc_fwd")
    return out


def pool3_linear_supported(x, out_features):
    """The fused tail needs 64 channels, a pooled map of one pixel and a multiple of 8 outputs."""
    return (x.dim() == 4 and x.shape[1] == 64 and x.shape[2] // 3 == 1 and x.shape[3] // 3 == 1 and out_features % 8 == 0)


def pool3_linear(x, weight, bias):
    """MaxPool2d(3, 3) -> flatten -> Linear of a channels_last [N, 64, H, W] CUDA tensor with 3 <= H, W < 6:
    out [N, J] = bias + pooled @ weight.T, weight [J, 64] (BatchNorm1d folded in by the caller)."""
    _need_cuda(x, "x")
    _need_cuda(weight, "weight")
    _need_cuda(bias, "bias")
    if not pool3_linear_supported(x, weight.shape[0]) or tuple(weight.shape[1:]) != (64,) or bias.numel() != weight.shape[0]:
        raise ValueError("pool3_linear: x must be [N, 64, H, W] with H // 3 == W // 3 == 1, weight [J, 64], J % 8 == 0")
    x = x.contiguous(memory_format=torch.channels_last)
    N, _, H, Wd = x.shape
    J = weight.shape[0]
    out = torch.empty((N, J), dtype=torch.float32, device=x.device)
    _lib.check(_lib.lib().afs_pool3_linear_fwd(_ptr(x), N, H, Wd, 64, _ptr(weight.contiguous()), _ptr(bias.contiguous()),
                                               J, _ptr(out), _stream()), "afs_pool3_linear_fwd")
    return out


def add_bias_act_pool(a, b=None, bias=None, negative_slope=0.0, k=1, inplace=False):
    """MaxPool2d(k)(LeakyReLU(a + b + bias[c])) on channels_last [N, C, H, W] CUDA tensors (b, bias optional;
    k in {1, 2, 3}).  inplace=True (k == 1 only) writes into `a`."""
    _need_cuda(a, "a")
    if a.dim() != 4 or a.shape[1] % 4 != 0:
        raise ValueError("a must be [N, C, H, W] with C % 4 == 0")
    if not a.is_contiguous(memory_format=torch.channels_last):
        a = a.contiguous(memory_format=torch.channels_last)  # a copy: "in place" then means into that copy
    if b is not None:
        _need_cuda(b, "b")
        if b.shape != a.shape:
            raise ValueError("a and b must have the same shape")
        b = b.contiguous(memory_format=torch.channels_last)
    if bias is not None:
        _need_cuda(bias, "bias")
        bias = bias.contiguous()
    N, Cc, H, Wd = a.shape
    if inplace and k != 1:
        raise ValueError("in-place only without pooling")
    out = a if inplace else torch.empty((N, Cc, H // k, Wd // k), dtype=torch.float32, device=a.device,
                                        memory_format=torch.channels_last)
    _lib.check(_lib.lib().afs_add_bias_act_pool_nhwc_fwd(_ptr(a), _ptr(b), _ptr(bias), N, H, Wd, Cc,
                                                         float(negative_slope), int(k), _ptr(out), _stream()),
               "afs_add_bias_act_pool_nhwc_fwd")
    return out


def add_bias_act_pool_bf16(a, b=None, bias=None, negative_slope=0.0, k=1, inplace=False, out_dtype=torch.bfloat16):
    """add_bias_act_pool for the bf16 trunk: a, b channels_last [N, C, H, W] CUDA bf16 (C % 8 == 0), bias fp32; the
    arithmetic is fp32; the result is bf16 (optionally in place when k == 1) or fp32."""
    _need_cuda(a, "a", torch.bfloat16)
    if a.dim() != 4 or a.shape[1] % 8 != 0:
        raise ValueError("a must be [N, C, H, W] with C % 8 == 0")
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("out_dtype must be float32 or bfloat16")
    if not a.is_contiguous(memory_format=torch.channels_last):
        a = a.contiguous(memory_format=torch.channels_last)
    if b is not None:
        _need_cuda(b, "b", torch.bfloat16)
        if b.shape != a.shape:
            raise ValueError("a and b must have the same shape")
        b = b.contiguous(memory_format=torch.channels_last)
    if bias is not None:
        _need_cuda(bias, "bias")
        bias = bias.contiguous()
    N, Cc, H, Wd = a.shape
    if inplace and (k != 1 or out_dtype != torch.bfloat16):
        raise ValueError("in-place only without pooling and with a bf16 result")
    out = a if inplace else torch.empty((N, Cc, H // k, Wd // k), dtype=out_dtype, device=a.device,
                                        memory_format=torch.channels_last)
    _lib.check(_lib.lib().afs_add_bias_act_pool_nhwc_bf16_fwd(_ptr(a), _ptr(b), _ptr(bias), N, H, Wd, Cc,
                                                              float(negative_slope), int(k), _ptr(out),
                                                              1 if out_dtype == torch.float32 else 0, _stream()),
               "afs_add_bias_act_pool_nhwc_bf16_fwd")
    return out


# --------------------------------------------------------------------------- heads
def _proto_call(feat, cls_row, E, W, S, mode, want_pred):
    _need_cuda(feat, "feat")
    _need_cuda(cls_row, "cls_row", torch.int32)
    if feat.dim() != 2:
        raise ValueError("feat must be [N, D]")
    if feat.stride(1) != 1 or feat.stride(0) % 4 != 0 or feat.data_ptr() % 16 != 0:
        feat = feat.contiguous()
    N, D = feat.shape
    if D % 4 != 0:
        raise ValueError("feature dim must be a multiple of 4")
    NQ = N - E * W * S
    logits = torch.empty((NQ, W), dtype=torch.float32, device=feat.device)
    pred = torch.empty((NQ,), dtype=torch.int32, device=feat.device) if want_pred else None
    h = _lib.lib()
    ws_bytes = int(h.afs_proto_workspace_bytes(E, W, S, D))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=feat.device) if ws_bytes else None
    _lib.check(h.afs_proto_fwd(_ptr(feat), feat.stride(0), _ptr(cls_row), N, E, W, S, D, PROTO_MODES[mode],
                               _ptr(logits), _ptr(pred), _ptr(ws), ws_bytes, _stream()), "afs_proto_fwd")
    return feat, logits, pred


class _ProtoFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, cls_row, E, W, S, mode):
        feat_c, logits, _ = _proto_call(feat.detach(), cls_row, E, W, S, mode, False)
        if mode == "cos_sim":
            ctx.save_for_backward(feat_c, cls_row, logits)
        else:
            ctx.save_for_backward(feat_c, cls_row)
        ctx.cfg = (E, W, S, mode)
        return logits

    @staticmethod
    def backward(ctx, grad_logits):
        E, W, S, mode = ctx.cfg
        feat, cls_row = ctx.saved_tensors[0], ctx.saved_tensors[1]
        N, D = feat.shape
        grad_logits = grad_logits.contiguous().float()
        grad_feat = torch.empty((N, D), dtype=torch.float32, device=feat.device)
        if mode == "cos_sim":
            logits = ctx.saved_tensors[2]
            h = _lib.lib()
            ws_bytes = int(h.afs_proto_bwd_cos_workspace_bytes(N, E, W, S))
            ws = torch.empty((max(ws_bytes, 16),), dtype=torch.uint8, device=feat.device)
            _lib.check(h.afs_proto_bwd_cos(_ptr(feat), feat.stride(0), _ptr(cls_row), N, E, W, S, D, _ptr(logits),
                                           _ptr(grad_logits), _ptr(grad_feat), D, _ptr(ws), ws_bytes, _stream()),
                       "afs_proto_bwd_cos")
            return grad_feat, None, None, None, None, None
        _lib.check(_lib.lib().afs_proto_bwd(_ptr(feat), feat.stride(0), _ptr(cls_row), N, E, W, S, D,
                                            PROTO_MODES[mode], _ptr(grad_logits), _ptr(grad_feat), D, _stream()),
                   "afs_proto_bwd")
        return grad_feat, None, None, None, None, None


def _proto_tc_call(feat, cls_row, E, W, S, want_pred):
    """Prototype head in the "tf32" precision class (csrc/proto_tc.cu): -(|q|^2 - 2 q.p + |p|^2) with q.p on the
    tcgen05 tensor cores.  Euclidean mode, W <= 8, D % 32 == 0."""
    _need_cuda(feat, "feat")
    _need_cuda(cls_row, "cls_row", torch.int32)
    if feat.dim() != 2:
        raise ValueError("feat must be [N, D]")
    if feat.stride(1) != 1 or feat.stride(0) % 4 != 0 or feat.data_ptr() % 16 != 0:
        feat = feat.contiguous()
    N, D = feat.shape
    NQ = N - E * W * S
    logits = torch.empty((NQ, W), dtype=torch.float32, device=feat.device)
    pred = torch.empty((NQ,), dtype=torch.int32, device=feat.device) if want_pred else None
    h = _lib.lib()
    ws_bytes = int(h.afs_proto_tc_workspace_bytes(E, W, D))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=feat.device)
    _lib.check(h.afs_proto_fwd_tc(_ptr(feat), feat.stride(0), _ptr(cls_row), N, E, W, S, D, _ptr(logits), _ptr(pred),
                                  _ptr(ws), ws_bytes, _stream()), "afs_proto_fwd_tc")
    return logits, pred


def proto_logits(feat, cls_row, E, W, S, mode="euclidean", want_pred=False, precision="fp32"):
    """Prototype head.  Differentiable w.r.t. feat (modes euclidean, dot) when feat requires grad.
    precision="tf32" (evaluation, euclidean only): the tensor-core GEMM-epilogue formulation, a separate precision
    class -- absolute logit error ~1e-3 |q| |p|, near-tie predictions may differ from the fp32 kernel."""
    if precision not in ("fp32", "tf32"):
        raise ValueError("precision must be 'fp32' or 'tf32'")
    if torch.is_grad_enabled() and feat.requires_grad:
        if precision != "fp32":
            raise ValueError("the tf32 prototype head has no backward: use precision='fp32' for training")
        logits = _ProtoFn.apply(feat, cls_row, E, W, S, mode)
        return (logits, None) if want_pred else logits
    if precision == "tf32":
        if mode != "euclidean":
            raise ValueError("the tf32 prototype head implements the euclidean mode only")
        logits, pred = _proto_tc_call(feat, cls_row, E, W, S, want_pred)
        return (logits, pred) if want_pred else logits
    _, logits, pred = _proto_call(feat, cls_row, E, W, S, mode, want_pred)
    return (logits, pred) if want_pred else logits


def dn4_tc_supported(C):
    """Channel counts the tensor-core DN4 head (precision="tf32") is built for: multiples of 32 up to 4096
    (csrc/dn4_tc2.cu) and multiples of 8 up to 128 (csrc/dn4_tc.cu).  Other maps run the fp32 head."""
    return C % 8 == 0 and (C <= 128 or (C % 32 == 0 and C <= 4096))


def _dn4_tc_call(feat, cls_row, E, W, S, n_k, want_topk, want_pred, staged=False):
    """Tensor-core (tcgen05 TF32) DN4 head; same outputs as _dn4_call.  C % 32 == 0 runs the TMA-fed
    pipeline (csrc/dn4_tc2.cu); other C % 8 == 0 widths (or staged=True) the register-staged kernel
    (csrc/dn4_tc.cu)."""
    _need_cuda(feat, "feat")
    _need_cuda(cls_row, "cls_row", torch.int32)
    feat = feat.contiguous()
    N, Cc = feat.shape[0], feat.shape[1]
    HW = int(np.prod(feat.shape[2:]))
    NQ = N - E * W * S
    score = torch.empty((NQ, W), dtype=torch.float32, device=feat.device)
    topk = torch.empty((NQ, W, HW, n_k), dtype=torch.int32, device=feat.device) if want_topk else None
    pred = torch.empty((NQ,), dtype=torch.int32, device=feat.device) if want_pred else None
    h = _lib.lib()
    if Cc % 32 == 0 and not staged:  # TMA-fed, warp-specialised pipeline
        ws_bytes = int(h.afs_dn4_tc2_workspace_bytes(N, E, W, S, Cc, HW))
        ws = torch.empty((max(ws_bytes, 256),), dtype=torch.uint8, device=feat.device)
        _lib.check(h.afs_dn4_fwd_tc2(_ptr(feat), _ptr(cls_row), N, E, W, S, Cc, HW, int(n_k), _ptr(score),
                                     _ptr(topk), _ptr(pred), _ptr(ws), ws_bytes, _stream()), "afs_dn4_fwd_tc2")
        return feat, score, topk, pred
    ws_bytes = int(h.afs_dn4_tc_workspace_bytes(N, E, W, S, HW))
    ws = torch.empty((max(ws_bytes, 16),), dtype=torch.uint8, device=feat.device)
    _lib.check(h.afs_dn4_fwd_tc(_ptr(feat), _ptr(cls_row), N, E, W, S, Cc, HW, int(n_k), _ptr(score), _ptr(topk),
                                _ptr(pred), _ptr(ws), ws_bytes, _stream()), "afs_dn4_fwd_tc")
    return feat, score, topk, pred


def _dn4_call(feat, cls_row, E, W, S, n_k, want_topk, want_pred):
    _need_cuda(feat, "feat")
    _need_cuda(cls_row, "cls_row", torch.int32)
    feat = feat.contiguous()
    N, Cc = feat.shape[0], feat.shape[1]
    HW = int(np.prod(feat.shape[2:]))
    NQ = N - E * W * S
    score = torch.empty((NQ, W), dtype=torch.float32, device=feat.device)
    topk = torch.empty((NQ, W, HW, n_k), dtype=torch.int32, device=feat.device) if want_topk else None
    pred = torch.empty((NQ,), dtype=torch.int32, device=feat.device) if want_pred else None
    h = _lib.lib()
    ws_bytes = int(h.afs_dn4_workspace_bytes(N, E, W, S, Cc, HW))
    ws = torch.empty((max(ws_bytes, 16),), dtype=torch.uint8, device=feat.device)
    _lib.check(h.afs_dn4_fwd(_ptr(feat), _ptr(cls_row), N, E, W, S, Cc, HW, int(n_k), _ptr(score), _ptr(topk),
                             _ptr(pred), _ptr(ws), ws_bytes, _stream()), "afs_dn4_fwd")
    return feat, score, topk, pred


class _Dn4Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, cls_row, E, W, S, n_k):
        feat_c, score, topk, _ = _dn4_call(feat.detach(), cls_row, E, W, S, n_k, True, False)
        ctx.save_for_backward(feat_c, cls_row, topk)
        ctx.cfg = (E, W, S, n_k)
        return score

    @staticmethod
    def backward(ctx, grad_score):
        feat, cls_row, topk = ctx.saved_tensors
        E, W, S, n_k = ctx.cfg
        N, Cc = feat.shape[0], feat.shape[1]
        HW = int(np.prod(feat.shape[2:]))
        grad_score = grad_score.contiguous().float()
        grad_feat = torch.empty_like(feat)
        h = _lib.lib()
        ws_bytes = int(h.afs_dn4_bwd_workspace_bytes(N, Cc, HW))
        ws = torch.empty((max(ws_bytes, 16),), dtype=torch.uint8, device=feat.device)
        _lib.check(h.afs_dn4_bwd(_ptr(feat), _ptr(cls_row), N, E, W, S, Cc, HW, int(n_k), _ptr(topk),
                                 _ptr(grad_score), _ptr(grad_feat), _ptr(ws), ws_bytes, _stream()), "afs_dn4_bwd")
        return grad_feat, None, None, None, None, None


def dn4_scores(feat, cls_row, E, W, S, n_k, want_topk=False, want_pred=False, precision="fp32"):
    """DN4 head.  feat [N, C, H, W] (or [N, C, HW]) -> score [NQ, W] (+ topk_idx [NQ, W, HW, n_k], pred).
    Differentiable w.r.t. feat when it requires grad (top-k selection held fixed, as torch.topk's backward).
    precision: "fp32" = bit-stable SIMT path (parity with the reference's indices); "tf32" = tcgen05 tensor-core
    path (the widths dn4_tc_supported accepts), scores to ~1e-4, indices may differ at near-ties."""
    if precision not in ("fp32", "tf32", "tf32_staged"):
        raise ValueError("precision must be 'fp32', 'tf32' or 'tf32_staged'")
    if torch.is_grad_enabled() and isinstance(feat, torch.Tensor) and feat.requires_grad:
        return _Dn4Fn.apply(feat, cls_row, E, W, S, n_k), None, None
    if precision == "tf32_staged":
        _, score, topk, pred = _dn4_tc_call(feat, cls_row, E, W, S, n_k, want_topk, want_pred, staged=True)
        return score, topk, pred
    call = _dn4_tc_call if precision == "tf32" else _dn4_call
    _, score, topk, pred = call(feat, cls_row, E, W, S, n_k, want_topk, want_pred)
    return score, topk, pred


def _bdc_wide_ws(B, Cc, backward, device):
    """Workspace of the 64-channel-block kernels (csrc/bdc_wide.cu) for C = 128, 192, ..., 640, else None: every other
    channel count stays with afs_bdc_fwd / afs_bdc_bwd."""
    h = _lib.lib()
    if h.afs_bdc_wide_workspace_bytes(1, Cc, 0) == 0:
        return None
    return torch.empty((int(h.afs_bdc_wide_workspace_bytes(B, Cc, 1 if backward else 0)),), dtype=torch.uint8,
                       device=device)


def _bdc_call(x, log_temp, triu):
    _need_cuda(x, "x")
    _need_cuda(log_temp, "log_temp")
    x = x.contiguous()
    B, Cc = x.shape[0], x.shape[1]
    M = int(np.prod(x.shape[2:]))
    out_dim = Cc * (Cc + 1) // 2 if triu else Cc * Cc
    out = torch.empty((B, out_dim), dtype=torch.float32, device=x.device)
    ws = _bdc_wide_ws(B, Cc, False, x.device)
    if ws is not None:
        _lib.check(_lib.lib().afs_bdc_wide_fwd(_ptr(x), B, Cc, M, _ptr(log_temp.contiguous()), 1 if triu else 0,
                                               _ptr(out), _ptr(ws), ws.numel(), _stream()), "afs_bdc_wide_fwd")
        return x, out
    _lib.check(_lib.lib().afs_bdc_fwd(_ptr(x), B, Cc, M, _ptr(log_temp.contiguous()), 1 if triu else 0, _ptr(out),
                                      _stream()), "afs_bdc_fwd")
    return x, out


class _BdcFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, log_temp, triu):
        x_c, out = _bdc_call(x.detach(), log_temp.detach(), triu)
        ctx.save_for_backward(x_c, log_temp.detach().contiguous())
        ctx.triu = triu
        ctx.t_shape = log_temp.shape
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, log_temp = ctx.saved_tensors
        B, Cc = x.shape[0], x.shape[1]
        M = int(np.prod(x.shape[2:]))
        grad_out = grad_out.contiguous().float()
        grad_x = torch.empty_like(x)
        grad_t = torch.empty((B,), dtype=torch.float32, device=x.device)
        ws = _bdc_wide_ws(B, Cc, True, x.device)
        if ws is not None:
            _lib.check(_lib.lib().afs_bdc_wide_bwd(_ptr(x), B, Cc, M, _ptr(log_temp), 1 if ctx.triu else 0,
                                                   _ptr(grad_out), _ptr(grad_x), _ptr(grad_t), _ptr(ws), ws.numel(),
                                                   _stream()), "afs_bdc_wide_bwd")
            return grad_x, grad_t.sum().reshape(ctx.t_shape), None
        _lib.check(_lib.lib().afs_bdc_bwd(_ptr(x), B, Cc, M, _ptr(log_temp), 1 if ctx.triu else 0, _ptr(grad_out),
                                          _ptr(grad_x), _ptr(grad_t), _stream()), "afs_bdc_bwd")
        return grad_x, grad_t.sum().reshape(ctx.t_shape), None


def bdc_pool(x, log_temp, triu=True):
    """BDC matrix of x [B, C, H, W] (or [B, C, M]) with log-temperature tensor (1 element).
    Differentiable w.r.t. x and log_temp when either requires grad."""
    if torch.is_grad_enabled() and (x.requires_grad or log_temp.requires_grad):
        return _BdcFn.apply(x, log_temp, triu)
    return _bdc_call(x, log_temp, triu)[1]


def bdc_set_tensor_core(enable):
    """Process-wide switch of afs_bdc_fwd: True (default) runs the Gram on tcgen05 where the shape allows
    (C == 64, M % 4 == 0), False always the fp32 FMA kernel.  C = 128, 192, ..., 640 always run the fp32 FMA kernels
    of csrc/bdc_wide.cu, with the same bits either way."""
    _lib.check(_lib.lib().afs_bdc_set_tensor_core(1 if enable else 0), "afs_bdc_set_tensor_core")


VOTE_TIE_RULES = {"smallest": 0, "torch_cuda": 1}


def vote_acc(logits, q_start, q_target, tie_rule="torch_cuda"):
    """-> (q_pred int32 [nq], acc_pct float32 0-dim tensor, stats int32 [4]) without any host sync.
    tie_rule: "torch_cuda" = torch.mode on a CUDA slice (the reference's live path, utils.py:443);
    "smallest" = torch.mode on a CPU tensor."""
    _need_cuda(logits, "logits")
    _need_cuda(q_start, "q_start", torch.int32)
    _need_cuda(q_target, "q_target", torch.int32)
    logits = logits.contiguous()
    nq = q_target.numel()
    W = logits.shape[1]
    q_pred = torch.empty((nq,), dtype=torch.int32, device=logits.device)
    stats = torch.empty((4,), dtype=torch.int32, device=logits.device)
    acc = torch.empty((), dtype=torch.float32, device=logits.device)
    _lib.check(_lib.lib().afs_vote_acc(_ptr(logits), W, _ptr(q_start), nq, _ptr(q_target), VOTE_TIE_RULES[tie_rule], _ptr(q_pred),
                                       _ptr(stats),
                                       _ptr(acc), _stream()), "afs_vote_acc")
    return q_pred, acc, stats


def energy_score(logits, q_start, nq):
    _need_cuda(logits, "logits")
    _need_cuda(q_start, "q_start", torch.int32)
    logits = logits.contiguous()
    out = torch.empty((nq,), dtype=torch.float32, device=logits.device)
    _lib.check(_lib.lib().afs_energy_score(_ptr(logits), logits.shape[1], _ptr(q_start), nq, _ptr(out), _stream()),
               "afs_energy_score")
    return out

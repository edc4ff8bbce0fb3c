#!/usr/bin/env python
"""Per-kernel roofline table at the BASELINE configs (SURVEY.md 8d): each head / front-end kernel timed
alone with CUDA events, inputs larger than L2 (or L2 flushed), algorithmic bytes / duration against the
measured HBM peak.  Prints one JSON line per kernel; `python bench_kernels.py > profiles/rNN_kernels.jsonl`.
bench.py is the contract benchmark; this is the supporting evidence for DESIGN.md section 3."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from audio_fewshot_b200 import ops  # noqa: E402
from audio_fewshot_b200.episode import EpisodeTable  # noqa: E402
from audio_fewshot_b200.frontend import LogMelFrontEnd  # noqa: E402


def peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return float(json.load(open(p))["hbm_gbs"]) if os.path.exists(p) else 6650.0


def timeit(fn, iters=20, warmup=3, flush=None):
    if os.environ.get("AFS_BENCH_ONCE"):  # under ncu: one warm launch + one profiled launch per kernel
        iters, warmup = 1, 1
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()  # > L2: evicts the previous iteration's lines
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def report(name, unit, units, bytes_per_unit, ms, ms_min, flops_per_unit=None, note=""):
    peak = peak_gbs()
    gbs = units * bytes_per_unit / (ms * 1e-3) / 1e9
    line = {"kernel": name, "unit": unit, "units_per_launch": units, "algorithmic_bytes_per_unit": bytes_per_unit,
            "ms_median": ms, "ms_min": ms_min, "achieved_gbs": gbs, "hbm_peak_gbs": peak, "frac_of_measured_hbm": gbs / peak,
            "units_per_s": units / (ms * 1e-3), "note": note}
    if flops_per_unit:
        line["tflops"] = units * flops_per_unit / (ms * 1e-3) / 1e12
    print(json.dumps(line), flush=True)


def main():
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    flush = torch.empty(160 * 2 ** 20 // 4, dtype=torch.float32, device=dev)  # 160 MB > 126 MB L2

    # ---- fused log-mel, shapes S5 and S1
    for tag, L, hop, B in (("S5 L=80000 hop=512", 80000, 512, 800), ("S5 L=80000 hop=512", 80000, 512, 3200),
                           ("S1 L=16000 hop=102", 16000, 102, 800)):
        fr = LogMelFrontEnd(hop_length=hop, n_mels=128, mean=-15.0, std=26.0).to(dev).eval()
        wav = torch.randn(B, L, device=dev) * 0.1
        T = 1 + L // hop
        out = torch.empty(B, 1, 128, T, device=dev)
        ms, mn = timeit(lambda: fr(wav, out=out), flush=flush)
        report("logmel_pair_kernel (warp-per-frame-pair engine, plain launches) %s B=%d" % (tag, B), "clip", B,
               4 * L + 4 * 128 * T, ms, mn, note="T=%d" % T)
        del wav, out
    fr = LogMelFrontEnd(hop_length=512, n_mels=128, mean=-15.0, std=26.0, seed=7,
                        aug={"gain_db": (-6.0, 6.0), "max_shift": 1600, "noise_std": (0.0, 0.02)}).to(dev).train()
    wav = torch.randn(800, 80000, device=dev) * 0.1
    out = torch.empty(800, 1, 128, 157, device=dev)
    ms, mn = timeit(lambda: fr(wav, out=out), flush=flush)
    report("logmel_kernel (radix-8 engine, augmented launches) S5 + Philox gain/shift/noise", "clip", 800, 4 * 80000 + 4 * 128 * 157, ms, mn)

    # ---- conv1 stem
    img = torch.randn(800, 1, 128, 157, device=dev)
    w = np.random.default_rng(0).standard_normal((64, 9)).astype(np.float32)
    b = np.zeros(64, np.float32)
    ms, mn = timeit(lambda: ops.conv1_bn_act_pool3(img, w, b, 0.0), flush=flush)
    report("conv1_bn_act_pool3_kernel", "clip", 800, 4 * 128 * 157 + 4 * 64 * 42 * 52, ms, mn,
           flops_per_unit=2 * 64 * 42 * 52 * 81, note="fp32 SIMT; flops count the 9 conv positions per pooled pixel")
    ms, mn = timeit(lambda: ops.conv1_bn_act_pool3(img, w, b, 0.0, tf32=True), flush=flush)
    report("conv1_tc_kernel (tcgen05 TF32)", "clip", 800, 4 * 128 * 157 + 4 * 64 * 42 * 52, ms, mn,
           flops_per_unit=2 * 64 * 42 * 52 * 81, note="useful flops; the MMAs pad K 9 -> 16")
    ms, mn = timeit(lambda: ops.conv1_bn_act_pool3(img, w, b, 0.0, tf32=True, out_dtype=torch.bfloat16), flush=flush)
    report("conv1_tc_kernel, bf16 output (stated separately)", "clip", 800, 4 * 128 * 157 + 2 * 64 * 42 * 52, ms, mn,
           flops_per_unit=2 * 64 * 42 * 52 * 81, note="same TF32 arithmetic, rounded to bf16 at the store")
    act = torch.randn(800, 64, 42, 52, device=dev).contiguous(memory_format=torch.channels_last)
    ms, mn = timeit(lambda: ops.maxpool3_channels_last(act), flush=flush)
    report("maxpool3_nhwc_kernel [800,64,42,52]", "clip", 800, 4 * 64 * (42 * 52 + 14 * 17), ms, mn)

    # ---- Conv64F blocks 2 and 3 on the tensor cores (conv + folded BN + ReLU + max-pool) vs cuDNN + our pool
    for tag, H, Wd in (("block 2 [800,64,42,52]", 42, 52), ("block 3 [800,64,14,17]", 14, 17)):
        act = torch.randn(800, 64, H, Wd, device=dev).contiguous(memory_format=torch.channels_last)
        wt = (torch.randn(64, 64, 3, 3, device=dev) * 0.06)
        wcl = wt.contiguous(memory_format=torch.channels_last)
        bias = torch.randn(64, device=dev)
        packed = torch.from_numpy(ops.conv3x3_c64_pack_weights(wt)).to(dev)
        flops = 2 * 64 * 64 * 9 * H * Wd
        nbytes = 4 * 64 * (H * Wd + (H // 3) * (Wd // 3))
        ms, mn = timeit(lambda: ops.conv3x3_c64_bn_act(act, packed, bias, 0.0, pool=True), flush=flush)
        report("conv3x3_c64_tc_kernel " + tag, "clip", 800, nbytes, ms, mn, flops_per_unit=flops,
               note="tcgen05 TF32, pool fused; useful flops")
        act16 = act.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        packed16 = torch.from_numpy(ops.conv3x3_c64_pack_weights_bf16(wt)).to(dev).view(torch.bfloat16)
        ms, mn = timeit(lambda: ops.conv3x3_c64_bn_act_bf16(act16, packed16, bias, 0.0, pool=True), flush=flush)
        report("conv3x3_c64_tc_kernel bf16 (stated separately) " + tag, "clip", 800, nbytes // 2, ms, mn, flops_per_unit=flops,
               note="tcgen05 kind::f16 bf16 operands, K = 16, two epilogue groups, bf16 in / bf16 out; useful flops")
        torch.backends.cudnn.allow_tf32 = True
        ms, mn = timeit(lambda: ops.maxpool3_channels_last(
            torch.cudnn_convolution_relu(act, wcl, bias, (1, 1), (1, 1), (1, 1), 1)), flush=flush)
        report("cuDNN conv+bias+ReLU (TF32) + maxpool3_nhwc " + tag, "clip", 800, nbytes, ms, mn, flops_per_unit=flops,
               note="library baseline for the kernel above")

    # ---- prototype head: C1 (D=1600, 5w5s15q), C2 (D=12800, 5w1s15q), C4 vectors (D=2080, 5w5s10q)
    for tag, E, W, S, Q, D, mode in (("C1 D=1600 5w5s15q", 256, 5, 5, 15, 1600, "euclidean"),
                                     ("C1 D=1600 5w5s15q", 2048, 5, 5, 15, 1600, "euclidean"),
                                     ("C2 D=12800 5w1s15q", 64, 5, 1, 15, 12800, "euclidean"),
                                     ("C2 D=12800 5w1s15q", 512, 5, 1, 15, 12800, "euclidean"),
                                     ("C4 D=2080 5w5s10q", 256, 5, 5, 10, 2080, "euclidean"),
                                     ("C1 cosine", 256, 5, 5, 15, 1600, "cos_sim")):
        N = E * W * (S + Q)
        feat = torch.randn(N, D, device=dev)
        tab = EpisodeTable(E, W, S, Q, np.ones(E * W * Q, dtype=np.int64), dev)
        ms, mn = timeit(lambda: ops.proto_logits(feat, tab.cls_row, E, W, S, mode), flush=flush)
        report("proto_mean_kernel + proto_fwd_kernel %s E=%d" % (tag, E), "episode", E, 4 * W * (S + Q) * D + 4 * W * Q * W, ms, mn,
               flops_per_unit=3 * W * Q * W * D + W * S * D, note="two launches; small batches are launch-bound")
        if mode == "euclidean" and D % 32 == 0:
            ms, mn = timeit(lambda: ops.proto_logits(feat, tab.cls_row, E, W, S, mode, precision="tf32"), flush=flush)
            report("proto_tc_kernel (TMA + tcgen05 TF32 GEMM epilogue) %s E=%d" % (tag, E), "episode", E,
                   4 * W * (S + Q) * D + 4 * W * Q * W, ms, mn, flops_per_unit=2 * W * (S + Q) * 32 * D,
                   note="precision class tf32; flops = executed MMA flops (N = 32 columns)")
        del feat

    # ---- DN4: C3 Conv64F maps [64,4,5], 5w5s15q n_k=3; ResNet-12 maps [640,8,9] 5w5s10q
    for tag, E, W, S, Q, C, H, Wd in (("C3 map 64x4x5 5w5s15q", 128, 5, 5, 15, 64, 4, 5),
                                      ("ResNet-12 map 640x8x9 5w5s10q", 4, 5, 5, 10, 640, 8, 9)):
        N = E * W * (S + Q)
        feat = torch.rand(N, C, H, Wd, device=dev)
        tab = EpisodeTable(E, W, S, Q, np.ones(E * W * Q, dtype=np.int64), dev)
        ms, mn = timeit(lambda: ops.dn4_scores(feat, tab.cls_row, E, W, S, 3), flush=flush)
        HW = H * Wd
        report("dn4 fp32 (normalize+main+reduce) " + tag, "episode", E, 4 * W * (S + Q) * C * HW + 4 * W * Q * W, ms, mn,
               flops_per_unit=2 * (W * Q * HW) * (W * S * HW) * C)
        if C % 32 == 0:
            ms, mn = timeit(lambda: ops.dn4_scores(feat, tab.cls_row, E, W, S, 3, precision="tf32"), flush=flush)
            report("dn4 tf32 TMA+tcgen05 (prep+main+reduce) " + tag, "episode", E,
                   4 * W * (S + Q) * C * HW + 4 * W * Q * W, ms, mn, flops_per_unit=2 * (W * Q * HW) * (W * S * HW) * C)

    # ---- BDC matrix: C4 map [64,16,19]
    x = torch.relu(torch.randn(2000, 64, 16, 19, device=dev))
    t = torch.full((1, 1), float(np.log(1 / 200.0)), device=dev)
    for B_ in (2000, 8000):
        x = torch.relu(torch.randn(B_, 64, 16, 19, device=dev))
        for tc in (False, True):
            ops.bdc_set_tensor_core(tc)
            ms, mn = timeit(lambda: ops.bdc_pool(x, t), flush=flush)
            report("%s C4 map 64x16x19 B=%d" % ("bdc_tc_kernel (tcgen05, 3xTF32)" if tc else "bdc_kernel (fp32 FMA)", B_), "clip", B_,
                   4 * 64 * 304 + 4 * 2080, ms, mn, flops_per_unit=2 * 64 * 64 * 304)
        ops.bdc_set_tensor_core(True)

    # ---- vote + accuracy, 5-way, one window per query
    nq = 75 * 4096
    logits = torch.randn(nq, 5, device=dev)
    q_start = torch.arange(nq + 1, dtype=torch.int32, device=dev)
    target = torch.randint(0, 5, (nq,), dtype=torch.int32, device=dev)
    ms, mn = timeit(lambda: ops.vote_acc(logits, q_start, target), flush=flush)
    report("vote_kernel 5-way", "episode", 4096, 4 * 75 * 5 + 4 * 75 * 3, ms, mn, note="logits + q_start + target + pred")


def extra():
    """Kernels outside the evaluation step: PCM16 front-end, spectrogram augmentation, ResNet-12 block tail, and the
    fused training block 1."""
    import random

    from audio_fewshot_b200 import augment as aug
    dev = torch.device("cuda", 0)
    flush = torch.empty(160 * 2 ** 20 // 4, dtype=torch.float32, device=dev)
    fr = LogMelFrontEnd(hop_length=512, n_mels=128, mean=-15.0, std=26.0).to(dev).eval()
    pcm = (torch.randn(800, 80000, device=dev) * 0.1 * 32768).round().clamp(-32768, 32767).to(torch.int16)
    out = torch.empty(800, 1, 128, 157, device=dev)
    ms, mn = timeit(lambda: fr(pcm, out=out), flush=flush)
    report("logmel_pair_kernel<int16> S5 (16-bit PCM input)", "clip", 800, 2 * 80000 + 4 * 128 * 157, ms, mn)

    img = torch.randn(800, 1, 128, 157, device=dev)
    for t in ("noise_suppression", "background_subtraction", "cutout"):
        random.seed(1)
        ms, mn = timeit(lambda: aug.augment_spectrogram(img, -15.0, 26.0, augmentation_type=t), flush=flush)
        report("spec_augment_kernel " + t + " [800,1,128,157]", "clip", 800, 2 * 4 * 128 * 157, ms, mn)

    a = torch.randn(320, 64, 128, 157, device=dev).contiguous(memory_format=torch.channels_last)
    b = torch.randn_like(a).contiguous(memory_format=torch.channels_last)
    bias = torch.randn(64, device=dev)
    ms, mn = timeit(lambda: ops.add_bias_act_pool(a, b, bias, 0.1, 2), flush=flush)
    report("add_bias_act_pool_nhwc_kernel k=2 [320,64,128,157] (ResNet-12 layer-1 tail)", "clip", 320,
           4 * 64 * 128 * 157 * 2 + 4 * 64 * 64 * 78, ms, mn)

    conv = torch.nn.Conv2d(1, 64, 3, padding=1).to(dev)
    bn = torch.nn.BatchNorm2d(64).to(dev).train()
    x = torch.randn(200, 1, 128, 157, device=dev)
    g = torch.randn(200, 64, 42, 52, device=dev).contiguous(memory_format=torch.channels_last)
    y = ops.conv1_bn_act_pool3_train(x, conv, bn, 0.0)
    ms, mn = timeit(lambda: ops.conv1_bn_act_pool3_train(x, conv, bn, 0.0), flush=flush)
    report("conv1 training block forward (autocorr + fwd kernels + batch-stat algebra) [200,1,128,157]", "clip", 200,
           4 * 128 * 157 * 2 + 4 * 64 * 42 * 52, ms, mn, flops_per_unit=2 * 64 * 42 * 52 * 81)

    def bwd():
        y = ops.conv1_bn_act_pool3_train(x, conv, bn, 0.0)
        y.backward(g)

    ms_fb, mn_fb = timeit(bwd, flush=flush)
    report("conv1 training block forward + backward [200,1,128,157]", "clip", 200,
           4 * 128 * 157 * 3 + 2 * 4 * 64 * 42 * 52, ms_fb, mn_fb, flops_per_unit=3 * 2 * 64 * 42 * 52 * 81)


def logmel_nfft():
    """The front-end at n_fft 512 (8 kHz, hop 256) and 2048 (32 kHz, hop 1024): 5 s clips -> [3200, 1, 128, 157], plain,
    augmented and int16 launches of logmel_nfft_kernel, the torch.stft -> |.|^2 -> matmul -> log10 sequence at the same
    shapes, and time per frame against the n_fft 1024 radix-8 engine (logmel_kernel, zero-range augmented launch) at
    16 kHz / hop 512, which transforms the same 3200 x 157 frames."""
    from oracle import frontend as ofe
    dev = torch.device("cuda", 0)
    flush = torch.empty(160 * 2 ** 20 // 4, dtype=torch.float32, device=dev)
    B, T = 3200, 157
    zero = {"gain_db": (0.0, 0.0), "max_shift": 0, "noise_std": (0.0, 0.0)}
    real = {"gain_db": (-6.0, 6.0), "max_shift": 1600, "noise_std": (0.0, 0.02)}
    fr = LogMelFrontEnd(hop_length=512, n_mels=128, mean=-15.0, std=26.0, aug=zero).to(dev).train()
    wav = torch.randn(B, 80000, device=dev) * 0.1
    out = torch.empty(B, 1, 128, T, device=dev)
    ms_1024, mn = timeit(lambda: fr(wav, out=out), flush=flush)
    report("logmel_kernel (n_fft 1024 radix-8 engine, zero-range augmented launch) 16 kHz hop 512 B=%d" % B, "clip", B,
           4 * 80000 + 4 * 128 * T, ms_1024, mn, note="reference for the per-frame ratios below")
    del wav
    for tag, sr, n_fft, hop, L in (("8 kHz n_fft 512 hop 256", 8000, 512, 256, 40000),
                                   ("32 kHz n_fft 2048 hop 1024", 32000, 2048, 1024, 160000)):
        wav = torch.randn(B, L, device=dev) * 0.1
        pcm = (wav * 32768).round().clamp(-32768, 32767).to(torch.int16)
        nb = 4 * L + 4 * 128 * T
        for launch, aug, x, nbytes in (("plain", None, wav, nb), ("augmented (Philox gain/shift/noise)", real, wav, nb),
                                       ("plain, int16 PCM input", None, pcm, nb - 2 * L)):
            f = LogMelFrontEnd(sr, n_fft=n_fft, hop_length=hop, n_mels=128, mean=-15.0, std=26.0, seed=7,
                               aug=aug).to(dev)
            f = f.train() if aug else f.eval()
            ms, mn = timeit(lambda: f(x, out=out), flush=flush)
            report("logmel_nfft_kernel<%d> %s, %s B=%d" % (n_fft, tag, launch, B), "clip", B, nbytes, ms, mn,
                   note="T=%d; time per frame / n_fft 1024 radix-8 engine = %.2f" % (T, ms / ms_1024))
        win = torch.from_numpy(ofe.hann_periodic(n_fft)).to(dev)
        fb = torch.from_numpy(ofe.mel_filterbank(n_fft // 2 + 1, 0.0, sr / 2.0, 128, sr)).to(dev)

        def torch_path():
            spec = torch.stft(wav, n_fft, hop, n_fft, win, center=True, pad_mode="reflect", return_complex=True)
            mel = torch.matmul((spec.real ** 2 + spec.imag ** 2).transpose(1, 2), fb).transpose(1, 2)
            return ((10 * torch.log10(mel + ofe.LOG_EPS) + 15.0) / 26.0).unsqueeze(1)

        ms, mn = timeit(torch_path, iters=5, flush=flush)
        report("torch.stft -> |.|^2 -> matmul -> log10 %s B=%d" % (tag, B), "clip", B, 4 * L + 4 * 128 * T, ms, mn,
               note="PyTorch op sequence at the same shape (cuFFT + GEMM; the spectrum goes through HBM)")
        del wav, pcm


def _bdc_reference_fp32(x, t):
    """The reference's op sequence (bdc_pool.py:69-93): BDCovpool's 7 bmm, 3 of them against an all-ones matrix, then
    Triuvec's gather."""
    B, C = x.shape[:2]
    x = x.reshape(B, C, -1)
    I = torch.eye(C, C, device=x.device).view(1, C, C).repeat(B, 1, 1)
    I_M = torch.ones(B, C, C, device=x.device)
    x_pow2 = x.bmm(x.transpose(1, 2))
    dcov = I_M.bmm(x_pow2 * I) + (x_pow2 * I).bmm(I_M) - 2 * x_pow2
    dcov = torch.sqrt(torch.exp(t) * torch.clamp(dcov, min=0.0) + 1e-5)
    dcov = dcov - 1.0 / C * dcov.bmm(I_M) - 1.0 / C * I_M.bmm(dcov) + 1.0 / (C * C) * I_M.bmm(dcov).bmm(I_M)
    index = torch.ones(C, C, device=x.device).triu().reshape(C * C).nonzero(as_tuple=False)
    return dcov.reshape(B, C * C)[:, index].squeeze(-1)


def bdc_wide():
    """BDC at C = 128, 256, 640 on the 16 x 19 map (M = 304, resnet12Bdc's trunk output), B = 300 (one C4 step) and
    2400 (input and output larger than L2): the 64-channel-block kernels of csrc/bdc_wide.cu, forward and forward +
    backward, against the reference's fp32 op sequence at the same shapes with TF32 off.  Useful flops: the Gram with
    its symmetry used, M C (C + 1) per clip, and for the backward also dX = S X, 2 C^2 M.  Bytes: x once, the
    triangle once (forward); the backward adds grad_out, x and grad_x."""
    dev = torch.device("cuda", 0)
    flush = torch.empty(160 * 2 ** 20 // 4, dtype=torch.float32, device=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    t = torch.full((1, 1), float(np.log(1 / 200.0)), device=dev)
    M = 304
    for C in (128, 256, 640):
        tri = C * (C + 1) // 2
        fwd_bytes, fwd_flops = 4 * C * M + 4 * tri, M * C * (C + 1)
        for B in (300, 2400):
            x = torch.relu(torch.randn(B, C, 16, 19, device=dev))
            ms, mn = timeit(lambda: ops.bdc_pool(x, t), flush=flush)
            report("bdc_wide forward (norms + gram + center, fp32 FMA) C=%d M=%d B=%d" % (C, M, B), "clip", B, fwd_bytes,
                   ms, mn, flops_per_unit=fwd_flops)
            ms_ref, mn_ref = timeit(lambda: _bdc_reference_fp32(x, t), iters=5, flush=flush)
            report("reference fp32 op sequence (7 bmm + Triuvec, TF32 off) C=%d M=%d B=%d" % (C, M, B), "clip", B,
                   fwd_bytes, ms_ref, mn_ref, flops_per_unit=fwd_flops,
                   note="same useful flops and bytes as the kernel row; bdc_wide forward is %.1fx faster" % (ms_ref / ms))
            xg = x.clone().requires_grad_(True)
            tg = t.clone().requires_grad_(True)
            g = torch.randn(B, tri, device=dev)

            def fwd_bwd():
                ops.bdc_pool(xg, tg).backward(g)

            ms, mn = timeit(fwd_bwd, flush=flush)
            report("bdc_wide forward + backward (norms, gram, center; norms, dbstats, bwd_tile, dx) C=%d M=%d B=%d"
                   % (C, M, B), "clip", B, fwd_bytes + 8 * C * M + 4 * tri, ms, mn,
                   flops_per_unit=2 * fwd_flops + 2 * C * C * M)
            del x, xg, g
            torch.cuda.empty_cache()


if __name__ == "__main__":
    if "--logmel-nfft" in sys.argv:
        logmel_nfft()
    elif "--bdc-wide" in sys.argv:
        bdc_wide()
    else:
        main()
        extra()
        logmel_nfft()
        bdc_wide()

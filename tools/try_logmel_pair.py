"""Bring-up check of the warp-per-frame-pair log-mel engine (csrc/logmel_pair.cu) on a B200: features against the float64
spec and the radix-8 engine, and the engines' times.
    python tools/try_logmel_pair.py [--quick]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from audio_fewshot_b200.frontend import LogMelFrontEnd
from oracle import frontend as fe

dev = torch.device("cuda", 0)
MEAN, STD = -15.0, 26.0


def check(B, L, hop, n_mels=128, seed=0):
    rng = np.random.default_rng(seed + L + hop)
    x = (rng.standard_normal((B, L)) * 0.1).astype(np.float32)
    xd = torch.from_numpy(x).to(dev)
    ref = fe.logmel_f64(x, hop=hop, n_mels=n_mels, mean=MEAN, std=STD)
    tol = 1e-4 * np.maximum(np.abs(ref * STD + MEAN), 1.0)
    msg = []
    for eng in ("pair", "fft"):
        fr = LogMelFrontEnd(hop_length=hop, n_mels=n_mels, mean=MEAN, std=STD, engine=eng).to(dev).eval()
        g = fr(xd).cpu().numpy()
        err = np.abs(g - ref) * STD
        msg.append("%s max dB err %.3e (worst err/tol %.3f, nan %d)" % (eng, err.max(), (err / tol).max(), int(np.isnan(g).sum())))
    print("B=%d L=%d hop=%d mels=%d: %s" % (B, L, hop, n_mels, "; ".join(msg)), flush=True)


def timeit(fr, wav, out, flush):
    for _ in range(3):
        fr(wav, out=out)
    ts = []
    for _ in range(20):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fr(wav, out=out); b.record(); b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[10]


if __name__ == "__main__":
    check(1, 80000, 512)
    check(3, 80000, 512)
    check(2, 16000, 102)
    check(1, 4099, 511)
    check(2, 12345, 160, n_mels=80)
    check(5, 33 * 512, 512)
    check(2, 3000, 256, n_mels=64)
    check(1, 513, 512, n_mels=64)
    if "--quick" not in sys.argv:
        flush = torch.empty(40 * 2 ** 20, device=dev)
        for B in ((3200,) if "--short" in sys.argv else (800, 3200)):
            wav = torch.randn(B, 80000, device=dev) * 0.1
            out = torch.empty(B, 1, 128, 157, device=dev)
            for eng in ("fft", "pair"):
                fr = LogMelFrontEnd(hop_length=512, n_mels=128, mean=MEAN, std=STD, engine=eng).to(dev).eval()
                t = timeit(fr, wav, out, flush)
                print("logmel %s B=%d: %.4f ms  %.0f GB/s  frac %.3f" % (eng, B, t, B * 400384 / t / 1e6, B * 400384 / t / 1e6 / 6555.5), flush=True)
        wav = torch.randn(3200, 16000, device=dev) * 0.1
        out = torch.empty(3200, 1, 128, 157, device=dev)
        for eng in ("fft", "pair"):
            fr = LogMelFrontEnd(hop_length=102, n_mels=128, mean=MEAN, std=STD, engine=eng).to(dev).eval()
            t = timeit(fr, wav, out, flush)
            print("logmel S1 %s B=3200: %.4f ms  %.0f GB/s  frac %.3f" % (eng, t, 3200 * (64000 + 4 * 128 * 157) / t / 1e6, 3200 * (64000 + 4 * 128 * 157) / t / 1e6 / 6555.5), flush=True)
        if "--short" in sys.argv:
            sys.exit(0)
        pcm = (torch.randn(3200, 80000, device=dev) * 3000).to(torch.int16)
        out = torch.empty(3200, 1, 128, 157, device=dev)
        for eng in ("fft", "pair"):
            fr = LogMelFrontEnd(hop_length=512, n_mels=128, mean=MEAN, std=STD, engine=eng).to(dev).eval()
            t = timeit(fr, pcm, out, flush)
            print("logmel pcm16 %s B=3200: %.4f ms" % (eng, t), flush=True)
        aug = {"gain_db": (-6.0, 6.0), "max_shift": 1600, "noise_std": (0.0, 0.02)}
        wav = torch.randn(800, 80000, device=dev) * 0.1
        out = torch.empty(800, 1, 128, 157, device=dev)
        for eng in ("fft", "pair"):
            fr = LogMelFrontEnd(hop_length=512, n_mels=128, mean=MEAN, std=STD, engine=eng, aug=aug, seed=7).to(dev).train()
            t = timeit(fr, wav, out, flush)
            print("logmel aug %s B=800: %.4f ms" % (eng, t), flush=True)

"""TEST INFRASTRUCTURE ONLY.  Writes tests/golden/logmel_torchaudio_nfft.npz: torchaudio.transforms.MelSpectrogram at
the FFT sizes other than 1024 that the front-end serves -- 8 kHz / n_fft 512 / hop 256, 32 kHz / 2048 / 1024 and
44.1 kHz / 2048 / 1411 (5 s clips -> 157 frames each), plus one odd shape at 2048 -- in the format of
make_frontend_golden.py (torchaudio's own fp32 filterbank and window per case, dB = 10 log10(mel + eps), and how far
torchaudio's fp32 pipeline sits from a float64 evaluation of the same formula and tables).

    python oracle/make_frontend_golden_nfft.py        (needs torchaudio)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import frontend as fe  # noqa: E402
from oracle import frontend_nfft as fen  # noqa: E402

CASES = {
    "sr8k": dict(seed=911, B=2, L=40000, sr=8000, n_fft=512, hop=256, n_mels=128),
    "sr32k": dict(seed=912, B=2, L=160000, sr=32000, n_fft=2048, hop=1024, n_mels=128),
    "sr44k": dict(seed=913, B=1, L=220500, sr=44100, n_fft=2048, hop=1411, n_mels=128),
    "odd": dict(seed=914, B=1, L=9999, sr=48000, n_fft=2048, hop=777, n_mels=80),
}


def waveform(c):
    rng = np.random.default_rng(c["seed"])
    t = np.arange(c["L"]) / float(c["sr"])
    x = rng.standard_normal((c["B"], c["L"])) * 0.1 + 0.05 * np.sin(2 * np.pi * 440.0 * t)[None, :]
    return x.astype(np.float32)


def meta(c):
    return [c["seed"], c["B"], c["L"], c["sr"], c["n_fft"], c["hop"], c["n_mels"]]


def main():
    import torch
    import torchaudio

    out = {}
    for name, c in CASES.items():
        x = waveform(c)
        ms = torchaudio.transforms.MelSpectrogram(c["sr"], n_fft=c["n_fft"], hop_length=c["hop"], n_mels=c["n_mels"],
                                                  f_min=0.0, f_max=c["sr"] / 2.0, power=2.0, norm="slaney",
                                                  mel_scale="slaney", center=True, pad_mode="reflect")
        with torch.no_grad():
            mel = ms(torch.from_numpy(x))  # [B, n_mels, T]
        db = (10.0 * torch.log10(mel + fe.LOG_EPS)).numpy().astype(np.float32)
        fb = ms.mel_scale.fb.numpy().astype(np.float32)          # [n_fft/2 + 1, n_mels], torchaudio's fp32 table
        win = ms.spectrogram.window.numpy().astype(np.float32)   # torch.hann_window(n_fft), periodic
        ref = fen.logmel_f64(x, c["hop"], c["n_fft"], n_mels=c["n_mels"], fb=fb, window=win)[:, 0]
        floor = float(np.abs(db - ref).max())
        print("%s: dB %s, torchaudio fp32 vs float64 of the same formula and tables: %.2e dB" % (name, db.shape, floor))
        out[name + "_db"] = db
        out[name + "_fb"] = fb
        out[name + "_window"] = win
        out[name + "_meta"] = np.asarray(meta(c), dtype=np.int64)
        out[name + "_fp32_floor_db"] = np.float64(floor)
    out["torchaudio_version"] = np.asarray(torchaudio.__version__)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "logmel_torchaudio_nfft.npz"), **out)


if __name__ == "__main__":
    main()

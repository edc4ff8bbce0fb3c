"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

The float64 log-mel spec of oracle/frontend.py (`logmel_f64`) at any FFT size: the same formula and the same
tables (periodic Hann window, slaney mel filterbank over n_fft/2 + 1 bins, reflect padding of n_fft/2), with n_fft
a parameter instead of 1024.  Used by the tests of the n_fft 512 / 2048 kernel and by make_frontend_golden_nfft.py.
"""
import numpy as np

from oracle.frontend import LOG_EPS, frames, hann_periodic, mel_filterbank


def logmel_f64(x, hop, n_fft, n_mels=128, sample_rate=16000, mean=None, std=None, center=True, log_mult=10.0,
               log_eps=LOG_EPS, fb=None, window=None):
    """[B, L] -> [B, 1, n_mels, T] in float64.  fb/window default to the fp32-rounded tables the kernel receives."""
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    if fb is None:
        fb = mel_filterbank(n_fft // 2 + 1, 0.0, sample_rate / 2.0, n_mels, sample_rate)
    if window is None:
        window = hann_periodic(n_fft)
    fr = frames(x, hop, center, n_fft) * np.asarray(window, dtype=np.float64)[None, None, :]
    spec = np.fft.rfft(fr, axis=-1)
    power = spec.real ** 2 + spec.imag ** 2  # [B, T, n_fft/2 + 1]
    mel = power @ np.asarray(fb, dtype=np.float64)  # [B, T, n_mels]
    db = np.transpose(log_mult * np.log10(mel + log_eps), (0, 2, 1))  # [B, n_mels, T]
    if mean is not None:
        mean = np.broadcast_to(np.asarray(mean, dtype=np.float64).reshape(-1), (n_mels,))
        std = np.broadcast_to(np.asarray(std, dtype=np.float64).reshape(-1), (n_mels,))
        db = (db - mean[None, :, None]) / std[None, :, None]
    return db[:, None, :, :]

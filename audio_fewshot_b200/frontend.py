"""Waveform -> normalised log-mel front-end module (the step before every set_forward).

The reference consumes pre-computed spectrogram folders and normalises them with the
[mean, std] pair of Auxiliary/*_Mean_Std.npy (libfewshot_core/test.py:398-399,
audio_augmentations.py:36-53); it has no waveform code (SURVEY.md F2).  This module
produces that `image` tensor [B, 1, 128, 157] directly from waveforms with ONE fused
sm_100a kernel (csrc/logmel_pair.cu; csrc/logmel.cu when augmenting; csrc/logmel_nfft.cu at n_fft 512 and 2048).  Tables (periodic Hann, slaney mel filterbank) are
computed here in float64 and rounded to fp32 once.
"""
import math

import numpy as np
import torch
from torch import nn

from . import ops

LOG_EPS = 2.220446049250313e-16


def hann_window(n_fft):
    k = np.arange(n_fft, dtype=np.float64)
    return (0.5 - 0.5 * np.cos(2.0 * np.pi * k / n_fft)).astype(np.float32)


def slaney_mel_filterbank(n_freqs, n_mels, sample_rate, f_min=0.0, f_max=None):
    """Triangular filters on the slaney mel scale with slaney (area) normalisation,
    [n_freqs, n_mels] -- the convention of librosa.filters.mel / MetaAudio."""
    f_max = sample_rate / 2.0 if f_max is None else f_max
    lin_step, knee_hz, log_step = 200.0 / 3.0, 1000.0, math.log(6.4) / 27.0
    knee_mel = knee_hz / lin_step

    def to_mel(f):
        f = np.asarray(f, dtype=np.float64)
        return np.where(f >= knee_hz, knee_mel + np.log(np.maximum(f, 1e-30) / knee_hz) / log_step, f / lin_step)

    def to_hz(m):
        m = np.asarray(m, dtype=np.float64)
        return np.where(m >= knee_mel, knee_hz * np.exp(log_step * (m - knee_mel)), m * lin_step)

    bin_hz = np.linspace(0.0, sample_rate // 2, n_freqs)
    edges = to_hz(np.linspace(to_mel(f_min), to_mel(f_max), n_mels + 2))
    widths = np.diff(edges)
    rise = (bin_hz[:, None] - edges[None, :-2]) / widths[None, :-1]
    fall = (edges[None, 2:] - bin_hz[:, None]) / widths[None, 1:]
    tri = np.clip(np.minimum(rise, fall), 0.0, None)
    tri *= (2.0 / (edges[2:] - edges[:-2]))[None, :]
    return tri.astype(np.float32)


def load_mean_std(path):
    """Auxiliary/*_Mean_Std.npy -> (mean, std) Python floats (test.py:398-399)."""
    mean, std = np.load(path).flatten().tolist()
    return float(mean), float(std)


class LogMelFrontEnd(nn.Module):
    """wav [B, L] (CUDA fp32, or int16 PCM read as pcm * pcm_scale) -> [B, 1, n_mels, T].
    mean/std: scalars or per-bin [n_mels].  n_fft 512, 1024 or 2048 (other sizes raise AfsError on the first call):
    e.g. 8 kHz audio with n_fft 512 / hop 256, 32 kHz with 2048 / 1024 -- 5 s clips give the [1, 128, 157] image of
    16 kHz / 1024 / 512 at the audio's own rate."""

    def __init__(self, sample_rate=16000, n_fft=1024, hop_length=512, n_mels=128, f_min=0.0, f_max=None,
                 mean=0.0, std=1.0, mean_std_file=None, center=True, log_mult=10.0, log_eps=LOG_EPS, aug=None,
                 seed=0, pcm_scale=1.0 / 32768.0):
        super().__init__()
        if mean_std_file is not None:
            mean, std = load_mean_std(mean_std_file)
        self.sample_rate, self.n_fft, self.hop_length, self.n_mels = sample_rate, n_fft, hop_length, n_mels
        self.center, self.log_mult, self.log_eps = center, log_mult, log_eps
        self.aug, self.seed, self.pcm_scale = aug, seed, pcm_scale
        self._fb = slaney_mel_filterbank(n_fft // 2 + 1, n_mels, sample_rate, f_min, f_max)
        self._window = hann_window(n_fft)
        self.register_buffer("mean", torch.full((n_mels,), 0.0) + torch.as_tensor(mean, dtype=torch.float32).reshape(-1))
        self.register_buffer("std", torch.full((n_mels,), 0.0) + torch.as_tensor(std, dtype=torch.float32).reshape(-1))
        self._plan = None

    def plan(self):
        if self._plan is None:
            self._plan = ops.LogMelPlan(self._fb, self._window, self.hop_length, self.n_mels, self.center,
                                        self.log_mult, self.log_eps, device=self.mean.device)
        return self._plan

    def forward(self, wav, first_clip_index=0, out=None):
        aug = self.aug if self.training else None
        return self.plan().forward(wav, self.mean, self.std, aug=aug, seed=self.seed,
                                   first_clip_index=first_clip_index, out=out, pcm_scale=self.pcm_scale)

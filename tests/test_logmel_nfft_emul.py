"""Host logic of the n_fft 512 / 2048 log-mel kernel (csrc/logmel_nfft.cu): its __host__ __device__ phase functions
(csrc/logmel_nfft.cuh) run on the CPU, 64 'threads' per phase, against the float64 spec; the shared-memory layouts of
its exchanges; the ELL table budget at the new sizes; the config keys that select them; and the oracle against the
torchaudio golden at those sizes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from oracle import frontend as fe
from oracle import frontend_nfft as fen

SRC = os.path.join(ROOT, "tests", "emul", "logmel_nfft_emul.cu")
OUT_DIR = os.path.join(ROOT, "tests", "emul", "_build")
LIB = os.path.join(OUT_DIR, "liblogmel_nfft_emul.so")
CSRC = os.path.join(ROOT, "audio_fewshot_b200", "csrc")

# (sample rate, n_fft): the sizes the kernel is built for, at the rates that use them
RATES = [(8000, 512), (32000, 2048), (44100, 2048), (48000, 2048)]


@pytest.fixture(scope="module")
def emul():
    os.makedirs(OUT_DIR, exist_ok=True)
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("logmel_core.cuh", "logmel_fft.cuh", "logmel_nfft.cuh")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-x", "cu",
                               "-Wno-deprecated-gpu-targets", "-I", CSRC, "-I", os.path.join(ROOT, "include"),
                               SRC, "-o", LIB])
    return C.CDLL(LIB)


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def run(lib, x, n_fft, hop, sr, n_mels=128, mean=-15.1, std=26.2, center=True):
    L = x.shape[0]
    bins = n_fft // 2 + 1
    fb = np.ascontiguousarray(fe.mel_filterbank(bins, 0.0, sr / 2.0, n_mels, sr))
    win = fe.hann_periodic(n_fft)
    T = fe.num_frames(L, hop, center, n_fft)
    out = np.zeros((n_mels, T), np.float32)
    power = np.zeros((T, bins), np.float32)
    m = np.full(n_mels, mean, np.float32)
    s = np.full(n_mels, std, np.float32)
    got_T = lib.emul_logmel_nfft(n_fft, vp(x), C.c_int64(L), hop, 1 if center else 0, vp(fb), vp(win), n_mels, vp(m),
                                 vp(s), C.c_float(10.0), C.c_float(fe.LOG_EPS), vp(out), vp(power))
    assert got_T == T
    return out, power, fb, m, s


@pytest.mark.parametrize("n_fft,sr,L,hop,n_mels,center", [
    (512, 8000, 6000, 256, 128, True),     # hop == n_fft/2
    (512, 8000, 2049, 131, 80, True),      # odd hop, fewer mels
    (512, 8000, 257, 100, 64, True),       # minimum legal length
    (512, 8000, 3000, 200, 128, False),
    (2048, 32000, 12000, 1024, 128, True),
    (2048, 44100, 9001, 1411, 128, True),  # odd length and hop
    (2048, 48000, 1025, 512, 64, True),    # minimum legal length
    (2048, 48000, 7000, 777, 80, False),
])
def test_phases_match_float64_spec(emul, n_fft, sr, L, hop, n_mels, center):
    rng = np.random.default_rng(L + hop)
    x = (rng.standard_normal(L) * 0.1).astype(np.float32)
    x[: L // 3] += (0.5 * np.sin(np.arange(L // 3) * 0.3)).astype(np.float32)
    out, power, fb, m, s = run(emul, x, n_fft, hop, sr, n_mels, center=center)
    fr = fe.frames(x[None].astype(np.float64), hop, center, n_fft)[0] * fe.hann_periodic(n_fft).astype(np.float64)
    pref = np.abs(np.fft.rfft(fr, axis=-1)) ** 2
    assert power.shape == pref.shape
    assert np.abs(power - pref).max() / pref.max() < 2e-6
    ref = fen.logmel_f64(x[None], hop, n_fft, n_mels=n_mels, sample_rate=sr, mean=m, std=s, center=center)
    db_err = np.abs(out - ref[0, 0]).max() * 26.2
    assert db_err < 1e-4, db_err  # north-star tolerance 1e-4 (de-normalised dB, SURVEY.md 7.3)


@pytest.mark.parametrize("n_fft", [512, 2048])
def test_exchange_layouts_are_bijective_and_conflict_free(emul, n_fft):
    """Every 64-bit access of the FFT phases puts the 16 words of a half-warp on 16 different 8-byte banks, the
    32-bit power stores of a warp on 32 banks, and the exchange-2 slot function is a bijection onto [0, n_fft/2)."""
    assert emul.emul_nfft_bank_check(n_fft) == 1


@pytest.mark.parametrize("sr,n_fft", RATES)
@pytest.mark.parametrize("n_mels", [64, 80, 128])
def test_ell_weight_table_fits_and_reproduces_the_filterbank(emul, sr, n_fft, n_mels):
    """pack_mel_ell over n_fft/2 + 1 bins expands back to exactly the slaney filterbank, every filter has one owner,
    every power read stays inside the written bins, and the table fits the kernel's budget (4 096 floats at 512,
    8 192 at 2048)."""
    bins = n_fft // 2 + 1
    fb = np.ascontiguousarray(fe.mel_filterbank(bins, 0.0, sr / 2.0, n_mels, sr))
    dense = np.zeros((bins, n_mels), np.float32)
    owners = np.zeros(n_mels, np.int32)
    n = emul.emul_mel_ell_dense_n(vp(fb), n_mels, bins, vp(dense), vp(owners))
    assert 0 < n <= (8192 if n_fft == 2048 else 4096) and n % 32 == 0, n
    assert (owners == 1).all()
    assert np.array_equal(dense, fb)


def test_pure_tone_lands_in_the_right_mel_bin(emul):
    sr, f0 = 32000, 3000.0
    x = np.sin(2 * np.pi * f0 * np.arange(32000) / sr).astype(np.float32)
    out, _, fb, _, _ = run(emul, x, 2048, 1024, sr, mean=0.0, std=1.0)
    k = int(round(f0 / (sr / 2048)))
    assert int(out[:, 5].argmax()) == int(fb[k].argmax())


def test_frontend_from_config_defaults_and_new_keys():
    """Without the new keys the front-end is exactly today's (16 kHz, n_fft 1024, hop 512); with them it is built at
    the requested rate, FFT size and hop."""
    from audio_fewshot_b200.config import frontend_from_config
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    old = LogMelFrontEnd(sample_rate=16000, n_fft=1024, hop_length=512, n_mels=128)
    fr = frontend_from_config({}, "cpu")
    assert (fr.sample_rate, fr.n_fft, fr.hop_length, fr.n_mels, fr.center) == (16000, 1024, 512, 128, True)
    assert np.array_equal(fr._window, old._window) and np.array_equal(fr._fb, old._fb)
    for sr, n_fft, hop in ((32000, 2048, 1024), (8000, 512, 256), (44100, 2048, 1411)):
        fr = frontend_from_config({"sample_rate": sr, "n_fft": n_fft, "hop_length": hop}, "cpu")
        assert (fr.sample_rate, fr.n_fft, fr.hop_length) == (sr, n_fft, hop)
        assert np.array_equal(fr._window, fe.hann_periodic(n_fft))
        assert fr._fb.shape == (n_fft // 2 + 1, 128)
        assert np.abs(fr._fb - fe.mel_filterbank(n_fft // 2 + 1, 0.0, sr / 2.0, 128, sr)).max() < 1e-6


@pytest.mark.parametrize("case", ["sr8k", "sr32k", "sr44k", "odd"])
def test_oracle_matches_torchaudio_golden_at_new_fft_sizes(case):
    """The float64 spec at n_fft 512 / 2048, fed torchaudio's own fp32 tables, reproduces torchaudio's MelSpectrogram
    (oracle/make_frontend_golden_nfft.py) to within the distance of torchaudio's fp32 pipeline from float64."""
    from oracle.make_frontend_golden_nfft import CASES, meta, waveform
    g = np.load(os.path.join(GOLDEN, "logmel_torchaudio_nfft.npz"), allow_pickle=False)
    c = CASES[case]
    assert meta(c) == g[case + "_meta"].tolist()
    floor = float(g[case + "_fp32_floor_db"])
    assert floor < 2e-5
    x = waveform(c)
    want = fen.logmel_f64(x, c["hop"], c["n_fft"], n_mels=c["n_mels"], fb=g[case + "_fb"],
                          window=g[case + "_window"])[:, 0]
    assert want.shape == g[case + "_db"].shape
    assert np.abs(want - g[case + "_db"]).max() <= floor * 1.0001 + 1e-9


@pytest.mark.parametrize("hop,center,n_mels", [(512, True, 128), (511, True, 80), (300, False, 64)])
def test_general_spec_at_1024_is_the_canonical_spec(hop, center, n_mels):
    """oracle.frontend_nfft restates oracle.frontend.logmel_f64 with n_fft as a parameter; at 1024 the two agree bit
    for bit, with and without per-bin statistics."""
    x = (np.random.default_rng(hop).standard_normal((2, 7000)) * 0.1).astype(np.float32)
    mean, std = np.linspace(-30, -5, n_mels), np.linspace(10, 30, n_mels)
    assert np.array_equal(fen.logmel_f64(x, hop, 1024, n_mels=n_mels, center=center),
                          fe.logmel_f64(x, hop=hop, n_mels=n_mels, center=center))
    assert np.array_equal(fen.logmel_f64(x, hop, 1024, n_mels=n_mels, center=center, mean=mean, std=std),
                          fe.logmel_f64(x, hop=hop, n_mels=n_mels, center=center, mean=mean, std=std))

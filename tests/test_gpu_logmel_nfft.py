"""The fused log-mel front-end at n_fft 512 (8 kHz audio) and 2048 (32-48 kHz audio), csrc/logmel_nfft.cu: parity with
the float64 spec (oracle/frontend_nfft.py) and with torchaudio (tests/golden/logmel_torchaudio_nfft.npz), Philox
augmentation against the oracle, int16 PCM, determinism, engine selection, refusals, and the model and data paths
at 32 kHz.  Every shape runs as a plain launch and as an augmented launch with zero-width ranges.

Tolerance (north star: 1e-4 relative, fp32; SURVEY.md 7.3): on the de-normalised dB value,
|a - b| <= 1e-4 * max(|b|, 1)."""
import os
import wave

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import frontend as fe
from oracle import frontend_nfft as fen
from oracle import philox

pytestmark = pytest.mark.gpu
LAUNCHES = ("plain", "augmented")
ZERO_AUG = dict(gain_db=(0.0, 0.0), max_shift=0, noise_std=(0.0, 0.0))
REAL_AUG = dict(gain_db=(-3.0, 3.0), max_shift=700, noise_std=(0.005, 0.02))
MEAN, STD = -15.114207, 26.22313  # Auxiliary/Clean_Mean_Std.npy


def make_frontend(cuda, sr, n_fft, hop, n_mels=128, launch="plain", mean=MEAN, std=STD, **kw):
    """launch="augmented": a training-mode front-end with zero-width augmentation ranges unless `aug` is given."""
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    if launch == "augmented":
        kw.setdefault("aug", ZERO_AUG)
    fr = LogMelFrontEnd(sample_rate=sr, n_fft=n_fft, hop_length=hop, n_mels=n_mels, mean=mean, std=std, **kw).to(cuda)
    return fr.train() if launch == "augmented" else fr.eval()


def spec(x, sr, n_fft, hop, n_mels=128, center=True):
    return fen.logmel_f64(x, hop, n_fft, n_mels=n_mels, sample_rate=sr, mean=MEAN, std=STD, center=center)


def assert_db_close(got, want_norm, tol=1e-4):
    got_db = got.astype(np.float64) * STD + MEAN
    want_db = want_norm * STD + MEAN
    err = np.abs(got_db - want_db)
    bound = tol * np.maximum(np.abs(want_db), 1.0)
    assert (err <= bound).all(), "max dB err %.3e (bound %.3e)" % (err.max(), bound[err.argmax()])


def signal(shape, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * 0.1).astype(np.float32)
    L = shape[1]
    x[0, : L // 3] += (0.5 * np.sin(np.arange(L // 3) * 0.3)).astype(np.float32)
    return x


SHAPES = [  # B, L, sample rate, n_fft, hop, n_mels, center
    (2, 40000, 8000, 512, 256, 128, True),       # 5 s at 8 kHz -> [1, 128, 157]; hop == n_fft/2
    (2, 160000, 32000, 2048, 1024, 128, True),   # 5 s at 32 kHz -> [1, 128, 157]; hop == n_fft/2
    (1, 220500, 44100, 2048, 1411, 128, True),   # 5 s at 44.1 kHz, odd hop -> 157 frames
    (1, 240000, 48000, 2048, 1536, 128, True),   # 5 s at 48 kHz -> 157 frames
    (1, 257, 8000, 512, 256, 64, True),          # minimum legal length n_fft/2 + 1
    (1, 1025, 32000, 2048, 1024, 64, True),
    (1, 4099, 8000, 512, 131, 80, True),         # odd length, odd hop: unaligned loads
    (2, 12345, 48000, 2048, 777, 80, True),
    (2, 20 * 256, 8000, 512, 256, 128, True),    # 21 frames: one partial chunk
    (3, 33 * 1024, 32000, 2048, 1024, 128, True),  # 34 frames: the second chunk holds 2
    (2, 16000, 8000, 512, 200, 128, False),
    (2, 40000, 32000, 2048, 1000, 80, False),
]


@pytest.mark.parametrize("B,L,sr,n_fft,hop,n_mels,center", SHAPES)
@pytest.mark.parametrize("launch", LAUNCHES)
def test_logmel_nfft_matches_float64_spec(cuda, B, L, sr, n_fft, hop, n_mels, center, launch):
    x = signal((B, L), L + hop)
    fr = make_frontend(cuda, sr, n_fft, hop, n_mels, launch, center=center)
    got = fr(torch.from_numpy(x).to(cuda)).cpu().numpy()
    want = spec(x, sr, n_fft, hop, n_mels, center)
    assert got.shape == want.shape == (B, 1, n_mels, fe.num_frames(L, hop, center, n_fft))
    assert_db_close(got, want)


@pytest.mark.parametrize("case", ["sr8k", "sr32k", "sr44k", "odd"])
@pytest.mark.parametrize("launch", LAUNCHES)
def test_logmel_nfft_matches_torchaudio_golden(cuda, case, launch):
    """torchaudio's MelSpectrogram at n_fft 512 / 2048 (oracle/make_frontend_golden_nfft.py), with torchaudio's own fp32
    filterbank and window handed to the kernel.  torchaudio's fp32 pipeline sits up to ~1.1e-5 dB from float64 at
    8 kHz / 512 (recorded in the golden), far inside the 1e-4 relative bound."""
    from audio_fewshot_b200 import ops
    from oracle.make_frontend_golden_nfft import CASES, meta, waveform
    g = np.load(os.path.join(GOLDEN, "logmel_torchaudio_nfft.npz"), allow_pickle=False)
    c = CASES[case]
    assert meta(c) == g[case + "_meta"].tolist()
    assert float(g[case + "_fp32_floor_db"]) < 2e-5
    x = waveform(c)
    plan = ops.LogMelPlan(g[case + "_fb"], g[case + "_window"], c["hop"], c["n_mels"], device=cuda)
    zero = torch.zeros(c["n_mels"], device=cuda)
    one = torch.ones(c["n_mels"], device=cuda)
    aug = ZERO_AUG if launch == "augmented" else None
    got = plan.forward(torch.from_numpy(x).to(cuda), zero, one, aug=aug).cpu().numpy()[:, 0]
    want = g[case + "_db"].astype(np.float64)
    err = np.abs(got - want)
    assert (err <= 1e-4 * np.maximum(np.abs(want), 1.0)).all(), err.max()


@pytest.mark.parametrize("sr,n_fft,hop", [(8000, 512, 256), (8000, 512, 255), (32000, 2048, 1024), (48000, 2048, 1535)])
@pytest.mark.parametrize("gain,shift,noise", [((-6.0, 6.0), 0, (0.0, 0.0)), ((0.0, 0.0), 0, (0.01, 0.05)),
                                              ((-3.0, 3.0), 1000, (0.005, 0.02))])
def test_logmel_nfft_augmentation_matches_oracle(cuda, sr, n_fft, hop, gain, shift, noise):
    """Philox gain / shift / noise keyed by (seed, global clip index), as oracle.philox.augment_waveform; an odd hop
    starts every other frame on an odd sample, off the paired Philox path."""
    B, L, seed, first = 4, 2 * sr, 1234567890123, 40
    x = signal((B, L), 21)
    aug = dict(gain_db=gain, max_shift=shift, noise_std=noise)
    fr = make_frontend(cuda, sr, n_fft, hop, aug=aug, seed=seed, launch="augmented")
    got = fr(torch.from_numpy(x).to(cuda), first_clip_index=first).cpu().numpy()
    y = philox.augment_waveform(x, seed, first, gain, shift, noise)
    assert_db_close(got, spec(y, sr, n_fft, hop), tol=3e-4)  # Box-Muller in fp32 on the device vs fp64 in the oracle
    fr.eval()
    assert_db_close(fr(torch.from_numpy(x).to(cuda)).cpu().numpy(), spec(x, sr, n_fft, hop))


@pytest.mark.parametrize("B,L,sr,n_fft,hop", [(3, 40000, 8000, 512, 256), (2, 4099, 8000, 512, 131),
                                             (2, 160000, 32000, 2048, 1024), (2, 12345, 48000, 2048, 777)])
@pytest.mark.parametrize("launch", ["plain", "augmented", "real_aug"])
def test_logmel_nfft_pcm16_is_bit_identical_to_converted_fp32(cuda, B, L, sr, n_fft, hop, launch):
    rng = np.random.default_rng(L + hop)
    pcm = np.clip(np.round(rng.standard_normal((B, L)) * 0.1 * 32768.0), -32768, 32767).astype(np.int16)
    pcm[0, :7] = [-32768, 32767, 0, 1, -1, 12345, -12345]
    x = pcm.astype(np.float32) / np.float32(32768.0)
    if launch == "real_aug":
        fr = make_frontend(cuda, sr, n_fft, hop, launch="augmented", aug=REAL_AUG, seed=77)
    else:
        fr = make_frontend(cuda, sr, n_fft, hop, launch=launch)
    a = fr(torch.from_numpy(pcm).to(cuda), first_clip_index=5)
    b = fr(torch.from_numpy(x).to(cuda), first_clip_index=5)
    assert a.dtype == torch.float32 and torch.equal(a, b)
    if launch != "real_aug":
        assert_db_close(a.cpu().numpy(), spec(x, sr, n_fft, hop))


@pytest.mark.parametrize("sr,n_fft,hop,L", [(8000, 512, 256, 40000), (32000, 2048, 1024, 160000),
                                            (44100, 2048, 1411, 220500)])
def test_logmel_nfft_is_deterministic_and_batch_independent(cuda, sr, n_fft, hop, L):
    """Repeated launches are bit-identical, plain and zero-range augmented launches agree bit for bit (the same kernel
    with the same gain of 1), and a clip's features do not depend on how the batch is sliced; with real augmentation
    ranges the global clip index keys the draw, so a slice launched with its own first_clip_index matches too."""
    B = 37
    x = torch.from_numpy(signal((B, L), 5)).to(cuda)
    fr = make_frontend(cuda, sr, n_fft, hop)
    a = fr(x)
    for _ in range(2):
        assert torch.equal(fr(x), a)
    for i, n in ((0, 1), (13, 5), (36, 1)):
        assert torch.equal(fr(x[i:i + n]), a[i:i + n])
    assert torch.equal(make_frontend(cuda, sr, n_fft, hop, launch="augmented")(x), a)
    fa = make_frontend(cuda, sr, n_fft, hop, launch="augmented", aug=REAL_AUG, seed=9)
    full = fa(x, first_clip_index=100)
    assert torch.equal(fa(x, first_clip_index=100), full)
    assert torch.equal(fa(x[13:18], first_clip_index=113), full[13:18])


def test_logmel_launch_selects_the_engine_by_fft_size(cuda):
    """n_fft 512 and 2048 run logmel_nfft_kernel for plain and augmented launches; n_fft 1024 still runs
    logmel_pair_kernel (plain) and logmel_kernel (augmented)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    def kernels(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]

    want = {(512, "plain"): "logmel_nfft_kernel<512", (512, "augmented"): "logmel_nfft_kernel<512",
            (2048, "plain"): "logmel_nfft_kernel<2048", (2048, "augmented"): "logmel_nfft_kernel<2048",
            (1024, "plain"): "logmel_pair_kernel<", (1024, "augmented"): "logmel_kernel<"}
    for (n_fft, launch), name in want.items():
        sr = {512: 8000, 1024: 16000, 2048: 32000}[n_fft]
        x = torch.from_numpy(signal((8, 5 * sr), 3)).to(cuda)
        fr = make_frontend(cuda, sr, n_fft, n_fft // 2, launch=launch, aug=REAL_AUG, seed=4) if launch == "augmented" \
            else make_frontend(cuda, sr, n_fft, n_fft // 2)
        fr(x)
        names = kernels(lambda: fr(x))
        assert len(names) == 1 and name in names[0], (n_fft, launch, names)
        pcm = (x * 32768).round().clamp(-32768, 32767).to(torch.int16)
        names = kernels(lambda: fr(pcm))
        assert len(names) == 1 and name in names[0], (n_fft, launch, names)


@pytest.mark.parametrize("n_fft,n_mels", [(256, 128), (4096, 128), (1000, 128), (512, 129), (2048, 129)])
def test_logmel_refuses_unbuilt_sizes(cuda, n_fft, n_mels):
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200._lib import AfsError
    fb = fe.mel_filterbank(n_fft // 2 + 1, 0.0, 8000.0, n_mels, 16000)
    with pytest.raises(AfsError):
        ops.LogMelPlan(fb, fe.hann_periodic(n_fft), n_fft // 2, n_mels, device=cuda)


def test_logmel_nfft_rejects_clips_shorter_than_the_padding(cuda):
    from audio_fewshot_b200._lib import AfsError
    fr = make_frontend(cuda, 32000, 2048, 1024)
    with pytest.raises(AfsError):
        fr(torch.zeros(1, 1024, device=cuda))  # reflect padding needs L > n_fft/2
    assert fr(torch.zeros(1, 1025, device=cuda)).shape == (1, 1, 128, 2)


def test_32khz_episodes_through_conv64f_and_protonet(cuda):
    """5 s synthetic episodes at 32 kHz through LogMelFrontEnd(32000, n_fft=2048, hop_length=1024) -> Conv64F ->
    ProtoNet.set_forward, against the same model fed the float64 oracle's features rounded to fp32."""
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.synthetic import name_seeded_weights_, synthetic_clip_batch
    W, S, Q, E, sr, L = 5, 2, 3, 2, 32000, 160000
    wav = synthetic_clip_batch(7, 0, E, W, S, Q, L, sample_rate=sr)
    torch.manual_seed(0)
    emb = name_seeded_weights_(arch.Conv64F(is_flatten=True, num_channels=1))
    model = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q, emb_func=emb,
                          device=cuda).to(cuda).eval()
    front = LogMelFrontEnd(sr, n_fft=2048, hop_length=1024, n_mels=128, mean=MEAN, std=STD).to(cuda).eval()
    repeats = torch.ones(E * W * Q, dtype=torch.long)
    with torch.no_grad():
        image = front(torch.from_numpy(wav).to(cuda))
        assert image.shape == (E * W * (S + Q), 1, 128, 157)
        got, _ = model.set_forward([image, None, repeats, E * W * S])
        ref_img = torch.from_numpy(spec(wav, sr, 2048, 1024).astype(np.float32)).to(cuda)
        want, _ = model.set_forward([ref_img, None, repeats, E * W * S])
    assert (got - want).abs().max().item() <= 1e-3 * want.abs().max().item()
    assert torch.equal(got.argmax(1), want.argmax(1))


def test_32khz_wav_config_runs_through_the_loader_and_front_end(cuda, tmp_path):
    """A `data_format: wav` config at sample_rate 32000 / audio_samples 160000 / n_fft 2048 / hop_length 1024:
    get_dataloader serves int16 windows and frontend_from_config turns them into the [rows, 1, 128, 157] image."""
    from audio_fewshot_b200.config import frontend_from_config
    from audio_fewshot_b200.data import get_dataloader
    rng = np.random.default_rng(8)
    for c in ["dog", "cat", "owl", "bat", "fox"]:
        os.makedirs(tmp_path / "wav" / c)
        for i in range(3):
            pcm = rng.integers(-20000, 20000, size=int(rng.integers(100000, 200000))).astype("<i2")
            with wave.open(str(tmp_path / "wav" / c / ("%d.wav" % i)), "wb") as w:
                w.setnchannels(1); w.setsampwidth(2); w.setframerate(32000)
                w.writeframes(pcm.tobytes())
    cfg = dict(way_num=5, shot_num=1, query_num=2, test_way=5, test_shot=1, test_query=2, train_episode=2,
               test_episode=2, episode_size=1, data_root=str(tmp_path / "wav"), data_format="wav",
               audio_samples=160000, sample_rate=32000, n_fft=2048, hop_length=1024)
    (loader,) = get_dataloader(cfg, "test")
    wav, target, repeats, support_size = next(iter(loader))
    rows = 5 + int(repeats.sum())
    assert wav.dtype == torch.int16 and wav.shape == (rows, 160000)
    front = frontend_from_config(cfg, cuda).eval()
    assert (front.sample_rate, front.n_fft, front.hop_length) == (32000, 2048, 1024)
    image = front(wav.to(cuda))
    assert image.shape == (rows, 1, 128, 157) and torch.isfinite(image).all()
    x = wav[:2].numpy().astype(np.float32) / np.float32(32768.0)
    want = fen.logmel_f64(x, 1024, 2048, sample_rate=32000)
    got_db = image[:2].cpu().numpy().astype(np.float64)  # mean 0, std 1: plain dB
    assert (np.abs(got_db - want) <= 1e-4 * np.maximum(np.abs(want), 1.0)).all()

"""Config merge rules, model construction by name, and the episode loaders (CPU)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT

FIX = os.path.join(GOLDEN, "config")


def test_includes_merge_and_overrides():
    from audio_fewshot_b200.config import Config
    cfg = Config(os.path.join(FIX, "proto_fixture.yaml"), {"test_episode": 4}).get_config_dict()
    assert cfg["backbone"]["name"] == "Conv64F"          # the file overrides the included resnet12 fragment
    assert cfg["classifier"] == {"name": "ProtoNet", "kwargs": None}
    assert (cfg["way_num"], cfg["shot_num"], cfg["query_num"]) == (5, 5, 3)   # file beats header
    assert (cfg["test_way"], cfg["test_shot"], cfg["test_query"]) == (5, 5, 3)  # "~" -> same as train
    assert cfg["test_episode"] == 4 and cfg["tb_scale"] == 10.0                 # variable_dict beats file
    assert "includes" not in cfg and 25000 <= cfg["port"] <= 55000


def test_build_model_by_name():
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.config import Config, build_model
    cfg = Config(os.path.join(FIX, "proto_fixture.yaml")).get_config_dict()
    m = build_model(cfg, "cpu")
    assert isinstance(m, arch.ProtoNet) and isinstance(m.emb_func, arch.Conv64F)
    assert (m.way_num, m.shot_num, m.query_num, m.num_channels, m.is_clap) == (5, 5, 3, 1, False)
    m_test = build_model(cfg, "cpu", mode="test")
    assert not hasattr(m_test, "num_channels")  # test.py:636-645 omits it


BASELINE_CONFIGS = [
    ("proto_5shot_iid.yaml", "ProtoNet", "Conv64F"), ("proto_1shot_ood.yaml", "ProtoNet", "Conv64F"),
    ("dn4.yaml", "DN4", "Conv64F"), ("deepbdc.yaml", "DeepBDC", "resnet12Bdc"), ("maml_5shot_iid.yaml", "MAML", "Conv64F"),
]


@pytest.mark.parametrize("name,cls,backbone", BASELINE_CONFIGS)
def test_baseline_config_fixtures_build(name, cls, backbone):
    """The classifier, backbone and episode shape of each BASELINE.json config (tests/golden/config/baseline/, restated
    from SURVEY.md 8a) merge with the header and build by name; the MAML inner lr written `1e-2` arrives as a float."""
    from audio_fewshot_b200.config import Config, build_model
    cfg = Config(os.path.join(FIX, "baseline", name)).get_config_dict()
    assert cfg["classifier"]["name"] == cls and cfg["backbone"]["name"] == backbone
    assert "includes" not in cfg and cfg["train_episode"] == 40  # from headers/model.yaml
    m = build_model(cfg, "cpu")
    assert type(m).__name__ == cls and type(m.emb_func).__name__ in (backbone, "ResNetBdc")
    assert (m.way_num, m.shot_num, m.query_num) == (cfg["way_num"], cfg["shot_num"], cfg["query_num"])
    if cls == "MAML":
        lr = cfg["classifier"]["kwargs"]["inner_param"]["lr"]
        assert isinstance(lr, float) and lr == 0.01 and m.feat_dim == 1600


@pytest.mark.parametrize("name,cls,backbone", BASELINE_CONFIGS)
def test_reference_baseline_configs_build(reference, name, cls, backbone):
    """The five BASELINE.json configs of the reference's own source tree parse and build (where it is installed)."""
    from audio_fewshot_b200.config import Config, _load_yaml, build_model
    from oracle.ref_import import REFERENCE_ROOT
    cfg = Config(os.path.join(REFERENCE_ROOT, "config", name)).get_config_dict()
    assert cfg["classifier"]["name"] == cls and cfg["backbone"]["name"] == backbone
    if cls == "MAML":
        cfg["classifier"]["kwargs"]["feat_dim"] = 1600  # the file's 4608 is stale (SURVEY.md 8a)
        lr = _load_yaml(os.path.join(REFERENCE_ROOT, "config", "classifiers", "MAML.yaml"))["classifier"]["kwargs"][
            "inner_param"]["lr"]
        assert isinstance(lr, float) and lr == 0.01
    m = build_model(cfg, "cpu")
    assert type(m).__name__ == cls and type(m.emb_func).__name__ in (backbone, "ResNet", "ResNetBdc")
    assert m.way_num == 5


def test_sampler_shards_by_global_index_and_loader_layout():
    from audio_fewshot_b200.data import EpisodeSampler, SyntheticSpectrogramEpisodes
    full = EpisodeSampler(12, 2, 0, 1, seed=3)
    parts = [EpisodeSampler(12, 2, r, 3, seed=3) for r in range(3)]
    assert sorted(sum([list(p) for p in parts], [])) == list(full) == list(range(6))
    assert len({len(p) for p in parts}) == 1  # every rank iterates the same number of batches (collectives per step)
    with pytest.raises(ValueError):
        EpisodeSampler(7, 2)
    with pytest.raises(ValueError):  # 6 batches over 4 ranks: the last step's collectives would deadlock
        EpisodeSampler(12, 2, 0, 4)
    one = SyntheticSpectrogramEpisodes(full, 5, 2, 3, max_windows=3)
    shard = SyntheticSpectrogramEpisodes(parts[1], 5, 2, 3, max_windows=3)
    batches = {b: one.batch(b) for b in full}
    for b in parts[1]:  # world-size invariance: same global batch -> same content
        for x, y in zip(batches[b], shard.batch(b)):
            assert (torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y)
    image, target, repeats, support_size = batches[0]
    assert support_size == 2 * 5 * 2 and repeats.numel() == 2 * 5 * 3
    assert image.shape == (support_size + int(repeats.sum()), 1, 128, 157) and target.shape[0] == image.shape[0]
    from audio_fewshot_b200.episode import EpisodeTable
    tab = EpisodeTable(2, 5, 2, 3, repeats.numpy(), "cpu")
    assert tab.N == image.shape[0]
    for g in range(10):  # rows of block g carry label g % 5
        assert (target[tab.cls_row_host[g]:tab.cls_row_host[g + 1]] == g % 5).all()


def test_spectrogram_folder_loader(tmp_path):
    from audio_fewshot_b200.data import get_dataloader, window_spectrogram
    rng = np.random.default_rng(0)
    names = ["dog", "cat", "owl", "bat", "fox", "cow"]
    for c in names:
        os.makedirs(tmp_path / "spec" / c)
        for i in range(4):
            T = int(rng.integers(100, 500))
            np.save(tmp_path / "spec" / c / ("%d.npy" % i), rng.standard_normal((128, T)).astype(np.float32) * 20 - 15)
    split = np.empty(3, dtype=object)
    split[0], split[1], split[2] = names, names[:5], names[1:]
    np.save(tmp_path / "splits.npy", split, allow_pickle=True)
    np.save(tmp_path / "ms.npy", np.asarray([-15.0, 20.0], dtype=np.float32).reshape(2, 1, 1))
    cfg = dict(way_num=5, shot_num=1, query_num=2, test_way=5, test_shot=1, test_query=2, train_episode=4,
               test_episode=2, episode_size=1, data_root=str(tmp_path / "spec"), class_per_split=str(tmp_path / "splits.npy"),
               mean_std_file=str(tmp_path / "ms.npy"), seed=1)
    (loader,) = get_dataloader(cfg, "test", None, False, "audio")
    assert len(loader) == 2
    loader.sampler.set_epoch(1)
    image, target, repeats, support_size = next(iter(loader))
    assert support_size == 5 and repeats.numel() == 10 and (repeats >= 1).all() and repeats.max() >= 2
    assert image.shape == (5 + int(repeats.sum()), 1, 128, 157)
    assert abs(float(image.mean())) < 0.5  # normalised with the (2,1,1) file
    w = window_spectrogram(np.arange(128 * 400, dtype=np.float32).reshape(128, 400))
    assert w.shape == (3, 128, 157) and w[2, 0, -1] == 399 and w[1, 0, 0] == 157
    assert window_spectrogram(np.ones((128, 50), np.float32)).shape == (1, 128, 157)


def test_synthetic_waveform_loader_matches_bench_recipe():
    from audio_fewshot_b200.data import get_dataloader
    cfg = dict(way_num=5, shot_num=1, query_num=2, test_way=5, test_shot=1, test_query=2, train_episode=2,
               test_episode=2, episode_size=2, synthetic_waveform=True, audio_samples=4000)
    (loader,) = get_dataloader(cfg, "train")
    wav, target, repeats, support_size = next(iter(loader))
    assert wav.shape == (2 * 5 * 3, 4000) and support_size == 10 and repeats.tolist() == [1] * 20
    spec = np.abs(np.fft.rfft(wav[3 * 2].numpy()))  # class 2 -> 600 Hz tone
    assert abs(np.argmax(spec[10:]) + 10 - 600 * 4000 / 16000) <= 1


def test_wav_folder_loader_serves_pcm16_windows(tmp_path):
    """`data_format: wav` -> int16 [rows, L] windows (first window for supports, all windows + repeats for queries)
    that LogMelFrontEnd consumes directly (afs_logmel_fwd_pcm16)."""
    import wave
    from audio_fewshot_b200.data import get_dataloader, read_wav_pcm16, window_waveform
    rng = np.random.default_rng(3)
    names = ["dog", "cat", "owl", "bat", "fox"]
    written = {}
    for c in names:
        os.makedirs(tmp_path / "wav" / c)
        for i in range(3):
            n = int(rng.integers(2000, 9000))
            pcm = rng.integers(-20000, 20000, size=n).astype("<i2")
            path = str(tmp_path / "wav" / c / ("%d.wav" % i))
            with wave.open(path, "wb") as w:
                w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000)
                w.writeframes(pcm.tobytes())
            written[path] = pcm
    p0 = sorted(written)[0]
    got, sr = read_wav_pcm16(p0)
    assert sr == 16000 and got.dtype == np.int16 and np.array_equal(got, written[p0])
    cfg = dict(way_num=5, shot_num=1, query_num=2, test_way=5, test_shot=1, test_query=2, train_episode=2,
               test_episode=2, episode_size=1, data_root=str(tmp_path / "wav"), data_format="wav", audio_samples=4000)
    (loader,) = get_dataloader(cfg, "test")
    wav, target, repeats, support_size = next(iter(loader))
    assert wav.dtype == torch.int16 and wav.shape == (5 + int(repeats.sum()), 4000)
    assert support_size == 5 and repeats.numel() == 10 and repeats.max() >= 2 and target.shape[0] == wav.shape[0]
    w = window_waveform(np.arange(9000, dtype=np.int16), 4000)
    assert w.shape == (3, 4000) and w[2, -1] == 8999 and w[1, 0] == 4000
    assert window_waveform(np.ones(100, np.int16), 4000).shape == (1, 4000)
    with wave.open(str(tmp_path / "bad.wav"), "wb") as w8:
        w8.setnchannels(1); w8.setsampwidth(1); w8.setframerate(16000); w8.writeframes(b"\x00" * 10)
    with pytest.raises(ValueError):
        read_wav_pcm16(str(tmp_path / "bad.wav"))


def test_yaml_scientific_notation_floats(tmp_path):
    """PyYAML's YAML-1.1 resolver reads `1e-2` as a string; the reference writes learning rates that way
    (config/classifiers/MAML.yaml inner_param.lr).  The loader must hand floats to the optimisers."""
    from audio_fewshot_b200 import config
    f = tmp_path / "c.yaml"
    f.write_text("lr: 1e-2\nwd: 5.0e-4\nn: 12\nname: 1e\nquoted: '1e-2'\n")
    d = config._load_yaml(str(f))
    assert d == {"lr": 0.01, "wd": 5.0e-4, "n": 12, "name": "1e", "quoted": "1e-2"}

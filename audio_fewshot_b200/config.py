"""YAML experiment configs of the reference, and building the hot-path model from one.

The reference's loader (`libfewshot_core.config.Config`) is NOT in the snapshot (its own .gitignore
drops every `config/` package, SURVEY.md F1), so the merge rules are restated from what the YAML
files and the call sites need (run_trainer.py:43-50, run_test.py:148-159, config/headers/README):

  * a config file may list `includes:` -- header fragments resolved against the config ROOT
    (`./config/` in the reference: config/headers/README:3), merged in list order, later wins;
  * keys of the file itself override anything included (config/proto_5shot_iid.yaml selects
    `backbones/resnet12.yaml` through an include and then overrides `backbone:` inline);
  * YAML duplicate keys resolve last-wins (PyYAML) -- the same file has two `includes:` keys;
  * a `variable_dict` (run_test.py VAR_DICT) overrides the file;
  * `test_way / test_shot / test_query: ~` mean "same as train" (config/headers/model.yaml:13);
  * derived: `tb_scale = train_episode / test_episode`, `resume`, `resume_path`.

`build_model` restates Trainer._init_model / Test._init_model (trainer.py:426-454, test.py:625-646):
classes are looked up BY NAME in one namespace -- here `audio_fewshot_b200.model`.
"""
import os
import random
import re

import yaml

DEFAULTS = {  # keys the callers read unconditionally; the reference takes them from its default.yaml
    "augment_times": 1, "augment_times_query": 1, "is_clap": False, "modality": "audio", "n_gpu": 1,
    "device_ids": 0, "episode_size": 1, "seed": 0, "deterministic": True, "port": None,
    "test_way": None, "test_shot": None, "test_query": None, "pretrain_path": None, "resume": False,
    "train_episode": 100, "test_episode": 100, "ood": False,
}


class _Loader(yaml.SafeLoader):
    """SafeLoader whose float resolver also accepts `1e-2` (PyYAML's YAML-1.1 rule demands a dot, so the reference's
    `inner_param.lr: 1e-2` in config/classifiers/MAML.yaml would load as a string).  Same regular expression as
    upstream LibFewShot's config loader."""


_Loader.add_implicit_resolver(
    "tag:yaml.org,2002:float",
    re.compile(r"""^(?:
     [-+]?(?:[0-9][0-9_]*)\.[0-9_]*(?:[eE][-+]?[0-9]+)?
    |[-+]?(?:[0-9][0-9_]*)(?:[eE][-+]?[0-9]+)
    |\.[0-9_]+(?:[eE][-+][0-9]+)?
    |[-+]?[0-9][0-9_]*(?::[0-5]?[0-9])+\.[0-9_]*
    |[-+]?\.(?:inf|Inf|INF)
    |\.(?:nan|NaN|NAN))$""", re.X),
    list("-+0123456789."),
)


def _load_yaml(path):
    with open(path, "r", encoding="utf-8") as fin:
        return yaml.load(fin.read(), Loader=_Loader) or {}


def find_config_root(config_file):
    """The directory `includes:` are relative to: the nearest ancestor named `config` of the file,
    else ./config (the reference's hard-coded choice), else the file's own directory."""
    d = os.path.dirname(os.path.abspath(config_file))
    probe = d
    while True:
        if os.path.basename(probe) == "config":
            return probe
        parent = os.path.dirname(probe)
        if parent == probe:
            break
        probe = parent
    return "./config" if os.path.isdir("./config") else d


class Config:
    def __init__(self, config_file=None, variable_dict=None, is_resume=False, config_root=None):
        self.is_resume = is_resume
        self.config_file = config_file
        self.config_root = config_root or (find_config_root(config_file) if config_file else "./config")
        self.file_dict = self._load_config_files(config_file)
        self.variable_dict = dict(variable_dict or {})
        self.config_dict = self._merge()

    def _load_config_files(self, config_file):
        merged = {}
        if config_file is None:
            return merged
        own = _load_yaml(config_file)
        for include in own.get("includes") or []:
            merged.update(_load_yaml(os.path.join(self.config_root, include)))
        merged.pop("includes", None)
        own = dict(own)
        own.pop("includes", None)
        merged.update(own)
        return merged

    def _merge(self):
        cfg = dict(DEFAULTS)
        cfg.update(self.file_dict)
        cfg.update(self.variable_dict)
        for test_key, train_key in (("test_way", "way_num"), ("test_shot", "shot_num"), ("test_query", "query_num")):
            if cfg.get(test_key) is None and train_key in cfg:
                cfg[test_key] = cfg[train_key]
        if cfg.get("port") is None:
            cfg["port"] = random.randint(25000, 55000)
        cfg["resume"] = self.is_resume
        if self.is_resume and self.config_file:
            cfg["resume_path"] = os.path.dirname(os.path.abspath(self.config_file))
        if cfg.get("test_episode"):
            cfg["tb_scale"] = float(cfg["train_episode"]) / cfg["test_episode"]
        return cfg

    def get_config_dict(self):
        return self.config_dict


def build_model(config, device, arch=None, mode="train"):
    """Backbone + classifier from a config dict.  mode="train" passes the Trainer's kwargs
    (trainer.py:442-453: num_channels, is_clap included), mode="test" the evaluator's (test.py:636-645)."""
    if arch is None:
        from . import model as arch
    if config.get("is_clap"):
        raise NotImplementedError("the CLAP backbone is outside the hot path (SURVEY.md 2)")
    emb_func = arch.get_instance(arch, "backbone", config)
    kwargs = {
        "way_num": config["way_num"],
        "shot_num": config["shot_num"] * config["augment_times"],
        "query_num": config["query_num"],
        "test_way": config["test_way"],
        "test_shot": config["test_shot"] * config["augment_times"],
        "test_query": config["test_query"],
        "emb_func": emb_func,
        "device": device,
    }
    if mode == "train":
        bk = config["backbone"].get("kwargs") or {}
        kwargs["num_channels"] = bk.get("num_channels", 3)
        kwargs["is_clap"] = config.get("is_clap", False)
    model = arch.get_instance(arch, "classifier", config, **kwargs)
    if config.get("pretrain_path"):
        import torch
        state = torch.load(config["pretrain_path"], map_location="cpu")
        model.emb_func.load_state_dict(state, strict=False)
    return model.to(device)


def frontend_from_config(config, device, **overrides):
    """LogMelFrontEnd normalised with the config's `mean_std_file` (Auxiliary/*_Mean_Std.npy), at the config's
    `sample_rate`, `n_fft` and `hop_length` (defaults 16000 / 1024 / 512; e.g. 32000 / 2048 / 1024 or
    8000 / 512 / 256 give the same 157 frames for 5 s clips at their own rate)."""
    from .frontend import LogMelFrontEnd
    kw = dict(sample_rate=int(config.get("sample_rate", 16000)), n_fft=int(config.get("n_fft", 1024)),
              hop_length=int(config.get("hop_length", 512)), n_mels=128)
    kw.update(overrides)
    path = config.get("mean_std_file")
    if path and os.path.exists(path):
        kw["mean_std_file"] = path
    return LogMelFrontEnd(**kw).to(device)

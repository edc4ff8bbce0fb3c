"""CPU tests of the host side: episode tables, config-free model plumbing, sharding."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import cases, heads


@pytest.mark.parametrize("name", sorted(cases.SPLIT_CASES))
def test_episode_table_equals_reference_split(golden, name):
    from audio_fewshot_b200.episode import EpisodeTable
    c = cases.SPLIT_CASES[name]
    g = golden("episode_vote.npz")
    rep = cases.split_repeats(c)
    tab = EpisodeTable(c["E"], c["W"], c["S"], c["Q"], rep, "cpu")
    S = c["S"]
    cls_row = tab.cls_row.numpy()
    sup = np.concatenate([np.arange(cls_row[k], cls_row[k] + S) for k in range(c["E"] * c["W"])])
    qry = np.concatenate([np.arange(cls_row[k] + S, cls_row[k + 1]) for k in range(c["E"] * c["W"])])
    assert np.array_equal(sup, g[name + "/support_rows"].reshape(-1))
    assert np.array_equal(qry, g[name + "/query_rows"])
    assert np.array_equal(tab.q_target.numpy(), g[name + "/query_target"].reshape(-1))
    assert tab.NQ == int(rep.sum()) and tab.N == len(sup) + len(qry)
    assert np.array_equal(np.diff(tab.q_start.numpy()), rep)
    assert np.array_equal(cls_row, heads.cls_row_table(rep, c["E"], c["W"], S))


def test_table_cache_and_errors():
    from audio_fewshot_b200.episode import EpisodeTableCache, EpisodeTable
    cache = EpisodeTableCache(max_entries=2)
    a = cache.get(2, 5, 5, 15, None, "cpu")
    assert cache.get(2, 5, 5, 15, torch.ones(150, dtype=torch.long), "cpu") is not a  # keyed separately
    assert cache.get(2, 5, 5, 15, None, "cpu") is a
    assert a.N == 200 and a.NQ == 150
    with pytest.raises(ValueError):
        EpisodeTable(2, 5, 5, 15, np.ones(10), "cpu")


def test_model_contract_on_cpu():
    """Constructor kwargs, reverse_setting_info, model_type, forward dispatch (no kernels launched)."""
    from audio_fewshot_b200 import model as arch
    cfg = {"backbone": {"name": "Conv64F", "kwargs": {"is_flatten": True, "num_channels": 1}},
           "classifier": {"name": "ProtoNet", "kwargs": None}}
    emb = arch.get_instance(arch, "backbone", cfg)
    m = arch.get_instance(arch, "classifier", cfg, way_num=5, shot_num=5, query_num=15, test_way=5, test_shot=1,
                          test_query=10, emb_func=emb, device="cpu", num_channels=1, is_clap=False)
    assert m.model_type == arch.ModelType.METRIC
    assert any(k.startswith("emb_func.layer1.0.weight") for k in m.state_dict())
    m.reverse_setting_info()
    assert (m.way_num, m.shot_num, m.query_num, m.test_shot) == (5, 1, 10, 5)
    assert m.get_uncertainty_threshold() is None
    assert m.eval() is m
    from audio_fewshot_b200._lib import AfsError
    with pytest.raises(AfsError):  # CPU tensors never silently fall back
        m([torch.zeros(55, 1, 128, 157), torch.zeros(55), torch.ones(50, dtype=torch.long), 5])


def test_finetuning_model_contract():
    """FinetuningModel (finetuning_model.py:10-31): model_type, the three abstract methods, sub_optimizer from a
    {"name", "kwargs"} block."""
    from audio_fewshot_b200 import model as arch

    class Probe(arch.FinetuningModel):
        def __init__(self, **kw):
            super().__init__(**kw)
            self.classifier = torch.nn.Linear(4, 2)

        def set_forward(self, batch):
            return "eval"

        def set_forward_loss(self, batch):
            return "train"

    m = Probe(way_num=5, shot_num=1, query_num=15, test_way=5, test_shot=1, test_query=15, device="cpu")
    assert m.model_type == arch.ModelType.FINETUNING and m.way_num == 5 and m.init_type == "normal"
    assert m.train()([0]) == "train" and m.eval()([0]) == "eval"
    with pytest.raises(NotImplementedError):
        m.set_forward_adaptation()
    opt = m.sub_optimizer(m.classifier, {"name": "SGD", "kwargs": {"lr": 0.01, "momentum": 0.9}})
    assert isinstance(opt, torch.optim.SGD) and opt.param_groups[0]["momentum"] == 0.9
    assert isinstance(m.sub_optimizer(m.classifier, {"name": "Adam", "kwargs": None}), torch.optim.Adam)


def test_finetuning_model_has_the_live_reference_public_names(reference):
    import importlib

    from audio_fewshot_b200 import model as arch
    ref_cls = importlib.import_module("libfewshot_core.model.finetuning.finetuning_model").FinetuningModel
    want = {n for n in vars(ref_cls) if not n.startswith("_")}
    assert want <= {n for n in dir(arch.FinetuningModel)}, want


def test_sharding_is_a_partition():
    from audio_fewshot_b200.dist import shard_episodes
    for n, ws in [(10, 1), (10, 4), (1250, 8), (3, 8)]:
        parts = [shard_episodes(n, r, ws) for r in range(ws)]
        assert sorted(sum(parts, [])) == list(range(n))


def test_ci_matches_reference_golden(golden):
    from audio_fewshot_b200.dist import mean_confidence_interval
    m, h = mean_confidence_interval(list(cases.CI_DATA))
    np.testing.assert_allclose([m, h], golden("episode_vote.npz")["ci/mean_h"], rtol=1e-12)


WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from audio_fewshot_b200.dist import shard_episodes, gather_episode_accuracies, mean_confidence_interval
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["PORT"], rank=int(os.environ["RANK"]),
                        world_size=int(os.environ["WORLD_SIZE"]))
rank, ws = dist.get_rank(), dist.get_world_size()
n = 11
mine = shard_episodes(n, rank, ws)
local = torch.tensor([50.0 + g for g in mine])          # accuracy is a function of the GLOBAL index
full = gather_episode_accuracies(local, n)
assert full.tolist() == [50.0 + g for g in range(n)], full
m, h = mean_confidence_interval(full.tolist())
from audio_fewshot_b200.model.proto_net import accuracy_percent
out = torch.eye(4)[torch.tensor([0, 1, 2, 3])]
acc = accuracy_percent(out, torch.tensor([0, 1, 2, 0]) if rank == 0 else torch.tensor([0, 1, 2, 3]))
assert abs(acc - 100.0 * 7 / 8) < 1e-4, acc             # summed over both ranks (utils.py:116-118)
if rank == 0:
    print("OK %%.6f %%.6f" %% (m, h))
dist.barrier(); dist.destroy_process_group()
""" % ROOT


def test_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=120) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    m, h = [float(v) for v in outs[0][0].split()[1:3]]
    assert m == pytest.approx(55.0) and h > 0


def test_tta_helpers_match_reference_golden(golden):
    """tta.map_q_to_s_runs / augment_images_with_mask against outputs of the reference's own functions
    (libfewshot_core/test.py:33-152; tests/golden/tta.npz from `python -m oracle.make_golden --tta`): same rows, same
    order, same number and order of augmentation calls."""
    from audio_fewshot_b200 import tta
    g = golden("tta.npz")
    n_cases = len({k.split("/")[0] for k in g.files})
    assert n_cases == 6
    for i in range(n_cases):
        s, r, q, img = g["%d/s" % i], g["%d/r" % i], g["%d/q" % i], g["%d/img" % i]
        assert np.array_equal(tta.map_q_to_s_runs(s, r, q), g["%d/mapped" % i])
        calls = [0]

        def fn(x):
            calls[0] += 1
            return x * 2 + calls[0]

        got = tta.augment_images_with_mask(torch.from_numpy(img), torch.from_numpy(r), s, q, fn, 3)
        assert np.array_equal(got.numpy(), g["%d/aug" % i])
        rep = tta.updated_repeats(torch.from_numpy(r), q, 3)
        assert int(rep.sum()) + int((~s).sum()) == got.shape[0]  # repeats describe exactly the rows that exist
    with pytest.raises(ValueError):
        tta.map_q_to_s_runs([True, True], [1], [True])


def test_tta_helpers_match_live_reference(reference):
    import libfewshot_core.test as rt
    from audio_fewshot_b200 import tta
    from oracle.make_golden import tta_cases
    for s, r, q, img in tta_cases():
        assert np.array_equal(tta.map_q_to_s_runs(s, r, q), rt.map_q_to_s_runs(s, r, q))
        a = rt.augment_images_with_mask(torch.from_numpy(img), torch.from_numpy(r), s, q, lambda x: x + 1, 2)
        b = tta.augment_images_with_mask(torch.from_numpy(img), torch.from_numpy(r), s, q, lambda x: x + 1, 2)
        assert torch.equal(a, b)


def test_bench_reference_arm_line_and_no_cuda_refusal(tmp_path):
    """`bench.py --impl reference` (the oracle port timed on the host cores) prints ONE JSON line with the contract's
    keys and dumps its last step's outputs; the B200 arm refuses to run without a CUDA device instead of falling back."""
    import json
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--episodes-per-step", "2", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "episodes/sec" and d["higher_is_better"] is True
    assert d["metric"].startswith("episodes/sec (5w5s15q") and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["config"]["episodes_per_step_per_gpu"] == 2  # the CPU arm runs the B200 arm's step, not one episode
    logits, acc = np.load(tmp_path / "dump" / "logits.npy"), np.load(tmp_path / "dump" / "accuracy_pct.npy")
    assert logits.dtype == acc.dtype == np.float32 and logits.shape == (2 * 5 * 15, 5) and acc.shape == ()
    assert np.isfinite(logits).all() and 0.0 <= acc <= 100.0
    # under torchrun only rank 0 runs the reference arm; the other ranks exit 0 without work or output
    other = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                            "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300,
                           env=dict(env, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2"))
    assert other.returncode == 0 and not [l for l in other.stdout.splitlines() if l.startswith("{")]
    ours = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, timeout=300)
    assert ours.returncode != 0 and "no CPU fallback" in (ours.stderr + ours.stdout)
    assert not [l for l in ours.stdout.splitlines() if l.startswith("{")]


def test_committed_bench_line_has_the_contract_keys():
    """profiles/r01_bench_n*.json are bench.py's JSON lines as measured on B200: every key of the bench contract is
    there, the numbers are mutually consistent, and the roofline entry is the algorithmic bytes over the measured time."""
    import glob
    import json
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r01_bench_n[1248].json")))
    assert paths
    for path in paths:
        d = json.loads(open(path).read())
        n = d["n_gpus"]
        assert d["metric"].startswith("episodes/sec (5w5s15q") and d["unit"] == "episodes/sec"
        assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
        assert d["data"] == "synthetic" and d["dtype"] == "f32" and d["warmup"] >= 3 and d["steps"] >= 1
        cfg = d["config"]
        assert "workload" in cfg and "model" not in cfg and "l2_policy" in cfg
        per_step = cfg["episodes_per_step_per_gpu"] * n
        assert abs(d["value"] - per_step / d["ms_per_step"] * 1e3) <= 1e-6 * d["value"]
        e2e = d["e2e"]
        assert e2e["unit"] == d["unit"] and 0 < e2e["value"] < d["value"]
        # host fp32 waveforms of one step, and its logits + accuracy back
        assert e2e["h2d_bytes_per_step"] == cfg["clips_per_step_per_gpu"] * cfg["clip_samples"] * 4
        assert e2e["d2h_bytes_per_step"] == cfg["episodes_per_step_per_gpu"] * cfg["way"] * cfg["query"] * cfg["way"] * 4 + 4
        assert d["gpu_launches"] > 0
        r = d["roofline"]
        assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert r["bytes_per_launch"] == cfg["clips_per_step_per_gpu"] * 400384  # SURVEY 8(d): 4 L + 4 n_mels T per clip
        assert abs(r["achieved"] - r["bytes_per_launch"] / r["ms_per_launch"] / 1e6) <= 1e-6 * r["achieved"]
        assert r["traffic"] is None or 0.5 * r["bytes_per_launch"] < r["traffic"] < 1.5 * r["bytes_per_launch"]
        c = d["clocks"]
        assert c["sm_mhz"] > 0.9 * c["sm_max_mhz"] and not set(c["reasons"]) & {
            "hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if n == 1:
            b = d["cpu_baseline"]
            assert b["kind"] == "port" and b["cores"] >= 1 and b["unit"] == d["unit"] and 0 < b["value"] < e2e["value"]

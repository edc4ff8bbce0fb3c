#!/usr/bin/env python
"""Headline benchmark: episodes/sec, 5-way 5-shot 15-query, waveform -> logits.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode eval|train|eval10k]
                    [--dump-outputs DIR]

Workload (BASELINE.json `metric`; SURVEY.md 8d, config C1 = config/proto_5shot_iid.yaml): ProtoNet on
Conv64F, 5w5s15q = 100 clips per episode, each clip 5 s @ 16 kHz (L = 80 000) -> log-mel [1,128,157]
(n_fft 1024, hop 512, 128 slaney mels, KOS_0.5_alpha mean/std).  One "step" = one pass of the hot path
over `--episodes-per-step` episodes per rank:
    fused log-mel kernel -> Conv64F (tcgen05 block-1 and block-2/3 kernels, cuDNN block 4) -> prototype head
    kernel -> vote/accuracy kernel.
Episodes are independent, so ranks never exchange data inside an evaluation step ("weak" scaling: per-GPU
work is fixed).  Synthetic seeded waveforms, weights derived from parameter names
(audio_fewshot_b200.synthetic).

Keys of the JSON line (default mode `eval`):
`value`    device-resident inputs (two rotating batches, each larger than L2).
`e2e`      the public call EpisodePipeline.stream(pinned host batches): every step's H2D of the waveforms and
           D2H of the logits + accuracy inside the timed region (3 rotating device buffers, copies overlap
           compute).  `h2d_probe_gbs` is a plain pinned cudaMemcpyAsync of the same buffers run by all ranks at
           once in this run; `host_roofline_frac` = the bytes/s the e2e leg moved over that probe.
`e2e_pcm16` the same call with the host waveforms as 16-bit PCM (extra key; `e2e` is the fp32-host figure).
`roofline` the fused log-mel kernel (the north-star kernel BASELINE's metric names): algorithmic bytes
           4*L + 4*128*T per clip over its CUDA-event duration inside the timed region, against
           MEASURED_PEAKS.json; `traffic` and the issue/FMA co-limits are stamped from the committed ncu capture.
`roofline_all` every kernel that takes >= 10 % of the step (torch-profiler device times of three extra steps):
           HBM kernels against the copy peak, tcgen05 TF32 kernels against a TF32 matmul peak measured in this run.
`gpu_eager_baseline` the reference's op sequence in plain PyTorch on the same GPU (torch.stft log-mel, the
           nn.Module graph, broadcast ProtoLayer arithmetic): SURVEY 8d's "real bar".
`bf16_backbone` the same step with Conv64F.precision = "bf16" (stem writes bf16, blocks 2-3 as bf16 tcgen05 MMAs):
           the reduced-precision path the north star asks to be stated separately, with its argmax-flip count and
           logit deviation against this run's TF32 logits.  Never folded into `value`.
`s1`       the same pipeline on BASELINE configs[0]'s clips (1 s @ 16 kHz, hop 102 -> the same [1,128,157]).
`cpu_baseline` / `--impl reference`: the oracle port of the reference path (torch.stft front-end spec ->
           reference Conv64F arithmetic -> ProtoLayer -> majority vote) on the box's host cores, at the same
           episodes per step.

Collective-bearing modes (their own JSON line, same contract keys):
  --mode train    C1 episodic training step from waveforms: log-mel -> set_forward_loss -> backward -> ONE flat
                  NCCL gradient all-reduce (dist.all_reduce_gradients; reference trainer.py:504-509) -> Adam; the
                  reference's 1-float accuracy all-reduce per step stays (utils.py:116-118).
  --mode eval10k  BASELINE configs[1]: ProtoNet/ResNet-12 5w1s15q, 10 000 episodes sharded over the ranks, ONE
                  all_gather of the per-episode accuracies + the 95 % CI at the end (test.py:210) inside the timing.

`--steps` is the number of timed steps of eval, train and --impl reference.  eval10k times the whole job instead,
--episodes / (episodes per step * ranks) steps, and refuses --steps.

`--dump-outputs DIR` writes what the timed path returned, on rank 0, as DIR/<name>.npy (float32, float64 where the
path computes in float64): for the last timed step, eval and --impl reference `logits` and `accuracy_pct`, train
`logits`, `loss` and `accuracy_pct`; for the whole eval10k job, `episode_accuracy_pct` (every episode, in global
order) and `accuracy_mean_ci95`.  Inputs and weights are seeded, so the same arguments give the same inputs on every
run and two builds can be compared output for output.  With equal --steps and episodes per step, the eval and
--impl reference dumps come from the same waveforms, unless --ref-seconds made the reference arm run fewer episodes
per step (its JSON note then says "bounded below").
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, S, Q = 5, 5, 15
L, HOP, N_MELS, SR = 80000, 512, 128, 16000
T_FRAMES = 1 + L // HOP
CLIPS_PER_EPISODE = W * (S + Q)
LOGMEL_BYTES_PER_CLIP = 4 * L + 4 * N_MELS * T_FRAMES  # 400 384 (SURVEY.md 8d)
L_S1, HOP_S1 = 16000, 102                               # BASELINE configs[0]: 1 s clips -> the same 157 frames
LOGMEL_BYTES_PER_CLIP_S1 = 4 * L_S1 + 4 * N_MELS * (1 + L_S1 // HOP_S1)
MEAN_STD_FILE = os.path.join(ROOT, "tests", "golden", "KOS_0.5_alpha_Mean_Std.npy")
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent
METRIC = "episodes/sec (5w5s15q, waveform->logits)"
WORKLOAD = "ProtoNet Conv64F 5w5s15q, 100 clips/episode, 5 s @ 16 kHz -> log-mel [1,128,157] (C1, shape S5)"
CONV1_FLOP_PER_CLIP = 2 * 9 * 64 * 128 * 157                 # block 1: 3x3, 1 -> 64 channels, useful flops
CONV1_BYTES_PER_CLIP = 4 * 128 * 157 + 4 * 64 * 42 * 52          # block 1: image read + pooled NHWC output written
CONV3_FLOP_PER_CLIP = 2 * 9 * 64 * 64 * (42 * 52 + 14 * 17)  # blocks 2 + 3: 3x3, 64 -> 64 channels


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 100; not in eval10k)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="eval", choices=["eval", "train", "eval10k"])
    ap.add_argument("--episodes-per-step", type=int, default=None,
                    help="episodes per rank per step (default: 32 for eval, 2 for train, 4 for eval10k)")
    ap.add_argument("--episodes", type=int, default=10000, help="eval10k: total episodes of the job")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bf16-backbone", action="store_true",
                    help="mode eval10k only: run the trunk on the separately stated bf16 path (emb_func.precision = "
                         "'bf16'); the line says so in dtype and config")
    ap.add_argument("--no-extras", action="store_true", help="skip roofline_all / gpu_eager_baseline / s1 / pcm16 legs")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="bound of the cpu_baseline sample")
    ap.add_argument("--ref-seconds", type=float, default=240.0,
                    help="--impl reference: bound of the whole run (the driver's --steps 20 --warmup 5 at the B200 arm's "
                         "32 episodes per step needs about 150 s on the box's 16 host threads)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.mode == "eval10k" and args.impl == "b200":
        if args.steps is not None:
            ap.error("--mode eval10k runs --episodes / (episodes per step * ranks) steps; set --episodes, not --steps")
    elif args.steps is None:
        args.steps = 100
    elif args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(directory, arrays):
    """Write {name: tensor or array} as directory/<name>.npy, float64 kept, every other dtype as float32."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a.detach().cpu() if hasattr(a, "detach") else a)
        np.save(os.path.join(directory, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def mean_std():
    m, s = np.load(MEAN_STD_FILE).flatten().tolist()
    return float(m), float(s)


def make_weights():
    """Conv64F with deterministic name-derived weights; returns the product module (CPU)."""
    import torch

    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200.synthetic import name_seeded_weights_

    torch.manual_seed(0)
    emb = arch.Conv64F(is_flatten=True, num_channels=1)
    name_seeded_weights_(emb)
    return emb


def base_config(E, n_clips, world):
    """The workload description both arms print (the driver compares the two arms' `config`)."""
    return {"workload": WORKLOAD, "episodes_per_step_per_gpu": E, "clips_per_step_per_gpu": n_clips,
            "way": W, "shot": S, "query": Q, "clip_samples": L, "n_fft": 1024, "hop": HOP, "n_mels": N_MELS}


def bind_to_gpu_cpus(local_rank):
    """Pin this process (and therefore its pinned-memory allocations, first touched from here) to the CPUs NVML
    reports as local to the GPU -- the per-rank affinity `nvidia-smi topo -m` shows.  Returns the CPU list or None."""
    try:
        import pynvml
        import torch

        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
        allowed = os.sched_getaffinity(0)
        cpus = sorted(c for c in (64 * i + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1)
                      if c in allowed)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


# ----------------------------------------------------------------------------------- CPU oracle arm
class CpuReferencePath:
    """The reference's op sequence on host cores (oracle port; /root/reference cannot travel to the box)."""

    def __init__(self):
        import torch

        from oracle import frontend as ofe

        self.torch = torch
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.sd = {k: v.clone() for k, v in make_weights().state_dict().items()}
        self.mean, self.std = mean_std()
        self.fb = ofe.mel_filterbank(513, 0.0, SR / 2.0, N_MELS, SR)
        self.win = ofe.hann_periodic()

    def episodes(self, wav, n_episodes):
        from oracle import backbones as obb
        from oracle import frontend as ofe
        from oracle import heads

        torch = self.torch
        with torch.no_grad():
            image = ofe.logmel_torch(wav, hop=HOP, n_mels=N_MELS, sample_rate=SR, mean=self.mean, std=self.std,
                                     fb=self.fb, window=self.win)
            feat = obb.conv64f_forward(self.sd, image)
            repeats = torch.ones(n_episodes * W * Q, dtype=torch.long)
            out, acc, _ = heads.proto_forward(feat, W, S, Q, repeats, n_episodes * W * S)
        return out, acc


def cpu_sample(seconds, E):
    """Time the oracle path on batches of up to E episodes until `seconds` of CPU work are done."""
    from audio_fewshot_b200.synthetic import synthetic_clip_batch

    path = CpuReferencePath()
    e_cpu = min(E, 8)
    wav = synthetic_clip_batch(1234, 0, e_cpu, W, S, Q, L)
    path.episodes(wav[:CLIPS_PER_EPISODE], 1)  # warm-up (thread pools, FFT plans)
    n, t0 = 0, time.perf_counter()
    while n < 3 * e_cpu and (n < e_cpu or time.perf_counter() - t0 < seconds):
        path.episodes(wav, e_cpu)
        n += e_cpu
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "episodes/sec", "cores": path.cores, "kind": "port",
            "sample": "%d episodes of the same workload in batches of %d, %.1f s on %d host threads "
                      "(oracle: torch.stft log-mel -> Conv64F -> ProtoLayer -> vote)" % (n, e_cpu, dt, path.cores)}


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path, rank 0 only, every step a bounded sample
    of the B200 arm's step (the same episodes per step when the time bound allows it, never fewer than 8)."""
    if rank != 0:
        return
    from audio_fewshot_b200.synthetic import synthetic_clip_batch

    path = CpuReferencePath()
    E = args.episodes_per_step or 32
    probe = synthetic_clip_batch(1234, 0, 2, W, S, Q, L)
    path.episodes(probe, 2)
    t0 = time.perf_counter()
    path.episodes(probe, 2)
    per_episode = (time.perf_counter() - t0) / 2
    fit = int(args.ref_seconds / max(per_episode * (args.steps + args.warmup), 1e-9))
    e_ref = max(min(E, fit), min(E, 8))
    wav = [synthetic_clip_batch(1234, i * e_ref, e_ref, W, S, Q, L) for i in range(2)]
    for i in range(args.warmup):
        path.episodes(wav[i % 2], e_ref)
    t0 = time.perf_counter()
    for i in range(args.steps):
        output, acc = path.episodes(wav[i % 2], e_ref)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": output, "accuracy_pct": acc})
    value = args.steps * e_ref / dt
    cfg = base_config(e_ref, e_ref * CLIPS_PER_EPISODE, 1)
    cfg["note"] = ("CPU oracle port of the reference path; runs on rank 0's host cores only, whatever --gpus says; "
                   "episodes per step %s the B200 arm's %d" % ("equal" if e_ref == E else "bounded below", E))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "episodes/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": "episodes/sec", "cores": path.cores, "kind": "port",
                         "sample": "%d steps x %d episodes on %d host threads" % (args.steps, e_ref, path.cores)},
        "e2e": {"value": value, "unit": "episodes/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="afs_clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for row in open(self.path):
                f = [c.strip() for c in row.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0]))
                    smax.append(float(f[1]))
                except ValueError:
                    continue
                for name, flag in zip(names, f[3:7]):
                    if flag.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# ----------------------------------------------------------------------------------- shared helpers of the B200 arm
class Ranks:
    def __init__(self, rank, world, dev):
        self.rank, self.world, self.dev = rank, world, dev

    def barrier(self):
        import torch
        import torch.distributed as dist

        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, value):
        import torch
        import torch.distributed as dist

        if self.world == 1:
            return value
        t = torch.tensor([value], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())


def timed(ranks, fn, steps):
    """barrier + synchronize, `steps` calls of fn(i) bracketed by CUDA events, barrier + synchronize; max over ranks."""
    import torch

    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ranks.barrier()
    t0.record()
    last = None
    for i in range(steps):
        last = fn(i)
    t1.record()
    ranks.barrier()
    return ranks.max(t0.elapsed_time(t1)), last


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def measure_tf32_peak(dev):
    """Dense TF32 matmul throughput of this GPU, measured here (MEASURED_PEAKS.json carries bf16 only)."""
    import torch

    n = 8192
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        torch.matmul(a, b)
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def kernel_shares(step, n=3):
    """Device time per kernel name over n extra steps (torch profiler / CUPTI); None when the profiler is unavailable."""
    import torch

    try:
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(n):
                step(i)
            torch.cuda.synchronize()
        rows = {}
        for ev in prof.key_averages():
            us = getattr(ev, "device_time_total", None)
            if us is None:
                us = getattr(ev, "cuda_time_total", 0.0)
            if us and us > 0:
                rows[ev.key] = rows.get(ev.key, 0.0) + float(us) / n
        return rows
    except Exception as exc:  # the number is an extra; never fail the bench for it
        sys.stderr.write("bench.py: kernel shares unavailable (%s)\n" % exc)
        return None


def roofline_all(rows, n_clips, hbm_peak, tf32_peak):
    total = sum(rows.values())
    out = []
    for name, us in sorted(rows.items(), key=lambda kv: -kv[1]):
        share = us / total
        if share < 0.10:
            continue
        entry = {"kernel": name[:120], "us_per_step": us, "share_of_kernel_time": share}
        if "logmel" in name:
            ach = LOGMEL_BYTES_PER_CLIP * n_clips / (us * 1e-6) / 1e9
            entry.update(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak)
        elif "conv1_tc" in name or "conv3x3_c64_tc" in name:
            flop = (CONV1_FLOP_PER_CLIP if "conv1_tc" in name else CONV3_FLOP_PER_CLIP) * n_clips
            ach = flop / (us * 1e-6) / 1e12
            entry.update(bound="tensor", achieved=ach, peak=tf32_peak, unit="TFLOP/s", frac=ach / tf32_peak,
                         note="useful TF32 flops (zero padding of K and junk GEMM rows not counted) over a TF32 "
                              "torch.matmul 8192^3 measured in this run")
            if "conv1_tc" in name:  # K = 9 taps: the stem's floor is its NHWC output, not the tensor pipe
                hb = CONV1_BYTES_PER_CLIP * n_clips / (us * 1e-6) / 1e9
                entry.update(hbm_achieved=hb, hbm_frac=hb / hbm_peak,
                             hbm_note="4*128*157 B read + 4*64*42*52 B written per clip over the copy peak")
        out.append(entry)
    return out


class TorchEagerPath:
    """The reference's op sequence in plain PyTorch on the GPU: torch.stft log-mel (the front-end a user of the
    reference would write), the nn.Module graph of Conv64F, ProtoLayer's broadcast arithmetic
    (libfewshot_core/model/metric/proto_net.py:49-57), argmax accuracy.  Used for `gpu_eager_baseline` only."""

    def __init__(self, emb, fb, window, mean, std, dev):
        import torch

        self.emb = emb
        self.fb = torch.as_tensor(fb, device=dev)
        self.win = torch.as_tensor(window, device=dev)
        self.mean, self.std = mean, std
        self.target = torch.arange(W, device=dev).repeat_interleave(Q)

    def __call__(self, wav, E):
        import torch

        spec = torch.stft(wav, n_fft=1024, hop_length=HOP, win_length=1024, window=self.win, center=True,
                          pad_mode="reflect", return_complex=True)
        power = spec.real ** 2 + spec.imag ** 2
        mel = torch.matmul(power.transpose(1, 2), self.fb).transpose(1, 2)
        image = ((10.0 * torch.log10(mel + 2.220446049250313e-16) - self.mean) / self.std).unsqueeze(1)
        feat = self.emb(image).view(E, W, S + Q, -1)
        proto = feat[:, :, :S].mean(2)                                       # [E, W, D]
        query = feat[:, :, S:].reshape(E, W * Q, -1)                         # [E, WQ, D]
        logits = -((query.unsqueeze(2) - proto.unsqueeze(1)) ** 2).sum(3)    # [E, WQ, W]
        acc = (logits.argmax(2) == self.target.unsqueeze(0)).float().mean() * 100.0
        return logits.reshape(E * W * Q, W), acc


# ----------------------------------------------------------------------------------- B200 arm, mode eval
def run_eval(args, rank, world, local_rank):
    import torch

    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.pipeline import EpisodePipeline
    from audio_fewshot_b200.synthetic import synthetic_clip_batch

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    cpus = bind_to_gpu_cpus(local_rank)  # before any pinned allocation
    ranks = Ranks(rank, world, dev)
    E = args.episodes_per_step or 32
    n_clips = E * CLIPS_PER_EPISODE
    mean, std = mean_std()

    emb = make_weights()
    model = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q,
                          emb_func=emb, device=dev).to(dev).eval()
    front = LogMelFrontEnd(sample_rate=SR, hop_length=HOP, n_mels=N_MELS, mean=mean, std=std).to(dev).eval()
    pipe = EpisodePipeline(front, model)
    repeats = torch.ones(E * W * Q, dtype=torch.long)
    support_size = E * W * S

    # two rotating batches per rank; content keyed by the GLOBAL episode index
    host = []
    for b in range(2):
        first = (b * world + rank) * E
        host.append(torch.from_numpy(synthetic_clip_batch(1234, first, E, W, S, Q, L)).pin_memory())
    devb = [h.to(dev) for h in host]
    wav_bytes = n_clips * L * 4

    def step_device(i, ev=None):
        wav = devb[i % 2]
        if ev is not None:
            ev[0].record()
        image = front(wav, first_clip_index=0)
        if ev is not None:
            ev[1].record()
        return model.set_forward([image, None, repeats, support_size])

    def run_e2e(n, batches):
        """n steps through the public streaming call: every step's waveforms go pinned host -> device on the
        copy stream, its logits and accuracy come back to pinned host memory; copies overlap compute."""
        last = None
        for last in pipe.stream((batches[i % 2] for i in range(n)), repeats, support_size):
            pass
        return last

    with torch.no_grad():
        # ---- device-resident: `value`
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        for i in range(args.warmup):
            step_device(i)
        ranks.barrier()
        launches0 = ops.launch_count()
        lm_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                     for _ in range(args.steps)]
        ms_dev, (output, acc) = timed(ranks, lambda i: step_device(i, lm_events[i]), args.steps)
        launches = ops.launch_count() - launches0
        logmel_ms = ranks.max(float(np.mean([a.elapsed_time(b) for a, b in lm_events])))
        acc_dev = float(acc.item())
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"logits": output, "accuracy_pct": acc})

        # ---- end to end through the public call: `e2e`
        run_e2e(args.warmup, host)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ranks.barrier()
        t0.record()
        out_host, acc_host = run_e2e(args.steps, host)
        t1.record()
        ranks.barrier()
        ms_e2e = ranks.max(t0.elapsed_time(t1))
        clocks = sampler.stop() if rank == 0 else None
        acc_e2e = float(acc_host.item())

        # ---- what the host side can deliver: plain pinned cudaMemcpyAsync of the same buffers, all ranks at once
        probe_dst = torch.empty_like(devb[0])
        probe_dst.copy_(host[0], non_blocking=True)
        ms_probe, _ = timed(ranks, lambda i: probe_dst.copy_(host[i % 2], non_blocking=True), 6)
        probe_gbs = 6 * wav_bytes / (ms_probe * 1e-3) / 1e9  # per rank, slowest rank
        del probe_dst

        extras = {}
        if not args.no_extras:
            # ---- the same call fed with int16 PCM host buffers: `e2e_pcm16` (extra key, not the headline)
            host_pcm = [(h * 32768.0).round_().clamp_(-32768, 32767).to(torch.int16).pin_memory() for h in host]
            run_e2e(args.warmup, host_pcm)
            ranks.barrier()
            t0.record()
            _, acc_pcm_host = run_e2e(args.steps, host_pcm)
            t1.record()
            ranks.barrier()
            ms_pcm = ranks.max(t0.elapsed_time(t1))
            extras["e2e_pcm16"] = {
                "value": args.steps * E * world / (ms_pcm * 1e-3), "unit": "episodes/sec",
                "h2d_bytes_per_step": wav_bytes // 2, "d2h_bytes_per_step": out_host.numel() * 4 + 4,
                "ms_per_step": ms_pcm / args.steps, "accuracy_pct": float(acc_pcm_host.item()),
                "note": "same public call, host waveforms quantised to int16 PCM (afs_logmel_fwd_pcm16 converts on "
                        "load); `e2e` above is the fp32-host-buffer figure"}
            del host_pcm

            # ---- the separately stated bf16 backbone path (north star; SURVEY 8f row 4): same step, same inputs,
            # Conv64F.precision = "bf16" (stem writes bf16, blocks 2-3 as bf16 tcgen05 MMAs).  Extra key, not `value`.
            ref_logits = [step_device(b)[0].clone() for b in range(2)]
            emb.precision = "bf16"
            try:
                for i in range(args.warmup):
                    step_device(i)
                ms_b16, (_, acc_b16) = timed(ranks, lambda i: step_device(i), args.steps)
                flips, dev_rel = 0, 0.0
                for b in range(2):
                    lb = step_device(b)[0]
                    flips += int((lb.argmax(1) != ref_logits[b].argmax(1)).sum().item())
                    dev_rel = max(dev_rel, float(((lb - ref_logits[b]).abs().max() / ref_logits[b].abs().max()).item()))
            finally:
                emb.precision = None
            extras["bf16_backbone"] = {
                "value": args.steps * E * world / (ms_b16 * 1e-3), "unit": "episodes/sec",
                "ms_per_step": ms_b16 / args.steps, "accuracy_pct": float(acc_b16.item()),
                "argmax_flips": flips, "queries_compared": 2 * E * W * Q, "max_logit_deviation_rel": dev_rel,
                "note": "reduced-precision path stated separately from `value` (which stays in the reference's TF32 "
                        "class): bf16 activations between blocks 1-3, bf16 weights, fp32 accumulation; flips and "
                        "deviation are against this run's TF32 logits on the two bench batches"}
            del ref_logits

        if rank == 0 and not args.no_extras:
            hbm_peak, _ = peaks()
            # ---- every kernel >= 10 % of the step
            tf32_peak = measure_tf32_peak(dev)
            rows = kernel_shares(step_device)
            if rows:
                extras["roofline_all"] = roofline_all(rows, n_clips, hbm_peak, tf32_peak)
                extras["kernel_time_us_per_step"] = sum(rows.values())
            extras["tf32_tflops_measured"] = tf32_peak
            # ---- the reference's op sequence in plain PyTorch on this GPU
            from audio_fewshot_b200.frontend import hann_window, slaney_mel_filterbank

            eager_emb = make_weights().to(dev).eval()
            eager_emb._inference_ok = lambda x: False  # plain nn.Module graph (cuDNN + elementwise kernels)
            eager = TorchEagerPath(eager_emb, slaney_mel_filterbank(513, N_MELS, SR), hann_window(1024), mean, std, dev)
            e_eager = min(E, 8)  # the eager graph materialises a 4 GB block-1 activation per 8 episodes
            n_eager = e_eager * CLIPS_PER_EPISODE
            for i in range(2):
                eager(devb[i % 2][:n_eager], e_eager)
            k_eager = max(3, min(args.steps, 10))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(k_eager):
                _, acc_eager = eager(devb[i % 2][:n_eager], e_eager)
            e1.record()
            torch.cuda.synchronize()
            ms_eager = e0.elapsed_time(e1)
            extras["gpu_eager_baseline"] = {
                "value": k_eager * e_eager / (ms_eager * 1e-3), "unit": "episodes/sec", "episodes_per_step": e_eager,
                "ms_per_step": ms_eager / k_eager, "accuracy_pct": float(acc_eager.item()),
                "what": "plain PyTorch on the same GPU, inputs resident: torch.stft log-mel -> Conv64F nn.Module graph "
                        "(cuDNN, TF32 allowed) -> broadcast ProtoLayer arithmetic -> argmax; the reference's op sequence "
                        "(proto_net.py:74-120) with the front-end a user would write"}
            del eager, eager_emb
            torch.cuda.empty_cache()

        if not args.no_extras:
            # ---- BASELINE configs[0]'s clip shape: 1 s @ 16 kHz, hop 102 (every rank runs it; rank 0 reports)
            front1 = LogMelFrontEnd(sample_rate=SR, hop_length=HOP_S1, n_mels=N_MELS, mean=mean, std=std).to(dev).eval()
            s1 = [torch.from_numpy(synthetic_clip_batch(4321, (b * world + rank) * E, E, W, S, Q, L_S1)).to(dev)
                  for b in range(2)]
            ev1 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]

            def step_s1(i, ev=None):
                if ev is not None:
                    ev[0].record()
                image = front1(s1[i % 2], first_clip_index=0)
                if ev is not None:
                    ev[1].record()
                return model.set_forward([image, None, repeats, support_size])

            for i in range(args.warmup):
                step_s1(i)
            ms_s1, (_, acc_s1) = timed(ranks, lambda i: step_s1(i, ev1[i]), args.steps)
            lm1 = ranks.max(float(np.mean([a.elapsed_time(b) for a, b in ev1])))
            if rank == 0:
                hbm_peak, _ = peaks()
                ach1 = LOGMEL_BYTES_PER_CLIP_S1 * n_clips / (lm1 * 1e-3) / 1e9
                extras["s1"] = {
                    "workload": "same model, 1 s @ 16 kHz clips, hop 102 -> [1,128,157] (BASELINE configs[0], shape S1)",
                    "value": args.steps * E * world / (ms_s1 * 1e-3), "unit": "episodes/sec",
                    "ms_per_step": ms_s1 / args.steps, "accuracy_pct": float(acc_s1.item()),
                    "logmel": {"ms_per_launch": lm1, "achieved": ach1, "unit": "GB/s", "frac": ach1 / hbm_peak,
                               "bytes_per_launch": LOGMEL_BYTES_PER_CLIP_S1 * n_clips,
                               "note": "10x frame overlap: 2.8x fewer algorithmic bytes per frame than S5, the same "
                                       "FFT work per frame -- the kernel is bound by the FMA pipe / shared-memory data "
                                       "path, the HBM fraction follows"}}

    total_eps = args.steps * E * world
    if rank != 0:
        return

    peak, peak_src = peaks()
    achieved = LOGMEL_BYTES_PER_CLIP * n_clips / (logmel_ms * 1e-3) / 1e9
    traffic, traffic_src, colimit = None, None, None
    tpath = os.path.join(ROOT, "profiles", "logmel_traffic.json")  # written from an ncu --set full capture
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))  # captured at `clips_per_launch` clips; DRAM bytes scale with the clip count
            traffic = tj["dram_bytes_per_launch"] / tj["clips_per_launch"] * n_clips
            traffic_src = "ncu --set full capture of this kernel at commit %s (%s), scaled to this launch's clip count" % (
                tj.get("commit", "?"), tj.get("report", "profiles/"))
            colimit = tj.get("co_limits")
        except Exception:
            traffic = None
    cfg = base_config(E, n_clips, world)
    cfg.update({
        "backbone": "Conv64F eval path: tcgen05 TF32 kernels for block 1 (conv+BN+ReLU+pool) and blocks 2-3 "
                    "(implicit GEMM+BN+ReLU+pool), cuDNN conv+bias+ReLU for block 4 (TF32 allowed, the "
                    "reference's PyTorch default)",
        "logmel_engine": "pair" if front.plan().engine == "auto" else front.plan().engine,
        "e2e_path": "EpisodePipeline.stream: H2D on a copy stream overlapped with compute, 3 device buffers",
        "l2_policy": "inputs larger than L2: %d MB of waveform per step, two rotating batches" % (wav_bytes // 2 ** 20),
        "parallelism": "episodes sharded over %d rank(s), no data-path collective; timing: barrier + 1-double MAX "
                       "all-reduce" % world,
        "cpu_affinity": ("rank 0 bound to %d CPUs local to its GPU (NVML)" % len(cpus)) if cpus else "not set",
        "accuracy_pct": acc_dev})
    e2e_gbs = wav_bytes / (ms_e2e / args.steps * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": total_eps / (ms_dev * 1e-3), "unit": "episodes/sec", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "e2e": {"value": total_eps / (ms_e2e * 1e-3), "unit": "episodes/sec", "h2d_bytes_per_step": wav_bytes,
                "d2h_bytes_per_step": out_host.numel() * 4 + 4, "ms_per_step": ms_e2e / args.steps,
                "accuracy_pct": acc_e2e, "h2d_gbs_per_gpu": e2e_gbs, "h2d_probe_gbs_per_gpu": probe_gbs,
                "host_roofline_frac": e2e_gbs / probe_gbs,
                "note": "h2d_probe = plain pinned cudaMemcpyAsync of the same buffers by all %d rank(s) at once "
                        "(slowest rank); the e2e leg is bound by that copy, not by the %.1f ms of device work"
                        % (world, ms_dev / args.steps)},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "logmel_pair_kernel<false, float, true> (fused waveform->log-mel, warp-per-frame-pair engine)",
                     "bound": "hbm",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src, "co_limits": colimit,
                     "peak_source": peak_src, "bytes_per_launch": LOGMEL_BYTES_PER_CLIP * n_clips,
                     "ms_per_launch": logmel_ms, "share_of_step": logmel_ms / (ms_dev / args.steps)},
        "clocks": clocks,
    }
    line.update(extras)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_sample(args.cpu_seconds, E)
    emit(line)


# ----------------------------------------------------------------------------------- B200 arm, mode train
def run_train(args, rank, world, local_rank):
    """C1 episodic TRAINING step from waveforms, data-parallel over episodes (reference trainer.py:186-192, :504-509)."""
    import torch

    from audio_fewshot_b200 import dist as afs_dist
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.synthetic import synthetic_clip_batch

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ranks = Ranks(rank, world, dev)
    E = args.episodes_per_step or 2
    mean, std = mean_std()
    emb = make_weights()
    model = arch.ProtoNet(way_num=W, shot_num=S, query_num=Q, test_way=W, test_shot=S, test_query=Q,
                          emb_func=emb, device=dev).to(dev).train()
    model.acc_on_device = True
    front = LogMelFrontEnd(sample_rate=SR, hop_length=HOP, n_mels=N_MELS, mean=mean, std=std).to(dev).eval()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    target = torch.arange(W).repeat_interleave(S + Q).repeat(E)
    wav = [torch.from_numpy(synthetic_clip_batch(1234, (b * world + rank) * E, E, W, S, Q, L)).to(dev) for b in range(2)]
    n_grad = sum(p.numel() for p in model.parameters() if p.requires_grad)

    def step(i):
        with torch.no_grad():
            image = front(wav[i % 2], first_clip_index=0)
        output, acc, loss = model.set_forward_loss([image, target])  # acc: 1-float all-reduce inside (utils.py:116-118)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        afs_dist.all_reduce_gradients(model.parameters())           # ONE flat collective (trainer.py:504-509)
        opt.step()
        return output, acc, loss

    for i in range(args.warmup):
        step(i)
    l0 = ops.launch_count()
    ms, (output, acc, loss) = timed(ranks, step, args.steps)
    launches = ops.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logits": output, "loss": loss, "accuracy_pct": acc})
    # replicas must stay identical: the same parameters on every rank after K data-parallel steps
    checksum = torch.stack([p.detach().double().sum() for p in model.parameters()]).sum()
    spread = 0.0
    if world > 1:
        import torch.distributed as dist

        lo, hi = checksum.clone(), checksum.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        spread = float((hi - lo).abs().item())
    if rank != 0:
        return
    cfg = base_config(E, E * CLIPS_PER_EPISODE, world)
    cfg.update({"mode": "train", "optimizer": "Adam lr 1e-3",
                "parallelism": "dp%d over episodes; per step ONE flat fp32 all-reduce of %d gradient elements (%d bytes, "
                               "NCCL) + the reference's 1-float accuracy all-reduce" % (world, n_grad, 4 * n_grad),
                "replica_parameter_checksum_spread": spread, "loss": float(loss.item()), "accuracy_pct": float(acc.item())})
    emit({"metric": "episodes/sec (5w5s15q, waveform->loss->backward->gradient all-reduce->Adam)",
          "value": args.steps * E * world / (ms * 1e-3), "unit": "episodes/sec", "n_gpus": world, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "gpu_launches": int(launches)})


# ----------------------------------------------------------------------------------- B200 arm, mode eval10k
def run_eval10k(args, rank, world, local_rank):
    """BASELINE configs[1]: ProtoNet/ResNet-12 5-way 1-shot 15-query, `--episodes` episodes sharded round-robin over
    the ranks; per-episode accuracies -> ONE all_gather -> mean and 95 % CI (reference test.py:210, utils.py:148-159)."""
    import torch

    from audio_fewshot_b200 import dist as afs_dist
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200 import ops
    from audio_fewshot_b200.frontend import LogMelFrontEnd
    from audio_fewshot_b200.synthetic import name_seeded_weights_, synthetic_clip_batch_device

    w, s, q = 5, 1, 15
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ranks = Ranks(rank, world, dev)
    E = args.episodes_per_step or 4
    n_total = args.episodes
    if n_total % (E * world):
        raise SystemExit("--episodes must be a multiple of episodes-per-step * world (%d)" % (E * world))
    steps = n_total // (E * world)
    mean, std = mean_std()
    torch.manual_seed(0)
    emb = name_seeded_weights_(arch.resnet12(keep_prob=0.0, avg_pool=True, is_flatten=True, maxpool_last2=True,
                                             num_channels=1))
    model = arch.ProtoNet(way_num=w, shot_num=s, query_num=q, test_way=w, test_shot=s, test_query=q,
                          emb_func=emb, device=dev).to(dev).eval()
    if args.bf16_backbone:
        emb.precision = "bf16"
    front = LogMelFrontEnd(sample_rate=SR, hop_length=HOP, n_mels=N_MELS, mean=mean, std=std).to(dev).eval()
    repeats = torch.ones(E * w * q, dtype=torch.long)
    target = torch.arange(w, device=dev).repeat_interleave(q)
    local = torch.empty(steps * E, device=dev)

    def step(i):
        # batch i of this rank covers the global episodes (i * world + rank) * E ... + E - 1
        first = (i * world + rank) * E
        wav = synthetic_clip_batch_device(77, first, E, w, s, q, L, dev)
        image = front(wav, first_clip_index=first * w * (s + q))
        output, _ = model.set_forward([image, None, repeats, E * w * s])
        local[i * E:(i + 1) * E] = (output.argmax(1).view(E, w * q) == target).float().mean(1) * 100.0

    with torch.no_grad():
        for i in range(min(args.warmup, steps)):
            step(i)
        l0 = ops.launch_count()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ranks.barrier()
        t0.record()
        for i in range(steps):
            step(i)
        # global order: episode g = (i * world + r) * E + e  ->  gather [steps, E] per rank, interleave ranks per batch
        per_rank = local.view(steps, E)
        if world > 1:
            import torch.distributed as dist

            bufs = [torch.empty_like(per_rank) for _ in range(world)]
            dist.all_gather(bufs, per_rank)
            full = torch.stack(bufs, dim=1).reshape(-1)
        else:
            full = per_rank.reshape(-1)
        acc_all = full.cpu()
        m, h = afs_dist.mean_confidence_interval(acc_all.tolist())
        t1.record()
        ranks.barrier()
        ms = ranks.max(t0.elapsed_time(t1))
        launches = ops.launch_count() - l0
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"episode_accuracy_pct": acc_all, "accuracy_mean_ci95": np.array([m, h])})
    emit({"metric": "episodes/sec (5w1s15q ResNet-12, waveform->logits, %d episodes incl. accuracy gather + 95%% CI)" % n_total,
          "value": n_total / (ms * 1e-3), "unit": "episodes/sec", "n_gpus": world, "steps": steps, "warmup": args.warmup,
          "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
          "dtype": "bf16 trunk (stated separately), f32 front-end and head" if args.bf16_backbone else "f32",
          "data": "synthetic",
          "config": {"workload": "ProtoNet ResNet-12 5w1s15q, 80 clips/episode, 5 s @ 16 kHz (BASELINE configs[1], C2)",
                     "mode": "eval10k", "episodes": n_total, "episodes_per_step_per_gpu": E,
                     "backbone_precision": "bf16 (opt-in reduced-precision path)" if args.bf16_backbone else "tf32 class (parity path)",
                     "parallelism": "episodes sharded round-robin over %d rank(s); ONE all_gather of %d per-episode "
                                    "accuracies per rank (%d bytes) at the end, then mean_confidence_interval"
                                    % (world, steps * E, 4 * steps * E),
                     "inputs": "generated on the device per step inside the timed region (torch Philox keyed by the "
                               "global episode index)",
                     "accuracy_pct_mean": float(m), "ci95_half_width": float(h),
                     "accuracy_checksum": float(acc_all.double().sum().item())},
          "gpu_launches": int(launches)})


_REAL_STDOUT = None


def _claim_stdout():
    """Libraries (NCCL's version banner, cuDNN warnings) print to fd 1; the contract is ONE JSON line on
    stdout.  Point fd 1 at stderr for the run and keep the real stdout for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    args = parse()
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback "
                         "(use --impl reference for the CPU oracle)")
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        {"eval": run_eval, "train": run_train, "eval10k": run_eval10k}[args.mode](args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

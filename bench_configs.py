"""Episodes/s of each BASELINE.json config through the reference-facing model API on one B200.

Not the contract bench (that is bench.py, config C1, waveform -> logits); this is the per-config evidence for
SURVEY.md 8(d): the `image` batches of the reference's own API ([N,1,128,157] normalised log-mel, synthetic,
resident on the device) go through `model(batch_list)` exactly as test.py:380 / trainer.py:186 call it.

    C1  ProtoNet / Conv64F   5w5s15q   eval   set_forward
    C2  ProtoNet / resnet12  5w1s15q   eval   set_forward            (D = 12 800)
    C3  DN4 / Conv64F maps   5w5s15q   eval   set_forward, n_k = 3   (fp32 parity head and tcgen05 TF32 head)
    C4  DeepBDC / resnet12Bdc reduce_dim 64, 5w5s10q  eval  set_forward
    C4w DeepBDC / resnet12Bdc at its default reduce_dim (640), 5w5s10q, eval, set_forward, with the BDC kernels' share
        of the step's device time from torch.profiler (opt-in: --only C4w)
    C5  MAML / Conv64F       5w5s10q   train  set_forward_loss + backward, episode_size 2, 5 inner steps

One JSON line per config on stdout; CUDA events, >= 3 warm-up steps, inputs rotate over two batches that together
exceed the 126 MB L2 wherever the config's batch allows it (stated per line).
"""
import argparse
import json
import sys

import numpy as np
import torch


def images(n, dev, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(n, 1, 128, 157, generator=g) * 0.7).to(dev)


def timeit(step, iters, warmup):
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(iters):
        step(i)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def card():
    """Name and power limit of the GPU the numbers were measured on."""
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return "card: %s" % (q or torch.cuda.get_device_name(0))


def bdc_share(model, E, W, S, Q, steps=5):
    """Share of the step's kernel time spent in the bdc* kernels, from torch.profiler over `steps` warm steps (a run
    of its own: the timed steps run without the profiler)."""
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda", 0)
    n = E * W * (S + Q)
    x = images(n, dev, 400)
    repeats = torch.ones(E * W * Q, dtype=torch.long)
    model.eval()
    with torch.no_grad():
        for _ in range(2):
            model([x, None, repeats, E * W * S])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                model([x, None, repeats, E * W * S])
            torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    total = sum(e.device_time_total for e in kernels)
    bdc = sum(e.device_time_total for e in kernels if "bdc" in e.name)
    return "BDC kernels %.3f ms of %.3f ms kernel time per step (%.1f %%)" % (
        bdc / 1e3 / steps, total / 1e3 / steps, 100.0 * bdc / max(total, 1e-9))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", default="")
    ap.add_argument("--module-graph", action="store_true",
                    help="run the backbones as the plain module graph (the reference's op sequence) for comparison")
    ap.add_argument("--bf16", action="store_true",
                    help="run the backbones on the separately stated bf16 path (emb_func.precision = 'bf16') and report "
                         "the argmax flips against the parity path on the same batches")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_configs.py needs a CUDA device (no CPU fallback)")
    from audio_fewshot_b200 import model as arch
    from audio_fewshot_b200 import ops
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)

    def emit(tag, what, E, ms, note, launches):
        print(json.dumps({"config": tag, "what": what, "episodes_per_step": E, "ms_per_step": ms,
                          "episodes_per_sec": E / (ms * 1e-3), "afs_launches_per_step": launches, "note": note}),
              flush=True)

    def run_eval(tag, what, model, E, W, S, Q, note, **fwd_kw):
        n = E * W * (S + Q)
        batches = [images(n, dev, 100 + b) for b in range(2)]
        repeats = torch.ones(E * W * Q, dtype=torch.long)
        model.eval()
        if args.module_graph:
            what += " [module graph]"
            if hasattr(model.emb_func, "fast_eval"):
                model.emb_func.fast_eval = False
            else:
                model.emb_func._inference_ok = lambda x: False
        with torch.no_grad():
            step = lambda i: model([batches[i % 2], None, repeats, E * W * S], **fwd_kw)
            if args.bf16 and hasattr(model.emb_func, "precision"):
                ref = [step(b)[0].clone() for b in range(2)]
                model.emb_func.precision = "bf16"
                flips = sum(int((step(b)[0].argmax(1) != ref[b].argmax(1)).sum().item()) for b in range(2))
                what += " [bf16 backbone]"
                note += "; argmax flips vs the parity path: %d of %d queries" % (flips, 2 * ref[0].shape[0])
                del ref
            step(0)
            l0 = ops.launch_count()
            step(1)
            per = ops.launch_count() - l0
            ms = timeit(step, args.steps, args.warmup)
        mb = 2 * n * 128 * 157 * 4 / 2 ** 20
        emit(tag, what, E, ms, note + "; two rotating image batches = %.0f MB" % mb, per)

    common = dict(way_num=5, test_way=5)
    only = set(args.only.split(",")) if args.only else None

    if only is None or "C1" in only:
        emb = arch.Conv64F(is_flatten=True, num_channels=1)
        m = arch.ProtoNet(shot_num=5, query_num=15, test_shot=5, test_query=15, emb_func=emb, device=dev, **common).to(dev)
        run_eval("C1", "ProtoNet/Conv64F 5w5s15q set_forward", m, 8, 5, 5, 15, "800 images per step")

    if only is None or "C1T" in only:
        # episodic TRAINING step of C1 (trainer.py:186-192): set_forward_loss + backward + Adam, episode_size 2
        from audio_fewshot_b200.graph_step import GraphedTrainStep
        E, W, S, Q = 2, 5, 5, 15
        n = E * W * (S + Q)
        target = torch.arange(W).repeat_interleave(S + Q).repeat(E)
        for tag, cl, graphed in (("eager launches", False, False), ("channels_last", True, False),
                                 ("ONE CUDA graph (GraphedTrainStep)", False, True),
                                 ("channels_last + ONE CUDA graph", True, True)):
            torch.manual_seed(0)
            emb = arch.Conv64F(is_flatten=True, num_channels=1)
            m = arch.ProtoNet(shot_num=S, query_num=Q, test_shot=S, test_query=Q, emb_func=emb, device=dev, **common).to(dev)
            if cl:
                m = m.to(memory_format=torch.channels_last)
            m.train()
            batches = [images(n, dev, 200 + b) for b in range(2)]
            if graphed:
                opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
                gstep = GraphedTrainStep(m, opt, batches[0].shape, target=target)
                step = lambda i: gstep(batches[i % 2])
            else:
                opt = torch.optim.Adam(m.parameters(), lr=1e-3)

                def step(i, m=m, opt=opt, batches=batches):
                    opt.zero_grad(set_to_none=True)
                    out, acc, loss = m([batches[i % 2], target])
                    loss.backward()
                    opt.step()

            ms = timeit(step, args.steps, args.warmup)
            emit("C1-train", "ProtoNet/Conv64F 5w5s15q train step + Adam, " + tag, E, ms, "200 images per step", 0)

    if only is None or "C2" in only:
        emb = arch.resnet12(keep_prob=0.0, avg_pool=True, is_flatten=True, maxpool_last2=True, num_channels=1)
        m = arch.ProtoNet(shot_num=1, query_num=15, test_shot=1, test_query=15, emb_func=emb, device=dev, **common).to(dev)
        run_eval("C2", "ProtoNet/resnet12 5w1s15q set_forward", m, 4, 5, 1, 15, "320 images per step, D = 12800")

    if only is None or "C3" in only:
        for prec in ("fp32", "tf32"):
            emb = arch.Conv64F(is_flatten=False, last_pool=False, num_channels=1)
            m = arch.DN4(n_k=3, shot_num=5, query_num=15, test_shot=5, test_query=15, emb_func=emb, device=dev, **common).to(dev)
            if hasattr(m, "precision"):
                m.precision = prec
            run_eval("C3", "DN4/Conv64F 5w5s15q n_k=3 set_forward, head " + prec, m, 8, 5, 5, 15, "800 images per step")

    if only is None or "C4" in only:
        emb = arch.resnet12Bdc(reduce_dim=64, num_channels=1)
        m = arch.DeepBDC(shot_num=5, query_num=10, test_shot=5, test_query=10, emb_func=emb, device=dev, **common).to(dev)
        run_eval("C4", "DeepBDC/resnet12Bdc(dr=64) 5w5s10q set_forward", m, 4, 5, 5, 10, "300 images per step")

    if only is not None and "C4w" in only:
        emb = arch.resnet12Bdc(num_channels=1)
        m = arch.DeepBDC(shot_num=5, query_num=10, test_shot=5, test_query=10, emb_func=emb, device=dev, **common).to(dev)
        run_eval("C4w", "DeepBDC/resnet12Bdc(default reduce_dim = 640) 5w5s10q set_forward", m, 4, 5, 5, 10,
                 "300 images per step; " + bdc_share(m, 4, 5, 5, 10) + "; " + card())

    if only is None or "C5" in only:
        emb = arch.Conv64F(is_flatten=True, num_channels=1)
        m = arch.MAML(inner_param={"lr": 0.01, "train_iter": 5, "test_iter": 10}, feat_dim=1600, shot_num=5,
                      query_num=10, test_shot=5, test_query=10, emb_func=emb, device=dev, **common).to(dev)
        E, W, S, Q = 2, 5, 5, 10
        n = E * W * (S + Q)
        batches = [images(n, dev, 300 + b) for b in range(2)]
        target = torch.arange(W).repeat_interleave(S + Q).repeat(E)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        m.train()

        def step(i):
            opt.zero_grad(set_to_none=True)
            out, acc, loss = m([batches[i % 2], target])
            loss.backward()
            opt.step()

        ms = timeit(step, max(3, args.steps // 4), 2)
        emit("C5", "MAML/Conv64F 5w5s10q train step (5 inner steps, second order) + Adam, eager launches", E, ms,
             "150 images per step; autograd through cuDNN (SURVEY a20)", 0)

        from audio_fewshot_b200.graph_step import GraphedTrainStep
        opt2 = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)
        gstep = GraphedTrainStep(m, opt2, batches[0].shape, target=target)
        ms = timeit(lambda i: gstep(batches[i % 2]), args.steps, 3)
        emit("C5", "MAML/Conv64F 5w5s10q train step as ONE CUDA graph (GraphedTrainStep)", E, ms,
             "same kernels and order as the eager step; launch path only", 0)


if __name__ == "__main__":
    sys.exit(main())

"""Time the tensor-core stem (csrc/conv1_tc.cu) alone, several builds side by side in one process.

    python tools/time_stem.py [--variant NAME=SOURCE.cu[:-DMACRO=1,...]] ... [--clips 3200] [--launches 50] [--rounds 7]

Each variant is one conv1_tc.cu compiled with nvcc for sm_100a into its own shared library in a temporary directory,
so an older revision of the file (e.g. `git show <rev>:audio_fewshot_b200/csrc/conv1_tc.cu` saved to a file) can be
timed against the current one.  Without --variant the script times the last commit's conv1_tc.cu (`git show HEAD:`,
so it needs a git checkout) against the working tree's.  Every round times every variant, in alternating order, with CUDA events around
--launches back-to-back launches at N x 1 x 128 x 157 (the bench's 3 200 clips: 257 MB of input and 1.8 GB of fp32
output, both larger than the 126 MB L2); the table gives the median over rounds and the spread (min - max).  All
variants must produce bit-identical output (fp32 and bf16) on the same input, or the script fails.
"""
import argparse
import ctypes
import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "audio_fewshot_b200", "csrc")
INCLUDE = os.path.join(ROOT, "include")

# the two symbols of csrc/abi.cu that conv1_tc.cu links against
STUB = r"""
namespace afs {
thread_local int g_last_cuda_error = 0;
void count_launch() {}
}
"""


def _compile(name, src, defines, tmp):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    stub = os.path.join(tmp, "stub.cu")
    so = os.path.join(tmp, name + ".so")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "--shared",
           "-I", INCLUDE, "-I", CSRC, *defines, src, stub, "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (name, r.stderr))
    return so


def _load(so):
    lib = ctypes.CDLL(so)
    for fn in (lib.afs_conv1_bn_act_pool3_fwd_tf32, lib.afs_conv1_bn_act_pool3_fwd_tf32_bf16out):
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                       ctypes.c_void_p, ctypes.c_int32, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]
    return lib


def _power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--variant", action="append", default=[],
                    help="NAME=SOURCE.cu[:-DA=1,-DB=0]; default: HEAD (git show) and the working tree")
    ap.add_argument("--clips", type=int, default=3200)
    ap.add_argument("--H", type=int, default=128)
    ap.add_argument("--W", type=int, default=157)
    ap.add_argument("--slope", type=float, default=0.0)
    ap.add_argument("--bf16", action="store_true", help="time the bf16-output instance")
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_stem.py needs a GPU"
    dev = torch.device("cuda", 0)
    print("device: %s, power limit / max SM clock: %s" % (torch.cuda.get_device_name(dev), _power_limit()))
    tmp = tempfile.mkdtemp(prefix="time_stem_")
    try:
        specs = args.variant
        if not specs:
            head = os.path.join(tmp, "conv1_tc_HEAD.cu")
            with open(head, "wb") as fh:
                fh.write(subprocess.run(["git", "-C", ROOT, "show", "HEAD:audio_fewshot_b200/csrc/conv1_tc.cu"],
                                        capture_output=True, check=True).stdout)
            specs = ["HEAD=" + head, "tree=" + os.path.join(CSRC, "conv1_tc.cu")]
        variants = []
        for s in specs:
            name, rest = s.split("=", 1)
            src, sep, defs = rest.partition(":-D")  # the defines start at the first ":-D", so paths may hold ':'
            defs = (sep[1:] + defs).split(",") if sep else []
            variants.append((name, os.path.abspath(src), [d for d in defs if d]))
        with open(os.path.join(tmp, "stub.cu"), "w") as fh:
            fh.write(STUB)
        with ThreadPoolExecutor(max_workers=len(variants)) as ex:
            sos = list(ex.map(lambda v: _compile(v[0], v[1], v[2], tmp), variants))
        libs = [_load(so) for so in sos]

        N, H, W = args.clips, args.H, args.W
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn((N, 1, H, W), generator=g, device=dev)
        rng = np.random.default_rng(1)
        w = np.ascontiguousarray((rng.standard_normal((64, 9)) * 0.3).astype(np.float32))
        shift = np.ascontiguousarray(rng.standard_normal(64).astype(np.float32))
        odt = torch.bfloat16 if args.bf16 else torch.float32
        out = torch.empty((N, H // 3, W // 3, 64), dtype=odt, device=dev)
        stream = torch.cuda.current_stream(dev)

        def launch(lib, dtype, dst):
            fn = lib.afs_conv1_bn_act_pool3_fwd_tf32_bf16out if dtype == torch.bfloat16 else lib.afs_conv1_bn_act_pool3_fwd_tf32
            rc = fn(x.data_ptr(), N, H, W, w.ctypes.data, shift.ctypes.data, 64, args.slope, dst.data_ptr(),
                    ctypes.c_void_p(stream.cuda_stream))
            if rc != 0:
                raise RuntimeError("stem launch failed: %d" % rc)

        # same bits from every variant, both output types
        for dtype in (torch.float32, torch.bfloat16):
            ref = None
            for (name, _, _), lib in zip(variants, libs):
                o = torch.full((N, H // 3, W // 3, 64), float("nan"), dtype=dtype, device=dev)
                launch(lib, dtype, o)
                torch.cuda.synchronize()
                if ref is None:
                    ref = o
                elif not torch.equal(o.view(torch.int16 if dtype == torch.bfloat16 else torch.int32),
                                     ref.view(torch.int16 if dtype == torch.bfloat16 else torch.int32)):
                    raise SystemExit("variant %s: %s output differs from %s" % (name, dtype, variants[0][0]))
            del ref, o
        print("outputs bit-identical across %d variants (fp32 and bf16)" % len(variants))

        for lib in libs:  # warm-up
            for _ in range(5):
                launch(lib, odt, out)
        torch.cuda.synchronize()
        times = {v[0]: [] for v in variants}
        order = list(range(len(variants)))
        for rnd in range(args.rounds):
            seq = order if rnd % 2 == 0 else order[::-1]
            for i in seq:
                start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                start.record(stream)
                for _ in range(args.launches):
                    launch(libs[i], odt, out)
                stop.record(stream)
                stop.synchronize()
                times[variants[i][0]].append(start.elapsed_time(stop) / args.launches)
        base = np.median(times[variants[0][0]])
        print("stem %s, %d x 1 x %d x %d, slope %g: ms per launch over %d launches, %d rounds"
              % ("bf16 out" if args.bf16 else "fp32 out", N, H, W, args.slope, args.launches, args.rounds))
        for name, _, defs in variants:
            t = np.array(times[name])
            print("  %-14s median %.4f  spread %.4f - %.4f  vs %s %.3f  %s"
                  % (name, np.median(t), t.min(), t.max(), variants[0][0], np.median(t) / base, " ".join(defs)))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    sys.exit(main())

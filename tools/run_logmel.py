"""Launch the log-mel front-end a few times (ncu target): plain launches run the pair engine, augmented ones the
radix-8 engine.  usage: python tools/run_logmel.py plain|augmented [B] [hop] [L]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from audio_fewshot_b200.frontend import LogMelFrontEnd

launch = sys.argv[1]
if launch not in ("plain", "augmented"):
    sys.exit("usage: python tools/run_logmel.py plain|augmented [B] [hop] [L]")
B = int(sys.argv[2]) if len(sys.argv) > 2 else 800
hop = int(sys.argv[3]) if len(sys.argv) > 3 else 512
L = int(sys.argv[4]) if len(sys.argv) > 4 else 80000
dev = torch.device("cuda", 0)
aug = {"gain_db": (-6.0, 6.0), "max_shift": 1600, "noise_std": (0.0, 0.02)}
fr = LogMelFrontEnd(hop_length=hop, n_mels=128, mean=-15.0, std=26.0, seed=7, aug=aug).to(dev)
fr.train(launch == "augmented")
wav = torch.randn(B, L, device=dev) * 0.1
out = torch.empty(B, 1, 128, 1 + L // hop, device=dev)
for _ in range(4):
    fr(wav, out=out)
torch.cuda.synchronize()

"""GPU probe: the cost of explanations.  MilAttentionFineTuneModel (ResNet50, 224 px, bf16 encoder) on 32 bags x 48 slices given as
slice arrays (no file I/O): wall time of `predict_proba` and of `explain` (attention, contributions, Grad-CAM maps on the slice grid,
copied to the host), alternated in one process and timed with CUDA events; then `gradcam_kernel` alone on the whole feature map
(CUDA events over 20 launches, best of 5; the 616 MB map does not fit the L2, so every launch reads it from HBM) with its achieved
bandwidth on the feature-map bytes.  Prints the card's name and power limit beside the numbers.
usage: explain_times.py [n_bags] [rounds]"""
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[2] / "robust-multimodal-pd_b200"))
import numpy as np
import torch

from pd_fusion_b200.heads import gradcam
from pd_fusion_b200.models.mil_attention_finetune import MilAttentionFineTuneModel

n_bags = int(sys.argv[1]) if len(sys.argv) > 1 else 32
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
L, S = 48, 160
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          timeout=30).stdout.strip().splitlines()[0]
except (OSError, subprocess.SubprocessError, IndexError):
    card = torch.cuda.get_device_name() + ", power limit unknown"
print(f"card: {card}")

torch.manual_seed(7)
m = MilAttentionFineTuneModel({"backbone": "resnet50", "pretrained": False, "input_size": 224, "slice_count": L, "batch_size": n_bags,
                               "train_aug": False})
rng = np.random.default_rng(1)
bags = [rng.random((L, S, S), dtype=np.float32) for _ in range(n_bags)]


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), r


for _ in range(2):                                      # warm-up of both paths (encoder build, module loads)
    m.predict_proba(bags)
    ex = m.explain(bags)
tp, te = [], []
for _ in range(rounds):
    tp.append(timed(lambda: m.predict_proba(bags))[0])
    te.append(timed(lambda: m.explain(bags))[0])
print(f"{n_bags} bags x {L} slices ({S}x{S} -> 224 px), resnet50 bf16, {rounds} alternating rounds (ms per call)")
print(f"  predict_proba: min {min(tp):.1f}  median {np.median(tp):.1f}  max {max(tp):.1f}")
print(f"  explain      : min {min(te):.1f}  median {np.median(te):.1f}  max {max(te):.1f}   (+{np.median(te) / np.median(tp) - 1:.0%} median)")
prob = m.predict_proba(bags)
print(f"  explain prob vs predict_proba: max |diff| {np.abs(ex['prob'] - prob).max():.2e}")

enc = next(v for k, v in m._native.items() if isinstance(k, tuple) and k[0] == "enc")
fmap = enc.feature_map()[: n_bags * L]
g = torch.randn((fmap.shape[0], fmap.shape[3]), device="cuda")
for _ in range(3):
    gradcam(fmap, g, (S, S))
best = 1e9
for _ in range(5):
    ms, _ = timed(lambda: [gradcam(fmap, g, (S, S)) for _ in range(20)])
    best = min(best, ms / 20)
fbytes = fmap.numel() * 4
print(f"gradcam_kernel: {fmap.shape[0]} slices, feature map {tuple(fmap.shape[1:])} f32 = {fbytes / 1e6:.0f} MB, maps {S}x{S}: "
      f"{best * 1e3:.0f} us = {fbytes / (best / 1e3) / 1e9:.0f} GB/s on the feature-map bytes "
      f"({(fbytes + fmap.shape[0] * S * S * 4) / (best / 1e3) / 1e9:.0f} GB/s with the map writes)")

"""GPU probe: training a deep ensemble of E heads in lockstep (HeadEnsemble.train) against E sequential single-model `train` calls, for
E in {1, 8, 32}, in the same process and alternated.  Cases: ModDrop at bench.py's heads-leg widths (mri 512 -> 256-128-64-1, dropout
0.3) on N = 10 000 subjects, batch 32, one epoch; MoE at bench.py's C4 widths (clinical 10 + mri 512, experts 32-16, router 16) on
N = 10 000, full batch, 20 epochs; the gated MIL head at uncertainty_times.py's widths (D 512, H 256, A 128, dropout 0.3) on 2048 bags
x 48 instances, batch 16, one epoch.  Wall time of each call closed by a device synchronise (median of `rounds` after one warm-up of
each), the library's kernel launches per training step, the dropout draws per step, and the card's name and power limit.
usage: ensemble_times.py [rounds]"""
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[2] / "robust-multimodal-pd_b200"))
import numpy as np
import torch

from pd_fusion_b200 import _lib
from pd_fusion_b200.models.ensemble import HeadEnsemble
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel
from pd_fusion_b200.models.mil_attention import MilAttentionModel
from pd_fusion_b200.models.moe import MoEModel

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          timeout=30).stdout.strip().splitlines()[0]
except (OSError, subprocess.SubprocessError, IndexError):
    card = torch.cuda.get_device_name() + ", power limit unknown"
print(f"card: {card}")

rng = np.random.default_rng(0)
N = 10_000
X_md = rng.standard_normal((N, 512)).astype(np.float32)
y = (rng.random(N) < 0.5).astype(np.float32)
md_args = ({"clinical": 0, "datspect": 0, "mri": 512}, {"hidden_dims": [256, 128, 64], "dropout": 0.3, "lr": 1e-3, "epochs": 1,
                                                       "batch_size": 32})
X_moe = {"clinical": rng.standard_normal((N, 10)).astype(np.float32), "mri": X_md}
mask_moe = (rng.random((N, 2)) < 0.7).astype(np.float32)
moe_args = ({"clinical": 10, "mri": 512}, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16], "lr": 1e-3, "epochs": 20})
bags = [rng.standard_normal((48, 512)).astype(np.float32) for _ in range(2048)]
y_mil = (rng.random(2048) < 0.5).astype(np.float32)
mil_args = (512, {"hidden_dim": 256, "attn_dim": 128, "gated": True, "dropout": 0.3, "lr": 1e-3, "epochs": 1, "batch_size": 16})
CASES = (("moddrop", ModalityDropoutModel, md_args, (X_md, y), 2),          # dropout layers per step (torch.rand launches per member)
         ("moe", MoEModel, moe_args, (X_moe, y, mask_moe), 0),
         ("mil", MilAttentionModel, mil_args, (bags, y_mil), 1))


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def ensemble(cls, args, targs, E):
    ens = HeadEnsemble(cls, args, list(range(E)))
    n0 = _lib.launch_count()
    ens.train(*targs)
    return (_lib.launch_count() - n0) / len(ens.last_losses)


def sequential(cls, args, targs, E):
    n0, steps = _lib.launch_count(), 0
    for s in range(E):
        torch.manual_seed(s)
        np.random.seed(s)
        m = cls(*args)
        m.train(*targs)
        steps += len(m.last_losses)
    return (_lib.launch_count() - n0) / steps


for name, cls, args, targs, drops in CASES:
    for E in (1, 8, 32):
        fns = {"ensemble": lambda: ensemble(cls, args, targs, E), "sequential": lambda: sequential(cls, args, targs, E)}
        per_step = {k: fn() for k, fn in fns.items()}                # warm-up
        t = {k: [] for k in fns}
        for _ in range(rounds):
            for k, fn in fns.items():
                t[k].append(wall(fn)[0])
        med = {k: float(np.median(v)) for k, v in t.items()}
        print(f"{name} E={E}: ensemble {med['ensemble']:.1f} ms, {E} sequential {med['sequential']:.1f} ms "
              f"({med['sequential'] / med['ensemble']:.2f}x); library launches per step: ensemble {per_step['ensemble']:.0f}, "
              f"single model {per_step['sequential']:.0f}; dropout draws per ensemble step: {drops * E} torch.rand")
        torch.cuda.empty_cache()

"""GPU probe: the cost of the fusion-head explanations.  bench.py's heads-leg nets (ModDrop at the C2 widths: mri 512 -> 256-128-64-1;
MoE {clinical: 10, mri: 512}, experts 32-16, router 16) under 7 random scenario masks.  CUDA-event times after warm-up (median of
`rounds`, the calls alternated) of the sweep (`forward`, i.e. predict_proba_sweep's launch) against `explain(steps=0)` (Shapley values)
at N = 10 000 and 1 000 000, and `explain(steps=32)` (Shapley values + integrated gradients) at N = 10 000 and 100 000.  Then one
torch.profiler pass over explain(steps=32) at N = 100 000 gives the device time per kernel, and mlp_ig_kernel's FLOP/s from the FLOP
count below.  Prints the card's name and power limit beside the numbers.
usage: fusion_explain_times.py [rounds]"""
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[2] / "robust-multimodal-pd_b200"))
import numpy as np
import torch

from pd_fusion_b200.heads import ModDropSweep, MoeSweep
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet
from pd_fusion_b200.models.moe import MoENet

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
S, K = 7, 32
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          timeout=30).stdout.strip().splitlines()[0]
except (OSError, subprocess.SubprocessError, IndexError):
    card = torch.cuda.get_device_name() + ", power limit unknown"
print(f"card: {card}")

dev = torch.device("cuda")
torch.manual_seed(4321)                                     # bench.py heads_leg's nets
dims_md = {"clinical": 0, "datspect": 0, "mri": 512}
hidden_md = [256, 128, 64]
md = ModDropSweep(ModalityDropoutNet(dims_md, hidden_md, 0.3).state_dict(), dims_md, device=dev)
dims_moe = {"clinical": 10, "mri": 512}
hidden_moe = [32, 16]
moe = MoeSweep(MoENet(dims_moe, {"expert_hidden_dims": hidden_moe, "router_hidden_dims": [16]}).state_dict(), list(dims_moe), device=dev)


def ig_flops(hidden, rows):
    """mlp_ig_kernel: per (pair, step) row, the forward and the backward GEMM of every layer between two hidden layers, 2 FLOP per
    multiply-add (layer 1 is an FMA per hidden unit, the last layer a dot product: not counted)"""
    macs = sum(a * b for a, b in zip(hidden[:-1], hidden[1:]))
    return rows * 2 * 2 * macs


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


g = torch.Generator(device=dev).manual_seed(3)
for N in (10_000, 100_000, 1_000_000):
    X = torch.randn((N, 512), generator=g, device=dev)
    Xc = torch.randn((N, 10), generator=g, device=dev)
    m3 = (torch.rand((S, N, 3), generator=g, device=dev) < 0.7).to(torch.uint8)
    m2 = m3[:, :, 1:].contiguous()
    cases = {"moddrop": {"sweep": lambda: md.forward(X, m3), "explain(0)": lambda: md.explain(X, m3, 0)},
             "moe": {"sweep": lambda: moe.forward({"clinical": Xc, "mri": X}, m2), "explain(0)": lambda: moe.explain({"clinical": Xc, "mri": X}, m2, 0)}}
    if N <= 100_000:
        cases["moddrop"][f"explain({K})"] = lambda: md.explain(X, m3, K)
        cases["moe"][f"explain({K})"] = lambda: moe.explain({"clinical": Xc, "mri": X}, m2, K)
    if N == 100_000:                                        # IG only: the sweep and Shapley sizes are N = 1e4 and 1e6
        for c in cases.values():
            del c["sweep"], c["explain(0)"]
    for head, fns in cases.items():
        for fn in fns.values():
            fn(); fn()
        t = {k: [] for k in fns}
        for _ in range(rounds):
            for k, fn in fns.items():
                t[k].append(timed(fn))
        print(f"{head} N={N} S={S}: " + "  ".join(f"{k} {np.median(v):.3f} ms (min {min(v):.3f})" for k, v in t.items()))
    if N == 100_000:
        from torch.profiler import ProfilerActivity, profile
        for head, fn, rows, hidden in (("moddrop", lambda: md.explain(X, m3, K), S * N * K, hidden_md),
                                       ("moe", lambda: moe.explain({"clinical": Xc, "mri": X}, m2, K), 2 * N * K, hidden_moe)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            per = {}
            for ev in prof.events():
                if ev.device_type.name == "CUDA":
                    per[ev.name] = per.get(ev.name, 0.0) + ev.device_time_total
            print(f"{head} explain({K}) N={N}: device time per kernel (us): " +
                  ", ".join(f"{k.split('(')[0][:60]} {v:.0f}" for k, v in sorted(per.items(), key=lambda kv: -kv[1])))
            ig_us = sum(v for k, v in per.items() if "mlp_ig_kernel" in k)
            fl = ig_flops(hidden, rows)
            print(f"  mlp_ig_kernel: {ig_us:.0f} us, {fl / 1e9:.1f} GFLOP counted -> {fl / (ig_us * 1e-6) / 1e12:.2f} TFLOP/s (FP32 FFMA)")
    del X, Xc, m3, m2
    torch.cuda.empty_cache()

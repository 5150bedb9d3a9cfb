"""GPU probe: the cost of Monte-Carlo dropout (pdf_moddrop_mc, pdf_mil_mc).  ModDrop at bench.py's heads-leg widths (mri 512 ->
256-128-64-1, dropout 0.3) under 7 random scenario masks with T = 32 samples at N = 10 000 and 100 000, timed against
`explain(steps=32)` of the same S, N (the same tile shape, forward and backward); the gated MIL head at bench.py's C3 widths (D 512,
H 256, A 128, dropout 0.3) on 2048 bags x 48 instances with T = 32, timed against its sweep.  CUDA-event times after warm-up (median of
`rounds`, the calls alternated), then one torch.profiler pass per call for the device time per kernel and the MC kernels' FLOP/s on
the counted forward FLOPs below.  Prints the card's name and power limit beside the numbers.
usage: uncertainty_times.py [rounds]"""
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[2] / "robust-multimodal-pd_b200"))
import numpy as np
import torch

from pd_fusion_b200.heads import MilHead, ModDropSweep
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet
from pd_fusion_b200.models.mil_attention import MILAttentionNet

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
S, T, P = 7, 32, 0.3
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          timeout=30).stdout.strip().splitlines()[0]
except (OSError, subprocess.SubprocessError, IndexError):
    card = torch.cuda.get_device_name() + ", power limit unknown"
print(f"card: {card}")

dev = torch.device("cuda")
torch.manual_seed(4321)                                     # bench.py heads_leg's net
dims_md = {"clinical": 0, "datspect": 0, "mri": 512}
hidden_md = [256, 128, 64]
md = ModDropSweep(ModalityDropoutNet(dims_md, hidden_md, P).state_dict(), dims_md, device=dev)
D, H, A, NB, L = 512, 256, 128, 2048, 48
torch.manual_seed(7)
mil = MilHead(MILAttentionNet(D, H, A, P, gated=True).state_dict(), True, 0.5, device=dev)


def moddrop_flops(rows):
    """moddrop_mc_kernel per (pair, sample) row: layers 2.. and the logit, 2 FLOP per multiply-add (layer 1 is the sweep's partials,
    added per row: not counted)"""
    return rows * 2 * (sum(a * b for a, b in zip(hidden_md[:-1], hidden_md[1:])) + hidden_md[-1])


def mil_flops(instances):
    """mil_mc_kernel per (instance, sample): the two attention layers (2A x H) and the pooling (H), 2 FLOP per multiply-add"""
    return instances * 2 * (2 * A * H + H)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def run(label, fns):
    for fn in fns.values():
        fn(); fn()
    t = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            t[k].append(timed(fn))
    print(f"{label}: " + "  ".join(f"{k} {np.median(v):.3f} ms (min {min(v):.3f})" for k, v in t.items()))


def profile(label, fn, kernel, flops):
    from torch.profiler import ProfilerActivity, profile as prof_
    with prof_(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA":
            per[ev.name] = per.get(ev.name, 0.0) + ev.device_time_total
    print(f"{label}: device time per kernel (us): " +
          ", ".join(f"{k.split('(')[0][:60]} {v:.0f}" for k, v in sorted(per.items(), key=lambda kv: -kv[1])))
    us = sum(v for k, v in per.items() if kernel in k)
    print(f"  {kernel}: {us:.0f} us, {flops / 1e9:.1f} GFLOP counted -> {flops / (us * 1e-6) / 1e12:.2f} TFLOP/s (FP32 FFMA)")


g = torch.Generator(device=dev).manual_seed(3)
for N in (10_000, 100_000):
    X = torch.randn((N, 512), generator=g, device=dev)
    m3 = (torch.rand((S, N, 3), generator=g, device=dev) < 0.7).to(torch.uint8)
    run(f"moddrop N={N} S={S} T={T}", {"sweep": lambda: md.forward(X, m3), f"mc(T={T})": lambda: md.mc(X, m3, T, 0, P),
                                          f"explain({T})": lambda: md.explain(X, m3, T)})
    profile(f"moddrop mc N={N}", lambda: md.mc(X, m3, T, 0, P), "moddrop_mc_kernel", moddrop_flops(S * N * T))
    del X, m3
    torch.cuda.empty_cache()

bags = torch.randn((NB, L, D), generator=g, device=dev)
lens = torch.full((NB,), L, dtype=torch.int32, device=dev)
live = (torch.rand((S, NB), generator=g, device=dev) < 0.8).to(torch.uint8)
run(f"mil gated D={D} H={H} A={A} {NB} bags x {L} S={S} T={T}", {"sweep": lambda: mil.sweep(bags, lens, live, S),
                                                                  f"mc(T={T})": lambda: mil.mc(bags, lens, live, S, T, 0, P)})
profile("mil mc", lambda: mil.mc(bags, lens, live, S, T, 0, P), "mil_mc_kernel", mil_flops(NB * L * T))

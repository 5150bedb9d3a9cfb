"""GPU probe: ResNet50 with block 0's projection shortcut inside its conv3 launch (PDFUSION_B200_SHORTCUT) against the separate
downsample launches, A/B inside ONE process (per-op times move by 10-20 % from process to process).  Per stage: the fused conv3
against the downsample + conv3 pair it replaces; then the whole stack per stage set, alternated over rounds.
usage: shortcut_ab.py [n_slices] [rounds]"""
import os
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[2] / "robust-multimodal-pd_b200"))
import torch
from pd_fusion_b200.backbone import ResNet2D, ResNetEncoder

n = int(sys.argv[1]) if len(sys.argv) > 1 else 768
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
torch.manual_seed(1234)
sd = {k: v for k, v in ResNet2D("resnet50").state_dict().items() if not k.startswith("fc.")}
x = (torch.rand(n, 224, 224, device="cuda") * 2 - 1).to(torch.bfloat16)
sets = ("none", "1", "1,2", "1,2,3", "1,2,3,4")
encs = {}
for sc in sets:
    os.environ["PDFUSION_B200_SHORTCUT"] = sc
    encs[sc] = ResNetEncoder(sd, n, 224, precision="bf16", arch="resnet50")
    encs[sc].forward(x)
del os.environ["PDFUSION_B200_SHORTCUT"]
torch.cuda.synchronize()


def t_ops(enc, idx, reps=30):
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            for i in idx:
                enc.run_range(i, 1)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps * 1e3)
    return best


sep, fus = encs["none"], encs["1,2,3,4"]
print("stage  downsample+conv3 (us)  fused conv3 (us)   per round")
for k in range(1, 5):
    pair = [sep.op_names.index(f"layer{k}.0.downsample.0"), sep.op_names.index(f"layer{k}.0.conv3")]
    one = [fus.op_names.index(f"layer{k}.0.conv3")]
    a, b = [], []
    for _ in range(rounds):
        a.append(t_ops(sep, pair))
        b.append(t_ops(fus, one))
    print(f"{k:5d}  {min(a):21.1f}  {min(b):16.1f}   " + " ".join(f"{u:.0f}/{v:.0f}" for u, v in zip(a, b)), flush=True)

stack = {sc: [] for sc in sets}
for _ in range(rounds):
    for sc in sets:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        encs[sc].forward(None)
        e0.record()
        for _ in range(20):
            encs[sc].forward(None)
        e1.record()
        torch.cuda.synchronize()
        stack[sc].append(e0.elapsed_time(e1) / 20 * 1e3)
for sc in sets:
    print(f"shortcut stages {sc:8s}: whole stack {min(stack[sc]):8.1f} us (rounds: {' '.join(f'{v:.0f}' for v in stack[sc])}), "
          f"{len(encs[sc].op_names)} ops")

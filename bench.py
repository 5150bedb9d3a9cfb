#!/usr/bin/env python
"""bench.py -- MRI subjects/s of the imaging-embedding hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c5] [--subjects B] [--impl b200|reference]
                    [--dump-outputs DIR]

The default workload is c3 = configs/openneuro_ds001907_resnet2d_mil.yaml (ResNet50, 48 slices, gated MIL attention): the
configuration BASELINE.json's metric ("ResNet2D-MIL embed+fuse") is quoted on.

A "step" = one pass of the hot path over one batch of B synthetic subjects per GPU:
raw T1 volumes f32[256,256,176] resident in HBM -> resample 160^3 -> p1/p99 normalise -> slice select ->
224x224 network input -> ResNet2D (bf16 tcgen05) -> per-slice embeddings (+ slice mean) -> fusion head (ModDrop for c2, gated
MIL attention for c3) under the 7 missing-modality scenarios of configs/eval_missingness_openneuro_ds001907.yaml [-> all-gather
of the embedding table and of the per-scenario probabilities when N > 1].  Prints ONE JSON line (rank 0).

  value        device-resident throughput (inputs already in HBM), CUDA-event timed, max over ranks
  e2e          same metric through the public host API, fed what the manifest's files hold -- the voxels as an int16 NIfTI stores them
               (x fastest), in pinned host memory: H2D inside the timed region, decode (nibabel's float64 scaling rule, cast,
               transpose) on the device, hot path, D2H of the results
  e2e_float32_volumes  the same call fed ready-made float32 host arrays (what `_load_volume` works on after nibabel): twice the PCIe
               bytes, PCIe-bound
  roofline     the dominant kernel family (tcgen05 implicit-GEMM convs): algorithmic FLOPs / CUDA-event time of the timed region
               against the measured BURST bf16 peak, with the DRAM traffic of the same launches (ncu capture, profiles/)
  sustained    >= 2 s of back-to-back steps / conv stacks (the regime of a 10 k-subject job: the board sits at its power cap):
               subjects/s, and the conv stack's TFLOP/s against the measured SUSTAINED bf16 peak
  roofline_preproc, roofline_preproc_dense  the preprocessing kernels against the measured copy bandwidth (SURVEY.md 8d
               algorithmic bytes) on the synthetic brains (73 % exact-zero background, which the kernels skip) and on volumes
               without background
  roofline_mil the MIL head (projection + attention + pooling, all 7 scenarios) on a bag table larger than L2: 4*L*D+4 bytes per bag
  heads        pdf_moddrop_sweep / pdf_moe_sweep at N = 10 000 and 1 000 000 subjects (SURVEY.md 8d), bytes-based roofline
  cpu_baseline the oracle port of the reference's CPU path on a bounded sample (rank 0, N = 1 only)

`--impl reference` times the reference's own CPU implementation of the path (the oracle port in oracle/oracle.py: the
reference is Python, so there is nothing to compile).

`--dump-outputs DIR` writes, after the timed steps, what the timed path returned in its last step as DIR/<name>.npy (float32),
64 MB at most, so that two builds can be compared output for output on identical inputs (the same arguments give the same
seeded inputs):
  c2 / c3      embeddings.npy (c3: [B*N, L, D] slice embeddings, c2: [B*N, D] slice means) and scenario_probs.npy [B*N, 7]
  c5           loss.npy, probs.npy [bags], and the updated weights: head_params.npy, backbone_params.npy (flat)
An array larger than its share of the 64 MB is replaced by a fixed, seeded sample of its rows (the same rows for the same
shapes), flattened to [rows, last axis] -- c3 embeddings to [k, D] rows of (subject, slice) pairs -- with the kept row indices in
<name>_rows.npy (row = subject * L + slice for the c3 table).
c3's last step depends only on the seeded inputs, so two runs of one build are expected to write the same files.  c5's weights
are not expected to match bit for bit between runs: the training kernels accumulate with atomicAdd (the head's gradients, the
loss and the gradient norm in float, BatchNorm statistics in double) in no fixed order, and Adam carries those last-bit
differences through the steps; compare c5 dumps with a tolerance.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (ROOT, ROOT / "robust-multimodal-pd_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np  # noqa: E402

WORKLOADS = {
    # configs/openneuro_ds001907_resnet2d.yaml + data_openneuro_ds001907_resnet2d.yaml (BASELINE configs[1])
    "c2": dict(arch="resnet18", axes=[2], counts=[24], batch_size=32, name="configs/openneuro_ds001907_resnet2d.yaml"),
    # configs/openneuro_ds001907_resnet2d_mil.yaml (BASELINE configs[2])
    "c3": dict(arch="resnet50", axes=[2], counts=[48], batch_size=16, name="configs/openneuro_ds001907_resnet2d_mil.yaml"),
    # BASELINE configs[4]: fine-tune forward/backward (configs/openneuro_ds001907_resnet2d_mil_ft.yaml: resnet50, 64 slices,
    # 4 bags per step, 16-slice chunks, gated MIL head, focal loss, clip 1.0, Adam 1e-4 / 3e-4) -- its own leg (run_c5)
    "c5": dict(arch="resnet50", axes=[2], counts=[64], batch_size=16, name="configs/openneuro_ds001907_resnet2d_mil_ft.yaml"),
}
IN_SHAPE, TARGET, INPUT_SIZE = (256, 256, 176), (160, 160, 160), 224
METRIC, UNIT = "mri_subjects_per_sec_resnet2d_embed_fuse", "subjects/s"


def conv_dram_traffic(workload: str, B: int):
    """DRAM bytes moved by the conv launches of ONE step: dram__bytes_read.sum + dram__bytes_write.sum summed over the launches
    of one `ncu --set full` capture of this command, written by scripts/ncu_traffic.py into profiles/conv_traffic.json (keyed
    by workload and subjects per step, with the capture's date and source file).  None when that configuration was not captured."""
    p = ROOT / "profiles" / "conv_traffic.json"
    if not p.exists():
        return None, None
    d = json.loads(p.read_text())
    e = d.get(f"{workload}_b{B}")
    return (float(e["dram_bytes"]), e.get("source")) if e else (None, None)


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm=float(d["hbm_gbs"]), tf=float(d["bf16_tflops"]), tf_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML; nvidia-smi as a fallback)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.index, self.sm, self.mx, self.reasons, self._stop, self._t = index, [], [], set(), threading.Event(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)))
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in self.BITS.items():
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            r = [c.strip() for c in out.splitlines()[0].split(",")]
            self.sm.append(float(r[0])); self.mx.append(float(r[1]))
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def _loop(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.02 if self.nvml else 0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml" if self.nvml else "nvidia-smi"}


DUMP_BYTES = 64 * 10**6 - 4096          # --dump-outputs budget, less room for the .npy headers


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each array as out_dir/<name>.npy in float32.  Smallest first, each array gets an equal share of what is left of
    DUMP_BYTES; one larger than its share is replaced by a sample of its rows drawn with a fixed seed (the same rows for the
    same shapes in every run): the array flattened to [rows, last axis] (a 1-D array: to its elements), the kept rows in
    ascending order, and their indices into that flattened array in out_dir/<name>_rows.npy (float64, exact)."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    arrays = sorted(((name, np.asarray(a, dtype=np.float32)) for name, a in arrays.items()), key=lambda kv: kv[1].nbytes)
    left = DUMP_BYTES
    for i, (name, a) in enumerate(arrays):
        share = left // (len(arrays) - i)
        if a.nbytes > share:
            rows = a.reshape(-1, a.shape[-1]) if a.ndim > 1 else a.reshape(-1, 1)
            keep = share // (rows.shape[1] * 4 + 8)                     # a row and its float64 index
            pick = np.sort(np.random.default_rng(0).choice(rows.shape[0], keep, replace=False))
            a = rows[pick] if a.ndim > 1 else rows[pick, 0]
            np.save(out / f"{name}_rows.npy", pick.astype(np.float64))
            left -= pick.size * 8
        np.save(out / f"{name}.npy", a)
        left -= a.nbytes


def host_pool(n: int):
    from pd_fusion_b200.synthetic import synthetic_volume
    return [synthetic_volume(i, IN_SHAPE) for i in range(n)]


def dense_volume(index: int):
    """A volume WITHOUT background: Gamma(4, 100) everywhere (no exact zeros for the kernels to skip)."""
    return np.random.default_rng(5000 + index).gamma(4.0, 100.0, size=IN_SHAPE).astype(np.float32)


def cpu_reference_rate(wl, n_subjects: int, pool):
    """The reference's CPU path (oracle port) on `n_subjects` subjects with every host thread."""
    import torch
    from oracle import oracle as O
    from pd_fusion_b200.backbone import ResNet2D
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(1234)
    sd = {k: v for k, v in ResNet2D(wl["arch"]).state_dict().items() if not k.startswith("fc.")}
    # the fuse half: the config's head under the 7 scenario masks, per subject as evaluate_model would (tiny next to the backbone)
    torch.manual_seed(4321)
    D = 2048 if wl["arch"] == "resnet50" else 512
    if wl["arch"] == "resnet18":
        from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet
        dims = {"clinical": 0, "datspect": 0, "mri": D}
        hsd = {k: v.numpy() for k, v in ModalityDropoutNet(dims, [256, 128, 64], 0.3).state_dict().items()}
    else:
        from pd_fusion_b200.models.mil_attention import MILAttentionNet
        hsd = {k: v.numpy() for k, v in MILAttentionNet(D, 256, 128, 0.2, gated=True).state_dict().items()}
    mri_masks = [1, 1, 0, 1, 0, 0, 1]                       # one subject's mri availability under the 7 scenarios (fixed draw)
    t0 = time.perf_counter()
    for i in range(n_subjects):
        _, emb = O.embed_subject(pool[i % len(pool)], sd, wl["arch"], TARGET, wl["axes"], wl["counts"], INPUT_SIZE, wl["batch_size"])
        for m in mri_masks:
            if wl["arch"] == "resnet18":
                O.moddrop_predict_proba(hsd, dims, emb.mean(axis=0, keepdims=True), {"clinical": np.zeros(1), "datspect": np.zeros(1), "mri": np.array([m])})
            else:
                O.mil_predict_proba(hsd, [emb], True, {"mri": np.array([m])})
    dt = time.perf_counter() - t0
    return n_subjects / dt, cores, dt


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    per_step = 1
    pool = host_pool(2)
    for _ in range(args.warmup):
        cpu_reference_rate(wl, 1, pool)
    t0 = time.perf_counter()
    rate, cores, _ = cpu_reference_rate(wl, per_step * args.steps, pool)
    dt = time.perf_counter() - t0
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "backbone": wl["arch"], "slices": sum(wl["counts"]), "subjects_per_step": per_step,
                       "volume": list(IN_SHAPE), "note": "reference CPU path (oracle port of the Python reference), all host threads"},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{per_step * args.steps} subjects, full {wl['arch']} path"},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def heads_leg(dev, peaks, timed):
    """pdf_moddrop_sweep (C2 dims: mri 512 -> 256-128-64-1) and pdf_moe_sweep (C4 dims: mri 512 + clinical 10) under the 7 scenarios
    of the ds001907 eval file and under the 8-mask power set, at N = 10 000 and 1 000 000 subjects.  Algorithmic bytes per subject
    (SURVEY.md 8d): features once (4F) + S*M mask bytes + 4S probabilities.  The reference's evaluate_model loop (oracle port) is
    timed next to the N = 10 000 ModDrop/MoE sweeps on the host."""
    import torch
    from oracle import oracle as O
    from pd_fusion_b200.heads import ModDropSweep, MoeSweep
    from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet
    from pd_fusion_b200.models.moe import MoENet
    out = []
    torch.manual_seed(4321)
    dims_md = {"clinical": 0, "datspect": 0, "mri": 512}
    md_sd = ModalityDropoutNet(dims_md, [256, 128, 64], 0.3).state_dict()
    md = ModDropSweep(md_sd, dims_md, device=dev)
    dims_moe = {"clinical": 10, "mri": 512}
    moe_sd = MoENet(dims_moe, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16]}).state_dict()   # configs/model_moe.yaml
    moe = MoeSweep(moe_sd, list(dims_moe), device=dev)
    g = torch.Generator(device=dev).manual_seed(3)
    for N in (10_000, 1_000_000):
        X = torch.randn((N, 512), generator=g, device=dev)
        Xc = torch.randn((N, 10), generator=g, device=dev)
        for S, label in ((7, "7 scenarios"), (8, "8-mask power set")):
            m3 = (torch.rand((S, N, 3), generator=g, device=dev) < 0.7).to(torch.uint8)
            m2 = m3[:, :, 1:].contiguous()
            reps = 20 if N <= 10_000 else 3
            for name, fn, F, M in (("moddrop", lambda: md.forward(X, m3), 512, 3), ("moe", lambda: moe.forward({"clinical": Xc, "mri": X}, m2), 522, 2)):
                fn(); fn()
                ms = timed(fn, reps) / reps
                nbytes = N * (4 * F + S * M + 4 * S)
                rec = {"head": name, "N": N, "S": S, "masks": label, "ms": ms, "pairs_per_s": N * S / (ms / 1e3),
                       "roofline": {"bound": "hbm", "achieved": nbytes / (ms / 1e3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
                                    "frac": nbytes / (ms / 1e3) / 1e9 / peaks["hbm"], "bytes_per_subject": 4 * F + S * M + 4 * S}}
                if N == 10_000 and S == 7:      # the reference's per-scenario loop on the host cores (oracle port), same inputs
                    Xh, mh = X.cpu().numpy(), m3.cpu().numpy()
                    t0 = time.perf_counter()
                    if name == "moddrop":
                        sdn = {k: v.numpy() for k, v in md_sd.items()}
                        for s_ in range(S):
                            O.moddrop_predict_proba(sdn, dims_md, Xh, {m: mh[s_][:, i] for i, m in enumerate(O.MODALITIES)})
                    else:
                        sdn = {k: v.numpy() for k, v in moe_sd.items()}
                        Xch, m2h = Xc.cpu().numpy(), m2.cpu().numpy()
                        for s_ in range(S):
                            O.moe_predict_proba(sdn, {"clinical": Xch * m2h[s_][:, :1], "mri": Xh * m2h[s_][:, 1:2]}, m2h[s_].astype(np.float32))
                    rec["cpu_reference_ms"] = (time.perf_counter() - t0) * 1e3
                out.append(rec)
        del X, Xc
    return out


def run_c5(args, wl):
    """Fine-tune training steps (BASELINE config 5): slices -> backbone in TRAIN mode (BatchNorm statistics per 16-slice chunk) -> MIL
    head -> focal loss -> backward -> clip -> Adam, all on the native FP32 kernels of csrc/train.cu; one process per GPU, bags
    sharded, gradients averaged with one NCCL all-reduce per flat buffer.  value = subjects (bags) per second, weak scaling."""
    import torch
    from pd_fusion_b200 import _lib
    from pd_fusion_b200.backbone import flops_per_image
    from pd_fusion_b200.models.mil_attention_finetune import MilAttentionFineTuneModel
    from pd_fusion_b200.parallel import barrier, init_distributed
    rank, local_rank, ws = init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    peaks = measured_peaks()
    bags_per_step, L = 4, sum(wl["counts"])
    params = {"backbone": wl["arch"], "pretrained": False, "target_shape": list(TARGET), "slice_axis": 2, "slice_count": L, "input_size": INPUT_SIZE,
              "slice_batch_size": 16, "batch_size": bags_per_step, "hidden_dim": 256, "attn_dim": 128, "dropout": 0.2, "gated": True,
              "loss_type": "focal", "focal_gamma": 2.0, "focal_alpha": 0.25, "lr": 3e-4, "lr_backbone": 1e-4, "weight_decay": 1e-3,
              "max_grad_norm": 1.0, "train_aug": False, "missing_prob": 0.5}
    torch.manual_seed(1234)
    model = MilAttentionFineTuneModel(params)
    precision = os.environ.get("PD_FUSION_B200_TRAIN_PRECISION", "bf16")      # training.ResNetTrainer reads the same variable
    rng = np.random.default_rng(100 + rank)
    host_bags = [rng.random((L, TARGET[0], TARGET[1])).astype(np.float32) for _ in range(bags_per_step)]
    dev_bags = [torch.from_numpy(b).to(dev) for b in host_bags]
    y = np.array([1.0, 0.0, 1.0, 0.0], dtype=np.float32)
    last = [None]                                      # what the last timed call returned

    def timed(fn, steps):
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last[0] = fn()
        e1.record()
        torch.cuda.synchronize(); barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if ws > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item())

    step_dev = lambda: model.train_step(dev_bags, y, frozen=False, clip=1.0)
    step_host = lambda: model.train_step(host_bags, y, frozen=False, clip=1.0)[0].item()     # loss read back: the step's result
    for _ in range(max(args.warmup, 3)):
        step_dev()
    torch.cuda.synchronize()
    steps = args.steps
    l0 = _lib.launch_count()
    with ClockSampler(local_rank) as clk:
        ms = timed(step_dev, steps)
    launches = _lib.launch_count() - l0
    if args.dump_outputs and rank == 0:            # before the host-fed steps below train the weights further
        loss, prob = last[0]
        rt, ht, _ = model._trainers()
        dump_outputs(args.dump_outputs, {"loss": loss.cpu().numpy(), "probs": prob.cpu().numpy(),
                                         "head_params": ht.flat_param.cpu().numpy(), "backbone_params": rt.flat_param.cpu().numpy()})
    step_host()
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host()
    torch.cuda.synchronize(); barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3
    flops = 3.0 * bags_per_step * L * flops_per_image(wl["arch"], INPUT_SIZE)              # forward + dgrad + wgrad
    tf = flops / (ms / steps / 1e3) / 1e12
    line = {"metric": "mri_subjects_per_sec_resnet2d_mil_finetune_fwd_bwd", "value": ws * bags_per_step * steps / (ms / 1e3), "unit": UNIT,
            "n_gpus": ws, "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "backbone": wl["arch"], "slices": L, "train_precision": precision, "bags_per_step_per_gpu": bags_per_step, "slice_batch_size": 16,
                       "input_size": INPUT_SIZE, "loss": "focal(2.0, 0.25)", "optimizer": "Adam 1e-4 / 3e-4, wd 1e-3, clip 1.0",
                       "l2": "activations of one step (~25 GB) exceed L2 many times over",
                       "parallelism": f"bags sharded x{ws}, one gradient all-reduce per flat buffer" if ws > 1 else "1 GPU"},
            "clocks": clk.summary(),
            "e2e": {"value": ws * bags_per_step * steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(sum(b.nbytes for b in host_bags)),
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor",
                         "kernel": ("whole training step: tcgen05 forward / data-gradient implicit GEMMs (conv_tc, conv_tc2) + wgrad_tc_kernel on bf16 "
                                    "operands, f32 BatchNorm / pooling / head / Adam kernels between them" if precision == "bf16" else
                                    "conv_f32 / conv_dgrad_f32 / conv_wgrad_f32 (CUDA-core FFMA implicit GEMMs: the FP32 parity path of training)"),
                         "achieved": tf, "peak": peaks["tf"], "unit": "TFLOP/s", "frac": tf / peaks["tf"], "traffic": None,
                         "flops_per_step": flops, "peak_source": peaks["src"] + " burst bf16 tensor peak; the numerator is the step's convolution "
                                                                               "FLOPs over the WHOLE step time"}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if ws > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--subjects", type=int, default=32, help="subjects per step per GPU")
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic volumes cycled by subject index")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-subjects", type=int, default=8, help="bounded CPU-baseline sample (subjects)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--overlap", action="store_true",
                    help="software-pipeline preprocessing of batch i+1 next to the convolutions of batch i on two streams (measured 2 %% SLOWER "
                         "than one stream since the conv stack is power-capped: profiles/r01_ab_overlap.txt)")
    ap.add_argument("--no-overlap", action="store_true", help="(default) one stream")
    ap.add_argument("--no-stored-e2e", action="store_true", help="skip the second end-to-end leg (int16 stored voxels decoded on the device)")
    ap.add_argument("--sustained-seconds", type=float, default=2.0, help="length of the sustained legs (0 = skip)")
    ap.add_argument("--no-heads", action="store_true", help="skip the fusion-head legs (ModDrop / MoE sweeps at N = 1e4, 1e6)")
    ap.add_argument("--mil-bags", type=int, default=2048, help="bags of the MIL roofline leg (c3)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 path; the reference arm keeps none")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)
    if args.workload == "c5":
        return run_c5(args, wl)

    import torch
    from pd_fusion_b200 import _lib
    from pd_fusion_b200.backbone import ResNet2D
    from pd_fusion_b200.parallel import all_gather_rows, barrier, init_distributed
    from pd_fusion_b200.pipeline import EmbeddingPipeline

    rank, local_rank, ws = init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, L = args.subjects, sum(wl["counts"])
    peaks = measured_peaks()

    torch.manual_seed(1234)
    sd = {k: v for k, v in ResNet2D(wl["arch"]).state_dict().items() if not k.startswith("fc.")}
    pipe = EmbeddingPipeline(sd, IN_SHAPE, TARGET, wl["axes"], wl["counts"], INPUT_SIZE, precision="bf16", max_subjects=B, device=dev)
    D = pipe.D

    pool = host_pool(args.pool)
    pinned = torch.empty((B,) + IN_SHAPE, dtype=torch.float32).pin_memory()
    for i in range(B):
        pinned[i].copy_(torch.from_numpy(pool[(rank * B + i) % len(pool)]))
    raw = pinned.to(dev, non_blocking=True)
    table = torch.empty((B, L, D) if args.workload == "c3" else (B, D), dtype=torch.float32, device=dev)
    host_out = torch.empty(table.shape, dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()

    overlap = args.overlap and not args.no_overlap
    fuse_stream = torch.cuda.Stream(dev)
    if overlap:
        pipe.enable_overlap()

    # --- the "fuse" half of the metric: the config's head evaluated under EVERY scenario mask of
    #     configs/eval_missingness_openneuro_ds001907.yaml in one masked-forward launch over the batch's embeddings
    #     (evaluation/evaluate.py:18-97 loops scenarios and subjects).  Masks are drawn on the host by the reference's
    #     rule (global numpy RNG), once; weights are random-init (seed 4321).
    import pandas as pd
    from pd_fusion_b200.data.missingness import scenario_mask_tensor
    from pd_fusion_b200.heads import MilHead, ModDropSweep
    scenarios = [{"name": "full_observation", "drop_modalities": []},
                 {"name": "mri_missing_25", "drop_modalities": ["mri"], "drop_rate": 0.25},
                 {"name": "mri_missing_50", "drop_modalities": ["mri"], "drop_rate": 0.50},
                 {"name": "mri_missing_75", "drop_modalities": ["mri"], "drop_rate": 0.75},
                 {"name": "mri_missing_100", "drop_modalities": ["mri"]},
                 {"name": "random_1_drop", "n_drop": 1, "type": "random"},
                 {"name": "random_2_drop", "n_drop": 2, "type": "random"}]
    mods = ["clinical", "datspect", "mri"]
    base = {"clinical": np.zeros(B, dtype=int), "datspect": np.zeros(B, dtype=int), "mri": np.ones(B, dtype=int)}   # openneuro_ds001907.py:77-81
    np.random.seed(11 + rank)
    mask_np, _ = scenario_mask_tensor(pd.DataFrame({"subject_id": np.arange(B)}), scenarios, base, mods)
    masks = torch.from_numpy(mask_np).to(dev)                                  # u8 [S, B, 3]
    S_scen = len(scenarios)
    torch.manual_seed(4321)
    if args.workload == "c2":
        from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet
        dims = {"clinical": 0, "datspect": 0, "mri": D}
        head = ModDropSweep(ModalityDropoutNet(dims, [256, 128, 64], 0.3).state_dict(), dims, device=dev)
    else:
        from pd_fusion_b200.models.mil_attention import MILAttentionNet
        head = MilHead(MILAttentionNet(D, 256, 128, 0.2, gated=True).state_dict(), True, 0.5, device=dev, precision="tf32")
        mri_col = masks[:, :, 2].contiguous()                  # [S, B] u8: the bag is present under scenario s
        full_len = torch.full((B,), L, dtype=torch.int32, device=dev)
        probs_sb = torch.empty((S_scen, B), dtype=torch.float32, device=dev)
    probs = torch.empty((B, S_scen), dtype=torch.float32, device=dev)

    def fuse(res, emb=None):
        """probabilities [B, S] of the batch under every scenario (emb: a stable copy of the embeddings to read instead of res)"""
        if args.workload == "c2":
            probs.copy_(head.forward(res.mean if emb is None else emb, masks).t())
        else:                                   # MIL: project + pool every bag ONCE, the scenario only selects missing_prob (pdf_mil_sweep)
            e = res.embeddings if emb is None else emb
            probs.copy_(head.sweep(e, full_len, mri_col, out=probs_sb).t())
        return probs

    def step_device():
        # The fusion head (a few small latency-bound launches) and the gathers run on a side stream, next to the preprocessing of
        # the following batch; they read `table`, this step's copy of the embeddings.
        cur = torch.cuda.current_stream()
        if not overlap:
            res = pipe.embed(raw)
            cur.wait_stream(fuse_stream)         # the previous step's head has finished reading `table` (long ago)
            table.copy_(res.embeddings if args.workload == "c3" else res.mean)
            fuse_stream.wait_stream(cur)
            with torch.cuda.stream(fuse_stream):
                pr = fuse(res, table)
                return (all_gather_rows(table, B * ws), all_gather_rows(pr, B * ws)) if ws > 1 else (table, pr)
        # --overlap: preprocessing of this batch additionally overlaps the convolutions of the previous one (two streams, two
        # encoder instances)
        res = pipe.embed_overlapped(raw)
        fuse_stream.wait_stream(pipe.conv_stream)
        with torch.cuda.stream(fuse_stream):
            table.copy_(res.embeddings if args.workload == "c3" else res.mean)
            pr = fuse(res)
            out = (all_gather_rows(table, B * ws), all_gather_rows(pr, B * ws)) if ws > 1 else (table, pr)
        pipe.hold_slot(fuse_stream)          # this batch's result slot may be reused only after the head has read it
        return out

    host_batches = [pinned] * args.steps

    def run_e2e():
        # public host API: pinned host volumes -> (H2D overlapped with the previous batch's kernels) -> hot path -> D2H
        outs = pipe.embed_host(host_batches, out_bags=(args.workload == "c3"), post=fuse)
        if ws > 1:
            all_gather_rows(outs[-1][0].to(dev), B * ws)
            all_gather_rows(outs[-1][1].to(dev), B * ws)
        return outs

    last = [None]                                      # what the last timed call returned

    def timed(fn, steps):
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if overlap:
            pipe.overlap_begin()
        fuse_stream.wait_stream(torch.cuda.current_stream())
        for _ in range(steps):
            last[0] = fn()
        if overlap:
            pipe.overlap_end()
        torch.cuda.current_stream().wait_stream(fuse_stream)
        e1.record()
        torch.cuda.synchronize(); barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if ws > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(args.warmup, 3)):
        step_device()
    torch.cuda.synchronize()
    launches0 = _lib.launch_count()
    with ClockSampler(local_rank) as clk:
        ms = timed(step_device, args.steps)
    launches = _lib.launch_count() - launches0
    value = ws * B * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:            # the legs below reuse these buffers
        emb, pr = last[0]
        dump_outputs(args.dump_outputs, {"embeddings": emb.cpu().numpy(), "scenario_probs": pr.cpu().numpy()})

    # --- per-kernel-family device time (same buffers, same launches): K2 conv stack and K1 preprocessing
    def enc_only():
        pipe.enc.forward(None)

    def pre_only():
        pipe.pre.run(raw, net_input=pipe._net_input)

    for _ in range(2):
        enc_only(); pre_only()
    ms_enc = timed(enc_only, args.steps) / args.steps
    ms_pre = timed(pre_only, args.steps) / args.steps
    flops = pipe.enc.algorithmic_flops()
    tf = flops / (ms_enc / 1e3) / 1e12
    gbs = pipe.algorithmic_bytes_per_subject() * B / (ms_pre / 1e3) / 1e9

    # --- sustained regime: >= `sustained_seconds` of back-to-back work, clocks sampled throughout.  A 10 k-subject job runs
    #     for seconds, not for the 0.1-0.5 s of the timed region above: the board settles at its power cap.
    sustained = None
    if args.sustained_seconds > 0:
        n_step = max(args.steps, int(np.ceil(args.sustained_seconds * 1e3 / max(ms / args.steps, 1e-3))))
        n_enc = max(args.steps, int(np.ceil(args.sustained_seconds * 1e3 / max(ms_enc, 1e-3))))
        with ClockSampler(local_rank) as clk_s:
            ms_s = timed(step_device, n_step)
        with ClockSampler(local_rank) as clk_c:
            ms_c = timed(enc_only, n_enc) / n_enc
        tf_s = flops / (ms_c / 1e3) / 1e12
        sustained = {"seconds": ms_s / 1e3, "steps": n_step, "value": ws * B * n_step / (ms_s / 1e3), "unit": UNIT,
                     "ms_per_step": ms_s / n_step, "clocks": clk_s.summary(),
                     "conv": {"achieved": tf_s, "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": tf_s / peaks["tf_sustained"],
                              "ms": ms_c, "launches_timed": n_enc, "seconds": ms_c * n_enc / 1e3, "clocks": clk_c.summary(),
                              "peak_source": peaks["src"] + " sustained bf16 (cuBLAS back to back for 4 s)"}}

    # --- preprocessing on volumes WITHOUT background (the synthetic brains are ~73 % exact zeros, which the resample and select
    #     kernels skip): same kernels, same algorithmic bytes
    pool_d = [dense_volume(i) for i in range(2)]
    raw_d = torch.empty_like(raw)
    for i in range(B):
        raw_d[i].copy_(torch.from_numpy(pool_d[i % 2]), non_blocking=False)

    def pre_dense():
        pipe.pre.run(raw_d, net_input=pipe._net_input)

    for _ in range(2):
        pre_dense()
    ms_pre_d = timed(pre_dense, args.steps) / args.steps
    gbs_d = pipe.algorithmic_bytes_per_subject() * B / (ms_pre_d / 1e3) / 1e9
    del raw_d

    # --- MIL head on a bag table larger than L2 (SURVEY.md 8d: 4*L*D + 4 bytes per bag): projection + attention (tcgen05
    #     kind::tf32 on the f32 bags) + softmax-pool + classifier ONCE, all scenarios selected on the device
    roofline_mil = None
    if args.workload == "c3" and args.mil_bags > 0:
        nb = args.mil_bags
        g = torch.Generator(device=dev).manual_seed(7)
        bag_tab = torch.randn((nb, L, D), generator=g, device=dev, dtype=torch.float32)
        lens_tab = torch.full((nb,), L, dtype=torch.int32, device=dev)
        live_tab = (torch.rand((S_scen, nb), generator=g, device=dev) < 0.6).to(torch.uint8)
        out_tab = torch.empty((S_scen, nb), dtype=torch.float32, device=dev)

        def mil_only():
            head.sweep(bag_tab, lens_tab, live_tab, out=out_tab)

        for _ in range(3):
            mil_only()
        l0 = _lib.launch_count()
        mil_only()
        mil_launches = _lib.launch_count() - l0
        ms_mil = timed(mil_only, max(args.steps, 10)) / max(args.steps, 10)
        b_mil = (4 * L * D + 4) * nb
        gbs_mil = b_mil / (ms_mil / 1e3) / 1e9
        roofline_mil = {"bound": "hbm", "kernel": "pdf_mil_sweep: gemm_tf32_kernel x2 (projection, attention scores) + mil_pool_kernel",
                        "achieved": gbs_mil, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs_mil / peaks["hbm"], "ms": ms_mil,
                        "bags": nb, "scenarios": S_scen, "launches": int(mil_launches), "bytes_per_bag": 4 * L * D + 4,
                        "table_bytes": int(bag_tab.numel() * 4), "peak_source": peaks["src"]}
        del bag_tab, out_tab

    # --- fusion heads (SURVEY.md 8d): every scenario in one call at N = 10 000 and 1 000 000 subjects
    heads = None
    if not args.no_heads and rank == 0:
        def timed_local(fn, steps):          # rank 0 only: NO collective inside (the other ranks are not here)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return float(e0.elapsed_time(e1))
        heads = heads_leg(dev, peaks, timed_local)
    barrier()

    run_e2e()                                            # warm-up (allocates the second device buffer)
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    run_e2e()
    torch.cuda.synchronize(); barrier()
    ms_e2e_t = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
    if ws > 1:
        torch.distributed.all_reduce(ms_e2e_t, op=torch.distributed.ReduceOp.MAX)
    ms_e2e = float(ms_e2e_t.item())
    e2e = ws * B * args.steps / (ms_e2e / 1e3)

    # --- the same end-to-end call fed the voxels AS AN int16 NIfTI STORES THEM (x fastest): half the PCIe bytes, decode
    #     (float64 scaling rule, cast, transpose) on the device -- SURVEY.md 8f rank 1.  Values are the pool volumes rounded to
    #     integers (NaN/Inf -> 0), so this is reported next to `e2e`, not instead of it.
    e2e_i16 = None
    if not args.no_stored_e2e:
        pinned_i16 = torch.empty((B, int(np.prod(IN_SHAPE))), dtype=torch.int16).pin_memory()
        for i in range(B):
            v = np.nan_to_num(pool[(rank * B + i) % len(pool)], nan=0.0, posinf=0.0, neginf=0.0)
            pinned_i16[i].copy_(torch.from_numpy(np.clip(np.round(v), -32768, 32767).astype(np.int16).reshape(-1, order="F")))
        stored_batches = [pinned_i16] * args.steps
        stored_desc = (4, 1, 1.0, 0.0)
        pipe.embed_host(stored_batches[:2], out_bags=(args.workload == "c3"), post=fuse, stored=stored_desc)
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        pipe.embed_host(stored_batches, out_bags=(args.workload == "c3"), post=fuse, stored=stored_desc)
        torch.cuda.synchronize(); barrier()
        t_i16 = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
        if ws > 1:
            torch.distributed.all_reduce(t_i16, op=torch.distributed.ReduceOp.MAX)
        e2e_i16 = {"value": ws * B * args.steps / (float(t_i16.item()) / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(pinned_i16.numel() * 2),
                   "d2h_bytes_per_step": int(host_out.numel() * 4 + B * S_scen * 4),
                   "h2d_gbs_per_gpu": pinned_i16.numel() * 2 / (float(t_i16.item()) / args.steps / 1e3) / 1e9,
                   "ms_per_step": float(t_i16.item()) / args.steps,
                   "overlap": "H2D of batch i+1 on a copy stream overlaps the kernels of batch i",
                   "timer": "host wall clock around K steps, device synchronised on both sides",
                   "input": "voxels as an int16 NIfTI stores them (Fortran order) in pinned host memory; float64 scaling rule, cast and "
                            "transpose on the device"}

    e2e_f32 = {"value": e2e, "unit": UNIT, "h2d_gbs_per_gpu": pinned.numel() * 4 / (ms_e2e / args.steps / 1e3) / 1e9,
               "h2d_bytes_per_step": int(pinned.numel() * 4), "d2h_bytes_per_step": int(host_out.numel() * 4 + B * S_scen * 4),
               "overlap": "H2D of batch i+1 on a copy stream overlaps the kernels of batch i",
               "timer": "host wall clock around K steps, device synchronised on both sides", "ms_per_step": ms_e2e / args.steps,
               "input": "float32 host arrays [256,256,176] in pinned memory (PCIe-bound: 46 MB per subject)"}
    traffic, traffic_src = conv_dram_traffic(args.workload, B)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ws, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl["name"], "backbone": wl["arch"], "slices": L, "subjects_per_step_per_gpu": B,
                   "volume": list(IN_SHAPE), "target": list(TARGET), "input_size": INPUT_SIZE, "volume_pool": args.pool,
                   "l2": "inputs larger than L2 (%.1f GB of volumes per step)" % (B * 4 * np.prod(IN_SHAPE) / 1e9),
                   "parallelism": f"subjects sharded x{ws}, all-gather of the embedding table" if ws > 1 else "1 GPU",
                   "fuse": ("Fusion-ModDrop 512-256-128-64-1" if args.workload == "c2" else "gated MIL attention 2048-256-128") +
                           f" under {S_scen} missingness scenarios, " + ("one launch" if args.workload == "c2" else "one pdf_mil_sweep call (tf32 tensor path)"),
                   "streams": ("preprocessing of batch i+1 overlaps the conv stack of batch i (2 streams); " if overlap else "preprocessing + conv stack on one stream; ") +
                              "fusion head and gathers on a side stream next to the following batch"},
        "clocks": clk.summary(),
        # the manifest's files hold int16 voxels: that leg is the end-to-end number; the float32-array leg is kept beside it
        "e2e": e2e_i16 if e2e_i16 is not None else e2e_f32,
        "e2e_float32_volumes": e2e_f32,
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "tcgen05 implicit-GEMM conv stack (stem_fused, conv3x3_c64, conv3x3_hs, conv_tc, conv_tc2, "
                                                  "conv_pw kernels: all launches of one step)",
                     "achieved": tf, "peak": peaks["tf"], "unit": "TFLOP/s", "frac": tf / peaks["tf"],
                     "traffic": traffic,
                     "traffic_source": traffic_src or "no ncu --set full capture of this configuration in profiles/conv_traffic.json",
                     "peak_source": peaks["src"] + " burst bf16 (numerator and denominator both from sub-second runs; the >= 2 s regime is "
                                                   "under `sustained`)",
                     "ms": ms_enc, "flops_per_step": flops},
        "sustained": sustained,
        "roofline_preproc": {"bound": "hbm", "kernel": "K1 resample/select/gather (all launches of one step)", "achieved": gbs,
                             "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"], "ms": ms_pre,
                             "bytes_per_subject": pipe.algorithmic_bytes_per_subject(), "peak_source": peaks["src"],
                             "input": "synthetic brains, ~73 % exact-zero background"},
        "roofline_preproc_dense": {"bound": "hbm", "achieved": gbs_d, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs_d / peaks["hbm"],
                                   "ms": ms_pre_d, "input": "Gamma(4,100) everywhere, no background"},
        "roofline_mil": roofline_mil,
        "heads": heads,
    }
    if rank == 0 and ws == 1 and not args.no_cpu_baseline:
        rate, cores, dt = cpu_reference_rate(wl, args.cpu_subjects, pool)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{args.cpu_subjects} subjects of the same workload in {dt:.1f} s (oracle port, torch fp32, all threads)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if ws > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

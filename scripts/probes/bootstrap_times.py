"""GPU probe: the cost of the device bootstrap (pdf_bootstrap_metrics) against the host metrics it replaces.  S = 7 scenarios of
random probabilities rounded to 1e-3 (ties, as real sweeps have), N in {10^4, 10^6}, B in {100, 1000}.  Each shape is warmed up, then
the whole call is timed with CUDA events (median of `rounds`); one torch.profiler pass per shape splits the device time into the sort
and gather (CUB radix sort, boot_copy_keys_kernel, boot_gather_kernel) and bootstrap_metrics_kernel.  The rate is the sorted positions
the replicate kernel walks, S (B + 1) N, over its time.  compute_metrics (sklearn, host) is timed on 3 resamples at the same N for the
per-replicate host cost.  Prints the card's name and power limit beside the numbers.
usage: bootstrap_times.py [rounds]"""
import ctypes as C
import statistics
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[2] / "robust-multimodal-pd_b200"))
import numpy as np
import torch

from pd_fusion_b200 import _lib
from pd_fusion_b200.utils.metrics import compute_metrics

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
S = 7
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          timeout=30).stdout.strip().splitlines()[0]
except (OSError, subprocess.SubprocessError, IndexError):
    card = torch.cuda.get_device_name() + ", power limit unknown"
print(f"card: {card}")

lib = _lib.load()
dev = torch.device("cuda")
rng = np.random.default_rng(0)
for N in (10 ** 4, 10 ** 6):
    y = rng.integers(0, 2, N)
    p = np.round(rng.random((S, N)), 3)
    d_prob = torch.from_numpy(p).to(dev)
    d_label = torch.from_numpy(y.astype(np.uint8)).to(dev)
    ws = torch.empty(int(lib.pdf_bootstrap_metrics_workspace_bytes(S, N)), dtype=torch.uint8, device=dev)
    idx = rng.integers(0, N, (3, N))
    compute_metrics(y[idx[0]], p[0, idx[0]])
    t0 = time.perf_counter()
    for r in range(3):
        compute_metrics(y[idx[r]], p[0, idx[r]])
    host = (time.perf_counter() - t0) / 3
    for B in (100, 1000):
        out = torch.empty((S, B + 1, 6), dtype=torch.float64, device=dev)

        def call():
            _lib.check(lib.pdf_bootstrap_metrics(S, N, B, C.c_uint64(1), d_prob.data_ptr(), d_label.data_ptr(), None, ws.data_ptr(),
                                                 out.data_ptr(), _lib.stream_ptr()), "pdf_bootstrap_metrics")

        call()
        torch.cuda.synchronize()
        times = []
        for _ in range(rounds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            call()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b))
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        kern = other = 0.0
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA":
                if "bootstrap_metrics_kernel" in ev.key:
                    kern += ev.device_time_total
                else:
                    other += ev.device_time_total
        kern_ms, other_ms = kern / 1e3, other / 1e3
        rate = S * (B + 1) * N / (kern_ms / 1e3)
        print(f"S={S} N={N} B={B}: call {statistics.median(times):.3f} ms (median of {rounds}; min {min(times):.3f}), "
              f"sort+gather {other_ms:.3f} ms, bootstrap_metrics_kernel {kern_ms:.3f} ms = {rate / 1e9:.1f} G sorted positions/s; "
              f"host compute_metrics {host * 1e3:.1f} ms per replicate -> {host * B * S:.1f} s for S x B, "
              f"device {statistics.median(times) / (B * S) * 1e3:.2f} us per replicate")

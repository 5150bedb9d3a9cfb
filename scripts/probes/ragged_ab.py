"""GPU probe: embed_manifest on a manifest whose rows interleave four scanner geometries (stored type and scaling differ too)
against a uniform manifest of the same size.  Reports subjects/s of the whole builder call (file read, upload, decode,
preprocessing, encoder; one untimed call first) and torch.cuda.max_memory_allocated of the timed call.

  python scripts/probes/ragged_ab.py [--trees TREE ...] [--rounds R] [--subjects N]

Every tree (a checkout of this repository with its library built) runs in its own process, the trees alternating round by round,
on the same manifests.  Backbone: randomly initialised (no weight download), resnet18, 160^3 target, 24 axis-2 slices, 224 px."""
import argparse
import json
import os
import struct
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

GEOMETRIES = [((256, 256, 176), "int16", 1.0, 0.0), ((240, 256, 160), "float32", 1.0, 0.0),
              ((192, 256, 256), "int16", 0.5, 10.0), ((176, 240, 256), "uint8", 1.0, 0.0)]
CODES = {"uint8": 2, "int16": 4, "float32": 16}


def _write_nifti(path, vol, slope, inter):
    hdr = bytearray(352)
    struct.pack_into("<i", hdr, 0, 348)
    struct.pack_into("<8h", hdr, 40, 3, *vol.shape, 1, 1, 1, 1)
    struct.pack_into("<h", hdr, 70, CODES[vol.dtype.name])
    struct.pack_into("<h", hdr, 72, vol.dtype.itemsize * 8)
    struct.pack_into("<f", hdr, 108, 352.0)
    struct.pack_into("<2f", hdr, 112, slope, inter)
    with open(path, "wb") as f:
        f.write(bytes(hdr) + vol.tobytes(order="F"))


def write_manifests(root: Path, n: int, src_root: Path):
    sys.path.insert(0, str(src_root))
    from pd_fusion_b200.synthetic import synthetic_volume
    rows = {"mixed": [], "uniform": []}
    for kind in rows:
        for i in range(n):
            shape, dtype, slope, inter = GEOMETRIES[i % 4 if kind == "mixed" else 0]
            v = np.nan_to_num(synthetic_volume(i % 8, shape, 1e-4), nan=0.0, posinf=0.0, neginf=0.0)
            v = np.clip(v * (200.0 / max(float(v.max()), 1e-6)), 0, 255) if dtype == "uint8" else v
            p = root / f"{kind}_{i:03d}.nii"
            _write_nifti(p, v.astype(dtype), slope, inter)
            rows[kind].append(f"sub-{i:03d},1,{i % 2},{p}")
    for kind, r in rows.items():
        (root / f"{kind}.csv").write_text("subject_id,session,label,t1wbrain_path\n" + "\n".join(r) + "\n")


def worker(tree: Path, manifest: Path):
    sys.path.insert(0, str(tree / "robust-multimodal-pd_b200"))
    import pandas as pd
    import torch
    from pd_fusion_b200.data import openneuro_features as F
    build = F._build_resnet_backbone
    F._build_resnet_backbone = lambda backbone, pretrained=True: build(backbone, pretrained=False)
    torch.manual_seed(0)
    df = pd.read_csv(manifest)
    kw = dict(backbone="resnet18", target_shape=(160, 160, 160), axes=[2], counts=[24], input_size=224)
    F.embed_manifest(df, **kw)                               # warm-up: modules, page cache, allocator
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    emb, _ = F.embed_manifest(df, **kw)                      # returns host arrays: ends in a device synchronise
    dt = time.perf_counter() - t0
    print(json.dumps({"subjects_per_s": len(df) / dt, "seconds": dt, "max_memory_allocated_gb": torch.cuda.max_memory_allocated() / 1e9,
                      "emb_checksum": float(np.abs(emb).sum())}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=[str(Path(__file__).resolve().parents[2])])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--subjects", type=int, default=64)
    ap.add_argument("--worker", nargs=2, metavar=("TREE", "MANIFEST"))
    a = ap.parse_args()
    if a.worker:
        worker(Path(a.worker[0]), Path(a.worker[1]))
        return
    with tempfile.TemporaryDirectory() as tmp:
        root = Path(tmp)
        write_manifests(root, a.subjects, Path(a.trees[0]).resolve() / "robust-multimodal-pd_b200")
        for r in range(a.rounds):
            for kind in ("mixed", "uniform"):
                for tree in a.trees:
                    out = subprocess.run([sys.executable, __file__, "--worker", str(Path(tree).resolve()), str(root / f"{kind}.csv")],
                                         capture_output=True, text=True, env=dict(os.environ))
                    line = out.stdout.strip().splitlines()[-1] if out.returncode == 0 and out.stdout.strip() else out.stderr[-2000:]
                    print(f"round {r} {kind:8s} {tree}: {line}", flush=True)


if __name__ == "__main__":
    main()

"""CLI of the `cnn3d` feature mode, drop-in for the reference's scripts/build_cnn3d_embeddings.py (same flags, same file names
`embeddings_<manifest-hash>_<config-hash>.parquet/.json`, same columns `mri_cnn_0.. , subject_id, session, label`): a 3-D conv
auto-encoder trained on the manifest's volumes with MSE + Adam, then the encoder's 128-d embedding of every volume.  Volumes are
decoded, resampled (scipy-exact) and standardised on the device and stay resident there; every training step runs on the native
kernels of pd_fusion_b200/cnn3d.py."""
import argparse
import json
from pathlib import Path

import _bootstrap  # noqa: F401  (puts the package on sys.path)
import numpy as np
import pandas as pd
import torch

from pd_fusion_b200 import _lib
from pd_fusion_b200.cnn3d import Simple3DAE, standardize_volumes, train_autoencoder
from pd_fusion_b200.data import openneuro_features as onf


def load_volumes(paths, target_shape, dev) -> torch.Tensor:
    """`load_volume` for every manifest row (scripts/build_cnn3d_embeddings.py:28-41) -> [S, D, H, W] f32 on the device."""
    out = []
    bsz = onf._subject_batch()
    reader = onf._ReadAhead(paths, 0, len(paths), window=2 * bsz)
    pre = onf._preprocessor(None, tuple(target_shape), max_batch=bsz)      # ragged: one batch mixes every raw geometry
    for i in range(0, len(paths), bsz):
        j = min(len(paths), i + bsz)
        batch = [reader.get(k) for k in range(i, j)]
        reader.release(i, j)
        zoomed = pre.resample(onf._decode_on_device(batch, dev))
        out.append(standardize_volumes(zoomed).clone())
    return torch.cat(out, dim=0)


def main():
    parser = argparse.ArgumentParser(description="Build CNN embeddings for ds001907")
    parser.add_argument("--manifest", type=str, required=True)
    parser.add_argument("--out-dir", type=str, default="data/processed/openneuro_ds001907/embeddings_cnn3d")
    parser.add_argument("--target-shape", type=int, nargs=3, default=[96, 96, 96])
    parser.add_argument("--embedding-dim", type=int, default=128)
    parser.add_argument("--epochs", type=int, default=10)
    parser.add_argument("--batch-size", type=int, default=4)
    parser.add_argument("--lr", type=float, default=1e-3)
    parser.add_argument("--seed", type=int, default=42)
    args = parser.parse_args()

    _lib.require_cuda()
    torch.manual_seed(args.seed)
    manifest_path, out_dir = Path(args.manifest), Path(args.out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    cfg = {"target_shape": args.target_shape, "embedding_dim": args.embedding_dim, "epochs": args.epochs, "batch_size": args.batch_size,
           "lr": args.lr}
    stem = f"embeddings_{onf._hash_file(manifest_path)}_{onf._hash_config(cfg)}"
    emb_path, meta_path = out_dir / f"{stem}.parquet", out_dir / f"{stem}.json"

    df = pd.read_csv(manifest_path)
    dev = torch.device("cuda", torch.cuda.current_device())
    model = Simple3DAE(input_shape=tuple(args.target_shape), embedding_dim=args.embedding_dim).to(dev)
    vols = load_volumes(df["t1wbrain_path"].tolist(), args.target_shape, dev)
    trainer = train_autoencoder(model, vols, args.epochs, args.batch_size, args.lr)

    emb = np.vstack([trainer.embed(vols[i:i + 1]).cpu().numpy().reshape(-1) for i in range(len(df))])
    emb_df = pd.DataFrame(emb, columns=[f"mri_cnn_{i}" for i in range(emb.shape[1])])
    emb_df["subject_id"] = df["subject_id"].values
    emb_df["session"] = df["session"].values
    emb_df["label"] = df["label"].values
    emb_df.to_parquet(emb_path, index=False)
    with open(meta_path, "w") as f:
        json.dump({"manifest": str(manifest_path), "config": cfg}, f, indent=2)
    print(f"Saved embeddings to {emb_path}")


if __name__ == "__main__":
    main()

"""Drop-in for `pd_fusion.data.openneuro_features` (reference: data/openneuro_features.py), hot-path part:
volume load + resample, intensity normalisation, slice selection, ResNet2D embedding builders and the
cache readers.  Same function names, arguments, return types, cache file names and on-disk formats;
the numerics run in libpdfusion_b200.so on the GPU, batched over subjects, and -- under torchrun -- sharded
over the GPUs of the box with an NCCL all-gather of the embedding table (rank 0 writes the cache).

Non-hashed runtime knobs (environment, so the cache key `sha256(str(sorted(cfg.items())))` is untouched):
  PD_FUSION_B200_PRECISION       bf16 (default, tcgen05 path) | fp32 (CUDA-core parity path)
  PD_FUSION_B200_SUBJECT_BATCH   subjects per device batch (default 8)
  PD_FUSION_B200_BACKBONE_WEIGHTS  path of a torchvision-layout state_dict to use instead of downloading
"""
from __future__ import annotations

import gzip
import hashlib
import os
import struct
from pathlib import Path
from typing import Dict, List, Sequence, Tuple

import numpy as np
import pandas as pd
import torch

from .. import _lib
from ..backbone import RESNET_SPECS, ResNet2D
from ..parallel import all_gather_rows, barrier, init_distributed, shard_range, world
from ..pipeline import EmbeddingPipeline
from ..preprocess import RaggedBatch, VolumePreprocessor, ragged_offsets
from ..utils.npz_writer import savez_compressed_parallel


def _hash_file(path: Path) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 20), b""):
            h.update(chunk)
    return h.hexdigest()[:12]


def _hash_config(cfg: Dict) -> str:
    return hashlib.sha256(str(sorted(cfg.items())).encode()).hexdigest()[:12]


# ---------------------------------------------------------------------------------------------------
# volume decode (host).  The reference delegates to nibabel (openneuro_features.py:23-25), which is not in
# this image; .npy and NIfTI-1 (.nii / .nii.gz) are decoded here.  SURVEY.md 8f rank 1 ("next" row).
# ---------------------------------------------------------------------------------------------------
_NIFTI_DTYPES = {2: "u1", 4: "i2", 8: "i4", 16: "f4", 64: "f8", 256: "i1", 512: "u2", 768: "u4", 1024: "i8", 1280: "u8"}


_NP_TO_NIFTI = {"uint8": 2, "int16": 4, "int32": 8, "float32": 16, "float64": 64, "int8": 256, "uint16": 512, "uint32": 768}


class StoredVolume:
    """Voxels as they are stored, plus what is needed to turn them into the reference's float32 array on the device
    (`pdf_decode_volumes`): NIfTI datatype code, [X, Y, Z], storage order, scl_slope / scl_inter."""
    __slots__ = ("voxels", "code", "shape", "fortran", "slope", "inter")

    def __init__(self, voxels, code, shape, fortran, slope=1.0, inter=0.0):
        self.voxels, self.code, self.shape, self.fortran, self.slope, self.inter = voxels, int(code), tuple(shape), bool(fortran), float(slope), float(inter)

    def to_float32(self) -> np.ndarray:
        """Host restatement of `get_fdata().astype(np.float32)` (C-order [X, Y, Z]); the batched path decodes on the device."""
        data = self.voxels.reshape(self.shape, order="F" if self.fortran else "C").astype(np.float64)
        if self.slope != 0 and np.isfinite(self.slope) and not (self.slope == 1.0 and self.inter == 0.0):
            data = data * self.slope + (self.inter if np.isfinite(self.inter) else 0.0)
        return np.ascontiguousarray(data.astype(np.float32))


def _read_nifti_stored(path: Path) -> StoredVolume:
    raw = gzip.open(path, "rb").read() if str(path).endswith(".gz") else Path(path).read_bytes()
    end = "<" if struct.unpack("<i", raw[:4])[0] == 348 else ">"
    if struct.unpack(end + "i", raw[:4])[0] != 348:
        raise ValueError(f"{path}: not a NIfTI-1 file")
    dim = struct.unpack(end + "8h", raw[40:56])
    datatype = struct.unpack(end + "h", raw[70:72])[0]
    vox_offset = int(struct.unpack(end + "f", raw[108:112])[0])
    slope, inter = struct.unpack(end + "2f", raw[112:120])
    if datatype not in _NIFTI_DTYPES:
        raise ValueError(f"{path}: unsupported NIfTI datatype {datatype}")
    shape = [int(d) for d in dim[1:1 + dim[0]]]
    while len(shape) > 3 and shape[-1] == 1:
        shape.pop()
    if len(shape) != 3:
        raise ValueError(f"{path}: expected a 3-D volume, got shape {shape}")
    arr = np.frombuffer(raw, dtype=np.dtype(end + _NIFTI_DTYPES[datatype]), count=int(np.prod(shape)), offset=vox_offset)
    if end == ">":
        arr = arr.astype(arr.dtype.newbyteorder("<"))             # the device kernel reads native (little-endian) voxels
    if datatype in (1024, 1280):                                   # 64-bit integers: no device decode, go through float64 on the host
        arr, datatype = arr.astype(np.float64), 64
    return StoredVolume(arr, datatype, shape, True, slope, inter)


def _read_volume_stored(path) -> StoredVolume:
    p = str(path)
    if p.endswith(".npy"):
        data = np.load(p)
        if data.dtype.name not in _NP_TO_NIFTI:
            data = data.astype(np.float32)
        return StoredVolume(np.ascontiguousarray(data).reshape(-1), _NP_TO_NIFTI[data.dtype.name], data.shape, False)
    return _read_nifti_stored(Path(p))


def _read_nifti(path: Path) -> np.ndarray:
    """float64 array as `get_fdata()` returns it (host path)."""
    v = _read_nifti_stored(path)
    data = v.voxels.reshape(v.shape, order="F").astype(np.float64)
    if v.slope != 0 and np.isfinite(v.slope) and not (v.slope == 1.0 and v.inter == 0.0):
        data = data * v.slope + (v.inter if np.isfinite(v.inter) else 0.0)
    return data


def _read_volume_host(path) -> np.ndarray:
    """Raw volume as C-contiguous float32 [X,Y,Z] (no scrub, no resample)."""
    p = str(path)
    data = np.load(p) if p.endswith(".npy") else _read_nifti(Path(p))
    return np.ascontiguousarray(data.astype(np.float32))


class _ReadAhead:
    """Volumes of manifest rows [lo, hi) read by a small thread pool, `window` rows ahead of the consumer (file I/O and zlib
    release the GIL; the reference reads serially through nibabel, `data/openneuro_features.py:23-27`).  get(j) returns row j's
    StoredVolume, blocking until it is there; release(i, j) drops rows [i, j) once they are on the device."""

    def __init__(self, paths, lo: int, hi: int, window: int):
        from concurrent.futures import ThreadPoolExecutor
        self.paths, self.hi, self.window = paths, hi, max(1, int(window))
        n_threads = max(1, int(os.environ.get("PD_FUSION_B200_IO_THREADS", "4")))
        self.pool = ThreadPoolExecutor(max_workers=n_threads, thread_name_prefix="pdf-read")
        self.futures: Dict[int, object] = {}
        self.next = lo

    def _fill(self, upto: int) -> None:
        while self.next < min(self.hi, upto):
            self.futures[self.next] = self.pool.submit(_read_volume_stored, self.paths[self.next])
            self.next += 1

    def get(self, j: int) -> "StoredVolume":
        self._fill(j + self.window)
        return self.futures[j].result()                  # a reader's exception (missing file, bad header) surfaces here

    def release(self, i: int, j: int) -> None:
        for k in range(i, j):
            self.futures.pop(k, None)
        if self.next >= self.hi and not self.futures:
            self.pool.shutdown(wait=False)


_DECODE_BUFS: Dict[torch.device, List[torch.Tensor]] = {}


def _decode_on_device(batch, dev) -> RaggedBatch:
    """StoredVolumes of any shapes, stored types, orders and scalings -> a RaggedBatch on `dev`.  One pinned upload carries the
    files' bytes, each volume at a 16-byte aligned offset (half of the float32 array for the usual int16 T1 image); one
    `pdf_decode_volumes` launch does the float64 scaling, the cast and the transpose of every subject.  The device buffers are
    reused by the next call on the current stream and grow only when a larger batch arrives: consume a batch before decoding the
    next one on another stream."""
    src_offs, n_src = [], 0
    for v in batch:
        src_offs.append(n_src)
        n_src += (v.voxels.nbytes + 15) // 16 * 16
    raw_offs, n_raw = ragged_offsets([v.shape for v in batch])
    descs = (_lib.VolumeDesc * len(batch))()
    host = torch.empty(n_src, dtype=torch.uint8, pin_memory=True)
    hb = host.numpy()
    for b, v in enumerate(batch):
        d = descs[b]
        d.shape[:] = list(v.shape)
        d.nifti_datatype, d.fortran_order, d.src_offset, d.raw_offset = v.code, int(v.fortran), src_offs[b], raw_offs[b]
        d.slope, d.inter = v.slope, v.inter
        hb[src_offs[b]:src_offs[b] + v.voxels.nbytes] = np.ascontiguousarray(v.voxels).reshape(-1).view(np.uint8)   # bytes as stored
    bufs = _DECODE_BUFS.get(dev)
    if bufs is None or bufs[0].numel() < n_src or bufs[1].numel() < n_raw:
        old = (0, 0) if bufs is None else (bufs[0].numel(), bufs[1].numel())
        bufs = _DECODE_BUFS[dev] = [torch.empty(max(old[0], n_src), dtype=torch.uint8, device=dev),
                                    torch.empty(max(old[1], n_raw), dtype=torch.float32, device=dev)]
    src, raw = bufs
    src[:n_src].copy_(host, non_blocking=True)
    _lib.check(_lib.load().pdf_decode_volumes(len(batch), descs, src.data_ptr(), raw.data_ptr(), _lib.stream_ptr()), "pdf_decode_volumes")
    return RaggedBatch(raw, descs)


# ---------------------------------------------------------------------------------------------------
# single-volume helpers with the reference's names (imported by CLI 2 and the fine-tune model)
# ---------------------------------------------------------------------------------------------------
_PRE_CACHE: Dict[tuple, VolumePreprocessor] = {}


def _preprocessor(in_shape, target_shape, axes=(2,), counts=(1,), input_size=8, mode=_lib.OUT_F32_NHWC3, max_batch: int = 1) -> VolumePreprocessor:
    key = (None if in_shape is None else tuple(in_shape), tuple(target_shape), tuple(axes), tuple(counts), int(input_size), mode, int(max_batch), torch.cuda.current_device())
    if key not in _PRE_CACHE:
        _PRE_CACHE[key] = VolumePreprocessor(in_shape, target_shape, axes, counts, input_size, out_mode=mode, max_batch=int(max_batch))
    return _PRE_CACHE[key]


def _load_volume(path: Path, target_shape=(96, 96, 96)):
    """decode -> float32 -> nan_to_num -> trilinear resample to `target_shape` (K1a on the device)."""
    raw = _read_volume_host(path)
    shape = tuple(target_shape) if target_shape is not None else raw.shape
    pre = _preprocessor(raw.shape, shape)
    return pre.resample(torch.from_numpy(raw[None]).to(pre.device))[0].cpu().numpy()


def _normalize_volume_for_resnet(volume: np.ndarray) -> np.ndarray:
    """p1/p99 clip + min-max of an already-resampled volume (K1b + normalise kernel)."""
    v = np.ascontiguousarray(volume, dtype=np.float32)
    pre = _preprocessor(v.shape, v.shape)                      # identity zoom: resample_kernel reproduces v bit for bit
    pre.resample(torch.from_numpy(v[None]).to(pre.device))
    pre.select(1)
    return pre.normalized_volume(1)[0].cpu().numpy()


def _select_slices(volume: np.ndarray, axis: int, slice_count: int) -> np.ndarray:
    """Slices [n,H,W] over the non-zero extent of an (already normalised) volume."""
    v = np.ascontiguousarray(volume, dtype=np.float32)
    pre = _preprocessor(v.shape, v.shape, (int(axis),), (int(slice_count),))
    idx, n = pre.select_raw(torch.from_numpy(v[None]).to(pre.device))
    idx = idx[0, : int(n[0, 0])].cpu().numpy()
    # the gather itself is a view operation on the caller's host array (the batched path gathers on the device)
    if axis == 0:
        return v[idx, :, :]
    if axis == 1:
        return v[:, idx, :].transpose(1, 0, 2)
    return v[:, :, idx].transpose(2, 0, 1)


def _build_resnet_backbone(backbone: str, pretrained: bool = True):
    """(nn.Module, emb_dim, weights) -- a torchvision-layout ResNet18/50 whose `fc` is Identity."""
    import torch.nn as nn
    arch = "resnet50" if backbone == "resnet50" else "resnet18"
    weights = None
    local = os.environ.get("PD_FUSION_B200_BACKBONE_WEIGHTS")
    if pretrained and not local:
        from torchvision.models import ResNet18_Weights, ResNet50_Weights, resnet18, resnet50
        weights = ResNet50_Weights.DEFAULT if arch == "resnet50" else ResNet18_Weights.DEFAULT
        model = (resnet50 if arch == "resnet50" else resnet18)(weights=weights)   # needs the torchvision cache / network
    else:
        model = ResNet2D(arch)
        if local:
            model.load_state_dict(torch.load(local, map_location="cpu", weights_only=True), strict=False)
    emb_dim = model.fc.in_features
    model.fc = nn.Identity()
    return model, emb_dim, weights


def _apply_affine_2d(slice_2d: np.ndarray, angle_deg: float, translate: np.ndarray) -> np.ndarray:
    """Rotation about the slice centre + translation, bilinear, zero outside (reference: openneuro_features.py:166-178;
    scipy.ndimage.affine_transform order 1, mode "constant") -- `pdf_tta_augment` with affine_only on the device."""
    from .tta import TtaDraw, affine_matrix, params_bytes
    img = np.ascontiguousarray(slice_2d, dtype=np.float32)
    rot, offset = affine_matrix(img.shape, angle_deg, np.asarray(translate, dtype=np.float64))
    pre = _preprocessor((8, 8, 8), (8, 8, 8))           # any instance: only its library handle and device are used
    dev = pre.device
    params = torch.from_numpy(params_bytes([TtaDraw(rot, offset, 1.0, 0.0, None)])).to(dev)
    out = pre.tta_augment(torch.from_numpy(img[None, None]).to(dev), params, None, affine_only=True)
    return out[0, 0].cpu().numpy().astype(slice_2d.dtype, copy=False)


# ---------------------------------------------------------------------------------------------------
# batched builders
# ---------------------------------------------------------------------------------------------------
def _subject_batch() -> int:
    """PD_FUSION_B200_SUBJECT_BATCH, capped at the largest ragged batch the library takes in one call"""
    return min(max(1, int(os.environ.get("PD_FUSION_B200_SUBJECT_BATCH", "8"))), _lib.PDF_RAGGED_MAX_BATCH)


def _mean_std(weights) -> Tuple[List[float], List[float]]:
    if hasattr(weights, "meta"):
        return list(weights.meta.get("mean", [0.5, 0.5, 0.5])), list(weights.meta.get("std", [0.5, 0.5, 0.5]))
    return [0.5, 0.5, 0.5], [0.5, 0.5, 0.5]


def embed_manifest(df: pd.DataFrame, backbone: str, target_shape: Sequence[int], axes: Sequence[int], counts: Sequence[int],
                   input_size: int, tta: int = 1, tta_cfg: Dict | None = None, tta_seeds: Sequence[int] | None = None
                   ) -> Tuple[np.ndarray, np.ndarray]:
    """Per-slice embeddings [S, L, D] f32 and slice-mean embeddings [S, D] f32 for every manifest row, in row order.
    Subjects are processed in device batches; under torchrun each rank embeds its contiguous shard of rows and the
    table is assembled with an all-gather."""
    from .tta import subject_seed, tta_config
    tta = int(tta)
    tta_cfg = tta_config(tta_cfg or {})
    if tta > 1 and tta_seeds is None:                   # the reference's per-subject Generator seed (process-salted hash)
        ids = df["subject_id"].tolist() if "subject_id" in df.columns else [""] * len(df)
        tta_seeds = [subject_seed(s) for s in ids]
    # a library caller under torchrun gets the same sharding as the CLIs: the process group is created here when the
    # environment says WORLD_SIZE > 1 (all_gather_rows would otherwise silently return the local shard)
    rank, local_rank, ws = init_distributed()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    precision = os.environ.get("PD_FUSION_B200_PRECISION", "bf16")
    bsz = _subject_batch()
    model, emb_dim, weights = _build_resnet_backbone(backbone)
    mean, std = _mean_std(weights)
    sd = {k: v for k, v in model.state_dict().items() if not k.startswith("fc.")}
    L = int(sum(counts))
    n_rows = len(df)
    lo, hi = shard_range(n_rows, rank, ws)
    emb = torch.zeros((hi - lo, L, emb_dim), dtype=torch.float32, device=dev)
    avg = torch.zeros((hi - lo, emb_dim), dtype=torch.float32, device=dev)
    nsl = torch.zeros((hi - lo,), dtype=torch.int32, device=dev)
    # one pipeline (one encoder) serves every raw shape: a batch is the next bsz rows, whatever their geometry and stored type
    pipe = EmbeddingPipeline(sd, None, target_shape, axes, counts, input_size, precision, bsz, mean, std,
                             "resnet50" if backbone == "resnet50" else "resnet18", dev)
    paths = df["t1wbrain_path"].tolist()
    reader = _ReadAhead(paths, lo, hi, window=2 * bsz)     # files are read and gunzipped by worker threads, ahead of the GPU
    for i in range(lo, hi, bsz):
        j = min(hi, i + bsz)
        batch = [reader.get(k) for k in range(i, j)]
        reader.release(i, j)
        raw = _decode_on_device(batch, dev)
        if tta > 1:
            res = pipe.embed_tta(raw, [tta_seeds[k] for k in range(i, j)], tta, tta_cfg)
        else:
            res = pipe.embed(raw)
        emb[i - lo:j - lo].copy_(res.embeddings)
        avg[i - lo:j - lo].copy_(res.mean)
        nsl[i - lo:j - lo].copy_(res.nslices.sum(dim=1))
    if ws > 1:
        emb, avg, nsl = all_gather_rows(emb, n_rows), all_gather_rows(avg, n_rows), all_gather_rows(nsl, n_rows)
    torch.cuda.synchronize()
    if emb.shape[0] != n_rows or avg.shape[0] != n_rows:
        raise RuntimeError(f"embedding table has {emb.shape[0]} rows for {n_rows} manifest rows (rank {rank} of {ws}): "
                           "the shards were not gathered")
    nsl_h = nsl.cpu().numpy()
    if (nsl_h != L).any():
        bad = int(np.argmax(nsl_h != L))
        # the reference's MIL builder raises in np.stack when bags differ in length (SURVEY.md Appendix C.4); the mean
        # builder tolerates it.  Keep the information for the callers.
        embed_manifest.short_bags = (bad, int(nsl_h[bad]))
    else:
        embed_manifest.short_bags = None
    return emb.cpu().numpy(), avg.cpu().numpy()


embed_manifest.short_bags = None


def build_resnet2d_embeddings(manifest_path: Path, cache_dir: Path, config: Dict) -> pd.DataFrame:
    """Slice-mean ResNet2D embeddings, cached as resnet2d_<manifest-hash>_<config-hash>.parquet
    (reference: openneuro_features.py:180-278)."""
    cache_dir = Path(cache_dir)
    cache_dir.mkdir(parents=True, exist_ok=True)
    out_path = cache_dir / f"resnet2d_{_hash_file(manifest_path)}_{_hash_config(config)}.parquet"
    if out_path.exists():
        return pd.read_parquet(out_path)
    df = pd.read_csv(manifest_path)
    _, avg = embed_manifest(df, config.get("backbone", "resnet18"), tuple(config.get("target_shape", (160, 160, 160))),
                            [int(config.get("slice_axis", 2))], [int(config.get("slice_count", 24))],
                            int(config.get("input_size", 224)), int(config.get("tta", 1)), config)
    cols = {"subject_id": df["subject_id"].values, "session": df["session"].values, "label": df["label"].astype(int).values}
    emb64 = avg.astype(np.float64)                      # the reference stores python floats -> float64 columns
    cols.update({f"mri_resnet_{k}": emb64[:, k] for k in range(emb64.shape[1])})
    emb_df = pd.DataFrame(cols)
    if world()[0] == 0:                                 # written under a temporary name and renamed: a reader never sees half a file
        tmp = out_path.with_name(out_path.name + f".tmp{os.getpid()}")
        emb_df.to_parquet(tmp, index=False)
        os.replace(tmp, out_path)
    barrier()                                           # every rank returns only once the cache file exists
    return emb_df


def build_resnet2d_mil_embeddings(manifest_path: Path, out_dir: Path, cfg: Dict, axes: Sequence[int], counts: Sequence[int]) -> Path:
    """Per-slice (MIL bag) embeddings -> resnet2d_mil_<mh>_<ch>.npz with arrays embeddings/subject_id/session/label
    (reference: scripts/build_resnet2d_mil_embeddings.py:90-168, which always recomputes)."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    out_path = out_dir / f"resnet2d_mil_{_hash_file(manifest_path)}_{_hash_config(cfg)}.npz"
    df = pd.read_csv(manifest_path)
    emb, _ = embed_manifest(df, cfg["backbone"], tuple(cfg["target_shape"]), list(axes), list(counts), int(cfg["input_size"]),
                            int(cfg.get("tta", 1)), cfg)
    if embed_manifest.short_bags is not None:
        row, n = embed_manifest.short_bags
        raise ValueError(f"all input arrays must have the same shape: subject row {row} has {n} slices, expected {emb.shape[1]}")
    if world()[0] == 0:
        # same npz as np.savez_compressed (scripts/build_resnet2d_mil_embeddings.py:162-168), deflated by a thread pool
        tmp = out_path.with_name(out_path.name + f".tmp{os.getpid()}.npz")
        savez_compressed_parallel(tmp, embeddings=emb.astype(np.float32), subject_id=df["subject_id"].values,
                                  session=df["session"].values, label=df["label"].values)
        os.replace(tmp, out_path)
    barrier()
    return out_path


def load_resnet2d_embeddings(manifest_path: Path, cache_dir: Path, config: Dict) -> pd.DataFrame:
    cache_dir = Path(cache_dir)
    cache_dir.mkdir(parents=True, exist_ok=True)
    out_path = cache_dir / f"resnet2d_{_hash_file(manifest_path)}_{_hash_config(config)}.parquet"
    if not out_path.exists():
        raise FileNotFoundError(f"ResNet2D embeddings not found at {out_path}. Run scripts/build_resnet2d_embeddings.py to generate them.")
    return pd.read_parquet(out_path)


def load_resnet2d_mil_embeddings(manifest_path: Path, cache_dir: Path, config: Dict) -> pd.DataFrame:
    cache_dir = Path(cache_dir)
    cache_dir.mkdir(parents=True, exist_ok=True)
    out_path = cache_dir / f"resnet2d_mil_{_hash_file(manifest_path)}_{_hash_config(config)}.npz"
    if not out_path.exists():
        raise FileNotFoundError(f"ResNet2D MIL embeddings not found at {out_path}. Run scripts/build_resnet2d_mil_embeddings.py to generate them.")
    data = np.load(out_path, allow_pickle=True)
    df = pd.DataFrame({"subject_id": data["subject_id"], "session": data["session"], "label": data["label"]})
    df["mri_mil"] = list(data["embeddings"])
    return df


def load_cnn_embeddings(manifest_path: Path, cache_dir: Path, config: Dict) -> pd.DataFrame:
    """Reader of the `cnn3d` cache (reference: data/openneuro_features.py:106-119); its builder is scripts/build_cnn3d_embeddings.py
    (the 3-D conv auto-encoder on the native kernels of pd_fusion_b200/cnn3d.py)."""
    cache_dir = Path(cache_dir)
    cache_dir.mkdir(parents=True, exist_ok=True)
    out_path = cache_dir / f"embeddings_{_hash_file(manifest_path)}_{_hash_config(config)}.parquet"
    if not out_path.exists():
        raise FileNotFoundError(f"Embeddings not found at {out_path}. Run scripts/build_cnn3d_embeddings.py to generate them.")
    return pd.read_parquet(out_path)


def _simple_features_device(vols: torch.Tensor, hist_bins: int, grid_size: int, extra_stats: bool) -> np.ndarray:
    """`_compute_simple_features` for a batch of resampled volumes [B, T0, T1, T2] f32 resident on the device -> [B, F] f32.
    The statistics come from `pdf_simple_stats` (one block per subject: exact order statistics by radix select, np.histogram's
    bin rule, float64 moments); the grid means are a second scipy-exact trilinear zoom through K1a's resample kernel; the host
    only assembles the feature vector the way the reference does (data/openneuro_features.py:34-73)."""
    lib = _lib.load()
    B = int(vols.shape[0])
    shape = tuple(int(v) for v in vols.shape[1:])
    stride = int(lib.pdf_simple_stats_stride())
    out = torch.empty((B, stride), dtype=torch.float64, device=vols.device)
    _lib.check(lib.pdf_simple_stats(B, shape[0] * shape[1] * shape[2], int(hist_bins), vols.data_ptr(), out.data_ptr(), _lib.stream_ptr()),
               "pdf_simple_stats")
    grid = None
    if grid_size:
        pre = _preprocessor(shape, (int(grid_size),) * 3, max_batch=B)
        grid = pre.resample(vols).reshape(B, -1).cpu().numpy()
    st = out.cpu().numpy()
    feats = []
    for b in range(B):
        r = st[b]
        n = r[0]
        mean = np.float32(r[1] / n)
        std = np.float32(np.sqrt(r[4] / n))
        counts = r[16:16 + hist_bins]
        edges = r[16 + hist_bins:16 + 2 * hist_bins + 1].astype(np.float32)
        hist = counts / np.array(np.diff(edges), float) / counts.sum()          # np.histogram(density=True)
        f = [float(mean), float(std), float(np.float32(r[2])), float(np.float32(r[3])), float(np.float32(r[7])), float(np.float32(r[8])),
             float(np.float32(r[9]))]
        f.extend(hist.tolist())
        if grid is not None:
            f.extend(grid[b].tolist())
        if extra_stats:
            m2, m3, m4 = r[4] / n, r[5] / n, r[6] / n
            sk = float(np.nan_to_num(np.float32(m3 / m2 ** 1.5) if m2 > 0 else np.nan, nan=0.0))       # scipy.stats.skew (biased)
            kt = float(np.nan_to_num(np.float32(m4 / m2 ** 2 - 3.0) if m2 > 0 else np.nan, nan=0.0))    # scipy.stats.kurtosis (Fisher)
            h = hist + 1e-12
            f.extend([sk, kt, float(-(h * np.log(h)).sum())])
        feats.append(np.array(f, dtype=np.float32))
    return np.stack(feats)


def _compute_simple_features(volume: np.ndarray, hist_bins=10, grid_size=8, extra_stats: bool = False) -> np.ndarray:
    """Histogram / grid statistics of one resampled volume (reference: data/openneuro_features.py:34-73), computed on the device."""
    _lib.require_cuda()
    vol = torch.from_numpy(np.ascontiguousarray(volume, dtype=np.float32)).cuda()
    return _simple_features_device(vol[None], int(hist_bins), int(grid_size) if grid_size else 0, bool(extra_stats))[0]


def load_simple_features(manifest_path: Path, cache_dir: Path, config: Dict) -> pd.DataFrame:
    """The `simple` feature mode: `features_<mh>_<ch>.parquet` with columns subject_id, session, label, mri_feat_0.. (reference:
    data/openneuro_features.py:75-104, which loops `_load_volume` + `_compute_simple_features` per row on the CPU).  Here the rows go
    through the device in batches: stored voxels -> decode -> scipy-exact resample -> statistics -> grid zoom."""
    cache_dir = Path(cache_dir)
    cache_dir.mkdir(parents=True, exist_ok=True)
    out_path = cache_dir / f"features_{_hash_file(manifest_path)}_{_hash_config(config)}.parquet"
    if out_path.exists():
        return pd.read_parquet(out_path)
    _lib.require_cuda()
    df = pd.read_csv(manifest_path)
    hist_bins, grid_size = int(config.get("hist_bins", 10)), int(config.get("grid_size", 8))
    target_shape = tuple(int(v) for v in config.get("target_shape", (96, 96, 96)))
    extra_stats = bool(config.get("extra_stats", False))
    dev = torch.device("cuda", torch.cuda.current_device())
    bsz = _subject_batch()
    paths = df["t1wbrain_path"].tolist()
    reader = _ReadAhead(paths, 0, len(paths), window=2 * bsz)
    pre = _preprocessor(None, target_shape, max_batch=bsz)
    feats: List[np.ndarray] = []
    for i in range(0, len(paths), bsz):
        j = min(len(paths), i + bsz)
        batch = [reader.get(k) for k in range(i, j)]
        reader.release(i, j)
        zoomed = pre.resample(_decode_on_device(batch, dev))
        feats.append(_simple_features_device(zoomed, hist_bins, grid_size, extra_stats))
    F = np.concatenate(feats, axis=0).astype(np.float64)          # the reference stores python floats -> float64 columns
    cols = {"subject_id": df["subject_id"].values, "session": df["session"].values, "label": df["label"].astype(int).values}
    cols.update({f"mri_feat_{k}": F[:, k] for k in range(F.shape[1])})
    feat_df = pd.DataFrame(cols)
    tmp = out_path.with_name(out_path.name + f".tmp{os.getpid()}")
    feat_df.to_parquet(tmp, index=False)
    os.replace(tmp, out_path)
    return feat_df

"""Ragged batches on the device: subjects of different raw shapes, stored types, byte orders and scalings in one batch give,
bit for bit, what the per-shape (uniform) path gives each of them -- decode, resample + select + gather, the manifest builders
and the fine-tune model's path bags."""
import gzip
import math
import struct

import numpy as np
import pandas as pd
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from pd_fusion_b200 import _lib
from pd_fusion_b200.data import openneuro_features as F
from pd_fusion_b200.preprocess import RaggedBatch, VolumePreprocessor
from pd_fusion_b200.synthetic import synthetic_volume

CODES = {"uint8": 2, "int16": 4, "int32": 8, "float32": 16, "float64": 64, "int8": 256, "uint16": 512, "uint32": 768}


def _write_nifti(path, vol, code, slope, inter, big_endian=False):
    e = ">" if big_endian else "<"
    hdr = bytearray(352)
    struct.pack_into(e + "i", hdr, 0, 348)
    struct.pack_into(e + "8h", hdr, 40, 3, *vol.shape, 1, 1, 1, 1)
    struct.pack_into(e + "h", hdr, 70, code)
    struct.pack_into(e + "h", hdr, 72, vol.dtype.itemsize * 8)
    struct.pack_into(e + "f", hdr, 108, 352.0)
    struct.pack_into(e + "2f", hdr, 112, slope, inter)
    with gzip.open(path, "wb") as f:
        f.write(bytes(hdr) + vol.astype(vol.dtype.newbyteorder(e)).tobytes(order="F"))


def _stored(dtype, shape, rng):
    n = int(np.prod(shape))
    if dtype.startswith("float"):
        v = (rng.standard_normal(n) * 1e3).astype(dtype)
        v[::97], v[5::211] = np.nan, np.inf
    else:
        info = np.iinfo(dtype)
        v = rng.integers(info.min, info.max, size=n, dtype=np.int64 if dtype != "uint32" else np.uint64).astype(dtype)
    return v.reshape(shape)


def _same_bits(a, b):
    nan = np.isnan(b)                                   # NaN payloads are not part of the contract (nan_to_num zeroes them next)
    return np.array_equal(np.isnan(a), nan) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32))


def test_decode_mixed_types_orders_scalings_shapes(tmp_path):
    rng = np.random.default_rng(7)
    shapes = [(37, 21, 45), (16, 33, 8), (40, 36, 44)]
    paths = []
    for k, dtype in enumerate(sorted(CODES)):
        v = _stored(dtype, shapes[k % 3], rng)
        p = tmp_path / f"n{k}.nii.gz"                   # Fortran order; every other file scaled, some big-endian
        slope, inter = ((0.0123456789, -3.25) if k % 2 else (1.0, 0.0))
        _write_nifti(p, v, CODES[dtype], slope, inter, big_endian=k % 3 == 1)
        q = tmp_path / f"c{k}.npy"                      # C order, unscaled
        np.save(q, _stored(dtype, shapes[(k + 1) % 3], rng))
        paths += [p, q]
    rb = F._decode_on_device([F._read_volume_stored(p) for p in paths], torch.device("cuda", 0))
    torch.cuda.synchronize()
    assert len(rb) == 16
    for b, p in enumerate(paths):
        assert _same_bits(rb[b].cpu().numpy(), F._read_volume_host(p)), p.name


def _volumes():
    """Larger and smaller than the 32^3 target, Z % 4 != 0, odd sizes, no positive voxel, NaN / Inf voxels."""
    vols = [synthetic_volume(1, (40, 36, 44), 1e-4), synthetic_volume(2, (20, 24, 16), 1e-4),
            synthetic_volume(3, (33, 27, 30), 1e-4), -np.abs(synthetic_volume(4, (24, 28, 20), 0.0)),
            synthetic_volume(5, (36, 32, 40), 1e-4)]
    vols[4][3, 4, 5], vols[4][10, 11, 12], vols[4][20, 2, 7] = np.nan, np.inf, -np.inf
    return [np.ascontiguousarray(v, dtype=np.float32) for v in vols]


def _c_order(z, slice_major):
    return z.permute(0, 2, 3, 1).contiguous() if slice_major else z


@pytest.mark.parametrize("axes,counts,pick,expect_sm", [
    ((2,), (6,), [0, 1, 4], True),                # single-axis, every subject bulk-copy eligible: slice-major
    ((2,), (6,), [0, 1, 2, 3, 4], False),         # one Z % 4 != 0 subject: the whole batch is C-order
    ((0, 1, 2), (3, 4, 5), [0, 1, 2, 3, 4], False),
])
def test_ragged_preprocess_equals_uniform_runs(axes, counts, pick, expect_sm):
    vols = [_volumes()[i] for i in pick]
    target, S = (32, 32, 32), 40
    dev = torch.device("cuda", 0)
    pre = VolumePreprocessor(None, target, axes, counts, S, out_mode=_lib.OUT_BF16_C1, max_batch=len(vols), device=dev, slice_major=True)
    res = pre.run(RaggedBatch.from_volumes(vols, dev))
    assert res.slice_major == expect_sm
    got = [t.clone() for t in (_c_order(res.zoomed, res.slice_major), res.lohi, res.indices, res.nslices, res.net_input)]
    for b, v in enumerate(vols):
        uni = VolumePreprocessor(v.shape, target, axes, counts, S, out_mode=_lib.OUT_BF16_C1, max_batch=1, device=dev,
                                 slice_major=res.slice_major)
        r = uni.run(torch.from_numpy(v[None]).to(dev))
        ref = (_c_order(r.zoomed, r.slice_major), r.lohi, r.indices, r.nslices, r.net_input)
        for name, g, w in zip(("zoomed", "lohi", "indices", "nslices", "net_input"), got, ref):
            assert torch.equal(g[b].view(torch.int16 if g.dtype == torch.bfloat16 else g.dtype).cpu(),
                               w[0].view(torch.int16 if w.dtype == torch.bfloat16 else w.dtype).cpu()), (name, b, v.shape)
    # the stage-level entry points on the same workspace: C-order resample, then select
    pre.resample(RaggedBatch.from_volumes(vols, dev))
    lohi, idx, ns = pre.select(len(vols))
    assert torch.equal(lohi.view(torch.int32), got[1].view(torch.int32)) and torch.equal(idx, got[2]) and torch.equal(ns, got[3])
    assert torch.equal(pre.zoomed[:len(vols)].view(torch.int32), got[0].view(torch.int32))


@pytest.fixture()
def seeded_backbone(monkeypatch):
    from pd_fusion_b200.backbone import ResNet2D

    def _bb(backbone, pretrained=True):
        torch.manual_seed(1234)
        m = ResNet2D("resnet50" if backbone == "resnet50" else "resnet18")
        dim = m.fc.in_features
        m.fc = torch.nn.Identity()
        return m, dim, None
    monkeypatch.setattr(F, "_build_resnet_backbone", _bb)


def _manifest(tmp_path, n=11):
    """Rows interleaving three shapes, int16 / float32 storage, two scalings."""
    shapes = [(40, 36, 44), (33, 27, 30), (24, 28, 20)]
    rows = []
    for i in range(n):
        v = synthetic_volume(40 + i, shapes[i % 3], 0.0)
        if i % 2:
            p = tmp_path / f"s{i}.nii.gz"
            _write_nifti(p, np.round(v).astype(np.int16), 4, 0.5 if i % 4 == 1 else 1.0, 2.0 if i % 4 == 1 else 0.0)
        else:
            p = tmp_path / f"s{i}.npy"
            np.save(p, v.astype(np.float32))
        rows.append({"subject_id": f"sub-{i:02d}", "session": 1, "label": i % 2, "t1wbrain_path": str(p), "group": i % 3})
    return pd.DataFrame(rows)


@pytest.mark.parametrize("tta", [1, 2])
def test_embed_manifest_mixed_equals_per_shape_groups(tmp_path, seeded_backbone, monkeypatch, tta):
    from pd_fusion_b200 import backbone as BB
    df = _manifest(tmp_path)
    monkeypatch.setenv("PD_FUSION_B200_SUBJECT_BATCH", "4")
    built, passes = [], [0]
    real_pipe, real_fwd = F.EmbeddingPipeline, BB.ResNetEncoder.forward

    def counting_pipe(*a, **k):
        built.append(1)
        return real_pipe(*a, **k)

    def counting_fwd(self, *a, **k):
        passes[0] += 1
        return real_fwd(self, *a, **k)
    monkeypatch.setattr(F, "EmbeddingPipeline", counting_pipe)
    monkeypatch.setattr(BB.ResNetEncoder, "forward", counting_fwd)
    kw = dict(backbone="resnet18", target_shape=(32, 32, 32), axes=[2], counts=[4], input_size=64, tta=tta)
    seeds = list(range(100, 100 + len(df)))
    emb, avg = F.embed_manifest(df, tta_seeds=seeds if tta > 1 else None, **kw)
    assert len(built) == 1
    assert passes[0] == math.ceil(len(df) / 4) * tta
    for g in range(3):
        rows = np.where(df["group"].values == g)[0]
        eg, ag = F.embed_manifest(df.iloc[rows].reset_index(drop=True), tta_seeds=[seeds[r] for r in rows] if tta > 1 else None, **kw)
        assert np.array_equal(emb[rows], eg) and np.array_equal(avg[rows], ag), g


def test_simple_features_of_mixed_manifest(tmp_path):
    df = _manifest(tmp_path, n=7)
    man = tmp_path / "manifest.csv"
    df.to_csv(man, index=False)
    cfg = {"target_shape": (24, 24, 24), "hist_bins": 10, "grid_size": 4}
    out = F.load_simple_features(man, tmp_path / "cache", cfg)
    got = out[[c for c in out.columns if c.startswith("mri_feat_")]].to_numpy()
    for i, p in enumerate(df["t1wbrain_path"]):
        ref = F._compute_simple_features(F._load_volume(p, target_shape=(24, 24, 24)), 10, 4)
        assert np.array_equal(got[i], ref.astype(np.float64)), i


def _ft_model():
    from pd_fusion_b200.models.mil_attention_finetune import MilAttentionFineTuneModel
    torch.manual_seed(99)
    return MilAttentionFineTuneModel({"backbone": "resnet18", "pretrained": False, "target_shape": (32, 32, 32), "slice_axis": 2,
                                      "slice_count": 6, "input_size": 64, "train_aug": False, "batch_size": 4})


def test_finetune_path_bags_equal_slice_arrays(tmp_path):
    df = _manifest(tmp_path, n=5)
    paths = df["t1wbrain_path"].tolist()
    m = _ft_model()
    arrays = [m._bag_slices(p) for p in paths]
    p_paths, p_arrays = m.predict_proba(paths), m.predict_proba(arrays)
    assert np.array_equal(p_paths, p_arrays)
    # the slice stacks themselves -- all the path route changes -- are bit-identical
    for s, a in zip(m._device_stacks(paths), arrays):
        assert np.array_equal(s.cpu().numpy().view(np.uint32), np.ascontiguousarray(a).view(np.uint32))
    y = np.array([0, 1, 1, 0, 1], dtype=np.float32)
    ma, mb = _ft_model(), _ft_model()
    torch.manual_seed(5)                               # the same dropout masks for both steps
    np.random.seed(5)
    la, _ = ma.train_step(paths, y, frozen=False)
    torch.manual_seed(5)
    np.random.seed(5)
    lb, _ = mb.train_step(arrays, y, frozen=False)
    torch.cuda.synchronize()
    assert torch.allclose(la.float().cpu(), lb.float().cpu(), rtol=1e-5, atol=1e-7)
    # The training kernels accumulate gradients with atomicAdd in no fixed order, and Adam's first step moves every weight by
    # about lr * sign(gradient): where a gradient is near zero its sign can differ between two runs.  Two first steps from the
    # same weights therefore agree to 2 * lr per element, and no closer.
    for mod_a, mod_b, lr in ((ma.backbone, mb.backbone, 1e-4), (ma.attn, mb.attn, 3e-4)):
        for (na, pa), (nb, pb) in zip(mod_a.named_parameters(), mod_b.named_parameters()):
            assert na == nb and float((pa - pb).abs().max()) <= 2 * lr + 1e-6, na

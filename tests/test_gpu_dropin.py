"""Drop-in boundary on the GPU: the reference's entry points (CLI scripts, helper functions, model predict_proba,
evaluate_model) served by the CUDA path, checked against outputs the reference itself produced (tests/golden)."""
import hashlib
import json
import runpy
import sys
from pathlib import Path

import numpy as np
import pandas as pd
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O
import pd_fusion_b200.data.openneuro_features as of
from pd_fusion_b200.backbone import ResNet2D
from pd_fusion_b200.synthetic import synthetic_table, synthetic_volume, write_synthetic_manifest

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture()
def seeded_backbone(monkeypatch):
    """Same two patch points the oracle recipe applies to the reference (SURVEY.md Appendix B): random init, seed 1234."""
    def _bb(backbone, pretrained=True):
        torch.manual_seed(1234)
        m = ResNet2D("resnet50" if backbone == "resnet50" else "resnet18")
        dim = m.fc.in_features
        m.fc = torch.nn.Identity()
        return m, dim, None
    monkeypatch.setattr(of, "_build_resnet_backbone", _bb)


def _run_script(name, argv):
    old = sys.argv
    sys.argv = [name] + argv
    sys.path.insert(0, str(ROOT / "scripts"))
    try:
        runpy.run_path(str(ROOT / "scripts" / name), run_name="__main__")
    finally:
        sys.argv = old
        sys.path.remove(str(ROOT / "scripts"))


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 1e-2)])
def test_cli_scripts_match_reference_outputs(golden, tmp_path, seeded_backbone, monkeypatch, precision, tol):
    g = golden("scripts")
    monkeypatch.setenv("PD_FUSION_B200_PRECISION", precision)
    # The reference run kept its volumes in a temporary directory (`manifest_dir`) whose path the manifest records, and the
    # manifest's hash names the cache files.  The same volumes are written under tmp_path instead: the manifest must differ from
    # the reference's by that directory alone, and the file names by the manifest hash alone.  The reference's key rule (first
    # 12 hex digits of the sha256 of the manifest bytes) is applied to both manifests here, not taken from the code under test.
    vols = tmp_path / "vols"
    manifest = write_synthetic_manifest(vols, 3, shape=(48, 40, 36))
    ref_manifest = g["manifest_bytes"].tobytes()
    assert manifest.read_bytes() == ref_manifest.replace(str(g["manifest_dir"]).encode(), str(vols).encode())
    ref_key, key = (hashlib.sha256(m).hexdigest()[:12] for m in (ref_manifest, manifest.read_bytes()))

    def ref_files(tag):
        assert all(f"_{ref_key}_" in str(f) for f in g[f"{tag}/files"])
        return sorted(str(f).replace(f"_{ref_key}_", f"_{key}_") for f in g[f"{tag}/files"])

    def ref_meta(tag):
        meta = json.loads(str(g[f"{tag}/json"]))
        assert meta["manifest"] == str(Path(str(g["manifest_dir"])) / "manifest.csv")
        return dict(meta, manifest=str(manifest))
    # CLI 1
    out1 = tmp_path / "c2"
    _run_script("build_resnet2d_embeddings.py", ["--manifest", str(manifest), "--out-dir", str(out1)] + [str(a) for a in g["c2/argv"]])
    assert sorted(p.name for p in out1.iterdir()) == ref_files("c2")
    df = pd.read_parquet(next(out1.glob("*.parquet")))
    assert list(df.columns) == [str(c) for c in g["c2/columns"]] and [str(t) for t in df.dtypes] == [str(t) for t in g["c2/dtypes"]]
    emb = df[[c for c in df.columns if c.startswith("mri_resnet_")]].values
    rel = np.linalg.norm(emb - g["c2/emb"], axis=1) / np.linalg.norm(g["c2/emb"], axis=1)
    assert rel.max() < tol, rel
    assert json.loads(next(out1.glob("*.json")).read_text()) == ref_meta("c2")
    # second call returns the cached parquet
    again = of.build_resnet2d_embeddings(manifest, out1, json.loads(str(g["c2/json"]))["config"])
    assert again.equals(df)
    # CLI 2 (multi-axis MIL bags)
    out2 = tmp_path / "mil"
    _run_script("build_resnet2d_mil_embeddings.py", ["--manifest", str(manifest), "--out-dir", str(out2)] + [str(a) for a in g["mil/argv"]])
    assert sorted(p.name for p in out2.iterdir()) == ref_files("mil")
    meta = json.loads(next(out2.glob("*.json")).read_text())
    assert meta == ref_meta("mil")
    cfg = meta["config"]
    bags = of.load_resnet2d_mil_embeddings(manifest, out2, cfg)
    got = np.stack(bags["mri_mil"].tolist())
    assert got.shape == g["mil/emb"].shape and got.dtype == np.float32
    rel = np.linalg.norm(got - g["mil/emb"], axis=2) / np.linalg.norm(g["mil/emb"], axis=2)
    assert rel.max() < tol, rel
    assert [str(s) for s in bags["subject_id"]] == [str(s) for s in g["mil/subject_id"]]
    with pytest.raises(FileNotFoundError):
        of.load_resnet2d_embeddings(manifest, tmp_path / "nowhere", cfg)


def test_helper_functions_bit_exact(tmp_path):
    raw = synthetic_volume(0, (64, 48, 44), 1e-4)
    np.save(tmp_path / "v.npy", raw)
    vol = of._load_volume(tmp_path / "v.npy", target_shape=(40, 40, 40))
    ref = O.load_volume(raw, (40, 40, 40))
    assert vol.dtype == np.float32 and np.array_equal(vol.view(np.uint32), ref.view(np.uint32))
    norm = of._normalize_volume_for_resnet(vol)
    ref_norm = O.normalize_volume_for_resnet(ref)
    assert np.array_equal(norm.view(np.uint32), ref_norm.view(np.uint32))
    for axis, count in [(0, 6), (1, 5), (2, 7), (2, 100)]:
        assert np.array_equal(of._select_slices(norm, axis, count), O.select_slices(ref_norm, axis, count))
    with pytest.raises(ValueError):
        sys_argv = sys.argv
        sys.argv = ["x", "--manifest", "m.csv", "--slice-axes", "0", "1", "--slice-counts", "3"]
        sys.path.insert(0, str(ROOT / "scripts"))
        try:
            runpy.run_path(str(ROOT / "scripts" / "build_resnet2d_mil_embeddings.py"), run_name="__main__")
        finally:
            sys.argv = sys_argv
            sys.path.remove(str(ROOT / "scripts"))


def test_model_api_and_evaluate_sweep(golden):
    """predict_proba of the three heads + evaluate_model over the whole scenario list, one launch per model,
    metrics equal to the reference's (AUC to 3 decimals) after the same np.random.seed."""
    from pd_fusion_b200.data.preprocess import NaNRobustScaler
    from pd_fusion_b200.evaluation.evaluate import evaluate_model, predict_proba_for_scenario
    from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel
    from pd_fusion_b200.models.mil_attention import MilAttentionModel
    from pd_fusion_b200.models.moe import MoEModel
    g = golden("heads")
    dims = json.loads(str(g["table/dims"]))
    df, masks = synthetic_table(int(g["table/n"]), dims, seed=42, mask_seed=7)
    scen = json.loads(str(g["scenarios"]))
    cols = [c for m in O.MODALITIES for c in df.columns if c.startswith(m + "_")]
    # ---- ModDrop
    md = ModalityDropoutModel(dims, {"hidden_dims": [64, 32], "dropout": 0.2, "lr": 1e-3, "epochs": 1})
    md.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moddrop/sd/")})
    scaler = NaNRobustScaler().fit(df[cols].values)
    np.random.seed(11)
    res = evaluate_model(md, df, masks, (None, scaler, cols), scen)
    ref = json.loads(str(g["moddrop/metrics"]))
    for name in ref:
        assert round(res[name]["roc_auc"], 3) == round(ref[name]["roc_auc"], 3), name
        for k in ("pr_auc", "brier_score", "ece", "balanced_accuracy", "f1"):
            assert abs(res[name][k] - ref[name][k]) < 1e-4, (name, k)
    X = scaler.transform(df[cols].values)
    cur = {m: g["masks_seed11"][2][:, i] for i, m in enumerate(O.MODALITIES)}
    p = md.predict_proba(X, masks=cur)
    np.testing.assert_allclose(p, g["moddrop/probs"][2], atol=5e-6)
    assert p.dtype == np.float32 and p.shape == (len(df),)
    # ---- MoE
    mods = [str(m) for m in g["moe/mods"]]
    moe = MoEModel({m: dims[m] for m in mods}, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16], "lr": 1e-3, "epochs": 1})
    moe.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moe/sd/")})
    prep = {}
    for m in mods:
        cm = [c for c in df.columns if c.startswith(m + "_")]
        prep[m] = (None, NaNRobustScaler().fit(df[cm].values), cm)
    np.random.seed(12)
    res = evaluate_model(moe, df, {m: masks[m] for m in mods}, prep, scen)
    ref = json.loads(str(g["moe/metrics"]))
    for name in ref:
        assert round(res[name]["roc_auc"], 3) == round(ref[name]["roc_auc"], 3), name
    mk = g["moe/masks_seed12"][1]
    Xd = {m: torch.FloatTensor(prep[m][1].transform(df[prep[m][2]].values) * mk[:, i:i + 1]) for i, m in enumerate(mods)}
    p = moe.predict_proba(Xd, torch.FloatTensor(mk.astype(np.float32)))
    np.testing.assert_allclose(p, g["moe/probs"][1], atol=5e-6)
    # ---- MIL (bags with missing entries, masks dict, single-scenario helper)
    tag = "mil_gated"
    cfg = json.loads(str(g[f"{tag}/cfg"]))
    mil = MilAttentionModel(cfg["D"], {"hidden_dim": cfg["H"], "attn_dim": cfg["A"], "gated": True, "missing_prob": 0.5})
    mil.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith(f"{tag}/sd/")})
    none = g[f"{tag}/none"]
    bags = [None if none[i] else g[f"{tag}/bag{i}"] for i in range(len(none))]
    p = mil.predict_proba(bags, masks={"mri": g[f"{tag}/mask_mri"]})
    assert p.dtype == np.float64
    np.testing.assert_allclose(p, g[f"{tag}/prob"], atol=5e-6)
    dfm = pd.DataFrame({"diagnosis": [0, 1, 0, 1, 0, 1], "mri_mil": [b if b is not None else g[f"{tag}/bag4"] for b in bags]})
    y, pp = predict_proba_for_scenario(mil, dfm, {"clinical": np.zeros(6, int), "datspect": np.zeros(6, int), "mri": np.ones(6, int)},
                                       ("mil", "mri_mil"), {"name": "no_mri", "drop_modalities": ["mri"]})
    assert np.all(pp == 0.5) and len(y) == 6


@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 2e-3)])
def test_finetune_model_predict_proba_matches_reference(golden, tmp_path, seeded_backbone, monkeypatch, precision, tol):
    """a13, inference: volume paths / slice-array / None / masked bags through the native pipeline + one MIL launch,
    against probabilities the reference's MilAttentionFineTuneModel produced with the same weights."""
    from pd_fusion_b200.models.mil_attention_finetune import MilAttentionFineTuneModel
    g = golden("ft")
    monkeypatch.setenv("PD_FUSION_B200_PRECISION", precision)
    params = json.loads(str(g["params"]))
    manifest = write_synthetic_manifest(tmp_path / "vols", 3, shape=(48, 40, 36))
    paths = pd.read_csv(manifest)["t1wbrain_path"].tolist()
    m = MilAttentionFineTuneModel(params)
    m.attn.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("attn/")})
    m.invalidate()
    bags = [paths[0], paths[1], None, g["arr_bag"], paths[2]]
    prob = m.predict_proba(bags, masks={"mri": np.array([1, 1, 1, 1, 0])})
    assert prob.shape == (5,) and prob[2] == params["missing_prob"] and prob[4] == params["missing_prob"]
    assert np.abs(prob - g["prob"]).max() < tol, (prob, g["prob"])
    # save / load round trip keeps the reference's checkpoint layout
    m.save(tmp_path / "ft.pt")
    state = torch.load(tmp_path / "ft.pt", map_location="cpu", weights_only=True)
    assert set(state) == {"backbone", "attn"} and "layer1.0.conv1.weight" in state["backbone"]
    m2 = MilAttentionFineTuneModel.load(tmp_path / "ft.pt", params)
    assert np.abs(m2.predict_proba(bags[:2]) - prob[:2]).max() < 1e-6
    # one short training run changes the head and the native path picks the new weights up
    torch.manual_seed(0); np.random.seed(0)
    m.params.update(epochs=1, freeze_backbone_epochs=5, batch_size=2)
    m.train([paths[0], paths[1], g["arr_bag"]], np.array([1, 0, 1]))
    assert np.abs(m.predict_proba(bags[:2]) - prob[:2]).max() > 1e-6

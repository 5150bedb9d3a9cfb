"""Monte-Carlo dropout on the GPU (pdf_moddrop_mc, pdf_mil_mc, predict_uncertainty, evaluation.evaluate.uncertainty_model) against
tests/mc_oracle.py: the same ModalityDropoutNet / MILAttentionNet in float64 torch with the restated keep masks."""
import json

import numpy as np
import pandas as pd
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mc_oracle as MO  # noqa: E402
from oracle import oracle as O  # noqa: E402
from pd_fusion_b200.heads import MilHead, ModDropSweep  # noqa: E402
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet  # noqa: E402
from pd_fusion_b200.models.mil_attention import MILAttentionNet  # noqa: E402

S = 7
SEED = 0x1234_5678_9ABC


def _md(dims, hidden, seed, p=0.3):
    torch.manual_seed(seed)
    net = ModalityDropoutNet(dims, hidden, p).eval()
    return net, ModDropSweep(net.state_dict(), dims, device="cuda")


def _inputs(N, dims, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, sum(dims.values()))).astype(np.float32)
    masks = (rng.random((S, N, len(dims))) < 0.6).astype(np.uint8)
    masks[0] = 1
    return X, masks, [dims[m] for m in sorted(dims)]


def _check_stats(stats, samples):
    assert np.all(np.abs(stats - MO.stats(samples)) <= 1e-12)


DIMS = {"clinical": 7, "datspect": 0, "mri": 512}


@pytest.mark.parametrize("hidden,T,N", [([], 16, 300), ([32], 16, 300), ([256, 128, 64], 16, 300), ([256, 128, 64], 1, 300),
                                        ([64, 48, 33], 100, 64)])
def test_moddrop_samples_equal_oracle(hidden, T, N):
    net, sw = _md(DIMS, hidden, 11)
    X, masks, sizes = _inputs(N, DIMS, 5)
    stats, smp = sw.mc(torch.from_numpy(X).cuda(), torch.from_numpy(masks).cuda(), T, SEED, 0.3, samples=True)
    smp, stats = smp.cpu().numpy(), stats.cpu().numpy()
    ref = MO.moddrop_samples(net, X, masks, sizes, T, SEED, 0.3)
    assert np.abs(smp - ref).max() <= 5e-6
    _check_stats(stats, smp)
    if hidden and T > 1:
        assert (stats[..., 1] > 0).mean() > 0.5       # the dropout does something


@pytest.mark.parametrize("gated,H,A,lmax", [(True, 64, 32, 48), (False, 30, 12, 48), (True, 30, 12, 1), (False, 64, 32, 200),
                                            (True, 64, 20, 200)])
def test_mil_samples_equal_oracle(gated, H, A, lmax):
    rng = np.random.default_rng(lmax + H)
    n, D, T = 40, 48, 12
    torch.manual_seed(3)
    net = MILAttentionNet(D, H, A, 0.3, gated=gated).eval()
    head = MilHead(net.state_dict(), gated, 0.25, device="cuda")
    lens = rng.integers(1, lmax + 1, n).astype(np.int32)
    lens[::7] = 0                                         # missing bags
    bags = np.zeros((n, lmax, D), np.float32)
    for b in range(n):
        bags[b, :lens[b]] = rng.standard_normal((lens[b], D))
    live = (rng.random((3, n)) < 0.7).astype(np.uint8)
    live[1] = 0                                           # a dead scenario
    stats, smp = head.mc(torch.from_numpy(bags).cuda(), torch.from_numpy(lens).cuda(), torch.from_numpy(live).cuda(), 3, T, SEED, 0.3,
                         samples=True)
    smp, stats = smp.cpu().numpy(), stats.cpu().numpy()
    ref = MO.mil_samples(net, bags, lens, live, 0.25, T, SEED, 0.3)
    assert np.abs(smp - ref).max() <= 5e-6
    _check_stats(stats, smp)
    dead = (live == 0) | (lens[None, :] == 0)
    assert np.all(stats[dead][:, 0] == np.float32(0.25)) and np.all(stats[dead][:, [1, 4]] == 0)
    assert np.all(smp[dead] == np.float32(0.25))
    assert (stats[~dead][:, 1] > 0).all()


def test_p0_equals_sweep():
    net, sw = _md(DIMS, [256, 128, 64], 2, 0.0)
    for N in (300, 3000):                                 # S N below and above the sweep's tiled-kernel threshold
        X, masks, _ = _inputs(N, DIMS, N)
        Xd, md = torch.from_numpy(X).cuda(), torch.from_numpy(masks).cuda()
        stats = sw.mc(Xd, md, 8, 1, 0.0)[0].cpu().numpy()
        prob = sw.forward(Xd, md).cpu().numpy()
        assert np.abs(stats[..., 0] - prob).max() <= 1e-6
        assert np.all(stats[..., 1] == 0) and np.all(stats[..., 4] == 0)
    torch.manual_seed(1)
    mil = MILAttentionNet(64, 64, 32, 0.0, gated=True).eval()
    head = MilHead(mil.state_dict(), True, 0.5, device="cuda")
    rng = np.random.default_rng(0)
    bags = torch.from_numpy(rng.standard_normal((50, 70, 64)).astype(np.float32)).cuda()
    lens = torch.from_numpy(rng.integers(0, 71, 50).astype(np.int32)).cuda()
    live = torch.from_numpy((rng.random((4, 50)) < 0.6).astype(np.uint8)).cuda()
    stats = head.mc(bags, lens, live, 4, 5, 9, 0.0)[0].cpu().numpy()
    prob = head.sweep(bags, lens, live, 4).cpu().numpy()
    assert np.abs(stats[..., 0] - prob).max() <= 1e-6
    assert np.all(stats[..., 1] == 0) and np.all(stats[..., 4] == 0)


def test_statelessness():
    net, sw = _md(DIMS, [256, 128, 64], 4)
    X, masks, _ = _inputs(500, DIMS, 8)
    masks[3] = masks[5]
    Xd, md = torch.from_numpy(X).cuda(), torch.from_numpy(masks).cuda()
    a_st, a_sm = (t.cpu().numpy() for t in sw.mc(Xd, md, 16, SEED, 0.3, samples=True))
    b_st, b_sm = (t.cpu().numpy() for t in sw.mc(Xd, md, 16, SEED, 0.3, samples=True))
    assert np.array_equal(a_st, b_st) and np.array_equal(a_sm, b_sm)
    long_sm = sw.mc(Xd, md, 100, SEED, 0.3, samples=True)[1].cpu().numpy()
    assert np.array_equal(long_sm[..., :16], a_sm)
    sub = [5, 2]
    s_st, s_sm = (t.cpu().numpy() for t in sw.mc(Xd, md[sub].contiguous(), 16, SEED, 0.3, samples=True))
    assert np.array_equal(s_st, a_st[sub]) and np.array_equal(s_sm, a_sm[sub])
    assert np.array_equal(a_st[3], a_st[5]) and np.array_equal(a_sm[3], a_sm[5])
    assert not np.array_equal(sw.mc(Xd, md, 16, SEED + 1, 0.3, samples=True)[1].cpu().numpy(), a_sm)
    # MIL: the same properties, and a bag's samples do not depend on the scenario that keeps it
    torch.manual_seed(6)
    mil = MILAttentionNet(32, 64, 32, 0.3, gated=True).eval()
    head = MilHead(mil.state_dict(), True, 0.5, device="cuda")
    rng = np.random.default_rng(1)
    bags = torch.from_numpy(rng.standard_normal((60, 90, 32)).astype(np.float32)).cuda()
    lens = torch.from_numpy(rng.integers(1, 91, 60).astype(np.int32)).cuda()
    live = torch.from_numpy((rng.random((4, 60)) < 0.6).astype(np.uint8)).cuda()
    a_st, a_sm = (t.cpu().numpy() for t in head.mc(bags, lens, live, 4, 16, SEED, 0.3, samples=True))
    b_st, b_sm = (t.cpu().numpy() for t in head.mc(bags, lens, live, 4, 16, SEED, 0.3, samples=True))
    assert np.array_equal(a_st, b_st) and np.array_equal(a_sm, b_sm)
    long_sm = head.mc(bags, lens, live, 4, 40, SEED, 0.3, samples=True)[1].cpu().numpy()
    assert np.array_equal(long_sm[..., :16], a_sm)
    s_st = head.mc(bags, lens, live[[3, 0]].contiguous(), 2, 16, SEED, 0.3)[0].cpu().numpy()
    assert np.array_equal(s_st, a_st[[3, 0]])
    on = live.cpu().numpy().astype(bool)
    both = on[0] & on[2]
    assert np.array_equal(a_sm[0][both], a_sm[2][both])


def test_bad_arguments_on_device():
    net, sw = _md(DIMS, [32], 4)
    X, masks, _ = _inputs(20, DIMS, 8)
    Xd, md = torch.from_numpy(X).cuda(), torch.from_numpy(masks).cuda()
    from pd_fusion_b200 import _lib
    for kw in (dict(p=1.0), dict(p=-0.5), dict(n_samples=0), dict(n_samples=4097)):
        args = dict(n_samples=4, seed=0, p=0.2)
        args.update(kw)
        with pytest.raises(_lib.PdfusionError, match="rc=-1"):
            sw.mc(Xd, md, **args)


# ------------------------------------------------------------------ uncertainty_model

def _table(golden):
    from pd_fusion_b200.synthetic import synthetic_table
    g = golden("heads")
    dims = json.loads(str(g["table/dims"]))
    df, masks = synthetic_table(int(g["table/n"]), dims, seed=42, mask_seed=7)
    return g, dims, df, masks, json.loads(str(g["scenarios"]))


def _check_uncertainty(model, df, masks, prep, cfg, seed, tol):
    from pd_fusion_b200.data.schema import TARGET_COL
    from pd_fusion_b200.evaluation.evaluate import _sweep_probs, evaluate_model, uncertainty_model
    np.random.seed(seed)
    evaluate_model(model, df, masks, prep, cfg)
    after_eval = np.random.get_state()
    np.random.seed(seed)
    probs, _ = _sweep_probs(model, df, masks, prep, cfg["scenarios"])
    np.random.seed(seed)
    res = uncertainty_model(model, df, masks, prep, cfg, n_samples=8, seed=3)
    after = np.random.get_state()
    assert after_eval[0] == after[0] and np.array_equal(after_eval[1], after[1]) and after_eval[2:] == after[2:]
    y = df[TARGET_COL].values
    for s, sc in enumerate(cfg["scenarios"]):
        r = res[sc["name"]]
        assert set(r) == set(MO.STATS) | {"risk_coverage"}
        assert all(r[k].shape == (len(df),) and r[k].dtype == np.float64 for k in MO.STATS)
        if tol is not None:                                # a model without dropout: mean = evaluate_model's probability
            assert np.abs(r["mean"] - np.asarray(probs[s], dtype=np.float64)).max() <= tol
            assert np.all(r["std"] == 0) and np.all(r["mutual_info"] == 0)
        order = np.argsort(r["entropy"], kind="stable")
        err = ((r["mean"] >= 0.5).astype(int) != y.astype(int))[order]
        risk = np.cumsum(err) / np.arange(1, len(y) + 1)
        assert np.allclose(r["risk_coverage"]["risk"], risk, rtol=0, atol=1e-15)
        assert np.array_equal(r["risk_coverage"]["coverage"], np.arange(1, len(y) + 1) / len(y))
        assert r["risk_coverage"]["aurc"] == pytest.approx(float(np.mean(risk)), abs=1e-15)
    return res


def test_uncertainty_model(golden):
    from pd_fusion_b200.data.preprocess import NaNRobustScaler
    from pd_fusion_b200.evaluation.evaluate import uncertainty_model
    from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel
    from pd_fusion_b200.models.mil_attention import MilAttentionModel
    from pd_fusion_b200.models.moe import MoEModel
    g, dims, df, masks, scen = _table(golden)
    cols = [c for m in O.MODALITIES for c in df.columns if c.startswith(m + "_")]
    prep = (None, NaNRobustScaler().fit(df[cols].values), cols)
    sd = {k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moddrop/sd/")}
    md0 = ModalityDropoutModel(dims, {"hidden_dims": [64, 32], "dropout": 0.0, "lr": 1e-3, "epochs": 1})
    md0.model.load_state_dict(sd)
    _check_uncertainty(md0, df, masks, prep, scen, 11, 1e-6)
    md = ModalityDropoutModel(dims, {"hidden_dims": [64, 32], "dropout": 0.2, "lr": 1e-3, "epochs": 1})
    md.model.load_state_dict(sd)
    res = _check_uncertainty(md, df, masks, prep, scen, 11, None)
    assert any((res[sc["name"]]["std"] > 0).any() for sc in scen["scenarios"])
    # the model-level call for one scenario's masks equals that scenario's row of the sweep
    from pd_fusion_b200.data.preprocess import preprocess_features
    one = md.predict_uncertainty(preprocess_features(df, cols, None, prep[1])[0], None, n_samples=8, seed=3, return_samples=True)
    assert one["samples"].shape == (len(df), 8)
    _check_stats(np.stack([one[k] for k in MO.STATS], -1), one["samples"])

    # MIL: missing bags get exactly missing_prob
    rng = np.random.default_rng(5)
    n, D = 300, 16
    mcfg = {"scenarios": [{"name": "baseline", "drop_modalities": []}, {"name": "half", "drop_modalities": ["mri"], "drop_rate": 0.5}]}
    bags = [None if i % 5 == 0 else rng.standard_normal((int(rng.integers(1, 6)), D)).astype(np.float32) for i in range(n)]
    dfm = pd.DataFrame({"diagnosis": rng.integers(0, 2, n), "mri_mil": bags})
    mmask = {"clinical": np.ones(n, int), "datspect": np.ones(n, int), "mri": (rng.random(n) < 0.8).astype(int)}
    for p, tol in ((0.0, 1e-6), (0.3, None)):
        torch.manual_seed(2)
        mil = MilAttentionModel(D, {"hidden_dim": 8, "attn_dim": 4, "gated": True, "missing_prob": 0.5, "dropout": p})
        res = _check_uncertainty(mil, dfm, mmask, ("mil", "mri_mil"), mcfg, 21, tol)
        none = np.array([b is None for b in bags])
        assert np.all(res["baseline"]["mean"][none] == 0.5) and np.all(res["baseline"]["std"][none] == 0)

    mods = [str(m) for m in g["moe/mods"]]
    moe = MoEModel({m: dims[m] for m in mods}, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16], "lr": 1e-3, "epochs": 1})
    with pytest.raises(ValueError, match="ModalityDropoutModel and MilAttentionModel"):
        uncertainty_model(moe, df, {m: masks[m] for m in mods}, {m: (None, None, []) for m in mods}, scen)

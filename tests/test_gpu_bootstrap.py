"""The device bootstrap (pdf_bootstrap_metrics, utils.metrics.bootstrap_metrics, evaluation.evaluate.bootstrap_model) on the GPU:
point estimates against compute_metrics, every replicate against sklearn with sample_weight = the restated weights, exact AUC
rationals, units, determinism, and bootstrap_model against evaluate_model."""
import json

import numpy as np
import pandas as pd
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from bootstrap_oracle import bootstrap_weights, exact_auc, weighted_metrics  # noqa: E402
from oracle import oracle as O  # noqa: E402
from pd_fusion_b200.utils.metrics import METRIC_NAMES, bootstrap_metrics, compute_metrics  # noqa: E402

S = 7


def _probs(kind, S, N, rng):
    p = rng.random((S, N))
    if kind == "rounded":
        p = np.round(p, 2)
    elif kind == "tie":                          # one tie group of 40 % of N at exactly 0.5, longer than any tile
        p[:, : int(0.4 * N)] = 0.5
    return p


def _close(got, want, tol=1e-12):
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    ok = ~np.isnan(want)
    assert np.all(np.abs(got[ok] - want[ok]) <= tol), (got, want)


@pytest.mark.parametrize("N", [1, 2, 17, 1000, 100003, 10 ** 6])
@pytest.mark.parametrize("kind", ["continuous", "rounded", "tie", "one_class"])
def test_point_estimate_equals_compute_metrics(N, kind):
    rng = np.random.default_rng(N)
    y = rng.integers(0, 2, N)
    if kind == "one_class":
        y[:] = N % 2
    p = _probs(kind, S, N, rng)
    point, reps = bootstrap_metrics(y, p, n_boot=0)
    assert point.shape == (S, 6) and reps.shape == (S, 0, 6)
    for s in range(S) if N <= 100003 else (0, S - 1):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = np.array([compute_metrics(y, p[s])[k] for k in METRIC_NAMES])
        _close(point[s], want)
        a = exact_auc(y, p[s], np.ones(N, np.int64))
        assert (a is None and np.isnan(point[s, 0])) or point[s, 0] == a


@pytest.mark.parametrize("N", [5, 20, 1000, 100003])
def test_replicates_equal_weighted_sklearn(N):
    rng = np.random.default_rng(7 + N)
    y = rng.integers(0, 2, N)
    p = _probs("rounded" if N > 20 else "continuous", 3, N, rng)
    if N == 100003:
        p[1, : N // 3] = 0.5
    B, seed = 64, 99
    point, reps = bootstrap_metrics(y, p, n_boot=B, seed=seed)
    assert reps.shape == (3, B, 6)
    lost = 0
    for b in range(B):
        w = bootstrap_weights(seed, b, np.arange(N))
        lost += (w[y == 1].sum() == 0) + (w[y == 0].sum() == 0)
        for s in range(3):
            _close(reps[s, b], weighted_metrics(y, p[s], w))
            a = exact_auc(y, p[s], w)
            assert (a is None and np.isnan(reps[s, b, 0])) or reps[s, b, 0] == a
    if N == 5:
        assert lost > 0                          # replicates that lose a class are covered


def test_units_share_weights_and_groups():
    rng = np.random.default_rng(3)
    G, N = 300, 2000
    units = rng.integers(0, G, N)
    y = rng.integers(0, 2, N)
    p = np.round(rng.random((2, N)), 3)
    B, seed = 32, 5
    _, reps = bootstrap_metrics(y, p, n_boot=B, seed=seed, units=units)
    for b in range(B):
        w = bootstrap_weights(seed, b, np.arange(G))[units]
        for s in range(2):
            _close(reps[s, b], weighted_metrics(y, p[s], w))


def test_determinism_and_independence_of_B_and_S():
    rng = np.random.default_rng(11)
    N = 50000
    y = rng.integers(0, 2, N)
    p = _probs("rounded", S, N, rng)
    a = bootstrap_metrics(y, p, n_boot=1000, seed=3)
    b = bootstrap_metrics(y, p, n_boot=1000, seed=3)
    assert np.array_equal(a[0], b[0], equal_nan=True) and np.array_equal(a[1], b[1], equal_nan=True)
    small = bootstrap_metrics(y, p, n_boot=10, seed=3)
    assert np.array_equal(small[1], a[1][:, :10], equal_nan=True)
    one = bootstrap_metrics(y, p[4], n_boot=1000, seed=3)
    assert np.array_equal(one[1][0], a[1][4], equal_nan=True) and np.array_equal(one[0][0], a[0][4], equal_nan=True)
    two = bootstrap_metrics(y, np.stack([p[2], p[2]]), n_boot=100, seed=3)
    assert np.array_equal(two[1][0] - two[1][1], np.zeros((100, 6)))


def test_input_validation():
    y = np.array([0, 1, 1])
    for bad in (np.array([0.1, np.nan, 0.3]), np.array([0.1, 1.2, 0.3]), np.array([-0.1, 0.2, 0.3]), np.array([0.1, np.inf, 0.3])):
        with pytest.raises(ValueError, match="probabilities"):
            bootstrap_metrics(y, bad)
    with pytest.raises(ValueError, match="y_true"):
        bootstrap_metrics(np.array([0, 2, 1]), np.array([0.1, 0.2, 0.3]))
    with pytest.raises(ValueError, match="units"):
        bootstrap_metrics(y, np.array([0.1, 0.2, 0.3]), units=np.array([0, -1, 2]))


# ------------------------------------------------------------------ bootstrap_model against evaluate_model

def _table(golden):
    g = golden("heads")
    dims = json.loads(str(g["table/dims"]))
    df, masks = O_table(int(g["table/n"]), dims)
    scen = json.loads(str(g["scenarios"]))
    return g, dims, df, masks, scen


def O_table(n, dims):
    from pd_fusion_b200.synthetic import synthetic_table
    return synthetic_table(n, dims, seed=42, mask_seed=7)


def _compare(res, boot, tol_ece=1e-12):
    for name, mets in res.items():
        for k, v in mets.items():
            got = boot[name][k]["value"]
            tol = tol_ece if k.endswith(("ece", "brier_score")) else 1e-12
            assert (np.isnan(v) and np.isnan(got)) or abs(got - v) <= tol, (name, k, got, v)
            assert boot[name][k]["lo"] <= boot[name][k]["hi"] or boot[name][k]["n_valid"] == 0


def _check_model(model, df, masks, prep, cfg, seed, tol_ece):
    from pd_fusion_b200.evaluation.evaluate import bootstrap_model, evaluate_model
    np.random.seed(seed)
    res = evaluate_model(model, df, masks, prep, cfg)
    after_eval = np.random.get_state()
    np.random.seed(seed)
    boot = bootstrap_model(model, df, masks, prep, cfg, n_boot=200, alpha=0.1, seed=4)
    after_boot = np.random.get_state()
    assert after_eval[0] == after_boot[0] and np.array_equal(after_eval[1], after_boot[1]) and after_eval[2:] == after_boot[2:]
    _compare(res, boot, tol_ece)
    names = [sc["name"] for sc in cfg["scenarios"]]
    assert "delta" not in boot[names[0]] and all("delta" in boot[n] for n in names[1:])
    for n in names[1:]:
        for k in boot[n]["delta"]:
            d = boot[n]["delta"][k]["value"]
            want = boot[n][k]["value"] - boot[names[0]][k]["value"]
            assert (np.isnan(d) and np.isnan(want)) or d == want
    return boot


def test_bootstrap_model_matches_evaluate_model(golden):
    from pd_fusion_b200.data.preprocess import NaNRobustScaler
    from pd_fusion_b200.evaluation.evaluate import bootstrap_model
    from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel
    from pd_fusion_b200.models.mil_attention import MilAttentionModel
    from pd_fusion_b200.models.moe import MoEModel
    g, dims, df, masks, scen = _table(golden)
    cols = [c for m in O.MODALITIES for c in df.columns if c.startswith(m + "_")]
    md = ModalityDropoutModel(dims, {"hidden_dims": [64, 32], "dropout": 0.2, "lr": 1e-3, "epochs": 1})
    md.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moddrop/sd/")})
    scaler = NaNRobustScaler().fit(df[cols].values)
    prep = (None, scaler, cols)
    # ModDrop returns float32: evaluate_model's ECE / Brier accumulate in float32 inside numpy
    _check_model(md, df, masks, prep, scen, 11, 2e-6)

    # two identical scenarios: every delta replicate is exactly 0
    same = {"scenarios": [{"name": "a", "drop_modalities": ["mri"]}, {"name": "b", "drop_modalities": ["mri"]}]}
    out = bootstrap_model(md, df, masks, prep, same, n_boot=50)
    assert all(out["b"]["delta"][k]["lo"] == 0 and out["b"]["delta"][k]["hi"] == 0 for k in METRIC_NAMES
               if out["b"]["delta"][k]["n_valid"])

    # with group_col: subject-level metrics under the same replicates; some rows without a group
    dfg = df.copy()
    subj = np.arange(len(df)) // 3
    dfg["subject"] = subj.astype(float)
    dfg.loc[dfg.index[::17], "subject"] = np.nan
    cfg = dict(scen, group_col="subject")
    boot = _check_model(md, dfg, masks, prep, cfg, 13, 2e-6)
    assert "subject_roc_auc" in boot[scen["scenarios"][0]["name"]]

    # wrapper without a sweep: the per-scenario fallback
    class Wrapper:
        def __init__(self, m):
            self.m = m

        def predict_proba(self, X, masks=None):
            return self.m.predict_proba(X, masks=masks)

    _check_model(Wrapper(md), df, masks, prep, scen, 15, 2e-6)

    mods = [str(m) for m in g["moe/mods"]]
    moe = MoEModel({m: dims[m] for m in mods}, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16], "lr": 1e-3, "epochs": 1})
    moe.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moe/sd/")})
    mprep = {}
    for m in mods:
        cm = [c for c in df.columns if c.startswith(m + "_")]
        mprep[m] = (None, NaNRobustScaler().fit(df[cm].values), cm)
    _check_model(moe, df, {m: masks[m] for m in mods}, mprep, scen, 12, 2e-6)

    # MIL: missing bags all get exactly missing_prob, one large tie group
    rng = np.random.default_rng(5)
    n, D = 400, 16
    mil = MilAttentionModel(D, {"hidden_dim": 8, "attn_dim": 4, "gated": True, "missing_prob": 0.5})
    bags = [None if i % 5 == 0 else rng.standard_normal((int(rng.integers(1, 6)), D)).astype(np.float32) for i in range(n)]
    dfm = pd.DataFrame({"diagnosis": rng.integers(0, 2, n), "mri_mil": bags})
    mmask = {"clinical": np.ones(n, int), "datspect": np.ones(n, int), "mri": (rng.random(n) < 0.8).astype(int)}
    mcfg = {"scenarios": [{"name": "baseline", "drop_modalities": []}, {"name": "half", "drop_modalities": ["mri"], "drop_rate": 0.5}]}
    _check_model(mil, dfm, mmask, ("mil", "mri_mil"), mcfg, 21, 1e-12)

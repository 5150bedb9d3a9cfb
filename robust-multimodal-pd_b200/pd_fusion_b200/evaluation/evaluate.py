"""The missingness sweep ("eval_missingness"; reference: evaluation/evaluate.py:11-138).

Same signatures and the same dispatch on the TYPE of `prep_info` (("mil", col) tuple -> MIL; dict -> MoE;
3-tuple -> matrix models).  What changes is the execution: every scenario's masks are drawn first (host, the
reference's RNG order), uploaded once as uint8 [S, N, M], and the model is evaluated under ALL of them in one
launch; tabular preprocessing runs once instead of once per scenario (evaluate.py:58,67).
Models that do not expose a sweep entry point (e.g. a CalibratedModel wrapper) fall back to the reference's
per-scenario `predict_proba` calls -- each of which still runs on the device.
`explain_model` explains a fusion head's predictions under the same scenario masks.
`bootstrap_model` adds bootstrap confidence intervals, and paired intervals of each scenario's difference to a reference scenario, to
`evaluate_model`'s metrics; the replicates are computed on the device (utils.metrics.bootstrap_metrics).
`uncertainty_model` estimates every subject's predictive uncertainty under every scenario by Monte-Carlo dropout on the device.
`ensemble_model` evaluates a deep ensemble (models.ensemble.HeadEnsemble): the mean's metrics, every member's, their spread across seeds
and the members' disagreement per subject.
"""
from __future__ import annotations

from typing import Dict, List, Tuple

import numpy as np
import pandas as pd

from ..data.feature_utils import apply_masks_to_matrix
from ..data.missingness import apply_missingness_scenario, get_modality_mask_matrix, scenario_mask_tensor
from ..data.preprocess import preprocess_features
from ..data.schema import MODALITIES, TARGET_COL
from ..utils.metrics import METRIC_NAMES, bootstrap_metrics, compute_metrics


def _kind(prep_info) -> str:
    if isinstance(prep_info, tuple) and len(prep_info) >= 2 and prep_info[0] == "mil":
        return "mil"
    return "moe" if isinstance(prep_info, dict) else "matrix"


def _fusion_inputs(df_test, mask_test, prep_info, scenarios: List[Dict]):
    """Preprocessed features (unmasked), uint8 scenario masks [S, N, M], the per-scenario mask dicts (drawn in scenario order) and
    the mask column order, for the "moe" and "matrix" kinds."""
    if _kind(prep_info) == "moe":
        mods = list(prep_info.keys())
        if mods != sorted(mods):
            # MoENet orders its experts by sorted(modality) while the reference's evaluate feeds the router in caller order
            # (evaluation/evaluate.py:54-63): an unsorted prep_info would silently pair router outputs with the wrong experts
            raise ValueError(f"MoE prep_info modalities must be in sorted order, got {mods}")
        masks, per = scenario_mask_tensor(df_test, scenarios, mask_test, mods)
        X = {m: preprocess_features(df_test, prep_info[m][2], prep_info[m][0], prep_info[m][1])[0] for m in mods}
        return X, masks, per, mods
    imputer, scaler, feature_cols = prep_info
    X, _, _ = preprocess_features(df_test, feature_cols, imputer, scaler)
    masks, per = scenario_mask_tensor(df_test, scenarios, mask_test, MODALITIES)
    return X, masks, per, MODALITIES


def _sweep_probs(model, df_test, mask_test, prep_info, scenarios: List[Dict]) -> Tuple[np.ndarray, List[Dict[str, np.ndarray]]]:
    """Probabilities [S, N] for all scenarios + the per-scenario mask dicts (drawn in scenario order)."""
    kind = _kind(prep_info)
    if kind == "mil":
        _, per = scenario_mask_tensor(df_test, scenarios, mask_test, list(mask_test.keys()))
        bags = df_test[prep_info[1]].tolist()
        if hasattr(model, "predict_proba_sweep") and all(b is None or isinstance(b, np.ndarray) for b in bags):
            # one upload, one projection, one pooling pass for ALL scenarios (pdf_mil_sweep): the scenario only decides where
            # missing_prob replaces the bag's probability
            n = len(bags)
            mri = np.stack([np.asarray(cur["mri"]) if "mri" in cur else np.ones(n, dtype=int) for cur in per])
            return model.predict_proba_sweep(bags, mri), per
        probs = []
        for cur in per:   # the bag tensor is padded once per call; a missing bag never reaches the device
            b = [bag if m == 1 else None for bag, m in zip(bags, cur["mri"])] if "mri" in cur else bags
            probs.append(model.predict_proba(b, masks=cur))
        return np.stack(probs), per
    if kind == "moe":
        X, masks, per, mods = _fusion_inputs(df_test, mask_test, prep_info, scenarios)
        if hasattr(model, "predict_proba_sweep"):
            return model.predict_proba_sweep(X, masks, mods), per
        import torch
        probs = []
        for s, cur in enumerate(per):
            Xd = {m: torch.FloatTensor(X[m] * cur[m].reshape(-1, 1) if m in cur else X[m]) for m in mods}
            probs.append(model.predict_proba(Xd, torch.FloatTensor(np.stack([cur[m] for m in mods], axis=1))))
        return np.stack(probs), per
    feature_cols = prep_info[2]
    X, masks, per, _ = _fusion_inputs(df_test, mask_test, prep_info, scenarios)
    if hasattr(model, "predict_proba_sweep") and not hasattr(model, "mask_dim"):
        return model.predict_proba_sweep(X, masks, MODALITIES), per
    probs = []
    for cur in per:
        Xm = apply_masks_to_matrix(X, cur, feature_cols)
        probs.append(model.predict_proba(Xm, masks=get_modality_mask_matrix(cur) if hasattr(model, "mask_dim") else cur))
    return np.stack(probs), per


def _with_groups(metrics: Dict, df_test, y_true, y_prob, group_col):
    if group_col and group_col in df_test.columns:
        t = pd.DataFrame({"group": df_test[group_col].values, "y_true": y_true, "y_prob": y_prob})
        g = compute_metrics(t.groupby("group")["y_true"].first().values, t.groupby("group")["y_prob"].mean().values)
        metrics.update({f"subject_{k}": v for k, v in g.items()})
    return metrics


def evaluate_model(model, df_test, mask_test, prep_info, config) -> Dict[str, Dict[str, float]]:
    scenarios = config.get("scenarios", [{"name": "baseline", "drop_modalities": []}])
    group_col = config.get("group_col")
    y_true = df_test[TARGET_COL].values
    probs, _ = _sweep_probs(model, df_test, mask_test, prep_info, scenarios)
    return {sc["name"]: _with_groups(compute_metrics(y_true, np.asarray(probs[s])), df_test, y_true, np.asarray(probs[s]), group_col)
            for s, sc in enumerate(scenarios)}


def _group_units(groups: np.ndarray) -> Tuple[np.ndarray, int]:
    """(unit id per row, G): the groups of _with_groups (groupby order, NaN keys dropped) are units 0..G-1, and each row whose key is
    NaN is a unit of its own, numbered after them."""
    ids = pd.DataFrame({"group": groups}).groupby("group").ngroup().to_numpy(dtype=np.float64, copy=True)
    G = int(np.nanmax(ids)) + 1 if np.any(~np.isnan(ids)) else 0
    lone = np.isnan(ids)
    ids[lone] = G + np.arange(int(lone.sum()))
    return ids.astype(np.int64), G


def _interval(value: float, reps: np.ndarray, alpha: float) -> Dict[str, float]:
    n = int(np.count_nonzero(~np.isnan(reps)))
    lo, hi = np.nanpercentile(reps, [100 * alpha / 2, 100 * (1 - alpha / 2)]) if n else (np.nan, np.nan)
    return {"value": float(value), "lo": float(lo), "hi": float(hi), "n_valid": n}


def summarize_bootstrap(names: List[str], keys: List[str], point: np.ndarray, reps: np.ndarray, alpha: float = 0.05,
                        ref: int = 0) -> Dict[str, Dict]:
    """{scenario: {metric: {"value", "lo", "hi", "n_valid"}, "delta": {...}}} from point [S, K] and replicates [S, B, K]: percentile
    intervals (np.nanpercentile, linear, at 100 alpha/2 and 100 (1 - alpha/2)) over the non-NaN replicates, and for every scenario but
    `ref` the paired difference point[s] - point[ref] with the interval of reps[s, b] - reps[ref, b]."""
    out = {}
    for s, name in enumerate(names):
        res = {k: _interval(point[s, j], reps[s, :, j], alpha) for j, k in enumerate(keys)}
        if s != ref:
            res["delta"] = {k: _interval(point[s, j] - point[ref, j], reps[s, :, j] - reps[ref, :, j], alpha) for j, k in enumerate(keys)}
        out[name] = res
    return out


def bootstrap_model(model, df_test, mask_test, prep_info, config, n_boot: int = 1000, alpha: float = 0.05, seed: int = 0,
                    reference=None) -> Dict[str, Dict]:
    """evaluate_model's metrics with Poisson-bootstrap confidence intervals, computed on the device (utils.metrics.bootstrap_metrics):
    {scenario: {metric: {"value", "lo", "hi", "n_valid"}, "subject_<metric>": ... (with config["group_col"]),
    "delta": {metric: {...}} (every scenario but the reference)}}.

    The probabilities come from the sweep exactly as in evaluate_model (same masks under the same numpy seed; nothing else draws from
    numpy's RNG), so each "value" is evaluate_model's metric.  "lo"/"hi" are the alpha/2 and 1 - alpha/2 percentiles of the n_boot
    replicates whose metric is defined ("n_valid" of them).  "delta" is the paired difference to the reference scenario (`reference`,
    a scenario name; default the first): the same replicate b in both, so it carries no between-scenario resampling noise.  With
    group_col the resampling unit is the group (rows without a group resample alone), and the subject_* metrics are computed on
    _with_groups' group rows under the same replicates."""
    if not 0 < alpha < 1:
        raise ValueError("alpha must lie in (0, 1)")
    scenarios = config.get("scenarios", [{"name": "baseline", "drop_modalities": []}])
    names = [sc["name"] for sc in scenarios]
    if reference is not None and reference not in names:
        raise ValueError(f"reference scenario {reference!r} is not one of {names}")
    ref = 0 if reference is None else names.index(reference)
    group_col = config.get("group_col")
    y_true = df_test[TARGET_COL].values
    probs, _ = _sweep_probs(model, df_test, mask_test, prep_info, scenarios)
    probs = [np.asarray(probs[s]) for s in range(len(scenarios))]
    keys = list(METRIC_NAMES)
    grouped = bool(group_col) and group_col in df_test.columns
    units = _group_units(df_test[group_col].values)[0] if grouped else None
    point, reps = bootstrap_metrics(y_true, np.stack([p.astype(np.float64) for p in probs]), n_boot, seed, units)
    if grouped:
        gy, gp = None, []
        for p in probs:        # _with_groups' group rows, from the same dtype it sees
            t = pd.DataFrame({"group": df_test[group_col].values, "y_true": y_true, "y_prob": p})
            gy = t.groupby("group")["y_true"].first().values
            gp.append(t.groupby("group")["y_prob"].mean().values.astype(np.float64))
        gpoint, greps = bootstrap_metrics(gy, np.stack(gp), n_boot, seed, np.arange(len(gy)))
        point, reps = np.concatenate([point, gpoint], axis=1), np.concatenate([reps, greps], axis=2)
        keys += [f"subject_{k}" for k in METRIC_NAMES]
    return summarize_bootstrap(names, keys, point, reps, alpha, ref)


def explain_model(model, df_test, mask_test, prep_info, config, steps: int = 32) -> Dict[str, Dict]:
    """{scenario name: explanation} of a fusion head (ModalityDropoutModel.explain / MoEModel.explain: probabilities, exact modality
    Shapley values, integrated gradients with `steps` midpoints) under every scenario of `config`, in one explain call for all of
    them.  The scenario masks are drawn as evaluate_model draws them (same helper, same RNG order), so with the same seed each
    scenario's "prob" is evaluate_model's probability."""
    if _kind(prep_info) == "mil":
        raise ValueError("explain_model explains the fusion heads (ModDrop, MoE); explain a MIL model with MilAttentionModel.explain "
                         "or MilAttentionFineTuneModel.explain")
    if not hasattr(model, "explain_sweep") or hasattr(model, "mask_dim"):
        raise ValueError(f"{type(model).__name__} has no fusion-head explanation: explain_model needs a ModalityDropoutModel or an "
                         "MoEModel (MIL models: MilAttentionModel.explain)")
    scenarios = config.get("scenarios", [{"name": "baseline", "drop_modalities": []}])
    X, masks, _, order = _fusion_inputs(df_test, mask_test, prep_info, scenarios)
    ex = model.explain_sweep(X, masks, order, steps)
    return {sc["name"]: ex[s] for s, sc in enumerate(scenarios)}


def _risk_coverage_by_entropy(y_true, mean, entropy) -> Dict:
    """subjects ranked by entropy ascending (stable): risk at coverage k/N = error rate of the first k predictions (mean >= 0.5),
    aurc = the mean risk"""
    order = np.argsort(entropy, kind="stable")
    err = ((np.asarray(mean) >= 0.5).astype(int) != np.asarray(y_true).astype(int)).astype(np.float64)[order]
    k = np.arange(1, len(err) + 1)
    risk = np.cumsum(err) / k
    return {"coverage": k / len(err), "risk": risk, "aurc": float(np.mean(risk))}


def uncertainty_model(model, df_test, mask_test, prep_info, config, n_samples: int = 32, seed: int = 0) -> Dict[str, Dict]:
    """Monte-Carlo dropout uncertainty of every test subject under every scenario of `config`, in one device call for all of them:
    {scenario: {"mean", "std", "entropy", "expected_entropy", "mutual_info": [N] float64, "risk_coverage": {"coverage", "risk",
    "aurc"}}}.  The scenario masks are drawn as evaluate_model draws them (same helper, same numpy RNG order, nothing else drawn), and
    the dropout masks come from a counter-based generator keyed by `seed`, so numpy's and torch's RNGs are left as evaluate_model
    leaves them.  risk_coverage ranks the subjects by entropy (most certain first) and gives the error rate of the prediction
    mean >= 0.5 among the first k, and its mean (aurc).  Needs a head with dropout: ModalityDropoutModel or MilAttentionModel."""
    if not hasattr(model, "predict_uncertainty_sweep") or hasattr(model, "mask_dim") or _kind(prep_info) == "moe":
        raise ValueError(f"{type(model).__name__} has no Monte-Carlo dropout uncertainty: uncertainty_model supports "
                         "ModalityDropoutModel and MilAttentionModel (MoENet has no dropout layer)")
    scenarios = config.get("scenarios", [{"name": "baseline", "drop_modalities": []}])
    y_true = df_test[TARGET_COL].values
    if _kind(prep_info) == "mil":
        _, per = scenario_mask_tensor(df_test, scenarios, mask_test, list(mask_test.keys()))
        bags = df_test[prep_info[1]].tolist()
        n = len(bags)
        mri = np.stack([np.asarray(cur["mri"]) if "mri" in cur else np.ones(n, dtype=int) for cur in per])
        res = model.predict_uncertainty_sweep(bags, mri, n_samples, seed)
    else:
        X, masks, _, order = _fusion_inputs(df_test, mask_test, prep_info, scenarios)
        res = model.predict_uncertainty_sweep(X, masks, order, n_samples, seed)
    out = {}
    for s, sc in enumerate(scenarios):
        r = dict(res[s])
        r["risk_coverage"] = _risk_coverage_by_entropy(y_true, r["mean"], r["entropy"])
        out[sc["name"]] = r
    return out


def ensemble_model(ens, df_test, mask_test, prep_info, config) -> Dict[str, Dict]:
    """A deep ensemble (models.ensemble.HeadEnsemble) under every scenario of `config`: {scenario: {"metrics": evaluate_model's
    metrics of the ensemble mean, "members": [each member's metrics], "member_mean" / "member_std": {metric: mean / population std
    over the members} (the spread across training seeds), "mean", "std", "entropy", "expected_entropy", "mutual_info": [N] float64
    ensemble statistics per subject, "risk_coverage": {"coverage", "risk", "aurc"} ranked by the entropy of the ensemble mean}}.
    With config["group_col"] the metrics include _with_groups' subject_* metrics.  The scenario masks are drawn as evaluate_model
    draws them (same helpers, same numpy RNG order, nothing else drawn), so each member's metrics are evaluate_model's of that member
    under the same seed."""
    if not hasattr(ens, "predict_ensemble_sweep"):
        raise ValueError(f"{type(ens).__name__} is not an ensemble: ensemble_model needs a HeadEnsemble")
    scenarios = config.get("scenarios", [{"name": "baseline", "drop_modalities": []}])
    group_col = config.get("group_col")
    y_true = df_test[TARGET_COL].values
    if _kind(prep_info) == "mil":
        _, per = scenario_mask_tensor(df_test, scenarios, mask_test, list(mask_test.keys()))
        bags = df_test[prep_info[1]].tolist()
        n = len(bags)
        mri = np.stack([np.asarray(cur["mri"]) if "mri" in cur else np.ones(n, dtype=int) for cur in per])
        members, stats = ens.predict_ensemble_sweep(bags, mri)
    else:
        X, masks, _, order = _fusion_inputs(df_test, mask_test, prep_info, scenarios)
        members, stats = ens.predict_ensemble_sweep(X, masks, order)
    mean = ens._mean(members)
    out = {}
    for s, sc in enumerate(scenarios):
        per_member = [_with_groups(compute_metrics(y_true, members[e, s]), df_test, y_true, members[e, s], group_col)
                      for e in range(members.shape[0])]
        keys = list(per_member[0])
        r = {"metrics": _with_groups(compute_metrics(y_true, mean[s]), df_test, y_true, mean[s], group_col),
             "members": per_member,
             "member_mean": {k: float(np.mean([m[k] for m in per_member])) for k in keys},
             "member_std": {k: float(np.std([m[k] for m in per_member])) for k in keys}}
        r.update(stats[s])
        r["risk_coverage"] = _risk_coverage_by_entropy(y_true, r["mean"], r["entropy"])
        out[sc["name"]] = r
    return out


def predict_proba_for_scenario(model, df_test, mask_test, prep_info, scenario):
    """(y_true, y_prob) for a single scenario."""
    probs, _ = _sweep_probs(model, df_test, mask_test, prep_info, [scenario])
    return df_test[TARGET_COL].values, np.asarray(probs[0])


def compute_risk_coverage(y_true, y_prob, masks):
    """Risk-coverage curve by descending confidence (reference: evaluate.py:140-169)."""
    conf = np.maximum(y_prob, 1 - y_prob)
    order = np.argsort(conf)[::-1]
    hits = ((y_prob >= 0.5).astype(int) == y_true).astype(int)[order]
    n = len(y_true)
    k = np.arange(1, n + 1)
    return {"coverage": k / n, "risk": 1 - np.cumsum(hits) / k}

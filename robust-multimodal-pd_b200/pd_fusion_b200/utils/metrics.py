"""Scenario metrics (reference: utils/metrics.py:10-36): sklearn on the host, 10-bin ECE.  `bootstrap_metrics` computes the same six
metrics for every bootstrap replicate on the device (pdf_bootstrap_metrics)."""
import numpy as np
from sklearn.metrics import average_precision_score, balanced_accuracy_score, brier_score_loss, f1_score, roc_auc_score


def compute_ece(y_true, y_prob, n_bins: int = 10) -> float:
    edges = np.linspace(0, 1, n_bins + 1)
    ece = 0.0
    for lo, hi in zip(edges[:-1], edges[1:]):
        sel = (y_prob > lo) & (y_prob <= hi)
        frac = np.mean(sel)
        if frac > 0:
            acc = np.mean(y_true[sel] == (y_prob[sel] >= 0.5))
            ece += frac * np.abs(acc - np.mean(y_prob[sel]))
    return ece


def compute_metrics(y_true, y_prob, threshold: float = 0.5):
    y_pred = (y_prob >= threshold).astype(int)
    return {
        "roc_auc": roc_auc_score(y_true, y_prob),
        "pr_auc": average_precision_score(y_true, y_prob),
        "balanced_accuracy": balanced_accuracy_score(y_true, y_pred),
        "f1": f1_score(y_true, y_pred),
        "brier_score": brier_score_loss(y_true, y_prob),
        "ece": compute_ece(y_true, y_prob),
    }


METRIC_NAMES = ("roc_auc", "pr_auc", "balanced_accuracy", "f1", "brier_score", "ece")   # compute_metrics' key order


def bootstrap_metrics(y_true, probs, n_boot: int = 1000, seed: int = 0, units=None):
    """Poisson(1) bootstrap of compute_metrics on the device: (point [S, 6], replicates [S, n_boot, 6]) float64, metrics in
    METRIC_NAMES order, for probs [N] (S = 1) or [S, N] against labels y_true [N] in {0, 1}.

    Replicate b weights sampling unit u by Poisson1(philox4x32_10(key=seed, counter=(u, b, 0, 0)).x) (see pdf_bootstrap_metrics):
    a stateless function of (seed, b, u), so replicate b is the same for any n_boot and any number of scenarios, scenarios are paired
    replicate by replicate, and numpy's and torch's RNGs are not touched.  `units` [N] (non-negative ints) gives rows that resample
    together (e.g. the subject of each row); None resamples rows.  Each replicate metric is the sklearn / numpy metric with
    sample_weight = w (ECE: compute_ece's bins weighted by w); the point estimate is every weight 1, i.e. compute_metrics on float64
    probabilities.  Degenerate replicates follow sklearn: roc_auc NaN without both classes, pr_auc 0 without positives, balanced
    accuracy the recall of the one class present, F1 0 on zero division; all NaN when every weight is 0."""
    import ctypes as C

    import torch

    from .. import _lib

    y = np.asarray(y_true)
    p = np.asarray(probs, dtype=np.float64)
    if p.ndim == 1:
        p = p[None]
    if p.ndim != 2 or y.ndim != 1 or p.shape[1] != y.shape[0] or y.shape[0] == 0:
        raise ValueError(f"probs must be [N] or [S, N] and y_true [N], N >= 1 (got {p.shape} and {y.shape})")
    if not np.all(np.isfinite(p)) or np.any(p < 0) or np.any(p > 1):
        raise ValueError("probabilities must be finite and in [0, 1]")
    if not np.all((y == 0) | (y == 1)):
        raise ValueError("y_true must hold only 0 and 1")
    n_boot = int(n_boot)
    if n_boot < 0:
        raise ValueError("n_boot must be >= 0")
    u = None
    if units is not None:
        u = np.asarray(units)
        if u.shape != y.shape or (u.size and not np.issubdtype(u.dtype, np.integer)):
            raise ValueError("units must be [N] integers")
        if np.any(u < 0) or np.any(u > np.iinfo(np.int32).max):
            raise ValueError("units must be non-negative int32 ids")
    _lib.require_cuda()
    lib = _lib.load()
    S, N = p.shape
    dev = torch.device("cuda", torch.cuda.current_device())
    d_prob = torch.from_numpy(np.ascontiguousarray(p)).to(dev)
    d_label = torch.from_numpy(y.astype(np.uint8)).to(dev)
    d_unit = torch.from_numpy(u.astype(np.int32)).to(dev) if u is not None else None
    need = int(lib.pdf_bootstrap_metrics_workspace_bytes(S, N))
    if need == 0:
        raise ValueError(f"pdf_bootstrap_metrics does not take {S} scenarios of {N} rows")
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    out = torch.empty((S, n_boot + 1, 6), dtype=torch.float64, device=dev)
    _lib.check(lib.pdf_bootstrap_metrics(S, N, n_boot, C.c_uint64(int(seed) & (2**64 - 1)), d_prob.data_ptr(), d_label.data_ptr(),
                                         _lib.ptr(d_unit), ws.data_ptr(), out.data_ptr(), _lib.stream_ptr()), "pdf_bootstrap_metrics")
    out = out.cpu().numpy()
    return out[:, 0].copy(), out[:, 1:].copy()

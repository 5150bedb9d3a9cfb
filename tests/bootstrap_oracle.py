"""Restatement of the device bootstrap's resampling weights and metrics for the tests (no GPU, no product code).

bootstrap_weights(seed, b, units): Philox4x32-10 (Salmon et al., SC'11; the constants and round of curand's curand_Philox4x32_10) in
numpy uint64 arithmetic, then inversion of the first 32-bit word against POISSON1 = floor(2^32 P(X <= k)), X ~ Poisson(1).
weighted_metrics: compute_metrics' six metrics through sklearn with sample_weight = w, the 10-bin ECE weighted by w.
"""
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def poisson1_thresholds():
    """T_k = floor(2^32 P(X <= k)), k = 0..12, X ~ Poisson(1), from e^-1 to 60 digits."""
    getcontext().prec = 60
    em1 = Decimal(-1).exp()
    out, cdf, fact = [], Decimal(0), 1
    for k in range(13):
        fact *= max(k, 1)
        cdf += em1 / fact
        out.append(int((cdf * 2 ** 32).to_integral_value(rounding="ROUND_FLOOR")))
    return out


POISSON1 = np.array(poisson1_thresholds(), dtype=np.uint64)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """first output word of Philox4x32-10 for counters (c0..c3) (uint64 arrays holding 32-bit values) and key (k0, k1)."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3))
    for r in range(10):
        ka, kb = np.uint64((k0 + r * W0) & 0xFFFFFFFF), np.uint64((k1 + r * W1) & 0xFFFFFFFF)
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = hi1 ^ c1 ^ ka, lo1, hi0 ^ c3 ^ kb, lo0
    return c0


def bootstrap_weights(seed: int, b: int, units) -> np.ndarray:
    """int64 weight of every unit id in `units` in replicate b: Poisson1(philox4x32_10(key=seed, counter=(u, b, 0, 0)).x)."""
    u = np.asarray(units, dtype=np.uint64)
    z = np.zeros_like(u)
    x = philox4x32_10(u, np.full_like(u, b), z, z, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return (x[:, None] >= POISSON1[None, :]).sum(axis=1).astype(np.int64)


def weighted_ece(y, p, w, n_bins=10):
    edges = np.linspace(0, 1, n_bins + 1)
    W, ece = w.sum(), 0.0
    for lo, hi in zip(edges[:-1], edges[1:]):
        sel = (p > lo) & (p <= hi)
        ws = w[sel].sum()
        if ws > 0:
            acc = (w[sel] * (y[sel] == (p[sel] >= 0.5))).sum() / ws
            ece += ws / W * abs(acc - (w[sel] * p[sel]).sum() / ws)
    return ece


def weighted_metrics(y, p, w):
    """[6] compute_metrics with sample_weight = w (NaN everywhere when sum(w) == 0)"""
    import warnings

    from sklearn.metrics import average_precision_score, balanced_accuracy_score, brier_score_loss, f1_score, roc_auc_score
    y, p, w = np.asarray(y).astype(int), np.asarray(p, dtype=np.float64), np.asarray(w, dtype=np.float64)
    if w.sum() == 0:
        return np.full(6, np.nan)
    pred = (p >= 0.5).astype(int)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return np.array([roc_auc_score(y, p, sample_weight=w), average_precision_score(y, p, sample_weight=w),
                         balanced_accuracy_score(y, pred, sample_weight=w), f1_score(y, pred, sample_weight=w),
                         brier_score_loss(y, p, sample_weight=w), weighted_ece(y, p, w)])


def exact_auc(y, p, w):
    """AUC with integer weights as the exact rational sum over tie groups of w_neg (TP_prev + TP_end) / (2 Wpos Wneg), rounded once
    (None without both classes)."""
    o = np.argsort(-np.asarray(p, dtype=np.float64), kind="stable")
    ps, ys, ws = np.asarray(p, dtype=np.float64)[o], np.asarray(y)[o], np.asarray(w, dtype=np.int64)[o]
    end = np.r_[ps[1:] != ps[:-1], True]
    tp, fp = np.cumsum(ws * (ys == 1)), np.cumsum(ws * (ys == 0))
    TPe, FPe = tp[end], fp[end]
    TPp, FPp = np.r_[0, TPe[:-1]], np.r_[0, FPe[:-1]]
    wp, wn = int(tp[-1]), int(fp[-1])
    if wp == 0 or wn == 0:
        return None
    num = sum(int(a) * int(b) for a, b in zip(FPe - FPp, TPp + TPe))
    return float(Fraction(num, 2 * wp * wn))

"""Restatement of the device's Monte-Carlo dropout for the tests (no GPU, no product code): the keep masks from Philox4x32-10 with
bootstrap_oracle's constants and round, and the ModalityDropoutNet / MILAttentionNet forward passes in float64 torch with those explicit
masks.

Unit j of row n, sample t, layer l, instance i is dropped iff
  philox4x32_10(key = seed, counter = (n, t, (l << 16) | i, 0x80000000 | (j >> 2))).word[j & 3] < floor(p 2^32)
with p the float32 value of the dropout probability; a kept unit is multiplied by the float32 value of 1 / (1 - p)."""
import numpy as np
import torch

from bootstrap_oracle import M0, M1, MASK, W0, W1

STATS = ("mean", "std", "entropy", "expected_entropy", "mutual_info")


def philox4x32_10_words(c0, c1, c2, c3, k0, k1):
    """all four output words of Philox4x32-10 (uint64 arrays holding 32-bit values), bootstrap_oracle.philox4x32_10's rounds"""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3))
    for r in range(10):
        ka, kb = np.uint64((k0 + r * W0) & 0xFFFFFFFF), np.uint64((k1 + r * W1) & 0xFFFFFFFF)
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = hi1 ^ c1 ^ ka, lo1, hi0 ^ c3 ^ kb, lo0
    return c0, c1, c2, c3


def threshold(p: float) -> int:
    return int(np.floor(float(np.float32(p)) * 2.0 ** 32))


def keep_scale(p: float) -> float:
    return float(np.float32(1.0 / (1.0 - float(np.float32(p)))))


def counters(n, t, word2, width):
    """the counters of units 0..width-1 for broadcastable n, t, word2 (= (l << 16) | i): four uint64 arrays [..., ceil(width / 4)]"""
    q = np.arange((width + 3) // 4, dtype=np.uint64)
    n, t, w2 = (np.asarray(v, dtype=np.uint64)[..., None] for v in (n, t, word2))
    shape = np.broadcast_shapes(n.shape, t.shape, w2.shape, q.shape)
    return (np.broadcast_to(n, shape), np.broadcast_to(t, shape), np.broadcast_to(w2, shape),
            np.broadcast_to(np.uint64(0x80000000) | q, shape))


def keep_mask(seed: int, p: float, n, t, word2, width: int) -> np.ndarray:
    """float64 [..., width]: scale where the unit is kept, 0 where dropped"""
    c = counters(n, t, word2, width)
    words = np.stack(philox4x32_10_words(*c, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF), axis=-1)    # [..., q, 4]
    words = words.reshape(words.shape[:-2] + (-1,))[..., :width]
    return np.where(words >= np.uint64(threshold(p)), keep_scale(p), 0.0)


def moddrop_samples(net, X, masks, sizes, T, seed, p):
    """ModalityDropoutNet `net`, X [N, F], masks [S, N, M] in sorted(modality) order, modality widths `sizes` -> sample probabilities
    [S, N, T] float64: the net in float64 with the hidden layers' dropout replaced by the explicit keep masks"""
    lins = [m.double() for m in net.net if isinstance(m, torch.nn.Linear)]
    N = X.shape[0]
    n_idx, t_idx = np.arange(N)[:, None], np.arange(T)[None, :]
    drop = [torch.from_numpy(keep_mask(seed, p, n_idx, t_idx, l << 16, lin.out_features)) for l, lin in enumerate(lins[:-1])]
    Xd = torch.from_numpy(np.asarray(X, dtype=np.float64))
    out = np.zeros((masks.shape[0], N, T))
    with torch.no_grad():
        for s in range(masks.shape[0]):
            h = (Xd * torch.from_numpy(np.repeat(masks[s].astype(np.float64), sizes, axis=1)))[:, None, :].expand(N, T, Xd.shape[1])
            for l, lin in enumerate(lins):
                h = lin(h)
                if l < len(lins) - 1:
                    h = torch.relu(h) * drop[l]
            out[s] = torch.sigmoid(h[..., 0]).numpy()
    return out


def mil_samples(net, bags, lens, live, missing_prob, T, seed, p):
    """MILAttentionNet `net`, bags [n, Lmax, D], lens [n], live [S, n] or None -> sample probabilities [S, n, T] float64 (missing_prob
    as a float32 value where live[s, b] == 0 or lens[b] == 0)"""
    net = net.double()
    n = bags.shape[0]
    S = 1 if live is None else live.shape[0]
    mp = float(np.float32(missing_prob))
    out = np.full((S, n, T), mp)
    with torch.no_grad():
        for b in range(n):
            L = int(lens[b])
            if L <= 0:
                continue
            h = net.instance[1](net.instance[0](torch.from_numpy(np.asarray(bags[b, :L], dtype=np.float64))))          # [L, H]
            hm = h[None] * torch.from_numpy(keep_mask(seed, p, b, np.arange(T)[:, None], np.arange(L)[None, :], h.shape[1]))
            sc = (net.attn_w(net.attn_v(hm) * net.attn_u(hm)) if net.gated else net.attn(hm))[..., 0]                # [T, L]
            a = torch.softmax(sc, dim=1)
            prob = net.classifier((a[..., None] * hm).sum(dim=1))[:, 0].numpy()
            for s in range(S):
                if live is None or live[s, b]:
                    out[s, b] = prob
    return out


def entropy(q):
    q = np.asarray(q, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        a = np.where(q > 0, q * np.log(np.where(q > 0, q, 1.0)), 0.0)
        b = np.where(q < 1, (1 - q) * np.log(np.where(q < 1, 1 - q, 1.0)), 0.0)
    return -a - b


def stats(samples):
    """[..., T] sample probabilities -> [..., 5] in STATS order, numpy float64"""
    s = np.asarray(samples, dtype=np.float64)
    mean = s.mean(-1)
    ent, eent = entropy(mean), entropy(s).mean(-1)
    return np.stack([mean, s.std(-1), ent, eent, np.maximum(0.0, ent - eent)], axis=-1)

"""MIL (gated-)attention pooling head (reference: models/mil_attention.py).

`MILAttentionNet` keeps the reference's parameter names so its `state_dict` is the weight-interchange format
(SURVEY.md A.6).  Inference (`predict_proba`) runs ALL bags in one launch of pdf_mil_forward instead of the
reference's per-bag B=1 loop with a `.cpu()` per bag (mil_attention.py:169-177).  Training (`train`) runs the native forward/backward/Adam
kernels of csrc/train.cu through pd_fusion_b200/training.py (SURVEY.md 8f rank 2).  `predict_uncertainty` estimates the predictive
uncertainty by Monte-Carlo dropout of the instance layer (pdf_mil_mc).
"""
from __future__ import annotations

from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from ..heads import MilHead, mc_dicts
from ..utils.torch_utils import get_torch_device
from .base import BaseModel


class MILAttentionNet(nn.Module):
    def __init__(self, input_dim: int, hidden_dim: int, attn_dim: int, dropout: float = 0.3, gated: bool = False):
        super().__init__()
        self.gated = gated
        self.instance = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.ReLU(), nn.Dropout(dropout))
        if gated:
            self.attn_v = nn.Sequential(nn.Linear(hidden_dim, attn_dim), nn.Tanh())
            self.attn_u = nn.Sequential(nn.Linear(hidden_dim, attn_dim), nn.Sigmoid())
            self.attn_w = nn.Linear(attn_dim, 1)
        else:
            self.attn = nn.Sequential(nn.Linear(hidden_dim, attn_dim), nn.Tanh(), nn.Linear(attn_dim, 1))
        self.classifier = nn.Sequential(nn.Linear(hidden_dim, 1), nn.Sigmoid())

    def forward(self, x: torch.Tensor, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Training-time (autograd) forward; x [B, L, D], mask [B, L]."""
        h = self.instance(x)
        s = (self.attn_w(self.attn_v(h) * self.attn_u(h)) if self.gated else self.attn(h)).squeeze(-1)
        if mask is not None:
            s = s.masked_fill(mask == 0, -1e9)
        a = torch.softmax(s, dim=1)
        return self.classifier((a.unsqueeze(-1) * h).sum(dim=1)).squeeze(-1)


def _pad_bags(bags):
    """Zero-pads bags [L_i, D] to [n, Lmax, D] + {0,1} mask [n, Lmax] (reference: mil_attention.py:54-63)."""
    lmax = max(b.shape[0] for b in bags)
    X = np.zeros((len(bags), lmax, bags[0].shape[1]), dtype=np.float32)
    M = np.zeros((len(bags), lmax), dtype=np.float32)
    for i, b in enumerate(bags):
        X[i, : b.shape[0]] = b
        M[i, : b.shape[0]] = 1.0
    return X, M


def _fill_explanation(out: dict, rows: List[int], lens: np.ndarray, logit: torch.Tensor, attn: torch.Tensor, contrib: torch.Tensor):
    """Copies a MilHead.explain result of the bags `rows` (in that order, lengths `lens`) into the per-bag lists / arrays of `out`.
    prob = sigmoid(logit) on the device in float32, the pooling kernel's own last step."""
    prob = torch.sigmoid(logit).cpu().numpy()
    logit, attn, contrib = logit.cpu().numpy(), attn.cpu().numpy(), contrib.cpu().numpy()
    for j, i in enumerate(rows):
        L = int(lens[j])
        out["prob"][i] = float(prob[j])
        out["logit"][i] = float(logit[j])
        out["attention"][i] = attn[j, :L].copy()
        out["contribution"][i] = contrib[j, :L].copy()


class MilAttentionModel(BaseModel):
    def __init__(self, input_dim: int, params: dict):
        self.params = params or {}
        p = self.params
        self.gated = bool(p.get("gated", False))
        self.missing_prob = float(p.get("missing_prob", 0.5))
        self.model = MILAttentionNet(input_dim, int(p.get("hidden_dim", 128)), int(p.get("attn_dim", 64)),
                                     float(p.get("dropout", 0.3)), gated=self.gated)
        self.pos_weight = float(p["pos_weight"]) if (p.get("class_weight") != "balanced" and p.get("pos_weight") is not None) else None
        # "fp32" (default: FFMA GEMMs, <= 5e-6 against the reference) | "tf32" (tcgen05 kind::tf32 projection, the throughput path)
        self.precision = str(p.get("precision", "fp32"))
        self._head: Optional[MilHead] = None
        self._train = None

    # -- training: native forward/backward/Adam kernels (csrc/train.cu) ---------------------------
    def _trainer(self):
        if self._train is None:
            from ..training import MilHeadTrainer, NativeAdam
            self.model.to(get_torch_device()).float()
            ht = MilHeadTrainer(self.model, self.gated)
            p = self.params
            self._train = (ht, NativeAdam([([q for q, _ in ht.param_grads()], float(p.get("lr", 1e-3)))],
                                          weight_decay=float(p.get("weight_decay", 0.0))))
        return self._train

    def train(self, bags, y, val_data=None):
        """Same loop as the reference (models/mil_attention.py:88-155: torch.randperm batches, BCE x pos_weight, mean, optional
        clip_grad_norm_, Adam, early stopping on validation AUC); each step is pdf_gemm_f32 / pdf_mil_pool_train / pdf_adam_step
        launches on the padded bag tensor resident on the device -- no autograd graph."""
        X, M = _pad_bags(bags)
        dev = get_torch_device()
        ht, opt = self._trainer()
        Xt = torch.from_numpy(X).to(dev)
        lens_all = torch.from_numpy(M.sum(axis=1).astype(np.int32)).to(dev)
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32, device=dev)
        p = self.params
        bs, epochs = int(p.get("batch_size", 16)), int(p.get("epochs", 30))
        clip, patience = p.get("max_grad_norm"), int(p.get("early_stopping_patience", 0))
        if self.pos_weight is None and p.get("class_weight") == "balanced":
            pos, neg = float((yt == 1).sum()), float((yt == 0).sum())
            if pos > 0:
                self.pos_weight = neg / pos
        lr = opt.groups[0][1]
        best_auc, best_state, bad = -1.0, None, 0
        self.last_losses = []
        for _ in range(epochs):
            self.model.train()
            order = torch.randperm(len(Xt), device="cpu").to(dev)
            for i in range(0, len(order), bs):
                sel = order[i:i + bs]
                ht.zero_grad()
                loss, _, _ = ht.forward_backward(Xt[sel], lens_all[sel], yt[sel], "bce", self.pos_weight)
                pg = [(q, g, lr) for q, g in ht.param_grads()]
                scale = opt.clip([g for _, g, _ in pg], float(clip)) if clip else None
                opt.step(pg, scale)
                self.last_losses.append(loss)
            self._head = None
            if val_data is not None and patience > 0:
                from sklearn.metrics import roc_auc_score
                try:
                    auc = float(roc_auc_score(val_data[1], self.predict_proba(val_data[0])))
                except Exception:
                    auc = -1.0
                if auc > best_auc:
                    best_auc, bad = auc, 0
                    # the reference keeps `self.model.state_dict()` WITHOUT cloning (models/mil_attention.py:147): it aliases the
                    # live parameters, so restoring it below is a no-op and the final weights are the last epoch's.  A drop-in
                    # trains to the same weights; MilAttentionFineTuneModel keeps the same quirk (SURVEY.md C.5).
                    best_state = self.model.state_dict()
                else:
                    bad += 1
                    if bad >= patience:
                        break
        if best_state is not None:
            self.model.load_state_dict(best_state)
        self._head = None

    # -- inference: one launch over all bags ------------------------------------------------------
    def _get_head(self) -> MilHead:
        if self._head is None:
            self._head = MilHead(self.model.state_dict(), self.gated, self.missing_prob, device=get_torch_device(),
                                 precision=self.precision)
        return self._head

    def invalidate(self):
        """Call after mutating `self.model` weights in place (load_state_dict etc.)."""
        self._head = None

    def _upload(self, bags, keep):
        """Pads the bags listed in `keep` into one [n, Lmax, D] device tensor (once per call, whatever the number of scenarios)."""
        head = self._get_head()
        lmax = max(bags[i].shape[0] for i in keep)
        X = np.zeros((len(keep), lmax, head.D), dtype=np.float32)
        lens = np.zeros(len(keep), dtype=np.int32)
        for j, i in enumerate(keep):
            b = np.asarray(bags[i], dtype=np.float32)
            X[j, : b.shape[0]] = b
            lens[j] = b.shape[0]
        return head, torch.from_numpy(X).to(head.device), torch.from_numpy(lens).to(head.device)

    def predict_proba(self, bags: List[Optional[np.ndarray]], masks=None) -> np.ndarray:
        mri = masks["mri"] if isinstance(masks, dict) and "mri" in masks else None
        n = len(bags)
        live = [i for i, b in enumerate(bags) if b is not None and not (mri is not None and mri[i] == 0)]
        out = np.full(n, self.missing_prob, dtype=np.float64)
        if not live:
            return out
        head, X, lens = self._upload(bags, live)
        out[live] = head.forward(X, lens).cpu().numpy().astype(np.float64)
        return out

    def explain(self, bags: List[Optional[np.ndarray]], masks=None) -> dict:
        """Why each bag got its probability (bag and mask semantics of `predict_proba`), one pdf_mil_explain over the live bags:
        {"prob": [N] float64 (as predict_proba; missing_prob for absent bags), "logit": [N] float64 (NaN where absent),
         "attention": [a_l] and "contribution": [a_l * (w_cls . h_l)] per bag as np.ndarray [L_i] (None where absent)}.
        The contributions of a bag add up to logit - classifier bias.  Explanations always use the FP32 head arithmetic: for a
        "tf32" model, prob and logit are those of the same weights under "fp32"."""
        mri = masks["mri"] if isinstance(masks, dict) and "mri" in masks else None
        n = len(bags)
        live = [i for i, b in enumerate(bags) if b is not None and not (mri is not None and mri[i] == 0)]
        out = {"prob": np.full(n, self.missing_prob, dtype=np.float64), "logit": np.full(n, np.nan, dtype=np.float64),
               "attention": [None] * n, "contribution": [None] * n}
        if not live:
            return out
        head, X, lens = self._upload(bags, live)
        logit, attn, contrib, _ = head.explain(X, lens)
        _fill_explanation(out, live, lens.cpu().numpy(), logit, attn, contrib)
        return out

    def predict_proba_sweep(self, bags: List[Optional[np.ndarray]], mri_masks: Optional[np.ndarray]) -> np.ndarray:
        """All scenarios of evaluate_model at once (evaluation/evaluate.py:32-37 re-runs predict_proba per scenario with the
        dropped bags set to None): mri_masks [S, N] {0,1} (None = one scenario, everything present) -> prob [S, N] float64.
        Bags are padded and uploaded ONCE, projected and pooled ONCE; the scenario only selects missing_prob."""
        n = len(bags)
        S = 1 if mri_masks is None else int(np.asarray(mri_masks).shape[0])
        out = np.full((S, n), self.missing_prob, dtype=np.float64)
        have = [i for i, b in enumerate(bags) if b is not None]
        if mri_masks is not None:
            mm = np.asarray(mri_masks)
            have = [i for i in have if mm[:, i].any()]              # a bag dropped by every scenario never reaches the device
        if not have:
            return out
        head, X, lens = self._upload(bags, have)
        live = None if mri_masks is None else torch.from_numpy(np.ascontiguousarray(np.asarray(mri_masks)[:, have] != 0).astype(np.uint8))
        out[:, have] = head.sweep(X, lens, live, S).cpu().numpy().astype(np.float64)
        return out

    def predict_uncertainty_sweep(self, bags: List[Optional[np.ndarray]], mri_masks: Optional[np.ndarray], n_samples: int = 32,
                                  seed: int = 0, return_samples: bool = False) -> List[dict]:
        """`predict_uncertainty` under every scenario of mri_masks ([S, N] {0,1} as predict_proba_sweep; None = one scenario,
        everything present) in one pdf_mil_mc call -> one dict per scenario.  Every bag position is uploaded (absent ones empty), so
        bag i's masks depend on (seed, i, sample) only and a bag's samples are the same under every scenario where it is present."""
        head = self._get_head()
        n = len(bags)
        S = 1 if mri_masks is None else int(np.asarray(mri_masks).shape[0])
        lmax = max([1] + [np.asarray(b).shape[0] for b in bags if b is not None])
        X = np.zeros((n, lmax, head.D), dtype=np.float32)
        lens = np.zeros(n, dtype=np.int32)
        for i, b in enumerate(bags):
            if b is not None:
                b = np.asarray(b, dtype=np.float32)
                X[i, : b.shape[0]] = b
                lens[i] = b.shape[0]
        live = None if mri_masks is None else torch.from_numpy(np.ascontiguousarray(np.asarray(mri_masks) != 0).astype(np.uint8))
        stats, smp = head.mc(torch.from_numpy(X).to(head.device), torch.from_numpy(lens).to(head.device), live, S, n_samples, seed,
                             float(self.model.instance[2].p), return_samples)
        return mc_dicts(stats, smp)

    def predict_uncertainty(self, bags: List[Optional[np.ndarray]], masks=None, n_samples: int = 32, seed: int = 0,
                            return_samples: bool = False) -> dict:
        """Monte-Carlo dropout for the arguments of `predict_proba` (a bag that is None or whose masks["mri"] is 0 is missing):
        n_samples forward passes with the instance layer's nn.Dropout active.  Returns [N] float64 arrays "mean", "std"
        (population), "entropy" (of the mean, nats), "expected_entropy" and "mutual_info" (max(0, entropy - expected_entropy)), and
        with return_samples "samples" [N, n_samples].  A missing bag gets mean = missing_prob, std = mutual_info = 0.  Always the
        FP32 head arithmetic, whatever `precision` says."""
        mri = masks["mri"] if isinstance(masks, dict) and "mri" in masks else None
        return self.predict_uncertainty_sweep(bags, None if mri is None else np.asarray(mri)[None], n_samples, seed, return_samples)[0]

    def save(self, path):
        torch.save(self.model.state_dict(), path)

    @classmethod
    def load(cls, path, input_dim, params):
        inst = cls(input_dim, params)
        inst.model.load_state_dict(torch.load(path, map_location="cpu", weights_only=True))
        return inst

"""Fusion-ModDrop (reference: models/fusion_moddrop.py).

`ModalityDropoutNet` keeps the reference's layout (feature blocks in sorted(modality) order, `net.{0,3,6,..}`
keys).  `predict_proba` runs on the device through pdf_moddrop_sweep; `predict_proba_sweep` evaluates every
scenario mask of a missingness sweep in ONE launch (layer-1 partials per modality computed once).  `explain`
returns the modalities' exact Shapley values and integrated gradients of the logit (pdf_moddrop_explain).  `predict_uncertainty`
estimates the predictive uncertainty by Monte-Carlo dropout (pdf_moddrop_mc).
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from ..heads import ModDropSweep, mc_dicts
from ..utils.torch_utils import get_torch_device
from .base import BaseModel


class ModalityDropoutNet(nn.Module):
    def __init__(self, modality_dims: Dict[str, int], hidden_dims: List[int], dropout: float = 0.2):
        super().__init__()
        self.modality_dims = modality_dims
        self.mod_names = sorted(modality_dims)
        self.slices, pos = {}, 0
        for mod in self.mod_names:
            self.slices[mod] = (pos, pos + modality_dims[mod])
            pos += modality_dims[mod]
        layers, width = [], pos
        for h in hidden_dims:
            layers += [nn.Linear(width, h), nn.ReLU(), nn.Dropout(dropout)]
            width = h
        layers += [nn.Linear(width, 1), nn.Sigmoid()]
        self.net = nn.Sequential(*layers)

    def forward(self, x, training_dropout: bool = False, drop_rate: float = 0.0):
        if training_dropout and self.training:
            keep = torch.ones_like(x)
            for mod in self.mod_names:          # one np.random.rand() per modality per batch, as the reference draws them
                if np.random.rand() < drop_rate:
                    a, b = self.slices[mod]
                    keep[:, a:b] = 0.0
            x = x * keep
        return self.net(x)


class ModalityDropoutModel(BaseModel):
    def __init__(self, modality_dims, params):
        self.params = params
        self.modality_dims = modality_dims
        self.model = ModalityDropoutNet(modality_dims, params["hidden_dims"], params.get("dropout", 0.2))
        self._sweep: Optional[ModDropSweep] = None
        self._train = None      # (MlpTrainer, NativeAdam): created on first train(), Adam moments persist like the reference's self.optimizer

    def train(self, X, y, val_data=None):
        """The reference's loop (models/fusion_moddrop.py:69-91: torch.randperm mini-batches, one np.random.rand() per modality per
        batch for the modality dropout, nn.BCELoss, Adam) with every step on the native kernels: pdf_gemm_f32 forward / dgrad / wgrad,
        pdf_bce_sigmoid_train, pdf_adam_step.  The table stays resident on the device."""
        from .. import _lib
        from ..training import MlpTrainer, NativeAdam
        dev = get_torch_device()
        if self._train is None:
            self.model.to(dev).float()
            mt = MlpTrainer(self.model.net, "net.")
            self._train = (mt, NativeAdam([([q for q, _ in mt.param_grads()], float(self.params["lr"]))],
                                          weight_decay=float(self.params.get("weight_decay", 0.0))))
        mt, opt = self._train
        lib = _lib.load()
        Xt = torch.as_tensor(np.asarray(X), dtype=torch.float32).to(dev)
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32).to(dev)
        rate, bs = self.params.get("moddrop_rate", 0.2), self.params.get("batch_size", 32)
        lr = opt.groups[0][1]
        net = self.model
        self.last_losses = []
        for _ in range(self.params["epochs"]):
            net.train()
            order = torch.randperm(len(Xt)).to(dev)
            for i in range(0, len(Xt), bs):
                sel = order[i:i + bs]
                xb, yb = Xt[sel].contiguous(), yt[sel].contiguous()
                keep = None
                for mod in net.mod_names:       # one np.random.rand() per modality per batch, as the reference draws them
                    if np.random.rand() < rate:
                        if keep is None:
                            keep = torch.ones_like(xb)
                        a, b = net.slices[mod]
                        keep[:, a:b] = 0.0
                if keep is not None:
                    _lib.check(lib.pdf_mul_f32(xb.data_ptr(), keep.data_ptr(), xb.numel(), _lib.stream_ptr()), "pdf_mul_f32")
                mt.zero_grad()
                z = mt.forward(xb, train=True)
                n = int(z.shape[0])
                prob, dz = torch.empty(n, dtype=torch.float32, device=dev), torch.empty((n, 1), dtype=torch.float32, device=dev)
                loss = torch.zeros(1, dtype=torch.float32, device=dev)
                _lib.check(lib.pdf_bce_sigmoid_train(n, z.data_ptr(), yb.data_ptr(), prob.data_ptr(), loss.data_ptr(), dz.data_ptr(),
                                                     _lib.stream_ptr()), "pdf_bce_sigmoid_train")
                mt.backward(dz)
                opt.step([(q, g, lr) for q, g in mt.param_grads()])
                self.last_losses.append(loss)
        self._sweep = None

    def invalidate(self):
        self._sweep = None

    def _get_sweep(self) -> ModDropSweep:
        if self._sweep is None:
            self._sweep = ModDropSweep(self.model.state_dict(), self.modality_dims, device=get_torch_device())
        return self._sweep

    def _sweep_masks(self, masks_snm: np.ndarray, order: List[str]) -> np.ndarray:
        """masks_snm [S,N,len(order)] -> [S,N,M] in the sweep's sorted(modality) order; modalities missing from `order` are present."""
        sw = self._get_sweep()
        cols = [order.index(m) if m in order else -1 for m in sw.mods]
        mk = np.ones(masks_snm.shape[:2] + (len(sw.mods),), dtype=np.uint8)
        for j, c in enumerate(cols):
            if c >= 0:
                mk[:, :, j] = masks_snm[:, :, c]
        return mk

    def _single_mask(self, n: int, masks) -> np.ndarray:
        mk = np.ones((1, n, len(self._get_sweep().mods)), dtype=np.uint8)
        if masks is not None:
            for j, mod in enumerate(self._get_sweep().mods):
                if mod in masks:
                    # the reference multiplies by the float mask value; masks are {0,1} on every call site
                    mk[0, :, j] = np.asarray(masks[mod]) != 0
        return mk

    def predict_proba_sweep(self, X: np.ndarray, masks_snm: np.ndarray, order: List[str]) -> np.ndarray:
        """X [N,F] (unmasked); masks_snm uint8 [S,N,len(order)] -> probabilities [S,N] f32, one launch."""
        sw = self._get_sweep()
        mk = self._sweep_masks(masks_snm, order)
        dev = sw.device
        prob = sw.forward(torch.as_tensor(np.asarray(X), dtype=torch.float32).to(dev), torch.from_numpy(mk).to(dev))
        return prob.cpu().numpy()

    def predict_proba(self, X, masks=None):
        X = np.asarray(X)
        sw = self._get_sweep()
        return self.predict_proba_sweep(X, self._single_mask(X.shape[0], masks), sw.mods)[0]

    def explain_sweep(self, X: np.ndarray, masks_snm: np.ndarray, order: List[str], steps: int = 32) -> List[Dict]:
        """`explain` under every scenario mask of masks_snm (uint8 [S,N,len(order)], as predict_proba_sweep) in one
        pdf_moddrop_explain call -> one explanation dict per scenario."""
        sw = self._get_sweep()
        dev = sw.device
        value, base, shap, ig = sw.explain(torch.as_tensor(np.asarray(X), dtype=torch.float32).to(dev),
                                           torch.from_numpy(self._sweep_masks(masks_snm, order)).to(dev), steps)
        prob = torch.sigmoid(value).cpu().numpy().astype(np.float64)
        value, shap = value.cpu().numpy(), shap.cpu().numpy()
        ig = ig.cpu().numpy() if ig is not None else None
        b = float(base.item())
        return [{"prob": prob[s], "logit": value[s], "base_logit": b, "shapley": {m: shap[s, :, j] for j, m in enumerate(sw.mods)},
                 "ig": ig[s] if ig is not None else None} for s in range(value.shape[0])]

    def explain(self, X, masks=None, steps: int = 32) -> Dict:
        """Why each subject got its probability, for the arguments of `predict_proba` (X [N,F] unmasked, masks {mod: [N]} or None):
        prob [N] (predict_proba's, as float64), logit [N] (before net's final sigmoid), base_logit (the logit of the all-zero input,
        i.e. with every modality missing), shapley {mod: [N]} = exact Shapley values of the modalities for the logit (they add up
        to logit - base_logit; 0 for a missing modality), and ig [N,F] = integrated gradients of the logit from the zero input
        with `steps` midpoints (None for steps = 0; 0 on a missing modality's features)."""
        X = np.asarray(X)
        return self.explain_sweep(X, self._single_mask(X.shape[0], masks), self._get_sweep().mods, steps)[0]

    def _dropout_p(self) -> float:
        """the probability of the net's nn.Dropout layers (0 for a net without hidden layers)"""
        ps = {float(m.p) for m in self.model.net if isinstance(m, nn.Dropout)}
        if len(ps) > 1:
            raise ValueError(f"Monte-Carlo dropout needs one dropout probability for every hidden layer, got {sorted(ps)}")
        return ps.pop() if ps else 0.0

    def predict_uncertainty_sweep(self, X: np.ndarray, masks_snm: np.ndarray, order: List[str], n_samples: int = 32, seed: int = 0,
                                  return_samples: bool = False) -> List[Dict]:
        """`predict_uncertainty` under every scenario mask of masks_snm (uint8 [S,N,len(order)], as predict_proba_sweep) in one
        pdf_moddrop_mc call -> one dict per scenario.  Sample t of a subject drops the same units under every scenario."""
        sw = self._get_sweep()
        dev = sw.device
        stats, smp = sw.mc(torch.as_tensor(np.asarray(X), dtype=torch.float32).to(dev), torch.from_numpy(self._sweep_masks(masks_snm, order)).to(dev),
                           n_samples, seed, self._dropout_p(), return_samples)
        return mc_dicts(stats, smp)

    def predict_uncertainty(self, X, masks=None, n_samples: int = 32, seed: int = 0, return_samples: bool = False) -> Dict:
        """Monte-Carlo dropout for the arguments of `predict_proba`: n_samples forward passes with the net's own nn.Dropout layers
        active (their probability p; the training-time modality dropout stays off, the masks decide which modalities are present).
        Returns [N] float64 arrays "mean" (of the sample probabilities), "std" (population), "entropy" (of the mean, nats),
        "expected_entropy" (mean entropy of the samples) and "mutual_info" (max(0, entropy - expected_entropy): the model's own,
        epistemic, part), and with return_samples "samples" [N, n_samples].  Stateless in (seed, subject row, sample)."""
        X = np.asarray(X)
        return self.predict_uncertainty_sweep(X, self._single_mask(X.shape[0], masks), self._get_sweep().mods, n_samples, seed,
                                              return_samples)[0]

    def save(self, path):
        torch.save(self.model.state_dict(), path)

    @classmethod
    def load(cls, path, modality_dims, params):
        """The reference's `load` is an empty stub (fusion_moddrop.py:119-123); this one restores the state_dict."""
        inst = cls(modality_dims, params)
        inst.model.load_state_dict(torch.load(path, map_location="cpu", weights_only=True))
        return inst

"""Mixture-of-experts fusion head (reference: models/moe.py): one MLP expert per modality, a router MLP on the
availability mask with softmax gating.  Inference runs through pdf_moe_sweep (router + experts + gated sum for
every (scenario, subject) pair in one launch); `explain` returns the modalities' exact Shapley values and integrated gradients
of the probability (pdf_moe_explain)."""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from ..heads import MoeSweep
from ..utils.torch_utils import get_torch_device
from .base import BaseModel


class Expert(nn.Module):
    def __init__(self, input_dim, hidden_dims):
        super().__init__()
        layers, width = [], input_dim
        for h in hidden_dims:
            layers += [nn.Linear(width, h), nn.ReLU()]
            width = h
        layers += [nn.Linear(width, 1), nn.Sigmoid()]
        self.net = nn.Sequential(*layers)

    def forward(self, x):
        return self.net(x)


class MoENet(nn.Module):
    def __init__(self, modality_dims: Dict[str, int], params):
        super().__init__()
        self.experts = nn.ModuleDict({m: Expert(d, params["expert_hidden_dims"]) for m, d in modality_dims.items()})
        r = params["router_hidden_dims"][0]
        self.router = nn.Sequential(nn.Linear(len(modality_dims), r), nn.ReLU(), nn.Linear(r, len(modality_dims)), nn.Softmax(dim=1))

    def forward(self, modality_inputs: Dict[str, torch.Tensor], mask: torch.Tensor):
        """Training-time (autograd) forward."""
        w = self.router(mask)
        parts = [self.experts[m](modality_inputs[m]) * w[:, i:i + 1] for i, m in enumerate(sorted(modality_inputs))]
        return torch.stack(parts, dim=2).sum(dim=2)


class MoEModel(BaseModel):
    def __init__(self, modality_dims, params):
        self.params = params
        self.modality_dims = dict(modality_dims)
        self.model = MoENet(modality_dims, params)
        self._sweep: Optional[MoeSweep] = None
        self._train = None      # (expert trainers, router trainer, NativeAdam), created on first train()

    def train(self, X_dict, y, mask, val_data=None):
        """Full-batch steps as the reference (models/moe.py:60-70), every step on the native kernels: the experts' and the router's
        linear layers through pdf_gemm_f32 (forward, dgrad, wgrad), the gated combination + BCE and their backward in
        pdf_moe_combine_train, then pdf_adam_step.  Inputs stay resident on the device."""
        from .. import _lib
        from ..training import MlpTrainer, NativeAdam
        dev = get_torch_device()
        mods = sorted(X_dict)                                # MoENet.forward pairs router output i with sorted(modality) i
        if self._train is None:
            self.model.to(dev).float()
            experts = {m: MlpTrainer(self.model.experts[m].net, f"experts.{m}.net.") for m in mods}
            router = MlpTrainer(self.model.router, "router.")
            allp = [q for t in list(experts.values()) + [router] for q, _ in t.param_grads()]
            self._train = (experts, router, NativeAdam([(allp, float(self.params["lr"]))], weight_decay=float(self.params.get("weight_decay", 0.0))))
        experts, router, opt = self._train
        lib = _lib.load()
        X = {m: torch.as_tensor(np.asarray(X_dict[m]), dtype=torch.float32).to(dev).contiguous() for m in mods}
        mk = torch.as_tensor(np.asarray(mask), dtype=torch.float32).to(dev).contiguous()
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32).to(dev).contiguous()
        n, E = int(yt.shape[0]), len(mods)
        lr = opt.groups[0][1]
        self.last_losses = []
        for _ in range(self.params["epochs"]):
            self.model.train()
            for t in list(experts.values()) + [router]:
                t.zero_grad()
            z = torch.stack([experts[m].forward(X[m])[:, 0] for m in mods], dim=1).contiguous()       # [n, E] expert logits (layout only)
            r = router.forward(mk)                                                                     # [n, E] router logits
            out, dz, dr = torch.empty(n, dtype=torch.float32, device=dev), torch.empty_like(z), torch.empty_like(r)
            loss = torch.zeros(1, dtype=torch.float32, device=dev)
            _lib.check(lib.pdf_moe_combine_train(n, E, z.data_ptr(), r.data_ptr(), yt.data_ptr(), out.data_ptr(), loss.data_ptr(),
                                                 dz.data_ptr(), dr.data_ptr(), _lib.stream_ptr()), "pdf_moe_combine_train")
            for e, m in enumerate(mods):
                experts[m].backward(dz[:, e:e + 1].contiguous())
            router.backward(dr)
            opt.step([(q, g, lr) for t in list(experts.values()) + [router] for q, g in t.param_grads()])
            self.last_losses.append(loss)
        self._sweep = None

    def invalidate(self):
        self._sweep = None

    def _get_sweep(self) -> MoeSweep:
        if self._sweep is None:
            self._sweep = MoeSweep(self.model.state_dict(), list(self.modality_dims), device=get_torch_device())
        return self._sweep

    def predict_proba_sweep(self, X_dict: Dict[str, np.ndarray], masks_snm: np.ndarray, order: List[str]) -> np.ndarray:
        """X_dict {mod: [N,d]} UNMASKED features; masks_snm uint8 [S,N,len(order)] -> [S,N] f32, one launch."""
        sw = self._get_sweep()
        mk = np.stack([masks_snm[:, :, order.index(m)] for m in sw.mods], axis=2).astype(np.uint8)
        dev = sw.device
        Xd = {m: torch.as_tensor(np.asarray(X_dict[m]), dtype=torch.float32).to(dev) for m in sw.mods}
        return sw.forward(Xd, torch.from_numpy(np.ascontiguousarray(mk)).to(dev)).cpu().numpy()

    def _single(self, X_dict, mask):
        mods_in = list(X_dict.keys())
        if mods_in != sorted(mods_in):
            # the reference feeds the router mask columns in caller order but gates experts in sorted order
            # (models/moe.py:39-44); the two coincide on every call site (SURVEY.md A.7).  Refuse the ambiguous case.
            raise ValueError("MoEModel.predict_proba expects modality inputs in sorted(modality) order")
        N = int(next(iter(X_dict.values())).shape[0])
        m = np.ones((N, len(mods_in)), dtype=np.float32) if mask is None else np.asarray(mask, dtype=np.float32)
        mk = (m != 0).astype(np.uint8)[None]
        Xn = {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in X_dict.items()}
        return Xn, mk, mods_in

    def predict_proba(self, X_dict, mask=None):
        """X_dict {mod: FloatTensor [N,d]} (already multiplied by the mask by the caller, evaluate.py:59-61),
        mask FloatTensor [N,M] with columns in the X_dict key order the caller stacked them in."""
        Xn, mk, mods_in = self._single(X_dict, mask)
        return self.predict_proba_sweep(Xn, mk, mods_in)[0]

    def explain_sweep(self, X_dict: Dict[str, np.ndarray], masks_snm: np.ndarray, order: List[str], steps: int = 32) -> List[Dict]:
        """`explain` under every scenario mask of masks_snm (uint8 [S,N,len(order)], as predict_proba_sweep; X_dict unmasked) in
        one pdf_moe_explain call -> one explanation dict per scenario."""
        sw = self._get_sweep()
        mk = np.stack([masks_snm[:, :, order.index(m)] for m in sw.mods], axis=2).astype(np.uint8)
        dev = sw.device
        Xd = {m: torch.as_tensor(np.asarray(X_dict[m]), dtype=torch.float32).to(dev) for m in sw.mods}
        value, base, shap, ig = sw.explain(Xd, torch.from_numpy(np.ascontiguousarray(mk)).to(dev), steps)
        prob = value.cpu().numpy().astype(np.float64)
        shap = shap.cpu().numpy()
        ig = [t.cpu().numpy() for t in ig] if ig is not None else None
        b = float(base.item())
        return [{"prob": prob[s], "base_prob": b, "shapley": {m: shap[s, :, j] for j, m in enumerate(sw.mods)},
                 "ig": {m: ig[j][s] for j, m in enumerate(sw.mods)} if ig is not None else None} for s in range(prob.shape[0])]

    def explain(self, X_dict, mask=None, steps: int = 32) -> Dict:
        """Why each subject got its probability, for the arguments of `predict_proba`: prob [N] (predict_proba's, as float64),
        base_prob (the output for the all-zero input, every modality missing), shapley {mod: [N]} = exact Shapley values of the
        modalities for the probability (they add up to prob - base_prob; 0 for a missing modality), and ig {mod: [N, d_m]} =
        integrated gradients of the probability from the zero input with `steps` midpoints (None for steps = 0)."""
        Xn, mk, mods_in = self._single(X_dict, mask)
        return self.explain_sweep(Xn, mk, mods_in, steps)[0]

    def save(self, path):
        torch.save(self.model.state_dict(), path)

    @classmethod
    def load(cls, path, modality_dims, params):
        inst = cls(modality_dims, params)
        inst.model.load_state_dict(torch.load(path, map_location="cpu", weights_only=True))
        return inst

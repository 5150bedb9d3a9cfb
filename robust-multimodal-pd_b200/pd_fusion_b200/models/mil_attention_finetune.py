"""End-to-end ResNet2D + MIL attention model (reference: models/mil_attention_finetune.py, SURVEY.md 8a row a13).

Bags are volume paths (str / Path) or ready slice stacks (np.ndarray [L, H, W] in [0, 1]).

* `predict_proba` -- the inference path -- runs natively: volumes go through the batched CUDA pipeline (resample,
  normalise, slice select, resize, tcgen05 ResNet in eval mode) and ALL bags are pooled by one `pdf_mil_forward`
  launch, instead of the reference's per-bag, per-16-slice-chunk loop (`_forward_bags`, :135-162).
  `tta_inference > 1` re-augments each bag with `pdf_tta_augment` (unseeded Generator, as in the reference :267-272).
* `train` -- forward/backward with train-mode BatchNorm, focal/BCE loss, gradient clipping, Adam with two learning rates
  (:164-253) -- runs on the native kernels of training.py (ResNetTrainer, MilHeadTrainer, NativeAdam); the nn.Modules only
  hold the parameters.  The `state_dict` layout ({"backbone": ..., "attn": ...}) is the reference's.
* Path bags of one `predict_proba` / `train_step` call are prepared together on the device: one ragged decode -> resample ->
  slice select -> slice gather over volumes of any shapes (`_device_stacks`), the same slices `_bag_slices` returns per bag.
"""
from __future__ import annotations

import os
from pathlib import Path
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from .. import _lib
from ..backbone import ResNetEncoder
from ..data import openneuro_features as onf
from ..data.tta import TtaDraw, affine_matrix, params_bytes
from ..heads import MilHead, gradcam
from ..preprocess import VolumePreprocessor
from ..utils.torch_utils import get_torch_device
from .base import BaseModel
from .mil_attention import MILAttentionNet, _fill_explanation


def _is_path(bag) -> bool:
    return isinstance(bag, (str, os.PathLike))


def _pad_embeddings(embs: Sequence[torch.Tensor], dim: int, device):
    """Per-bag slice embeddings [L_i, D] -> zero-padded bags [n, Lmax, D] f32 and lengths [n] i32 on the device."""
    lmax = max(int(e.shape[0]) for e in embs)
    X = torch.zeros((len(embs), lmax, dim), dtype=torch.float32, device=device)
    for j, e in enumerate(embs):
        X[j, : e.shape[0]] = e
    return X, torch.tensor([int(e.shape[0]) for e in embs], dtype=torch.int32, device=device)


class MilAttentionFineTuneModel(BaseModel):
    def __init__(self, params: dict):
        p = self.params = params or {}
        self.backbone_name = p.get("backbone", "resnet50")
        self.target_shape = tuple(p.get("target_shape", (160, 160, 160)))
        axes, counts = p.get("slice_axes"), p.get("slice_counts")
        if axes and counts:
            self.axes, self.counts = [int(a) for a in axes], [int(c) for c in counts]
        else:
            self.axes, self.counts = [int(p.get("slice_axis", 2))], [int(p.get("slice_count", 48))]
        self.input_size = int(p.get("input_size", 224))
        self.slice_batch_size = int(p.get("slice_batch_size", 16))
        self.bag_batch_size = int(p.get("batch_size", 4))
        self.tta_inference = int(p.get("tta_inference", 1))
        self.aug = dict(max_rotation_deg=float(p.get("max_rotation_deg", 5.0)), max_translation=float(p.get("max_translation", 0.05)),
                        intensity_scale=float(p.get("intensity_scale", 0.1)), intensity_shift=float(p.get("intensity_shift", 0.1)),
                        noise_std=float(p.get("noise_std", 0.01)))
        self.missing_prob = float(p.get("missing_prob", 0.5))
        self.freeze_backbone_epochs = int(p.get("freeze_backbone_epochs", 2))
        self.train_aug = bool(p.get("train_aug", True))
        self.balanced_batches = bool(p.get("balanced_batches", False))
        self.loss_type = str(p.get("loss_type", "bce")).lower()
        self.focal_gamma = float(p.get("focal_gamma", 2.0))
        self.focal_alpha = p.get("focal_alpha")
        self.gated = bool(p.get("gated", False))
        self.device = get_torch_device()
        self.backbone, self.emb_dim, self.weights = onf._build_resnet_backbone(self.backbone_name, pretrained=bool(p.get("pretrained", True)))
        self.backbone = self.backbone.to(self.device).float()
        self.attn = MILAttentionNet(self.emb_dim, int(p.get("hidden_dim", 256)), int(p.get("attn_dim", 128)), float(p.get("dropout", 0.2)),
                                    gated=self.gated).to(self.device).float()
        self.mean_vals, self.std_vals = onf._mean_std(self.weights)
        # (the optimiser -- Adam, two learning-rate groups, L2 weight decay, `:73-79` -- is the native one of training.py, created
        #  on first use by _trainers(); its moments persist across train() calls like the reference's self.optimizer)
        self.pos_weight = None if (p.get("class_weight") == "balanced" or p.get("pos_weight") is None) else float(p["pos_weight"])
        self._native: Dict[str, object] = {}
        self._slicer: Optional[VolumePreprocessor] = None
        self._trainer = None

    # ------------------------------------------------------------------------------------------ native inference
    def invalidate(self):
        """Weights changed (training step, load): the lowered encoder / head are rebuilt on the next predict_proba."""
        self._native = {}

    def _precision(self) -> str:
        return os.environ.get("PD_FUSION_B200_PRECISION", "bf16")

    def _encoder(self, n_images: int) -> ResNetEncoder:
        key = ("enc", n_images)
        if key not in self._native:
            sd = {k: v for k, v in self.backbone.state_dict().items() if not k.startswith("fc.")}
            self._native[key] = ResNetEncoder(sd, n_images, self.input_size, self._precision(), "resnet50" if self.backbone_name == "resnet50"
                                              else "resnet18", self.device, mean=self.mean_vals, std=self.std_vals)
        return self._native[key]

    def _head(self) -> MilHead:
        if "head" not in self._native:
            self._native["head"] = MilHead(self.attn.state_dict(), self.gated, self.missing_prob, device=self.device)
        return self._native["head"]

    def _resizer(self, H: int, W: int) -> VolumePreprocessor:
        """A preprocessor instance used only for `resize_slices` / `tta_augment` of ready slice stacks."""
        bf16 = self._precision() == "bf16"
        key = ("resize", bf16)
        if key not in self._native:
            m, s = self.mean_vals, self.std_vals
            if bf16:
                m_avg, s_avg = sum(m) / 3.0, sum(s) / 3.0
                m, s = (m_avg,) * 3, (s_avg,) * 3
            self._native[key] = VolumePreprocessor((8, 8, 8), (8, 8, 8), (2,), (1,), self.input_size, m, s,
                                                   _lib.OUT_BF16_C1_PAD if bf16 else _lib.OUT_F32_NHWC3, 1, self.device)
        return self._native[key]

    def _bag_slices(self, bag) -> np.ndarray:
        """Normalised slice stack [L, H, W] f32 of one bag (the reference's `_load_bag`, without augmentation)."""
        if isinstance(bag, np.ndarray):
            return bag.astype(np.float32, copy=False)
        vol = onf._normalize_volume_for_resnet(onf._load_volume(bag, target_shape=self.target_shape))
        return np.concatenate([onf._select_slices(vol, a, c) for a, c in zip(self.axes, self.counts)], axis=0).astype(np.float32, copy=False)

    def _path_stacks(self, paths) -> List[torch.Tensor]:
        """`_bag_slices` of volume paths, computed together: ragged batches of stored volumes are decoded, resampled, normalised,
        sliced and gathered on the device ([n_i, H, W] f32 each, the valid slices of every axis group in order)."""
        bsz = onf._subject_batch()
        if not paths:
            return []
        if self._slicer is None:          # only resample / select / gather_slices are used: the network-input size is moot
            self._slicer = VolumePreprocessor(None, self.target_shape, self.axes, self.counts, 8, out_mode=_lib.OUT_F32_NHWC3,
                                              max_batch=bsz, device=self.device)
        pre = self._slicer
        out: List[torch.Tensor] = []
        for i in range(0, len(paths), bsz):
            raw = onf._decode_on_device([onf._read_volume_stored(p) for p in paths[i:i + bsz]], self.device)
            B = len(raw)
            pre.resample(raw)
            _, _, nslices = pre.select(B)
            slices = pre.gather_slices(B)
            ns = nslices.cpu().numpy()
            for b in range(B):
                offs = np.cumsum([0] + self.counts[:-1])
                out.append(torch.cat([slices[b, o:o + int(ns[b, a])] for a, o in enumerate(offs)], dim=0).clone())
        return out

    def _device_stacks(self, bags) -> List[Optional[torch.Tensor]]:
        """Slice stacks [L, H, W] f32 on the device of every bag (None stays None): path bags through `_path_stacks` in one go,
        tensors as they are, arrays uploaded."""
        from_paths = iter(self._path_stacks([b for b in bags if _is_path(b)]))
        out: List[Optional[torch.Tensor]] = []
        for bag in bags:
            if bag is None:
                out.append(None)
            elif _is_path(bag):
                out.append(next(from_paths))
            elif isinstance(bag, torch.Tensor):
                out.append(bag.to(device=self.device, dtype=torch.float32))
            else:
                out.append(torch.from_numpy(np.ascontiguousarray(self._bag_slices(bag))).to(self.device))
        return out

    def _capacity(self, longest: int) -> int:
        """Images per encoder pass: a FIXED capacity (bag_batch_size bags of the nominal length, at least 256 images), so that ONE
        encoder instance -- weights plus activation buffers -- serves every call whatever the number of live bags.  The reference
        goes bag by bag in 16-slice chunks (mil_attention_finetune.py:141-150); memory here is bounded the same way."""
        cap = int(os.environ.get("PD_FUSION_B200_FT_IMAGES", "0")) or max(256, self.bag_batch_size * int(sum(self.counts)))
        return max(cap, int(longest))

    def _embed_slices(self, stacks: Sequence[torch.Tensor], on_pass: Optional[Callable] = None) -> List[torch.Tensor]:
        """Per-slice embeddings of ready slice stacks ([L_i, H, W] f32 CUDA tensors in [0,1]): the bags go through ONE
        fixed-capacity encoder in groups of whole bags, the unused tail of the input buffer zeroed (as EmbeddingPipeline.embed does).
        on_pass(enc, first, embs), if given, runs after each encoder pass, while the pass's feature map is still in the encoder:
        bags [first, first + len(embs)) went through it, their rows in order from 0."""
        cap = self._capacity(max(int(s.shape[0]) for s in stacks))
        enc = self._encoder(cap)
        H, W = int(stacks[0].shape[1]), int(stacks[0].shape[2])
        pre = self._resizer(H, W)
        dst = enc.input_padded if enc.input_padded is not None else enc.input
        out: List[torch.Tensor] = []
        i = 0
        while i < len(stacks):
            j, total = i, 0
            while j < len(stacks) and total + int(stacks[j].shape[0]) <= cap:
                total += int(stacks[j].shape[0])
                j += 1
            allsl = torch.cat(list(stacks[i:j]), dim=0).contiguous().view(1, total, H, W)
            pre.resize_slices(allsl, out=dst[:total].view((1, total) + tuple(dst.shape[1:])))
            if total < cap:
                enc.input[total:].zero_()
            emb = enc.forward(None)[:total].clone()          # the encoder's output buffer is reused by the next group
            k = 0
            for s in stacks[i:j]:
                out.append(emb[k:k + int(s.shape[0])])
                k += int(s.shape[0])
            if on_pass is not None:
                on_pass(enc, i, out[i:j])
            i = j
        return out

    def _augment(self, stack: torch.Tensor, rng: np.random.Generator) -> torch.Tensor:
        """One random augmentation of a slice stack on the device (draw order of the reference's `_augment_slices`)."""
        L, H, W = (int(v) for v in stack.shape)
        a = self.aug
        angle = rng.uniform(-a["max_rotation_deg"], a["max_rotation_deg"])
        translate = rng.uniform(-a["max_translation"], a["max_translation"], size=2) * np.array([H, W])
        rot, offset = affine_matrix((H, W), angle, translate)
        scale = 1.0 + rng.uniform(-a["intensity_scale"], a["intensity_scale"])
        shift = rng.uniform(-a["intensity_shift"], a["intensity_shift"])
        noise = rng.normal(0.0, a["noise_std"], size=(L, H, W)) if a["noise_std"] > 0 else None
        params = torch.from_numpy(params_bytes([TtaDraw(rot, offset, float(scale), float(shift), None)])).to(self.device)
        nz = torch.from_numpy(noise[None]).to(self.device) if noise is not None else None
        return self._resizer(H, W).tta_augment(stack.view(1, L, H, W), params, nz)[0]

    def predict_proba(self, bags, masks=None):
        mri = masks["mri"] if isinstance(masks, dict) and "mri" in masks else None
        n = len(bags)
        out = np.full(n, self.missing_prob, dtype=np.float64)
        live = [i for i, b in enumerate(bags) if b is not None and not (mri is not None and mri[i] == 0)]
        if not live:
            return out
        self.backbone.eval()
        self.attn.eval()
        stacks = self._device_stacks([bags[i] for i in live])
        passes = max(1, self.tta_inference)
        acc = torch.zeros(len(live), dtype=torch.float32, device=self.device)
        head = self._head()
        rng = np.random.default_rng()
        for _ in range(passes):
            # the reference augments inside _load_bag only when train_aug is on AND the bag is a path (ndarray bags return before
            # the augmentation, mil_attention_finetune.py:114-125)
            cur = [self._augment(s, rng) if (self.tta_inference > 1 and self.train_aug and not isinstance(bags[i], np.ndarray)) else s
                   for s, i in zip(stacks, live)]
            X, lens = _pad_embeddings(self._embed_slices(cur), self.emb_dim, self.device)
            acc += head.forward(X, lens)
        out[live] = (acc / passes).cpu().numpy().astype(np.float64)
        return out

    def explain(self, bags, masks=None) -> dict:
        """Why each bag got its probability (bag and mask semantics of `predict_proba`):
        {"prob": [N] float64 (predict_proba's with tta_inference = 1; missing_prob for absent bags), "logit": [N] float64 (NaN where
         absent), and per bag (None where absent): "attention" / "contribution" np.ndarray [L_i] (attention weights a_l and
         a_l * (w_cls . h_l), which add up to logit - classifier bias), "slices" [L_i, H, W] (the stack `_bag_slices` returns) and
         "cam" [L_i, H, W]: the Grad-CAM map of the logit at the backbone's last stage, upsampled to the slice grid, unnormalised
         (a ReLU output)}.
        Explanations use no test-time augmentation, whatever tta_inference says, and the FP32 head arithmetic.  They run pass by
        pass inside the encoder's whole-bag grouping: after each pass, while its last feature map is live, the head's explanation
        (with the gradient of the logit with respect to every slice embedding) and pdf_gradcam of that pass's slices."""
        mri = masks["mri"] if isinstance(masks, dict) and "mri" in masks else None
        n = len(bags)
        out = {"prob": np.full(n, self.missing_prob, dtype=np.float64), "logit": np.full(n, np.nan, dtype=np.float64),
               "attention": [None] * n, "contribution": [None] * n, "slices": [None] * n, "cam": [None] * n}
        live = [i for i, b in enumerate(bags) if b is not None and not (mri is not None and mri[i] == 0)]
        if not live:
            return out
        self.backbone.eval()
        self.attn.eval()
        stacks = self._device_stacks([bags[i] for i in live])
        head = self._head()
        H, W = int(stacks[0].shape[1]), int(stacks[0].shape[2])

        def explain_pass(enc, first, embs):
            rows = live[first:first + len(embs)]
            X, lens = _pad_embeddings(embs, self.emb_dim, self.device)
            logit, attn, contrib, dX = head.explain(X, lens, need_grad=True)
            g = torch.cat([dX[j, : e.shape[0]] for j, e in enumerate(embs)], dim=0)
            cam, _ = gradcam(enc.feature_map()[: g.shape[0]], g, (H, W))
            lens_h = lens.cpu().numpy()
            _fill_explanation(out, rows, lens_h, logit, attn, contrib)
            cam = cam.cpu().numpy()
            k = 0
            for j, i in enumerate(rows):
                L = int(lens_h[j])
                out["cam"][i] = cam[k:k + L]
                out["slices"][i] = stacks[first + j].cpu().numpy()
                k += L

        self._embed_slices(stacks, on_pass=explain_pass)
        return out

    # ------------------------------------------------------------------------------------------ training (native kernels)
    def _train_resizer(self) -> VolumePreprocessor:
        """slices [L,H,W] in [0,1] -> the reference's float32 3-channel network input [L,S,S,3] ((x-mean)/std per channel)."""
        if "resize_f32" not in self._native:
            self._native["resize_f32"] = VolumePreprocessor((8, 8, 8), (8, 8, 8), (2,), (1,), self.input_size, self.mean_vals, self.std_vals,
                                                            _lib.OUT_F32_NHWC3, 1, self.device)
        return self._native["resize_f32"]

    def _epoch_batches(self, y: np.ndarray) -> List[np.ndarray]:
        n, bs = len(y), self.bag_batch_size
        pos, neg = np.where(y >= 0.5)[0], np.where(y < 0.5)[0]
        if self.balanced_batches and len(pos) and len(neg):
            rng, half = np.random.default_rng(), max(1, bs // 2)
            return [np.concatenate([rng.choice(pos, size=half, replace=len(pos) < half),
                                    rng.choice(neg, size=bs - half, replace=len(neg) < bs - half)]) for _ in range(max(1, -(-n // bs)))]
        order = np.random.permutation(n)
        return [order[s:s + bs] for s in range(0, n, bs)]

    def _trainers(self):
        """Native trainers over the live nn.Module parameters (created once; Adam state persists across train() calls like the
        reference's self.optimizer)."""
        if self._trainer is None:
            from ..training import MilHeadTrainer, NativeAdam, ResNetTrainer
            p = self.params
            rt = ResNetTrainer(self.backbone, "resnet50" if self.backbone_name == "resnet50" else "resnet18", self.input_size)
            ht = MilHeadTrainer(self.attn, self.gated)
            # (the trainers keep every parameter / gradient of a module in one flat buffer: one Adam launch per group)
            opt = NativeAdam([([rt.flat_param], float(p.get("lr_backbone", 1e-4))), ([ht.flat_param], float(p.get("lr", 3e-4)))],
                             weight_decay=float(p.get("weight_decay", 1e-3)))
            self._trainer = (rt, ht, opt)
        return self._trainer

    def train_step(self, batch_bags, y_batch: np.ndarray, frozen: bool, clip=None, augment: bool = True):
        """One optimisation step on a batch of bags (reference: the loop body of train(), mil_attention_finetune.py:206-229):
        slices -> network input -> backbone in TRAIN mode, 16-slice chunks -> MIL head -> loss -> backward -> clip -> Adam.
        Returns (loss, probabilities) as device tensors."""
        rt, ht, opt = self._trainers()
        pre = self._train_resizer()
        stacks, groups = [], [0]
        for bag, sl in zip(batch_bags, self._device_stacks(batch_bags)):
            if bag is None:
                stacks.append(None)
                continue
            if augment and self.train_aug and not isinstance(bag, (np.ndarray, torch.Tensor)):   # the reference augments bags it loads itself
                sl = self._augment(sl, np.random.default_rng())
            stacks.append(sl)
            L = int(sl.shape[0])
            for c0 in range(0, L, self.slice_batch_size):                          # BatchNorm statistics per chunk of one bag
                groups.append(groups[-1] + min(self.slice_batch_size, L - c0))
        live = [s for s in stacks if s is not None]
        total = groups[-1]
        H, W = int(live[0].shape[1]), int(live[0].shape[2])
        x = torch.empty((total, self.input_size, self.input_size, 3), dtype=torch.float32, device=self.device)
        pre.resize_slices(torch.cat(live, dim=0).contiguous().view(1, total, H, W), out=x.view(1, total, self.input_size, self.input_size, 3))
        emb = rt.forward(x, groups)
        B, lmax = len(stacks), max(int(s.shape[0]) for s in live)
        X = torch.zeros((B, lmax, self.emb_dim), dtype=torch.float32, device=self.device)
        lens = torch.zeros(B, dtype=torch.int32)
        k = 0
        for i, sl in enumerate(stacks):
            if sl is not None:
                L = int(sl.shape[0])
                X[i, :L].copy_(emb[k:k + L])
                lens[i] = L
                k += L
        ht.zero_grad()
        loss, prob, dX = ht.forward_backward(X, lens, torch.from_numpy(np.asarray(y_batch, dtype=np.float32)), self.loss_type, self.pos_weight,
                                             self.focal_gamma, self.focal_alpha, need_dx=not frozen)
        pg = [(ht.flat_param, ht.flat_grad, opt.groups[1][1])]
        if not frozen:
            rt.zero_grad()
            demb = torch.empty((total, self.emb_dim), dtype=torch.float32, device=self.device)
            k = 0
            for i, sl in enumerate(stacks):
                if sl is not None:
                    L = int(sl.shape[0])
                    demb[k:k + L].copy_(dX[i, :L])
                    k += L
            # data-parallel over bags under torchrun: every residual block's gradients are averaged on a side stream as soon as the
            # backward has left the block (training.BucketedAllReduce); the head's small buffer follows in one call
            from ..training import BucketedAllReduce
            reducer = BucketedAllReduce(rt.flat_grad)
            rt.backward(demb, reducer)
            reducer.finish()
            pg = [(rt.flat_param, rt.flat_grad, opt.groups[0][1])] + pg
        from ..training import allreduce_mean
        allreduce_mean([ht.flat_grad])
        scale = opt.clip([g for _, g, _ in pg], float(clip)) if clip else None
        opt.step(pg, scale)
        if not frozen:
            rt.sync_weights()
        return loss, prob

    def train(self, bags, y, val_data=None):
        y = np.asarray(y, dtype=np.float32)
        p = self.params
        clip, patience = p.get("max_grad_norm"), int(p.get("early_stopping_patience", 0))
        if self.pos_weight is None and p.get("class_weight") == "balanced" and (y == 1).sum() > 0:
            self.pos_weight = float((y == 0).sum()) / float((y == 1).sum())
        best_auc, best, stale = -1.0, None, 0
        for epoch in range(int(p.get("epochs", 20))):
            self.backbone.train()
            self.attn.train()
            frozen = epoch < self.freeze_backbone_epochs
            for q in self.backbone.parameters():
                q.requires_grad = not frozen
            for sel in self._epoch_batches(y):
                self.train_step([bags[i] for i in sel], y[sel], frozen, clip)
            self.invalidate()
            if val_data is not None and patience > 0:
                from sklearn.metrics import roc_auc_score
                try:
                    auc = float(roc_auc_score(val_data[1], self.predict_proba(val_data[0])))
                except Exception:
                    auc = -1.0
                if auc > best_auc:
                    # (the reference keeps `state_dict()` by reference, which aliases the live parameters -- SURVEY.md C.5;
                    #  restoring it is a no-op there.  Same here: no clone.)
                    best_auc, stale = auc, 0
                    best = {"backbone": self.backbone.state_dict(), "attn": self.attn.state_dict()}
                else:
                    stale += 1
                    if stale >= patience:
                        break
        if best is not None:
            self.backbone.load_state_dict(best["backbone"])
            self.attn.load_state_dict(best["attn"])
        self.invalidate()

    def save(self, path):
        torch.save({"backbone": self.backbone.state_dict(), "attn": self.attn.state_dict()}, path)

    @classmethod
    def load(cls, path, params):
        inst = cls(params)
        state = torch.load(path, map_location="cpu", weights_only=True)
        inst.backbone.load_state_dict(state["backbone"])
        inst.attn.load_state_dict(state["attn"])
        inst.invalidate()
        return inst

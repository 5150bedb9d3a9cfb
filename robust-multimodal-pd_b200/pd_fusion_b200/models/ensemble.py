"""Deep ensembles of the fusion and MIL heads: the same head trained from several seeds, as one batched device run.

`HeadEnsemble(member_cls, args, seeds)` holds E ordinary instances of `member_cls` (ModalityDropoutModel, MoEModel or
MilAttentionModel) built from the same constructor arguments.  `train` runs the member class's own training loop for all members in
lockstep: every launch of a step covers all members (csrc/train.cu), so a step costs the same number of kernel launches whatever E
is.  Member e ends up with the weights of

    torch.manual_seed(s_e); np.random.seed(s_e); m = member_cls(*args); m.train(*train_args)

because each member draws from private streams in the single path's order: a CPU torch.Generator captured right after its weights
were built (initial weights, then every epoch's torch.randperm), a CUDA torch.Generator seeded s_e (the dropout masks) and an
np.random.RandomState(s_e) (ModDrop's modality drops).  The global torch and numpy RNGs are left untouched.

Inference runs each member's own sweep into one [E, S, N] buffer; `predict_proba[_sweep]` return the float64 mean of the members
(summed in ascending member order), so the evaluation helpers accept an ensemble where they accept a member, and
`predict_ensemble_sweep` adds the per-subject spread of the members (pdf_ensemble_stats).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import _lib
from ..heads import mc_dicts
from ..utils.torch_utils import get_torch_device
from .fusion_moddrop import ModalityDropoutModel
from .mil_attention import MilAttentionModel, _pad_bags
from .moe import MoEModel

_SUPPORTED = (ModalityDropoutModel, MoEModel, MilAttentionModel)
MAX_MEMBERS = 1024


class HeadEnsemble:
    def __init__(self, member_cls, args: Sequence, seeds: Sequence[int]):
        if member_cls not in _SUPPORTED:
            raise ValueError(f"HeadEnsemble supports {', '.join(c.__name__ for c in _SUPPORTED)}, not {getattr(member_cls, '__name__', member_cls)}")
        seeds = [int(s) for s in seeds]
        if not 1 <= len(seeds) <= MAX_MEMBERS:
            raise ValueError(f"HeadEnsemble needs 1..{MAX_MEMBERS} seeds, got {len(seeds)}")
        if len(set(seeds)) != len(seeds):
            raise ValueError(f"HeadEnsemble seeds must be distinct, got {seeds}")
        self.member_cls, self.args, self.seeds = member_cls, tuple(args), seeds
        self._members, self._cpu_gens = [], []
        for s in seeds:
            with torch.random.fork_rng(devices=[]):
                torch.random.default_generator.manual_seed(s)
                self._members.append(member_cls(*self.args))
                g = torch.Generator()
                g.set_state(torch.get_rng_state())
            self._cpu_gens.append(g)
        self._np_rngs = [np.random.RandomState(s) for s in seeds]
        self._cuda_gens: Optional[List[torch.Generator]] = None
        self._state = None          # (BatchedGemm, trainer(s), BatchedAdam): built on the first train(), Adam state persists
        self.last_losses: List[torch.Tensor] = []

    @property
    def members(self) -> List:
        """the E trained heads, ordinary instances of member_cls (predict_proba, explain, predict_uncertainty, save work as usual)"""
        return list(self._members)

    def __len__(self) -> int:
        return len(self._members)

    # -- training -------------------------------------------------------------------------------------------------------------------
    def _setup(self, dev):
        from ..training import BatchedAdam, BatchedGemm, BatchedMilHeadTrainer, BatchedMlpTrainer, flatten_members
        if self._cuda_gens is None:
            self._cuda_gens = [torch.Generator(device=dev) for _ in self.seeds]
            for g, s in zip(self._cuda_gens, self.seeds):
                g.manual_seed(s)
        if self._state is not None:
            return self._state
        for m in self._members:
            m.model.to(dev).float()
        flat, offs = flatten_members([dict(m.model.named_parameters()) for m in self._members])
        bg = BatchedGemm(flat, torch.zeros_like(flat), offs)
        m0, p = self._members[0], self._members[0].params
        if self.member_cls is ModalityDropoutModel:
            tr = BatchedMlpTrainer(m0.model.net, "net.", bg)
            lr = float(p["lr"])
        elif self.member_cls is MoEModel:
            mods = sorted(m0.modality_dims)
            tr = ({m: BatchedMlpTrainer(m0.model.experts[m].net, f"experts.{m}.net.", bg) for m in mods},
                  BatchedMlpTrainer(m0.model.router, "router.", bg))
            lr = float(p["lr"])
        else:
            tr = BatchedMilHeadTrainer(m0.model, m0.gated, bg)
            lr = float(p.get("lr", 1e-3))
        self._state = (bg, tr, BatchedAdam(flat, lr, weight_decay=float(p.get("weight_decay", 0.0))))
        return self._state

    def train(self, *args, **kwargs):
        """The member class's `train(...)` arguments; trains every member as that class's loop would, all in lockstep."""
        dev = get_torch_device()
        bg, tr, opt = self._setup(dev)
        if self.member_cls is ModalityDropoutModel:
            self._train_moddrop(dev, bg, tr, opt, *args, **kwargs)
        elif self.member_cls is MoEModel:
            self._train_moe(dev, bg, tr, opt, *args, **kwargs)
        else:
            self._train_mil(dev, bg, tr, opt, *args, **kwargs)
        for m in self._members:
            m.invalidate()

    def _record(self, losses: List[torch.Tensor], active_per_step: Optional[List[Tuple[bool, ...]]] = None):
        """last_losses: [E] loss tensor per step; each member's last_losses: its own [1] losses of the steps it trained"""
        self.last_losses = losses
        for e, m in enumerate(self._members):
            m.last_losses = [l[e:e + 1] for i, l in enumerate(losses) if active_per_step is None or active_per_step[i][e]]

    def _train_moddrop(self, dev, bg, tr, opt, X, y, val_data=None):
        """models/fusion_moddrop.py's loop: per epoch a torch.randperm per member, minibatches with one modality-drop draw per
        modality per batch (numpy), nn.BCELoss, Adam"""
        lib, E = _lib.load(), len(self._members)
        m0 = self._members[0]
        net0 = m0.model
        Xt = torch.as_tensor(np.asarray(X), dtype=torch.float32).to(dev)
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32).to(dev)
        n, F = int(Xt.shape[0]), int(Xt.shape[1])
        rate, bs = m0.params.get("moddrop_rate", 0.2), m0.params.get("batch_size", 32)
        M, nb = len(net0.mod_names), (n + bs - 1) // bs
        losses = []
        for _ in range(m0.params["epochs"]):
            for m in self._members:
                m.model.train()
            order = torch.stack([torch.randperm(n, generator=g) for g in self._cpu_gens]).to(dev)          # [E, n]
            # the epoch's modality drops: member e's RandomState draws them batch by batch, modality by modality, as the single loop
            drop = np.stack([r.rand(nb * M).reshape(nb, M) < rate for r in self._np_rngs])                 # [E, nb, M]
            keep = np.ones((E, nb, F), dtype=np.float32)
            for j, mod in enumerate(net0.mod_names):
                a, b = net0.slices[mod]
                keep[:, :, a:b] = np.where(drop[:, :, j:j + 1], 0.0, 1.0)
            keep = torch.from_numpy(keep).to(dev)
            for bi, i in enumerate(range(0, n, bs)):
                sel = order[:, i:i + bs]
                xb, yb = Xt[sel].contiguous(), yt[sel].contiguous()                                       # [E, b, F], [E, b]
                b = int(xb.shape[1])
                kb = keep[:, bi:bi + 1, :].expand(E, b, F).contiguous()
                _lib.check(lib.pdf_mul_f32(xb.data_ptr(), kb.data_ptr(), xb.numel(), _lib.stream_ptr()), "pdf_mul_f32")
                bg.flat_grad.zero_()
                z = tr.forward(xb, self._cuda_gens)
                prob, dz = torch.empty((E, b), dtype=torch.float32, device=dev), torch.empty((E, b, 1), dtype=torch.float32, device=dev)
                loss = torch.empty(E, dtype=torch.float32, device=dev)
                _lib.check(lib.pdf_bce_sigmoid_train_batched(E, b, z.data_ptr(), yb.data_ptr(), b, prob.data_ptr(), loss.data_ptr(),
                                                             dz.data_ptr(), _lib.stream_ptr()), "pdf_bce_sigmoid_train_batched")
                tr.backward(dz)
                opt.step(bg.flat_grad)
                losses.append(loss)
        self._record(losses)

    def _train_moe(self, dev, bg, tr, opt, X_dict, y, mask, val_data=None):
        """models/moe.py's loop: full-batch steps; the inputs, the availability mask and the labels are shared by every member"""
        lib, E = _lib.load(), len(self._members)
        experts, router = tr
        mods = sorted(X_dict)
        X = {m: torch.as_tensor(np.asarray(X_dict[m]), dtype=torch.float32).to(dev).contiguous() for m in mods}
        mk = torch.as_tensor(np.asarray(mask), dtype=torch.float32).to(dev).contiguous()
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32).to(dev).contiguous()
        n, M = int(yt.shape[0]), len(mods)
        losses = []
        for _ in range(self._members[0].params["epochs"]):
            for m in self._members:
                m.model.train()
            bg.flat_grad.zero_()
            z = torch.cat([experts[m].forward(X[m]) for m in mods], dim=2).contiguous()          # [E, n, M] expert logits
            r = router.forward(mk)                                                                # [E, n, M] router logits
            out, dz, dr = torch.empty((E, n), dtype=torch.float32, device=dev), torch.empty_like(z), torch.empty_like(r)
            loss = torch.empty(E, dtype=torch.float32, device=dev)
            _lib.check(lib.pdf_moe_combine_train_batched(E, n, M, z.data_ptr(), r.data_ptr(), yt.data_ptr(), 0, out.data_ptr(), loss.data_ptr(),
                                                         dz.data_ptr(), dr.data_ptr(), _lib.stream_ptr()), "pdf_moe_combine_train_batched")
            for j, m in enumerate(mods):
                experts[m].backward(dz[:, :, j:j + 1].contiguous())
            router.backward(dr)
            opt.step(bg.flat_grad)
            losses.append(loss)
        self._record(losses)

    def _val_probs(self, bags, active: List[bool]) -> Dict[int, np.ndarray]:
        """every active member's predict_proba(bags), the bags padded and uploaded once"""
        n = len(bags)
        live = [i for i, b in enumerate(bags) if b is not None]
        out = {}
        X = lens = None
        if live:
            _, X, lens = self._members[0]._upload(bags, live)
        for e, m in enumerate(self._members):
            if not active[e]:
                continue
            p = np.full(n, m.missing_prob, dtype=np.float64)
            if live:
                p[live] = m._get_head().forward(X, lens).cpu().numpy().astype(np.float64)
            out[e] = p
        return out

    def _train_mil(self, dev, bg, tr, opt, bags, y, val_data=None):
        """models/mil_attention.py's loop: per epoch a torch.randperm per member, minibatches (BCE x pos_weight), optional
        clip_grad_norm_ per member, Adam, and early stopping on each member's own validation AUC.  A stopped member keeps its
        weights and Adam moments; as in the reference the final weights are those of the last epoch a member trained."""
        from sklearn.metrics import roc_auc_score
        E = len(self._members)
        m0 = self._members[0]
        Xp, Mp = _pad_bags(bags)
        Xt = torch.from_numpy(Xp).to(dev)
        lens_all = torch.from_numpy(Mp.sum(axis=1).astype(np.int32)).to(dev)
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32, device=dev)
        p = m0.params
        bs, epochs = int(p.get("batch_size", 16)), int(p.get("epochs", 30))
        clip, patience = p.get("max_grad_norm"), int(p.get("early_stopping_patience", 0))
        if m0.pos_weight is None and p.get("class_weight") == "balanced":
            pos, neg = float((yt == 1).sum()), float((yt == 0).sum())
            if pos > 0:
                for m in self._members:
                    m.pos_weight = neg / pos
        n = int(Xt.shape[0])
        active = [True] * E
        best_auc, bad = [-1.0] * E, [0] * E
        orders: List[Optional[torch.Tensor]] = [None] * E
        losses, steps_active = [], []
        self.stopped_epoch = [None] * E
        for epoch in range(epochs):
            if not any(active):
                break
            for m in self._members:
                m.model.train()
            for e in range(E):       # a stopped member draws nothing more; its (discarded) steps reuse its last permutation
                if active[e] or orders[e] is None:
                    orders[e] = torch.randperm(n, generator=self._cpu_gens[e])
            order = torch.stack(orders).to(dev)
            flags = tuple(active)
            for i in range(0, n, bs):
                sel = order[:, i:i + bs]
                bg.flat_grad.zero_()
                loss, _ = tr.forward_backward(Xt[sel], lens_all[sel], yt[sel], m0.pos_weight, self._cuda_gens)
                scale = opt.clip(bg.flat_grad, float(clip)) if clip else None
                opt.step(bg.flat_grad, scale, flags)
                losses.append(loss)
                steps_active.append(flags)
            for m in self._members:
                m.invalidate()
            if val_data is not None and patience > 0:
                probs = self._val_probs(val_data[0], active)
                for e, pr in probs.items():
                    try:
                        auc = float(roc_auc_score(val_data[1], pr))
                    except Exception:
                        auc = -1.0
                    if auc > best_auc[e]:
                        best_auc[e], bad[e] = auc, 0
                    else:
                        bad[e] += 1
                        if bad[e] >= patience:
                            active[e] = False
                            self.stopped_epoch[e] = epoch
        self._record(losses, steps_active)

    # -- inference ------------------------------------------------------------------------------------------------------------------
    def _member_probs(self, *args) -> Tuple[torch.Tensor, np.ndarray]:
        """(device f32 [E, S, N], host [E, S, N]): every member's predict_proba_sweep(*args), the inputs uploaded once and one sweep
        launch per member.  The host array has the dtype and values of the members' own predict_proba_sweep."""
        E = len(self._members)
        m0 = self._members[0]
        if self.member_cls is MilAttentionModel:
            bags, mri_masks = args
            n = len(bags)
            S = 1 if mri_masks is None else int(np.asarray(mri_masks).shape[0])
            have = [i for i, b in enumerate(bags) if b is not None]
            if mri_masks is not None:
                mm = np.asarray(mri_masks)
                have = [i for i in have if mm[:, i].any()]
            host = np.stack([np.full((S, n), m.missing_prob, dtype=np.float64) for m in self._members])
            dev = get_torch_device()
            full = torch.empty((E, S, n), dtype=torch.float32, device=dev)
            for e, m in enumerate(self._members):
                full[e].fill_(m.missing_prob)
            if have:
                _, X, lens = m0._upload(bags, have)
                live = None if mri_masks is None else torch.from_numpy(np.ascontiguousarray(np.asarray(mri_masks)[:, have] != 0).astype(np.uint8))
                buf = torch.empty((E, S, len(have)), dtype=torch.float32, device=dev)
                for e, m in enumerate(self._members):
                    m._get_head().sweep(X, lens, live, S, out=buf[e])
                full[:, :, have] = buf
                host[:, :, have] = buf.cpu().numpy().astype(np.float64)
            return full, host
        if self.member_cls is ModalityDropoutModel:
            X, masks_snm, order = args
            sw0 = m0._get_sweep()
            mk = torch.from_numpy(m0._sweep_masks(masks_snm, order)).to(sw0.device)
            Xd = torch.as_tensor(np.asarray(X), dtype=torch.float32).to(sw0.device)
        else:
            X, masks_snm, order = args
            sw0 = m0._get_sweep()
            mk = torch.from_numpy(np.ascontiguousarray(np.stack([masks_snm[:, :, order.index(m)] for m in sw0.mods], axis=2).astype(np.uint8)))
            mk = mk.to(sw0.device)
            Xd = {m: torch.as_tensor(np.asarray(X[m]), dtype=torch.float32).to(sw0.device) for m in sw0.mods}
        S, N = int(mk.shape[0]), int(mk.shape[1])
        buf = torch.empty((E, S, N), dtype=torch.float32, device=sw0.device)
        for e, m in enumerate(self._members):
            m._get_sweep().forward(Xd, mk, out=buf[e])
        return buf, buf.cpu().numpy()

    def predict_member_proba_sweep(self, *args) -> np.ndarray:
        """[E, S, N]: member e's predict_proba_sweep(*args) (the member class's arguments) in row e"""
        return self._member_probs(*args)[1]

    @staticmethod
    def _mean(host: np.ndarray) -> np.ndarray:
        acc = host[0].astype(np.float64)
        for e in range(1, host.shape[0]):
            acc = acc + host[e]
        return acc / host.shape[0]

    def predict_proba_sweep(self, *args) -> np.ndarray:
        """The member class's predict_proba_sweep arguments -> [S, N] float64: the mean of the members' probabilities, summed in
        ascending member order"""
        return self._mean(self._member_probs(*args)[1])

    def predict_ensemble_sweep(self, *args) -> Tuple[np.ndarray, List[Dict[str, np.ndarray]]]:
        """The member class's predict_proba_sweep arguments -> (member probabilities [E, S, N], one dict per scenario with [N]
        float64 "mean", "std" (population, over the members), "entropy" (of the mean, nats), "expected_entropy" (mean member
        entropy) and "mutual_info" (max(0, entropy - expected_entropy): the members' disagreement)).  The statistics use Monte-Carlo
        dropout's formulas (pdf_ensemble_stats) in float64 over the members' float32 probabilities, so equal members give exactly
        std = mutual_info = 0; for MIL a missing bag counts as float32(missing_prob)."""
        dev_probs, host = self._member_probs(*args)
        E, S, N = (int(v) for v in dev_probs.shape)
        stats = torch.empty((S, N, 5), dtype=torch.float64, device=dev_probs.device)
        lib = _lib.load()
        _lib.check(lib.pdf_ensemble_stats(E, S * N, dev_probs.data_ptr(), stats.data_ptr(), _lib.stream_ptr()), "pdf_ensemble_stats")
        return host, mc_dicts(stats, None)

    def _single_args(self, *args, **kwargs):
        """predict_proba's arguments (the member class's) -> predict_proba_sweep's, one scenario"""
        m0 = self._members[0]
        if self.member_cls is ModalityDropoutModel:
            X = np.asarray(args[0])
            masks = args[1] if len(args) > 1 else kwargs.get("masks")
            return X, m0._single_mask(X.shape[0], masks), m0._get_sweep().mods
        if self.member_cls is MoEModel:
            mask = args[1] if len(args) > 1 else kwargs.get("mask")
            return m0._single(args[0], mask)
        bags = args[0]
        masks = args[1] if len(args) > 1 else kwargs.get("masks")
        mri = masks["mri"] if isinstance(masks, dict) and "mri" in masks else None
        return list(bags), None if mri is None else np.asarray(mri)[None]

    def predict_proba(self, *args, **kwargs) -> np.ndarray:
        """The member class's predict_proba arguments -> [N] float64 mean of the members' probabilities"""
        return self.predict_proba_sweep(*self._single_args(*args, **kwargs))[0]

    # -- persistence ----------------------------------------------------------------------------------------------------------------
    def save(self, path):
        torch.save({"seeds": list(self.seeds),
                    "members": [{k: v.detach().cpu().clone() for k, v in m.model.state_dict().items()} for m in self._members]}, path)

    @classmethod
    def load(cls, path, member_cls, args) -> "HeadEnsemble":
        d = torch.load(path, map_location="cpu", weights_only=True)
        ens = cls(member_cls, args, d["seeds"])
        for m, sd in zip(ens._members, d["members"]):
            m.model.load_state_dict(sd)
            m.invalidate()
        return ens

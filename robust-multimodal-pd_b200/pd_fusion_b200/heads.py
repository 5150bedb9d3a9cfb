"""Host side of K3/K4: thin wrappers that marshal state_dict tensors into the C structs of
pdf_mil_forward / pdf_mil_explain / pdf_gradcam / pdf_moddrop_sweep / pdf_moe_sweep / pdf_moddrop_explain / pdf_moe_explain /
pdf_moddrop_mc / pdf_mil_mc.  No arithmetic happens here.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib


MC_STATS = ("mean", "std", "entropy", "expected_entropy", "mutual_info")     # the last axis of pdf_moddrop_mc / pdf_mil_mc's stats


def mc_dicts(stats: torch.Tensor, samples: Optional[torch.Tensor]) -> List[Dict[str, np.ndarray]]:
    """stats [S, N, 5] (and samples [S, N, T] or None) of an `mc` call -> one dict per scenario: the five statistics as [N] float64
    arrays (MC_STATS order), plus "samples" [N, T] float64 when samples were returned."""
    st = stats.cpu().numpy()
    sm = samples.cpu().numpy().astype(np.float64) if samples is not None else None
    out = []
    for s in range(st.shape[0]):
        d = {k: st[s, :, j].copy() for j, k in enumerate(MC_STATS)}
        if sm is not None:
            d["samples"] = sm[s]
        out.append(d)
    return out


def _dev_f32(t, device) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t))
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


class MilHead:
    """MILAttentionNet (models/mil_attention.py:10-51) in eval mode for a batch of padded bags.

    precision "fp32": FFMA GEMMs, <= 5e-6 against the reference; "tf32": both linear layers as tcgen05 kind::tf32 GEMMs on the
    f32 bags (the throughput path; needs H, (2)A in {64,128,256} and D, H multiples of 32 -- `tensor_path_ok`)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], gated: bool, missing_prob: float = 0.5, device=None,
                 precision: str = "fp32"):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        g = {k: _dev_f32(v, self.device) for k, v in state_dict.items()}
        self._keep = g
        w = _lib.MilWeights()
        w.H, w.D = g["instance.0.weight"].shape
        w.gated = 1 if gated else 0
        w.w_inst, w.b_inst = g["instance.0.weight"].data_ptr(), g["instance.0.bias"].data_ptr()
        if gated:
            w.A = g["attn_v.0.weight"].shape[0]
            # [W_v; W_u] and [b_v; b_u] packed: the tensor path runs both attention layers as ONE [2A, H] GEMM
            g["_attn_vu.weight"] = torch.cat([g["attn_v.0.weight"], g["attn_u.0.weight"]], dim=0).contiguous()
            g["_attn_vu.bias"] = torch.cat([g["attn_v.0.bias"], g["attn_u.0.bias"]], dim=0).contiguous()
            esz = 4
            w.w_v, w.b_v = g["_attn_vu.weight"].data_ptr(), g["_attn_vu.bias"].data_ptr()
            w.w_u, w.b_u = w.w_v + int(w.A) * int(w.H) * esz, w.b_v + int(w.A) * esz
            w.w_w, w.b_w = g["attn_w.weight"].data_ptr(), g["attn_w.bias"].data_ptr()
        else:
            w.A = g["attn.0.weight"].shape[0]
            w.w_v, w.b_v = g["attn.0.weight"].data_ptr(), g["attn.0.bias"].data_ptr()
            w.w_u, w.b_u = None, None
            w.w_w, w.b_w = g["attn.2.weight"].data_ptr(), g["attn.2.bias"].data_ptr()
        w.w_cls, w.b_cls = g["classifier.0.weight"].data_ptr(), g["classifier.0.bias"].data_ptr()
        w.missing_prob = float(missing_prob)
        self.w = w
        self.D = int(w.D)
        na = int(w.A) * (2 if gated else 1)
        self.tensor_path_ok = int(w.H) in (64, 128, 256) and na in (64, 128, 256) and self.D % 32 == 0 and int(w.H) % 32 == 0
        if precision not in ("fp32", "tf32"):
            raise ValueError("precision must be 'fp32' or 'tf32'")
        if precision == "tf32" and not self.tensor_path_ok:
            raise ValueError("the tf32 tensor path needs H and (2)A in {64,128,256}, D and H multiples of 32")
        self.precision = precision
        self._ws: Optional[torch.Tensor] = None

    def _workspace(self, n: int, lmax: int, device) -> torch.Tensor:
        need = int(self.lib.pdf_mil_workspace_bytes(C.byref(self.w), n, lmax))
        if self._ws is None or self._ws.numel() < need or self._ws.device != device:
            self._ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self._ws

    def sweep(self, bags: torch.Tensor, lens: torch.Tensor, live: Optional[torch.Tensor] = None, n_scenarios: int = 1,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """bags [n, Lmax, D] f32 cuda (zero padded), lens [n] i32 (0 = no bag), live [S, n] u8 (1 = the bag is present under
        scenario s; None = present everywhere) -> prob [S, n] f32: ONE projection + pooling pass for all scenarios."""
        if bags.dtype != torch.float32 or not bags.is_cuda or not bags.is_contiguous() or bags.shape[2] != self.D:
            raise ValueError("bags must be a contiguous float32 CUDA tensor [n, Lmax, D]")
        n, lmax = int(bags.shape[0]), int(bags.shape[1])
        lens = lens.to(device=bags.device, dtype=torch.int32).contiguous()
        if live is not None:
            live = live.to(device=bags.device, dtype=torch.uint8).contiguous()
            n_scenarios = int(live.shape[0])
            if tuple(live.shape) != (n_scenarios, n):
                raise ValueError("live must be [S, n]")
        ws = self._workspace(n, lmax, bags.device)
        prob = out if out is not None else torch.empty((n_scenarios, n), dtype=torch.float32, device=bags.device)
        prec = _lib.PREC_TF32 if self.precision == "tf32" else _lib.PREC_F32
        _lib.check(self.lib.pdf_mil_sweep(C.byref(self.w), n, lmax, bags.data_ptr(), lens.data_ptr(), n_scenarios, _lib.ptr(live), prec,
                                          ws.data_ptr(), prob.data_ptr(), _lib.stream_ptr()), "pdf_mil_sweep")
        return prob

    def forward(self, bags: torch.Tensor, lens: torch.Tensor) -> torch.Tensor:
        """bags [n, Lmax, D] f32 cuda (zero padded), lens [n] i32 cuda (0 = missing) -> prob [n] f32."""
        return self.sweep(bags, lens)[0]

    def explain(self, bags: torch.Tensor, lens: torch.Tensor, need_grad: bool = False):
        """bags [n, Lmax, D] f32 cuda (zero padded), lens [n] i32 (0 = missing) -> device tensors (logit [n], attn [n, Lmax],
        contrib [n, Lmax], dX [n, Lmax, D] or None) of pdf_mil_explain: attention weights, per-instance logit contributions
        (sum + b_cls = logit), and with need_grad the gradient of the logit with respect to every instance.  Always the FP32 head
        arithmetic, whatever `precision` says: sigmoid(logit) is the probability of the "fp32" sweep.  Missing bags: NaN logit,
        zero attention, contributions and gradient."""
        if bags.dtype != torch.float32 or not bags.is_cuda or not bags.is_contiguous() or bags.shape[2] != self.D:
            raise ValueError("bags must be a contiguous float32 CUDA tensor [n, Lmax, D]")
        n, lmax = int(bags.shape[0]), int(bags.shape[1])
        lens = lens.to(device=bags.device, dtype=torch.int32).contiguous()
        need = int(self.lib.pdf_mil_explain_workspace_bytes(C.byref(self.w), n, lmax))
        ws = torch.empty(need, dtype=torch.uint8, device=bags.device)
        logit = torch.empty(n, dtype=torch.float32, device=bags.device)
        attn = torch.empty((n, lmax), dtype=torch.float32, device=bags.device)
        contrib = torch.empty((n, lmax), dtype=torch.float32, device=bags.device)
        dX = torch.empty_like(bags) if need_grad else None
        _lib.check(self.lib.pdf_mil_explain(C.byref(self.w), n, lmax, bags.data_ptr(), lens.data_ptr(), ws.data_ptr(), logit.data_ptr(),
                                            attn.data_ptr(), contrib.data_ptr(), _lib.ptr(dX), _lib.stream_ptr()), "pdf_mil_explain")
        return logit, attn, contrib, dX

    def mc(self, bags: torch.Tensor, lens: torch.Tensor, live: Optional[torch.Tensor] = None, n_scenarios: int = 1, n_samples: int = 32,
           seed: int = 0, p: float = 0.0, samples: bool = False):
        """Monte-Carlo dropout of pdf_mil_mc: n_samples forward passes with the instance layer's dropout (probability p) active.
        bags, lens and live as `sweep` -> device tensors (stats [S, n, 5] float64: mean, std, entropy, expected_entropy, mutual_info;
        sample probabilities [S, n, T] f32 with `samples`, else None).  Bag b's masks are a function of (seed, b, sample) only.  Always
        the FP32 head arithmetic, whatever `precision` says."""
        if bags.dtype != torch.float32 or not bags.is_cuda or not bags.is_contiguous() or bags.shape[2] != self.D:
            raise ValueError("bags must be a contiguous float32 CUDA tensor [n, Lmax, D]")
        n, lmax = int(bags.shape[0]), int(bags.shape[1])
        lens = lens.to(device=bags.device, dtype=torch.int32).contiguous()
        if live is not None:
            live = live.to(device=bags.device, dtype=torch.uint8).contiguous()
            n_scenarios = int(live.shape[0])
            if tuple(live.shape) != (n_scenarios, n):
                raise ValueError("live must be [S, n]")
        need = int(self.lib.pdf_mil_mc_workspace_bytes(C.byref(self.w), n, lmax, int(n_samples)))
        ws = torch.empty(max(need, 1), dtype=torch.uint8, device=bags.device)
        stats = torch.empty((n_scenarios, n, 5), dtype=torch.float64, device=bags.device)
        smp = torch.empty((n_scenarios, n, int(n_samples)), dtype=torch.float32, device=bags.device) if samples else None
        _lib.check(self.lib.pdf_mil_mc(C.byref(self.w), float(p), n, lmax, bags.data_ptr(), lens.data_ptr(), n_scenarios, _lib.ptr(live),
                                       int(n_samples), int(seed) & (2 ** 64 - 1), ws.data_ptr(), stats.data_ptr(), _lib.ptr(smp),
                                       _lib.stream_ptr()), "pdf_mil_mc")
        return stats, smp


def gradcam(fmap: torch.Tensor, g: torch.Tensor, out_hw, cam_small: bool = False):
    """Grad-CAM of pdf_gradcam: fmap [n, hw, hw, C] f32 cuda (the feature map whose spatial mean is the embedding), g [n, C] f32 =
    d logit / d embedding -> cam [n, out_h, out_w] = bilinear upsample (align_corners=False) of ReLU(sum_c g fmap / hw^2),
    unnormalised; with cam_small also that [n, hw, hw] map: (cam, cam_small or None)."""
    n, hw, hw2, c = (int(v) for v in fmap.shape)
    if hw != hw2 or fmap.dtype != torch.float32 or not fmap.is_cuda or not fmap.is_contiguous():
        raise ValueError("fmap must be a contiguous float32 CUDA tensor [n, hw, hw, C]")
    if tuple(g.shape) != (n, c):
        raise ValueError("g must be [n, C]")
    g = g.to(device=fmap.device, dtype=torch.float32).contiguous()
    oh, ow = (int(v) for v in out_hw)
    cam = torch.empty((n, oh, ow), dtype=torch.float32, device=fmap.device)
    small = torch.empty((n, hw, hw), dtype=torch.float32, device=fmap.device) if cam_small else None
    _lib.check(_lib.load().pdf_gradcam(n, hw, c, fmap.data_ptr(), g.data_ptr(), oh, ow, _lib.ptr(small), cam.data_ptr(), _lib.stream_ptr()),
               "pdf_gradcam")
    return cam, small


def _fill_mlp(m: "_lib.Mlp", weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor]) -> None:
    if len(weights) > _lib.PDF_MAX_LAYERS:
        raise ValueError(f"at most {_lib.PDF_MAX_LAYERS} linear layers are supported")
    m.n_layers = len(weights)
    m.dims[0] = int(weights[0].shape[1])
    for i, (w, b) in enumerate(zip(weights, biases)):
        m.dims[i + 1] = int(w.shape[0])
        m.w[i] = w.data_ptr()
        m.b[i] = b.data_ptr()


class ModDropSweep:
    """ModalityDropoutNet (models/fusion_moddrop.py:8-55) evaluated under S scenario masks at once."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], modality_dims: Dict[str, int], device=None):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        idx = sorted({int(k.split(".")[1]) for k in state_dict if k.startswith("net.") and k.endswith(".weight")})
        self.weights = [_dev_f32(state_dict[f"net.{i}.weight"], self.device) for i in idx]
        self.biases = [_dev_f32(state_dict[f"net.{i}.bias"], self.device) for i in idx]
        self.mods = sorted(modality_dims)                       # fusion_moddrop.py:12 -- sorted(modality) feature layout
        m = _lib.Mlp()
        _fill_mlp(m, self.weights, self.biases)
        m.n_mods = len(self.mods)
        off = 0
        for i, mod in enumerate(self.mods):
            m.mod_off[i] = off
            off += int(modality_dims[mod])
        m.mod_off[len(self.mods)] = off
        if off != int(m.dims[0]):
            raise ValueError("modality_dims do not add up to the network input width")
        self.net = m

    def forward(self, X: torch.Tensor, masks: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """X [N,F] f32 cuda; masks [S,N,M] u8 cuda in self.mods order -> prob [S,N] f32 (written into `out`, a contiguous
        [S,N] f32 cuda tensor, when given)."""
        N, S = int(X.shape[0]), int(masks.shape[0])
        X = X.to(dtype=torch.float32).contiguous()
        masks = masks.to(dtype=torch.uint8).contiguous()
        ws = torch.empty(self.lib.pdf_moddrop_workspace_bytes(C.byref(self.net), N), dtype=torch.uint8, device=X.device)
        prob = out if out is not None else torch.empty((S, N), dtype=torch.float32, device=X.device)
        _lib.check(self.lib.pdf_moddrop_sweep(C.byref(self.net), N, S, X.data_ptr(), masks.data_ptr(), ws.data_ptr(),
                                              prob.data_ptr(), _lib.stream_ptr()), "pdf_moddrop_sweep")
        return prob

    def explain(self, X: torch.Tensor, masks: torch.Tensor, steps: int = 0):
        """X [N,F] f32 cuda (unmasked); masks [S,N,M] u8 cuda in self.mods order -> device tensors of pdf_moddrop_explain:
        (logit [S,N], base logit [1], Shapley values [S,N,M] of the logit, integrated gradients [S,N,F] with `steps` midpoints or
        None for steps = 0).  The Shapley values of a scenario add up to logit - base."""
        N, S = int(X.shape[0]), int(masks.shape[0])
        X = X.to(dtype=torch.float32).contiguous()
        masks = masks.to(dtype=torch.uint8).contiguous()
        if tuple(masks.shape) != (S, N, len(self.mods)) or X.shape[1] != int(self.net.dims[0]):
            raise ValueError("X must be [N, F] and masks [S, N, M]")
        need = int(self.lib.pdf_moddrop_explain_workspace_bytes(C.byref(self.net), N, S, steps))
        ws = torch.empty(need, dtype=torch.uint8, device=X.device)
        value = torch.empty((S, N), dtype=torch.float32, device=X.device)
        base = torch.empty(1, dtype=torch.float32, device=X.device)
        shap = torch.empty((S, N, len(self.mods)), dtype=torch.float32, device=X.device)
        ig = torch.empty((S, N, X.shape[1]), dtype=torch.float32, device=X.device) if steps > 0 else None
        _lib.check(self.lib.pdf_moddrop_explain(C.byref(self.net), N, S, X.data_ptr(), masks.data_ptr(), steps, ws.data_ptr(),
                                                value.data_ptr(), base.data_ptr(), shap.data_ptr(), _lib.ptr(ig), _lib.stream_ptr()),
                   "pdf_moddrop_explain")
        return value, base, shap, ig

    def mc(self, X: torch.Tensor, masks: torch.Tensor, n_samples: int = 32, seed: int = 0, p: float = 0.0, samples: bool = False):
        """Monte-Carlo dropout of pdf_moddrop_mc: n_samples forward passes with every hidden layer's dropout (probability p) active.
        X [N,F] f32 cuda (unmasked); masks [S,N,M] u8 cuda in self.mods order -> device tensors (stats [S,N,5] float64: mean, std,
        entropy, expected_entropy, mutual_info; sample probabilities [S,N,T] f32 with `samples`, else None).  Subject n's masks
        are a function of (seed, n, sample) only, the same under every scenario."""
        N, S = int(X.shape[0]), int(masks.shape[0])
        X = X.to(dtype=torch.float32).contiguous()
        masks = masks.to(dtype=torch.uint8).contiguous()
        if tuple(masks.shape) != (S, N, len(self.mods)) or X.shape[1] != int(self.net.dims[0]):
            raise ValueError("X must be [N, F] and masks [S, N, M]")
        need = int(self.lib.pdf_moddrop_mc_workspace_bytes(C.byref(self.net), N, S, int(n_samples)))
        ws = torch.empty(max(need, 1), dtype=torch.uint8, device=X.device)
        stats = torch.empty((S, N, 5), dtype=torch.float64, device=X.device)
        smp = torch.empty((S, N, int(n_samples)), dtype=torch.float32, device=X.device) if samples else None
        _lib.check(self.lib.pdf_moddrop_mc(C.byref(self.net), float(p), N, S, X.data_ptr(), masks.data_ptr(), int(n_samples),
                                           int(seed) & (2 ** 64 - 1), ws.data_ptr(), stats.data_ptr(), _lib.ptr(smp), _lib.stream_ptr()),
                   "pdf_moddrop_mc")
        return stats, smp


class MoeSweep:
    """MoENet (models/moe.py:23-47) evaluated under S scenario masks at once; experts in sorted(modality) order."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], modalities: Sequence[str], device=None):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.mods = sorted(modalities)
        if len(self.mods) > _lib.PDF_MAX_MODS:
            raise ValueError(f"at most {_lib.PDF_MAX_MODS} experts are supported")
        self._keep: List[torch.Tensor] = []
        net = _lib.Moe()
        net.n_experts = len(self.mods)
        for e, mod in enumerate(self.mods):
            idx = sorted({int(k.split(".")[3]) for k in state_dict if k.startswith(f"experts.{mod}.net.") and k.endswith(".weight")})
            ws = [_dev_f32(state_dict[f"experts.{mod}.net.{i}.weight"], self.device) for i in idx]
            bs = [_dev_f32(state_dict[f"experts.{mod}.net.{i}.bias"], self.device) for i in idx]
            self._keep += ws + bs
            _fill_mlp(net.expert[e], ws, bs)
        r = [_dev_f32(state_dict[k], self.device) for k in ("router.0.weight", "router.0.bias", "router.2.weight", "router.2.bias")]
        self._keep += r
        net.router_hidden = int(r[0].shape[0])
        net.w_r0, net.b_r0, net.w_r1, net.b_r1 = (t.data_ptr() for t in r)
        self.net = net

    def forward(self, X: Dict[str, torch.Tensor], masks: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """X {mod: [N,d] f32 cuda, UNMASKED}; masks [S,N,M] u8 in self.mods order -> prob [S,N] f32 (written into `out`, a
        contiguous [S,N] f32 cuda tensor, when given)."""
        xs = [X[m].to(dtype=torch.float32).contiguous() for m in self.mods]
        N, S = int(xs[0].shape[0]), int(masks.shape[0])
        masks = masks.to(dtype=torch.uint8).contiguous()
        ptrs = (C.c_void_p * len(xs))(*[x.data_ptr() for x in xs])
        prob = out if out is not None else torch.empty((S, N), dtype=torch.float32, device=xs[0].device)
        _lib.check(self.lib.pdf_moe_sweep(C.byref(self.net), N, S, ptrs, masks.data_ptr(), prob.data_ptr(), _lib.stream_ptr()),
                   "pdf_moe_sweep")
        return prob

    def explain(self, X: Dict[str, torch.Tensor], masks: torch.Tensor, steps: int = 0):
        """X {mod: [N,d] f32 cuda, UNMASKED}; masks [S,N,M] u8 in self.mods order -> device tensors of pdf_moe_explain:
        (prob [S,N], base prob [1], Shapley values [S,N,M] of the probability, integrated gradients [[S,N,d_e] per expert] with
        `steps` midpoints or None for steps = 0)."""
        xs = [X[m].to(dtype=torch.float32).contiguous() for m in self.mods]
        N, S = int(xs[0].shape[0]), int(masks.shape[0])
        masks = masks.to(dtype=torch.uint8).contiguous()
        if tuple(masks.shape) != (S, N, len(self.mods)):
            raise ValueError("masks must be [S, N, M]")
        dev = xs[0].device
        ptrs = (C.c_void_p * len(xs))(*[x.data_ptr() for x in xs])
        need = int(self.lib.pdf_moe_explain_workspace_bytes(C.byref(self.net), N, S, steps))
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        value = torch.empty((S, N), dtype=torch.float32, device=dev)
        base = torch.empty(1, dtype=torch.float32, device=dev)
        shap = torch.empty((S, N, len(self.mods)), dtype=torch.float32, device=dev)
        ig = [torch.empty((S, N, x.shape[1]), dtype=torch.float32, device=dev) for x in xs] if steps > 0 else None
        igp = (C.c_void_p * len(xs))(*[t.data_ptr() for t in ig]) if ig is not None else None
        _lib.check(self.lib.pdf_moe_explain(C.byref(self.net), N, S, ptrs, masks.data_ptr(), steps, ws.data_ptr(), value.data_ptr(),
                                            base.data_ptr(), shap.data_ptr(), igp, _lib.stream_ptr()), "pdf_moe_explain")
        return value, base, shap, ig

"""Host side of K5: device-native training steps built from the hand-written backward kernels of csrc/train.cu.

Replaces torch autograd under
  * `MilAttentionFineTuneModel.train` / `_forward_bags` (models/mil_attention_finetune.py:135-162, 164-253): ResNet backbone in
    TRAIN mode (BatchNorm statistics per 16-slice chunk of one bag), MIL head, BCE / focal loss, backward, clip_grad_norm_, Adam
    with two learning-rate groups;
  * `MilAttentionModel.train` (models/mil_attention.py:88-155).

Parameters stay where the reference keeps them -- in the `nn.Module`s, whose `state_dict` is the weight-interchange format --
and are updated in place by `pdf_adam_step`; torch supplies device memory and the random draws (permutations, dropout masks),
nothing on the arithmetic path.  FP32 throughout (gradients are checked against torch autograd in tests/test_gpu_training.py).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from . import _lib
from .backbone import RESNET_SPECS, conv_list


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _flat_like(params: Dict[str, torch.Tensor]):
    """One flat gradient buffer with a view per parameter: zeroing and the data-parallel all-reduce are ONE call each."""
    first = next(iter(params.values()))
    offs, total = {}, 0
    for k, v in params.items():
        offs[k] = total
        total += (v.numel() + 7) // 8 * 8                    # 32-byte aligned views
    flat = torch.zeros(total, dtype=torch.float32, device=first.device)
    _flat_like.last_offsets = dict(offs)                         # (layout of the buffer just built: used for the gradient buckets)
    return flat, {k: flat[offs[k]:offs[k] + v.numel()].view(v.shape) for k, v in params.items()}


_flat_like.last_offsets = {}


def flatten_parameters(params: Dict[str, torch.Tensor]) -> torch.Tensor:
    """Moves the parameters into ONE flat f32 buffer with `_flat_like`'s layout and re-points every `param.data` at its view, so
    that the global gradient norm and the Adam update are one launch per buffer instead of one per tensor (ResNet50: 161).
    The nn.Module keeps working unchanged: state_dict / load_state_dict / save see the same tensors."""
    flat, views = _flat_like({k: v.data for k, v in params.items()})
    for k, v in params.items():
        views[k].copy_(v.data)
        v.data = views[k]
    return flat


def block_of(param_name: str) -> str:
    """Bucket key of a backbone parameter: the residual block it belongs to ("layer3.4"), or "stem" (conv1 / bn1)."""
    parts = param_name.split(".")
    return ".".join(parts[:2]) if parts[0].startswith("layer") else "stem"


def bucket_ranges(offsets: Dict[str, int], sizes: Dict[str, int]) -> Dict[str, Tuple[int, int]]:
    """Flat-buffer range [lo, hi) of every block's parameters (`_flat_like` lays the parameters out in named_parameters order, so
    a block is one contiguous range; hi includes the alignment padding up to the next block)."""
    names = list(offsets)
    out: Dict[str, List[int]] = {}
    for i, k in enumerate(names):
        b = block_of(k)
        hi = offsets[names[i + 1]] if i + 1 < len(names) else offsets[k] + (sizes[k] + 7) // 8 * 8
        if b not in out:
            out[b] = [offsets[k], hi]
        else:
            assert offsets[k] == out[b][1], f"block {b} is not contiguous in the flat buffer ({k})"
            out[b][1] = hi
    return {b: (lo, hi) for b, (lo, hi) in out.items()}


class BucketedAllReduce:
    """DDP-style overlap for the fine-tune step (SURVEY.md 8e): the backward walks the blocks from layer4 down to the stem, and as soon
    as a block's last gradient (its weight gradients copied out of the wgrad accumulators, its BatchNorm gradients) is final, the
    block's contiguous range of the flat gradient buffer is averaged over the ranks on a SIDE stream, under the kernels of the
    blocks below it.  `finish()` makes the compute stream wait for the last bucket."""

    def __init__(self, flat: torch.Tensor):
        self.flat = flat
        self.enabled = torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1
        self.stream = torch.cuda.Stream(device=flat.device) if (self.enabled and flat.is_cuda) else None
        self.calls = 0

    def ready(self, lo: int, hi: int) -> None:
        if not self.enabled or hi <= lo:
            return
        self.calls += 1
        if self.stream is None:                                    # CPU tensors (gloo tests): no streams
            allreduce_mean([self.flat[lo:hi]])
            return
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            allreduce_mean([self.flat[lo:hi]])

    def finish(self) -> None:
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)


def allreduce_mean(flat_grads: Sequence[torch.Tensor]) -> None:
    """Data-parallel fine-tuning (SURVEY.md 8e): every rank runs its own bags, the gradients are averaged with one NCCL
    all-reduce per flat buffer before clip + Adam.  No-op in a single process."""
    if not (torch.distributed.is_available() and torch.distributed.is_initialized()):
        return
    ws = torch.distributed.get_world_size()
    if ws == 1:
        return
    nccl = torch.distributed.get_backend() == "nccl"
    for f in flat_grads:
        if nccl:
            torch.distributed.all_reduce(f, op=torch.distributed.ReduceOp.AVG)       # averaged inside the collective
        else:                                                                          # gloo (CPU tests) has no AVG
            torch.distributed.all_reduce(f, op=torch.distributed.ReduceOp.SUM)
            f.mul_(1.0 / ws)


class NativeAdam:
    """torch.optim.Adam (betas 0.9/0.999, eps 1e-8, L2-style weight decay) + clip_grad_norm_ on device tensors.
    groups: [(params: List[Tensor], lr)], gradients in `grads` (same order)."""

    def __init__(self, groups: Sequence[Tuple[List[torch.Tensor], float]], weight_decay: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8):
        self.lib = _lib.load()
        self.groups = [(list(ps), float(lr)) for ps, lr in groups]
        self.wd, self.b1, self.b2, self.eps = float(weight_decay), float(betas[0]), float(betas[1]), float(eps)
        self.state: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        self.steps: Dict[int, int] = {}
        dev = self.groups[0][0][0].device
        self._acc = torch.zeros(1, dtype=torch.float32, device=dev)
        self._scale = torch.ones(2, dtype=torch.float32, device=dev)

    def clip(self, grads: Sequence[torch.Tensor], max_norm: float) -> torch.Tensor:
        """Global L2 norm over `grads`; returns the device tensor [scale, norm] consumed by step()."""
        s = _lib.stream_ptr()
        self._acc.zero_()
        for g in grads:
            _lib.check(self.lib.pdf_sumsq_f32(g.data_ptr(), g.numel(), self._acc.data_ptr(), s), "pdf_sumsq_f32")
        _lib.check(self.lib.pdf_clip_scale(self._acc.data_ptr(), float(max_norm), self._scale.data_ptr(), s), "pdf_clip_scale")
        return self._scale

    def step(self, params_and_grads: Sequence[Tuple[torch.Tensor, torch.Tensor, float]], scale: Optional[torch.Tensor] = None):
        """params_and_grads: (param, grad, lr); parameters without an entry are left alone (as torch skips grad=None)."""
        s = _lib.stream_ptr()
        for p, g, lr in params_and_grads:
            key = p.data_ptr()
            if key not in self.state:
                self.state[key] = (torch.zeros_like(p), torch.zeros_like(p))
                self.steps[key] = 0
            self.steps[key] += 1
            m, v = self.state[key]
            _lib.check(self.lib.pdf_adam_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), float(lr), self.b1, self.b2,
                                              self.eps, self.wd, self.steps[key], _p(scale), s), "pdf_adam_step")


class MilHeadTrainer:
    """Forward + backward of MILAttentionNet (models/mil_attention.py:10-51) in train mode on [B, Lmax, D] padded bags."""

    def __init__(self, net: nn.Module, gated: bool):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.net, self.gated = net, bool(gated)
        sd = dict(net.named_parameters())
        for v in sd.values():
            if not (v.data.is_cuda and v.data.dtype == torch.float32 and v.data.is_contiguous()):
                raise ValueError("MilHeadTrainer needs contiguous float32 CUDA parameters")
        self.flat_param = flatten_parameters(sd)                 # same layout as flat_grad: clip / Adam in one launch each
        self.p = {k: v.data for k, v in sd.items()}
        self.flat_grad, self.g = _flat_like(self.p)
        self.H, self.D = self.p["instance.0.weight"].shape
        self.A = (self.p["attn_v.0.weight"] if self.gated else self.p["attn.0.weight"]).shape[0]
        self.NA = 2 * self.A if self.gated else self.A
        self.dropout = float(net.instance[2].p) if len(net.instance) > 2 else 0.0
        self.dev = self.p["instance.0.weight"].device

    def param_grads(self) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        return [(self.p[k], self.g[k]) for k in self.p]

    def zero_grad(self):
        self.flat_grad.zero_()

    def _gemm(self, M, N, K, A, a_rs, a_cs, B, b_rs, b_cs, Cm, c_rs, bias=None, act=0, acc=0):
        _lib.check(self.lib.pdf_gemm_f32(M, N, K, A.data_ptr() if isinstance(A, torch.Tensor) else A, a_rs, a_cs,
                                         B.data_ptr() if isinstance(B, torch.Tensor) else B, b_rs, b_cs,
                                         Cm.data_ptr() if isinstance(Cm, torch.Tensor) else Cm, c_rs, _p(bias), act, acc, _lib.stream_ptr()),
                   "pdf_gemm_f32")

    def forward_backward(self, X: torch.Tensor, lens: torch.Tensor, y: torch.Tensor, loss_type: str = "bce", pos_weight: Optional[float] = None,
                         focal_gamma: float = 2.0, focal_alpha: Optional[float] = None, need_dx: bool = False, train: bool = True):
        """X [B, Lmax, D] f32 (zero padded), lens [B] i32, y [B] f32 -> (loss [1] device tensor, prob [B], dX or None).
        Gradients are ACCUMULATED into self.g (call zero_grad() first)."""
        B, Lmax, D = (int(v) for v in X.shape)
        rows, H, A, NA = B * Lmax, self.H, self.A, self.NA
        dev, p, g = self.dev, self.p, self.g
        X = X.contiguous()
        h = torch.empty((rows, H), dtype=torch.float32, device=dev)
        self._gemm(rows, H, D, X, D, 1, p["instance.0.weight"], 1, D, h, H, p["instance.0.bias"], act=1)
        mask = None
        if train and self.dropout > 0:
            keep = 1.0 - self.dropout
            mask = (torch.rand((rows, H), device=dev) < keep).to(torch.float32) / keep        # inverted dropout (random draw only)
            _lib.check(self.lib.pdf_mul_f32(h.data_ptr(), mask.data_ptr(), h.numel(), _lib.stream_ptr()), "pdf_mul_f32")
        vu = torch.empty((rows, NA), dtype=torch.float32, device=dev)
        if self.gated:
            self._gemm(rows, A, H, h, H, 1, p["attn_v.0.weight"], 1, H, vu, NA, p["attn_v.0.bias"])
            self._gemm(rows, A, H, h, H, 1, p["attn_u.0.weight"], 1, H, vu.data_ptr() + 4 * A, NA, p["attn_u.0.bias"])
            w_w, b_w, gw_w, gb_w = p["attn_w.weight"], p["attn_w.bias"], g["attn_w.weight"], g["attn_w.bias"]
        else:
            self._gemm(rows, A, H, h, H, 1, p["attn.0.weight"], 1, H, vu, NA, p["attn.0.bias"])
            w_w, b_w, gw_w, gb_w = p["attn.2.weight"], p["attn.2.bias"], g["attn.2.weight"], g["attn.2.bias"]
        w = _lib.MilWeights()
        w.D, w.H, w.A, w.gated = D, H, A, 1 if self.gated else 0
        w.w_w, w.b_w, w.w_cls, w.b_cls = w_w.data_ptr(), b_w.data_ptr(), p["classifier.0.weight"].data_ptr(), p["classifier.0.bias"].data_ptr()
        t = _lib.MilTrain()
        t.loss_type = 1 if loss_type == "focal" else 0
        t.pos_weight = 1.0 if pos_weight is None else float(pos_weight)
        t.focal_gamma = float(focal_gamma)
        t.focal_alpha = -1.0 if focal_alpha is None else float(focal_alpha)
        t.d_w_w, t.d_b_w = gw_w.data_ptr(), gb_w.data_ptr()
        t.d_w_cls, t.d_b_cls = g["classifier.0.weight"].data_ptr(), g["classifier.0.bias"].data_ptr()
        prob = torch.empty(B, dtype=torch.float32, device=dev)
        loss = torch.zeros(1, dtype=torch.float32, device=dev)
        dh = torch.empty((rows, H), dtype=torch.float32, device=dev)
        dvu = torch.empty((rows, NA), dtype=torch.float32, device=dev)
        lens = lens.to(device=dev, dtype=torch.int32).contiguous()
        y = y.to(device=dev, dtype=torch.float32).contiguous()
        _lib.check(self.lib.pdf_mil_pool_train(C.byref(w), C.byref(t), B, Lmax, h.data_ptr(), vu.data_ptr(), lens.data_ptr(), y.data_ptr(),
                                               prob.data_ptr(), loss.data_ptr(), dh.data_ptr(), dvu.data_ptr(), _lib.stream_ptr()),
                   "pdf_mil_pool_train")
        # attention layers: dW = dvu^T h, db = colsum(dvu), dh += dvu W
        s = _lib.stream_ptr()
        names = [("attn_v.0", 0), ("attn_u.0", A)] if self.gated else [("attn.0", 0)]
        for name, off in names:
            dv = dvu.data_ptr() + 4 * off
            self._gemm(A, H, rows, dv, 1, NA, h, H, 1, g[name + ".weight"], H, acc=1)                 # dW[a, i] += sum_r dv[r, a] h[r, i]
            _lib.check(self.lib.pdf_gemm_f32(1, A, rows, self._ones(rows).data_ptr(), 0, 1, dv, NA, 1, g[name + ".bias"].data_ptr(), A, None, 0, 1, s),
                       "pdf_gemm_f32")
            self._gemm(rows, H, A, dv, NA, 1, p[name + ".weight"], H, 1, dh, H, acc=1)                # dh[r, i] += sum_a dv[r, a] W[a, i]
        # instance layer: ReLU (+ dropout) backward, dW_i = dh^T X, db_i, (dX = dh W_i)
        _lib.check(self.lib.pdf_relu_mask_backward(dh.data_ptr(), h.data_ptr(), _p(mask), dh.numel(), s), "pdf_relu_mask_backward")
        self._gemm(H, D, rows, dh, 1, H, X, D, 1, g["instance.0.weight"], D, acc=1)
        _lib.check(self.lib.pdf_colsum_f32(rows, H, dh.data_ptr(), g["instance.0.bias"].data_ptr(), 1, s), "pdf_colsum_f32")
        dX = None
        if need_dx:
            dX = torch.empty((B, Lmax, D), dtype=torch.float32, device=dev)
            self._gemm(rows, D, H, dh, H, 1, p["instance.0.weight"], D, 1, dX, D)
        return loss, prob, dX

    def _ones(self, n: int) -> torch.Tensor:
        if getattr(self, "_ones_buf", None) is None or self._ones_buf.numel() < n:
            self._ones_buf = torch.ones(n, dtype=torch.float32, device=self.dev)
        return self._ones_buf


class MlpTrainer:
    """Forward to the LOGITS and backward from d(logits) of an `nn.Sequential` MLP made of Linear / ReLU / Dropout / (final Sigmoid or
    Softmax, which the loss kernels own): the fusion heads' networks (models/fusion_moddrop.py:25-35, models/moe.py:7-35).
    Parameters are the module's tensors; gradients live in one flat buffer."""

    def __init__(self, seq: nn.Sequential, prefix: str = ""):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.layers: List[Tuple[str, nn.Linear, bool, float]] = []        # (name, linear, relu after, dropout p after)
        mods = list(seq)
        for i, m in enumerate(mods):
            if isinstance(m, nn.Linear):
                relu = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
                drop = float(mods[i + 2].p) if relu and i + 2 < len(mods) and isinstance(mods[i + 2], nn.Dropout) else 0.0
                self.layers.append((f"{prefix}{i}", m, relu, drop))
        self.p = {}
        for name, lin, _, _ in self.layers:
            self.p[name + ".weight"], self.p[name + ".bias"] = lin.weight.data, lin.bias.data
        for v in self.p.values():
            if not (v.is_cuda and v.dtype == torch.float32 and v.is_contiguous()):
                raise ValueError("MlpTrainer needs contiguous float32 CUDA parameters")
        self.flat_grad, self.g = _flat_like(self.p)
        self.dev = next(iter(self.p.values())).device

    def param_grads(self):
        return [(self.p[k], self.g[k]) for k in self.p]

    def zero_grad(self):
        self.flat_grad.zero_()

    def forward(self, X: torch.Tensor, train: bool = True) -> torch.Tensor:
        s = _lib.stream_ptr()
        a = X.contiguous()
        self.saved = []
        for name, lin, relu, drop in self.layers:
            n_out, n_in = lin.weight.shape
            out = torch.empty((a.shape[0], n_out), dtype=torch.float32, device=self.dev)
            _lib.check(self.lib.pdf_gemm_f32(a.shape[0], n_out, n_in, a.data_ptr(), n_in, 1, lin.weight.data.data_ptr(), 1, n_in, out.data_ptr(), n_out,
                                             lin.bias.data.data_ptr(), 1 if relu else 0, 0, s), "pdf_gemm_f32")
            mask = None
            if train and relu and drop > 0:
                keep = 1.0 - drop
                mask = (torch.rand(out.shape, device=self.dev) < keep).to(torch.float32) / keep       # random draw only
                _lib.check(self.lib.pdf_mul_f32(out.data_ptr(), mask.data_ptr(), out.numel(), s), "pdf_mul_f32")
            self.saved.append((a, out, mask))
            a = out
        return a

    def backward(self, dlogits: torch.Tensor) -> None:
        s = _lib.stream_ptr()
        d = dlogits.contiguous()
        for (name, lin, relu, drop), (a_in, out, mask) in zip(reversed(self.layers), reversed(self.saved)):
            n_out, n_in = lin.weight.shape
            rows = a_in.shape[0]
            if relu:
                _lib.check(self.lib.pdf_relu_mask_backward(d.data_ptr(), out.data_ptr(), _p(mask), d.numel(), s), "pdf_relu_mask_backward")
            _lib.check(self.lib.pdf_gemm_f32(n_out, n_in, rows, d.data_ptr(), 1, n_out, a_in.data_ptr(), n_in, 1, self.g[name + ".weight"].data_ptr(), n_in,
                                             None, 0, 1, s), "pdf_gemm_f32")
            _lib.check(self.lib.pdf_colsum_f32(rows, n_out, d.data_ptr(), self.g[name + ".bias"].data_ptr(), 1, s), "pdf_colsum_f32")
            if name != self.layers[0][0]:
                dn = torch.empty((rows, n_in), dtype=torch.float32, device=self.dev)
                _lib.check(self.lib.pdf_gemm_f32(rows, n_in, n_out, d.data_ptr(), n_out, 1, lin.weight.data.data_ptr(), n_in, 1, dn.data_ptr(), n_in,
                                                 None, 0, 0, s), "pdf_gemm_f32")
                d = dn
        self.saved = []


class _Act:
    __slots__ = ("data", "grad", "n", "hw", "c", "relu_bits")

    def __init__(self, data, n, hw, c, relu_bits=None):
        self.data, self.grad, self.n, self.hw, self.c = data, None, n, hw, c     # data / grad: f32 (fp32 path) or bf16 (tensor path)
        self.relu_bits = relu_bits      # tensor path: the producing BatchNorm's ReLU mask, one bit per element (read by its backward)


class ResNetTrainer:
    """Train-mode forward and backward of a torchvision-layout ResNet18/50 (fc = Identity) on NHWC float32 images.

    BatchNorm uses BATCH statistics over each group of images (`groups`: image offsets; one group = one 16-slice chunk of one
    bag, the unit the reference pushes through `self.backbone(batch)`, mil_attention_finetune.py:147-150) and updates the
    module's running statistics group by group.  Parameters are read from / updated in the nn.Module (torchvision layout
    [K,C,R,S]); the kernels consume re-laid-out copies refreshed by `sync_weights()`.

    precision "bf16" (default; PD_FUSION_B200_TRAIN_PRECISION overrides) -- the tensor-core path: every convolution runs on the
    tcgen05 kernels with bf16 operands and f32 accumulation.  Forward and data gradient go through the inference path's
    implicit-GEMM kernels (the data gradient as a stride-1 convolution of dY with the 180-degree-rotated, transposed filter; for
    the stride-2 3x3 convolutions dY is zero-dilated first, the stride-2 1x1 downsamples are a GEMM on dY scattered onto the even
    pixels), the weight gradient through wgrad_tc.cu, the 3-channel stem as a [M,192] patch-matrix GEMM.  Activations, conv
    outputs and activation gradients are STORED in bf16; BatchNorm statistics (float64 sums), normalisation, parameter gradients,
    master weights and the optimiser are f32 -- the numerics of torch's bf16 autocast (csrc/train_bf16.cu).
    precision "fp32": the CUDA-core parity path (csrc/train.cu), f32 everywhere."""

    def __init__(self, module: nn.Module, arch: str, input_size: int = 224, precision: Optional[str] = None):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.precision = precision or os.environ.get("PD_FUSION_B200_TRAIN_PRECISION", "bf16")
        if self.precision not in ("bf16", "fp32"):
            raise ValueError(f"ResNetTrainer: precision {self.precision!r} (bf16 | fp32)")
        self.bf16 = self.precision == "bf16"
        self.m, self.arch, self.S = module, arch, int(input_size)
        self.kind, self.layers, self.emb_dim = RESNET_SPECS[arch]
        self.params = dict(module.named_parameters())
        self.buffers = dict(module.named_buffers())
        self.dev = self.params["conv1.weight"].device
        self.convs = {cv["name"]: cv for cv in conv_list(arch)}
        self.wk: Dict[str, torch.Tensor] = {}         # fp32 path: [R,S,C,K] f32
        self.wk16: Dict[str, torch.Tensor] = {}       # tensor path: [K][R][S][C] bf16 (forward / wgrad layout; the stem: [64][192])
        self.wrot16: Dict[str, torch.Tensor] = {}     # tensor path: [C][R][S][K] bf16, taps rotated by 180 degrees (data-gradient operand)
        trainable = {k: v for k, v in self.params.items() if not k.startswith("fc.")}
        self.flat_param = flatten_parameters(trainable)              # same layout as flat_grad: clip / Adam in one launch each
        self.flat_grad, self.grad = _flat_like({k: v.data for k, v in trainable.items()})
        self.buckets = bucket_ranges(_flat_like.last_offsets, {k: v.numel() for k, v in trainable.items()})
        self._zero_bias = torch.zeros(4096, dtype=torch.float32, device=self.dev)
        self._scr = None
        if self.bf16:
            for name, cv in self.convs.items():
                if name == "conv1":
                    self.wk16[name] = torch.zeros((cv["cout"], 192), dtype=torch.bfloat16, device=self.dev)
                    continue
                assert cv["cin"] % 64 == 0 and cv["cout"] % 64 == 0, name
                self.wk16[name] = torch.empty((cv["cout"], cv["k"], cv["k"], cv["cin"]), dtype=torch.bfloat16, device=self.dev)
                self.wrot16[name] = torch.empty((cv["cin"], cv["k"], cv["k"], cv["cout"]), dtype=torch.bfloat16, device=self.dev)
            # weight-gradient accumulators [K][R][S][C] f32 of every convolution in ONE buffer (zeroed with one memset per step)
            sizes = {n: (192 * cv["cout"] if n == "conv1" else cv["cout"] * cv["k"] * cv["k"] * cv["cin"]) for n, cv in self.convs.items()}
            self._gw_flat = torch.zeros(sum(sizes.values()), dtype=torch.float32, device=self.dev)
            self._gw, off = {}, 0
            for n, cv in self.convs.items():
                shape = (cv["cout"], 192) if n == "conv1" else (cv["cout"], cv["k"], cv["k"], cv["cin"])
                self._gw[n] = self._gw_flat[off:off + sizes[n]].view(shape)
                off += sizes[n]
        self.sync_weights()

    # -- parameters --------------------------------------------------------------------------------
    def sync_weights(self):
        s = _lib.stream_ptr()
        for name, cv in self.convs.items():
            w = self.params[name + ".weight"].data
            if not self.bf16:
                self.wk[name] = w.permute(2, 3, 1, 0).contiguous()      # [R,S,C,K] (layout change only)
            elif name == "conv1":                                       # [64][7][7][3] -> 147 of the 192 patch-matrix columns
                self.wk16[name][:, :147].copy_(w.permute(0, 2, 3, 1).reshape(w.shape[0], 147))
            else:
                _lib.check(self.lib.pdf_pack_conv_weights(cv["cout"], cv["cin"], cv["k"], cv["k"], w.data_ptr(), self.wk16[name].data_ptr(),
                                                          self.wrot16[name].data_ptr(), s), "pdf_pack_conv_weights")

    def zero_grad(self):
        self.flat_grad.zero_()

    def param_grads(self) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        return [(self.params[k].data, self.grad[k]) for k in self.grad]

    # -- shared helpers ----------------------------------------------------------------------------
    def _op(self, n, h, c, cv, ho) -> "_lib.Op":
        op = _lib.Op()
        op.kind, op.precision = _lib.OP_CONV, _lib.PREC_F32
        op.n, op.h, op.w, op.c, op.k, op.r, op.s = n, h, h, c, cv["cout"], cv["k"], cv["k"]
        op.stride, op.pad, op.ho, op.wo, op.relu = cv["stride"], cv["pad"], ho, ho, 0
        return op

    def _run_op(self, op: "_lib.Op") -> None:
        plan = C.c_void_p()
        _lib.check(self.lib.pdf_plan_create(C.byref(plan), (_lib.Op * 1)(op), 1), "pdf_plan_create")
        _lib.check(self.lib.pdf_plan_run(plan, _lib.stream_ptr()), "pdf_plan_run")
        self.lib.pdf_plan_destroy(plan)

    def _pool_op(self, kind, prec, n, h, c, ho, d_in, d_out):
        op = _lib.Op()
        op.kind, op.precision = kind, prec
        op.n, op.h, op.w, op.c, op.ho, op.wo = n, h, h, c, ho, ho
        op.d_in, op.d_out = d_in, d_out
        self._run_op(op)

    def _scratch(self, n_doubles: int) -> torch.Tensor:
        if self._scr is None or self._scr.numel() < n_doubles:
            self._scr = torch.empty(max(n_doubles, 3 * 16 * 2048), dtype=torch.float64, device=self.dev)
        return self._scr

    def _goff(self, groups: Sequence[int], hw: int) -> torch.Tensor:
        key = (tuple(groups), hw)
        if key not in self._goff_cache:
            self._goff_cache[key] = torch.tensor([g * hw for g in groups], dtype=torch.int32, device=self.dev)
        return self._goff_cache[key]

    def _bn_module(self, bn: str) -> nn.BatchNorm2d:
        mod = self.m
        for part in bn.split("."):
            mod = mod[int(part)] if part.isdigit() else getattr(mod, part)
        return mod

    # -- forward ---------------------------------------------------------------------------------------
    def _bn_forward(self, bn: str, conv_out: torch.Tensor, res: Optional[_Act], relu: bool, groups, hw: int):
        """Train-mode BatchNorm (+ residual, ReLU) of a conv output [M, K] in the path's storage type; returns (y, goff, mean, invstd, max_rows, relu_bits)."""
        G, K = len(groups) - 1, int(conv_out.shape[1])
        goff = self._goff(groups, hw)
        max_rows = max(b - a for a, b in zip(groups[:-1], groups[1:])) * hw
        y = torch.empty_like(conv_out)
        mean = torch.empty((G, K), dtype=torch.float32, device=self.dev)
        invstd, varu = torch.empty_like(mean), torch.empty_like(mean)
        bnm = self._bn_module(bn)
        args = (G, goff.data_ptr(), max_rows, K, conv_out.data_ptr(), self.params[bn + ".weight"].data.data_ptr(),
                self.params[bn + ".bias"].data.data_ptr(), float(bnm.eps), _p(res.data if res else None), 1 if relu else 0, y.data_ptr())
        tail = (mean.data_ptr(), invstd.data_ptr(), varu.data_ptr(), self._scratch(3 * G * K).data_ptr(), _lib.stream_ptr())
        bits = None
        if self.bf16:        # the ReLU mask as one bit per element: what the backward reads instead of y
            bits = torch.empty(conv_out.numel() // 8, dtype=torch.uint8, device=self.dev) if relu else None
            _lib.check(self.lib.pdf_bn_train_forward_bf16(*args, _p(bits), *tail), "pdf_bn_train_forward_bf16")
        else:
            _lib.check(self.lib.pdf_bn_train_forward(*args, *tail), "pdf_bn_train_forward")
        if self.update_running:
            _lib.check(self.lib.pdf_bn_update_running(G, K, mean.data_ptr(), varu.data_ptr(), float(bnm.momentum),
                                                      self.buffers[bn + ".running_mean"].data_ptr(), self.buffers[bn + ".running_var"].data_ptr(),
                                                      _lib.stream_ptr()), "pdf_bn_update_running")
            self.buffers[bn + ".num_batches_tracked"] += G
        return y, goff, mean, invstd, max_rows, bits

    def _convbn(self, x: _Act, h: int, name: str, bn: str, relu: bool, res: Optional[_Act], groups) -> Tuple[_Act, int]:
        cv = self.convs[name]
        ho = (h + 2 * cv["pad"] - cv["k"]) // cv["stride"] + 1
        n, K = x.n, cv["cout"]
        op = self._op(n, h, x.c, cv, ho)
        if self.bf16:
            conv_out = torch.empty((n * ho * ho, K), dtype=torch.bfloat16, device=self.dev)
            op.precision = _lib.PREC_BF16
            op.d_in, op.d_weight, op.d_bias, op.d_out = x.data.data_ptr(), self.wk16[name].data_ptr(), self._zero_bias.data_ptr(), conv_out.data_ptr()
        else:
            conv_out = torch.empty((n * ho * ho, K), dtype=torch.float32, device=self.dev)
            op.d_in, op.d_weight, op.d_out = x.data.data_ptr(), self.wk[name].data_ptr(), conv_out.data_ptr()
        self._run_op(op)
        y, goff, mean, invstd, max_rows, bits = self._bn_forward(bn, conv_out, res, relu, groups, ho * ho)
        out = _Act(y, n, ho * ho, K, bits)
        self.tape.append(("convbn", name, bn, x, conv_out, out, relu, res, op, goff, mean, invstd, h, max_rows))
        return out, ho

    def _stem_tc(self, x: torch.Tensor, n: int, groups) -> Tuple[_Act, int]:
        """conv1 7x7/2 on the 3-channel f32 input as a tensor-core GEMM: patch matrix [M, 192] bf16 (147 columns + zero padding)
        x W1^T [192, 64]; the same matrix is the X operand of the stem's weight gradient."""
        S = self.S
        ho = (S + 6 - 7) // 2 + 1
        patches = torch.empty((n * ho * ho, 192), dtype=torch.bfloat16, device=self.dev)
        _lib.check(self.lib.pdf_stem_im2col3_bf16(n, S, S, x.data_ptr(), patches.data_ptr(), _lib.stream_ptr()), "pdf_stem_im2col3_bf16")
        conv_out = torch.empty((n * ho * ho, 64), dtype=torch.bfloat16, device=self.dev)
        op = _lib.Op()
        op.kind, op.precision = _lib.OP_CONV, _lib.PREC_BF16
        op.n, op.h, op.w, op.c, op.k, op.r, op.s, op.stride, op.pad, op.ho, op.wo, op.relu = n, ho, ho, 192, 64, 1, 1, 1, 0, ho, ho, 0
        op.d_in, op.d_weight, op.d_bias, op.d_out = patches.data_ptr(), self.wk16["conv1"].data_ptr(), self._zero_bias.data_ptr(), conv_out.data_ptr()
        self._run_op(op)
        y, goff, mean, invstd, max_rows, bits = self._bn_forward("bn1", conv_out, None, True, groups, ho * ho)
        out = _Act(y, n, ho * ho, 64, bits)
        self.tape.append(("stem", patches, conv_out, out, op, goff, mean, invstd, max_rows))
        return out, ho

    def forward(self, x: torch.Tensor, groups: Sequence[int], update_running: bool = True) -> torch.Tensor:
        """x [n, S, S, 3] f32 NHWC (the reference's (x-mean)/std 3-channel input); groups: image offsets [0, ..., n] of the
        BatchNorm groups.  Returns the embeddings [n, D] f32 and records the tape for backward()."""
        n = int(x.shape[0])
        assert groups[0] == 0 and groups[-1] == n
        self.tape, self._goff_cache, self.update_running = [], {}, bool(update_running)
        prec = _lib.PREC_BF16 if self.bf16 else _lib.PREC_F32
        adt = torch.bfloat16 if self.bf16 else torch.float32
        x = x.contiguous()
        if self.bf16:
            t, h = self._stem_tc(x, n, groups)
        else:
            t, h = self._convbn(_Act(x, n, self.S * self.S, 3), self.S, "conv1", "bn1", True, None, groups)
        ho = (h + 2 - 3) // 2 + 1
        pooled = torch.empty((n * ho * ho, 64), dtype=adt, device=self.dev)
        widx = None
        if self.bf16:                              # records the winning window position: the backward is a gather through it
            widx = torch.empty((n * ho * ho, 64), dtype=torch.uint8, device=self.dev)
            _lib.check(self.lib.pdf_maxpool_train_forward_bf16(n, h, h, 64, t.data.data_ptr(), pooled.data_ptr(), widx.data_ptr(), _lib.stream_ptr()),
                       "pdf_maxpool_train_forward_bf16")
        else:
            self._pool_op(_lib.OP_MAXPOOL, prec, n, h, 64, ho, t.data.data_ptr(), pooled.data_ptr())
        t2 = _Act(pooled, n, ho * ho, 64)
        self.tape.append(("maxpool", t, t2, h, widx))
        t, h = t2, ho
        for li, nblocks in enumerate(self.layers, start=1):
            for bi in range(nblocks):
                pfx = f"layer{li}.{bi}"
                idn, h_in = t, h
                if pfx + ".downsample.0" in self.convs:
                    idn, _ = self._convbn(t, h_in, pfx + ".downsample.0", pfx + ".downsample.1", False, None, groups)
                o, h = self._convbn(t, h_in, pfx + ".conv1", pfx + ".bn1", True, None, groups)
                if self.kind == "basic":
                    o, h = self._convbn(o, h, pfx + ".conv2", pfx + ".bn2", True, idn, groups)
                else:
                    o, h = self._convbn(o, h, pfx + ".conv2", pfx + ".bn2", True, None, groups)
                    o, h = self._convbn(o, h, pfx + ".conv3", pfx + ".bn3", True, idn, groups)
                t = o
        emb = torch.empty((t.n, t.c), dtype=torch.float32, device=self.dev)
        hw = int(round(t.hw ** 0.5))
        self._pool_op(_lib.OP_AVGPOOL, prec, t.n, hw, t.c, 1, t.data.data_ptr(), emb.data_ptr())
        self.tape.append(("avgpool", t))
        return emb

    # -- backward --------------------------------------------------------------------------------------
    def _bn_backward(self, bn, out: _Act, conv_out, relu, res: Optional[_Act], goff, mean, invstd, max_rows) -> torch.Tensor:
        """BatchNorm (+ReLU, + residual branch) backward: returns d(conv output) in the path's storage type; the residual
        branch's gradient is written / accumulated into res.grad."""
        G, K = int(mean.shape[0]), int(mean.shape[1])
        dconv = torch.empty_like(conv_out)
        dres, acc = None, 0
        if res is not None:
            if res.grad is None:
                res.grad = torch.empty_like(res.data)
            else:
                acc = 1
            dres = res.grad
        fn = self.lib.pdf_bn_train_backward_bf16 if self.bf16 else self.lib.pdf_bn_train_backward
        act = _p(out.relu_bits) if self.bf16 else out.data.data_ptr()              # bf16 path: the forward's bit mask; fp32 path: y itself
        _lib.check(fn(G, goff.data_ptr(), max_rows, K, out.grad.data_ptr(), act, conv_out.data_ptr(),
                      self.params[bn + ".weight"].data.data_ptr(), mean.data_ptr(), invstd.data_ptr(), 1 if relu else 0,
                      self._scratch(3 * G * K).data_ptr(), dconv.data_ptr(), _p(dres), acc, self.grad[bn + ".weight"].data_ptr(),
                      self.grad[bn + ".bias"].data_ptr(), _lib.stream_ptr()), "pdf_bn_train_backward")
        out.grad = None
        return dconv

    def _finalize_weight_grad(self, name: str, gwk) -> None:
        """-> torchvision [K,C,R,S] (layout change only; one backward per zero_grad, as the reference's step)"""
        if self.bf16:                                                # tensor path accumulated [K,R,S,C]
            gw = self._gw[name]
            if name == "conv1":
                self.grad[name + ".weight"].copy_(gw[:, :147].reshape(gw.shape[0], 7, 7, 3).permute(0, 3, 1, 2))
            else:
                self.grad[name + ".weight"].copy_(gw.permute(0, 3, 1, 2))
        else:                                                        # FP32 path accumulated [R,S,C,K]
            self.grad[name + ".weight"].copy_(gwk[name].permute(3, 2, 0, 1))

    def backward(self, demb: torch.Tensor, reducer: Optional["BucketedAllReduce"] = None):
        """demb [n, D] f32: gradient of the loss w.r.t. the embeddings.  Accumulates parameter gradients into self.grad
        (torchvision layout).  reducer: data-parallel runs hand in a BucketedAllReduce over self.flat_grad -- every residual block's
        range of the flat buffer is all-reduced on a side stream as soon as the backward has left the block."""
        s = _lib.stream_ptr()
        lib = self.lib
        gwk: Dict[str, torch.Tensor] = {}
        if self.bf16:
            self._gw_flat.zero_()
        cur_block = None

        def leave(block):
            if reducer is not None and block is not None:
                reducer.ready(*self.buckets[block])

        for entry in reversed(self.tape):
            kind = entry[0]
            if kind in ("stem", "convbn"):
                blk = "stem" if kind == "stem" else block_of(entry[1])
                if blk != cur_block:
                    leave(cur_block)
                    cur_block = blk
            if kind == "avgpool":
                t = entry[1]
                t.grad = torch.empty_like(t.data)
                fn = lib.pdf_avgpool_backward_bf16 if self.bf16 else lib.pdf_avgpool_backward_f32
                _lib.check(fn(t.n, t.hw, t.c, demb.contiguous().data_ptr(), t.grad.data_ptr(), s), "pdf_avgpool_backward")
            elif kind == "maxpool":
                _, tin, tout, h, widx = entry
                tin.grad = torch.empty_like(tin.data)
                if self.bf16:
                    _lib.check(lib.pdf_maxpool_backward_bf16(tin.n, h, h, tin.c, widx.data_ptr(), tout.grad.data_ptr(), tin.grad.data_ptr(), s),
                               "pdf_maxpool_backward_bf16")
                else:
                    _lib.check(lib.pdf_maxpool_backward_f32(tin.n, h, h, tin.c, tin.data.data_ptr(), tout.grad.data_ptr(), tin.grad.data_ptr(), s),
                               "pdf_maxpool_backward_f32")
                tout.grad = None
            elif kind == "stem":                                     # tensor path: the network input needs no gradient
                _, patches, conv_out, out, op, goff, mean, invstd, max_rows = entry
                dconv = self._bn_backward("bn1", out, conv_out, True, None, goff, mean, invstd, max_rows)
                _lib.check(lib.pdf_conv_wgrad_bf16(C.byref(op), patches.data_ptr(), dconv.data_ptr(), self._gw["conv1"].data_ptr(), s),
                           "pdf_conv_wgrad_bf16")
                self._finalize_weight_grad("conv1", gwk)
            else:
                _, name, bn, x, conv_out, out, relu, res, op, goff, mean, invstd, h, max_rows = entry
                dconv = self._bn_backward(bn, out, conv_out, relu, res, goff, mean, invstd, max_rows)
                if self.bf16:
                    self._backward_conv_tc(name, op, x, dconv, h)
                    self._finalize_weight_grad(name, gwk)
                    continue
                if name not in gwk:
                    gwk[name] = torch.zeros_like(self.wk[name])
                _lib.check(lib.pdf_conv_wgrad_f32(C.byref(op), x.data.data_ptr(), dconv.data_ptr(), gwk[name].data_ptr(), s), "pdf_conv_wgrad_f32")
                if name != "conv1":                                  # the network input needs no gradient
                    acc = 0 if x.grad is None else 1
                    if x.grad is None:
                        x.grad = torch.empty_like(x.data)
                    _lib.check(lib.pdf_conv_dgrad_f32(C.byref(op), dconv.data_ptr(), self.wk[name].data_ptr(), x.grad.data_ptr(), acc, s),
                               "pdf_conv_dgrad_f32")
                self._finalize_weight_grad(name, gwk)
        leave(cur_block)
        self.tape = []

    def _backward_conv_tc(self, name: str, op: "_lib.Op", x: _Act, dconv: torch.Tensor, h: int) -> None:
        """Weight and data gradient of one convolution on the tensor cores (bf16 operands and results, f32 accumulation).
        wgrad: dW[k][r][s][c] += dY^T im2col(X) (wgrad_tc.cu).  dgrad: a stride-1 convolution of dY with the 180-degree-rotated,
        transposed filter through the forward implicit-GEMM kernels (pad' = R-1-pad), a gradient already present in x.grad riding
        in as the kernel's residual operand; stride-2 3x3: dY zero-dilated to the input's size first (dY[p,q] at (2p, 2q));
        stride-2 1x1 (downsample): a GEMM on dY whose result is scatter-added onto the even pixels."""
        lib, s = self.lib, _lib.stream_ptr()
        cv = self.convs[name]
        n, C_in, K, R, stride, pad, ho = x.n, x.c, cv["cout"], cv["k"], cv["stride"], cv["pad"], int(op.ho)
        _lib.check(lib.pdf_conv_wgrad_bf16(C.byref(op), x.data.data_ptr(), dconv.data_ptr(), self._gw[name].data_ptr(), s), "pdf_conv_wgrad_bf16")
        assert stride in (1, 2), name
        dop = _lib.Op()
        dop.kind, dop.precision = _lib.OP_CONV, _lib.PREC_BF16
        dop.c, dop.k, dop.r, dop.s, dop.stride, dop.relu = K, C_in, R, R, 1, 0
        dop.d_weight, dop.d_bias = self.wrot16[name].data_ptr(), self._zero_bias.data_ptr()
        if stride == 2 and R == 1:
            tmp = torch.empty((n * ho * ho, C_in), dtype=torch.bfloat16, device=self.dev)
            dop.n, dop.h, dop.w, dop.pad, dop.ho, dop.wo = n, ho, ho, 0, ho, ho
            dop.d_in, dop.d_out = dconv.data_ptr(), tmp.data_ptr()
            self._run_op(dop)
            if x.grad is None:
                x.grad = torch.zeros_like(x.data)
            _lib.check(lib.pdf_scatter_add2_bf16(n, ho, ho, C_in, h, h, tmp.data_ptr(), x.grad.data_ptr(), s), "pdf_scatter_add2_bf16")
            return
        if stride == 1:
            src, hs = dconv, ho
        else:
            src, hs = torch.empty((n * h * h, K), dtype=torch.bfloat16, device=self.dev), h
            _lib.check(lib.pdf_dilate2_bf16(n, ho, ho, K, h, h, dconv.data_ptr(), src.data_ptr(), s), "pdf_dilate2_bf16")
        dop.n, dop.h, dop.w, dop.pad, dop.ho, dop.wo = n, hs, hs, R - 1 - pad, h, h
        assert hs + 2 * (R - 1 - pad) - R + 1 == h, (name, hs, h)
        dst = torch.empty_like(x.data)
        dop.d_in, dop.d_out = src.data_ptr(), dst.data_ptr()
        if x.grad is not None:
            dop.d_residual = x.grad.data_ptr()                       # accumulate: out = conv + the gradient already there
        self._run_op(dop)
        x.grad = dst


# -- deep ensembles: E members of one architecture trained in lockstep (csrc/train.cu) ----------------------------------------
def flatten_members(member_params: Sequence[Dict[str, torch.Tensor]]) -> Tuple[torch.Tensor, Dict[str, int]]:
    """Moves the parameters of E members of one architecture into ONE flat f32 buffer [E, P] (row e = member e, each row in
    `_flat_like`'s layout) and re-points every member's `param.data` at its view.  Returns (buffer, offset of each parameter in a
    row).  The members' nn.Modules keep working unchanged; every launch of a training step covers all rows."""
    first = member_params[0]
    offs, P = {}, 0
    for k, v in first.items():
        offs[k] = P
        P += (v.numel() + 7) // 8 * 8
    flat = torch.zeros((len(member_params), P), dtype=torch.float32, device=first[next(iter(first))].device)
    for e, params in enumerate(member_params):
        if list(params) != list(first) or any(params[k].shape != first[k].shape for k in first):
            raise ValueError("ensemble members must have the same parameters")
        for k, v in params.items():
            view = flat[e, offs[k]:offs[k] + v.numel()].view(v.shape)
            view.copy_(v.data)
            v.data = view
    return flat, offs


def _dropout_mask(shape, gens: Sequence[torch.Generator], keep: float, dev) -> torch.Tensor:
    """[E, *shape] inverted-dropout masks, member e's drawn from its own CUDA generator exactly as the single trainers draw theirs"""
    return torch.stack([torch.rand(shape, device=dev, generator=g) < keep for g in gens]).to(torch.float32) / keep


class BatchedGemm:
    """pdf_gemm_f32_batched over the members of a flat [E, P] parameter / gradient buffer pair"""

    def __init__(self, flat_param: torch.Tensor, flat_grad: torch.Tensor, offs: Dict[str, int]):
        self.lib = _lib.load()
        self.E, self.P = int(flat_param.shape[0]), int(flat_param.shape[1])
        self.flat_param, self.flat_grad, self.offs = flat_param, flat_grad, offs
        self.dev = flat_param.device
        self._ones_buf = None

    def param(self, name: str) -> int:
        return self.flat_param.data_ptr() + 4 * self.offs[name]

    def grad(self, name: str) -> int:
        return self.flat_grad.data_ptr() + 4 * self.offs[name]

    def gemm(self, M, N, K, A, a_rs, a_cs, a_es, B, b_rs, b_cs, b_es, Cm, c_rs, c_es, bias=None, bias_es=0, act=0, acc=0):
        ptr = lambda t: t.data_ptr() if isinstance(t, torch.Tensor) else t
        _lib.check(self.lib.pdf_gemm_f32_batched(self.E, M, N, K, ptr(A), a_rs, a_cs, a_es, ptr(B), b_rs, b_cs, b_es, ptr(Cm), c_rs, c_es,
                                                 bias, bias_es, act, acc, _lib.stream_ptr()), "pdf_gemm_f32_batched")

    def colsum(self, rows: int, n: int, d, d_es: int, out_name: str, d_rs: Optional[int] = None):
        """gradient[out_name] (+)= the column sums of every member's d [rows, n] (row stride d_rs): a GEMM with a shared row of ones,
        whose k-ascending accumulation adds the rows in pdf_colsum_f32's order"""
        self.gemm(1, n, rows, self.ones(rows), 0, 1, 0, d, n if d_rs is None else d_rs, 1, d_es, self.grad(out_name), n, self.P, acc=1)

    def ones(self, n: int) -> torch.Tensor:
        if self._ones_buf is None or self._ones_buf.numel() < n:
            self._ones_buf = torch.ones(n, dtype=torch.float32, device=self.dev)
        return self._ones_buf


class BatchedMlpTrainer:
    """MlpTrainer for the same `nn.Sequential` of E members at once: activations [E, rows, width], member e's weights in row e of
    the shared flat buffers.  The input of `forward` is [E, rows, F] or one [rows, F] matrix every member reads (MoE's full batch)."""

    def __init__(self, seq: nn.Sequential, prefix: str, bg: BatchedGemm):
        self.bg, self.lib = bg, bg.lib
        self.layers: List[Tuple[str, int, int, bool, float]] = []      # (name, n_out, n_in, relu after, dropout p after)
        mods = list(seq)
        for i, m in enumerate(mods):
            if isinstance(m, nn.Linear):
                relu = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
                drop = float(mods[i + 2].p) if relu and i + 2 < len(mods) and isinstance(mods[i + 2], nn.Dropout) else 0.0
                self.layers.append((f"{prefix}{i}", int(m.weight.shape[0]), int(m.weight.shape[1]), relu, drop))

    def forward(self, X: torch.Tensor, gens: Optional[Sequence[torch.Generator]] = None) -> torch.Tensor:
        """-> logits [E, rows, n_out]; gens: the members' CUDA generators for the dropout masks (None = no dropout, eval)"""
        bg, E, s = self.bg, self.bg.E, _lib.stream_ptr()
        a = X.contiguous()
        rows = int(a.shape[-2])
        a_es = 0 if a.dim() == 2 else rows * int(a.shape[-1])
        self.saved = []
        for name, n_out, n_in, relu, drop in self.layers:
            out = torch.empty((E, rows, n_out), dtype=torch.float32, device=bg.dev)
            bg.gemm(rows, n_out, n_in, a, n_in, 1, a_es, bg.param(name + ".weight"), 1, n_in, bg.P, out, n_out, rows * n_out,
                    bg.param(name + ".bias"), bg.P, 1 if relu else 0)
            mask = None
            if gens is not None and relu and drop > 0:
                mask = _dropout_mask((rows, n_out), gens, 1.0 - drop, bg.dev)
                _lib.check(self.lib.pdf_mul_f32(out.data_ptr(), mask.data_ptr(), out.numel(), s), "pdf_mul_f32")
            self.saved.append((a, a_es, out, mask))
            a, a_es = out, rows * n_out
        return a

    def backward(self, dlogits: torch.Tensor) -> None:
        bg, E, s = self.bg, self.bg.E, _lib.stream_ptr()
        d = dlogits.contiguous()
        for (name, n_out, n_in, relu, drop), (a_in, a_es, out, mask) in zip(reversed(self.layers), reversed(self.saved)):
            rows = int(out.shape[1])
            if relu:
                _lib.check(self.lib.pdf_relu_mask_backward(d.data_ptr(), out.data_ptr(), _p(mask), d.numel(), s), "pdf_relu_mask_backward")
            bg.gemm(n_out, n_in, rows, d, 1, n_out, rows * n_out, a_in, n_in, 1, a_es, bg.grad(name + ".weight"), n_in, bg.P, acc=1)
            bg.colsum(rows, n_out, d, rows * n_out, name + ".bias")
            if name != self.layers[0][0]:
                dn = torch.empty((E, rows, n_in), dtype=torch.float32, device=bg.dev)
                bg.gemm(rows, n_in, n_out, d, n_out, 1, rows * n_out, bg.param(name + ".weight"), n_in, 1, bg.P, dn, n_in, rows * n_in)
                d = dn
        self.saved = []


class BatchedMilHeadTrainer:
    """MilHeadTrainer.forward_backward for E members of one MILAttentionNet architecture at once (BCE loss): bags [E, B, Lmax, D]
    (each member its own minibatch), member e's parameters and gradients in row e of the flat buffers."""

    def __init__(self, net: nn.Module, gated: bool, bg: BatchedGemm):
        self.bg, self.lib, self.gated = bg, bg.lib, bool(gated)
        self.H, self.D = (int(v) for v in net.instance[0].weight.shape)
        self.A = int((net.attn_v[0] if self.gated else net.attn[0]).weight.shape[0])
        self.NA = 2 * self.A if self.gated else self.A
        self.dropout = float(net.instance[2].p) if len(net.instance) > 2 else 0.0

    def forward_backward(self, X: torch.Tensor, lens: torch.Tensor, y: torch.Tensor, pos_weight: Optional[float],
                         gens: Sequence[torch.Generator]) -> Tuple[torch.Tensor, torch.Tensor]:
        """X [E, B, Lmax, D], lens [E, B] i32, y [E, B] f32 -> (loss [E], prob [E, B]); gradients ACCUMULATED into the flat buffer"""
        bg, E, s = self.bg, self.bg.E, _lib.stream_ptr()
        B, Lmax, D = (int(v) for v in X.shape[1:])
        rows, H, A, NA, P = B * Lmax, self.H, self.A, self.NA, bg.P
        X = X.contiguous()
        h = torch.empty((E, rows, H), dtype=torch.float32, device=bg.dev)
        bg.gemm(rows, H, D, X, D, 1, rows * D, bg.param("instance.0.weight"), 1, D, P, h, H, rows * H, bg.param("instance.0.bias"), P, act=1)
        mask = None
        if self.dropout > 0:
            mask = _dropout_mask((rows, H), gens, 1.0 - self.dropout, bg.dev)
            _lib.check(self.lib.pdf_mul_f32(h.data_ptr(), mask.data_ptr(), h.numel(), s), "pdf_mul_f32")
        vu = torch.empty((E, rows, NA), dtype=torch.float32, device=bg.dev)
        names = [("attn_v.0", 0), ("attn_u.0", A)] if self.gated else [("attn.0", 0)]
        for name, off in names:
            bg.gemm(rows, A, H, h, H, 1, rows * H, bg.param(name + ".weight"), 1, H, P, vu.data_ptr() + 4 * off, NA, rows * NA,
                    bg.param(name + ".bias"), P)
        ww, bw = ("attn_w.weight", "attn_w.bias") if self.gated else ("attn.2.weight", "attn.2.bias")
        w = _lib.MilWeights()
        w.D, w.H, w.A, w.gated = D, H, A, 1 if self.gated else 0
        w.w_w, w.b_w, w.w_cls, w.b_cls = bg.param(ww), bg.param(bw), bg.param("classifier.0.weight"), bg.param("classifier.0.bias")
        t = _lib.MilTrain()
        t.loss_type, t.pos_weight, t.focal_gamma, t.focal_alpha = 0, 1.0 if pos_weight is None else float(pos_weight), 2.0, -1.0
        t.d_w_w, t.d_b_w = bg.grad(ww), bg.grad(bw)
        t.d_w_cls, t.d_b_cls = bg.grad("classifier.0.weight"), bg.grad("classifier.0.bias")
        prob = torch.empty((E, B), dtype=torch.float32, device=bg.dev)
        loss = torch.empty(E, dtype=torch.float32, device=bg.dev)
        dh = torch.empty((E, rows, H), dtype=torch.float32, device=bg.dev)
        dvu = torch.empty((E, rows, NA), dtype=torch.float32, device=bg.dev)
        ws = torch.empty(int(self.lib.pdf_mil_pool_train_batched_workspace_bytes(E, C.byref(w), B)), dtype=torch.uint8, device=bg.dev)
        lens = lens.to(device=bg.dev, dtype=torch.int32).contiguous()
        y = y.to(device=bg.dev, dtype=torch.float32).contiguous()
        _lib.check(self.lib.pdf_mil_pool_train_batched(E, C.byref(w), P, C.byref(t), P, B, Lmax, h.data_ptr(), vu.data_ptr(), lens.data_ptr(),
                                                       y.data_ptr(), prob.data_ptr(), loss.data_ptr(), dh.data_ptr(), dvu.data_ptr(),
                                                       ws.data_ptr(), s), "pdf_mil_pool_train_batched")
        # attention layers: dW = dvu^T h, db = colsum(dvu), dh += dvu W
        for name, off in names:
            dv = dvu.data_ptr() + 4 * off
            bg.gemm(A, H, rows, dv, 1, NA, rows * NA, h, H, 1, rows * H, bg.grad(name + ".weight"), H, P, acc=1)
            bg.colsum(rows, A, dv, rows * NA, name + ".bias", d_rs=NA)
            bg.gemm(rows, H, A, dv, NA, 1, rows * NA, bg.param(name + ".weight"), H, 1, P, dh, H, rows * H, acc=1)
        # instance layer: ReLU (+ dropout) backward, dW_i = dh^T X, db_i
        _lib.check(self.lib.pdf_relu_mask_backward(dh.data_ptr(), h.data_ptr(), _p(mask), dh.numel(), s), "pdf_relu_mask_backward")
        bg.gemm(H, D, rows, dh, 1, H, rows * H, X, D, 1, rows * D, bg.grad("instance.0.weight"), D, P, acc=1)
        bg.colsum(rows, H, dh, rows * H, "instance.0.bias")
        return loss, prob


class BatchedAdam:
    """NativeAdam (+ clip_grad_norm_) per member over flat [E, P] parameters: one pdf_clip_scale_batched and one pdf_adam_step_batched
    per step.  Each member keeps its own step count; a member that is not active (stopped early) keeps its weights and moments."""

    def __init__(self, flat_param: torch.Tensor, lr: float, weight_decay: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8):
        self.lib = _lib.load()
        self.p = flat_param
        self.E, self.P = int(flat_param.shape[0]), int(flat_param.shape[1])
        self.lr, self.wd, self.b1, self.b2, self.eps = float(lr), float(weight_decay), float(betas[0]), float(betas[1]), float(eps)
        self.m, self.v = torch.zeros_like(flat_param), torch.zeros_like(flat_param)
        self.steps = [0] * self.E
        self._scale = torch.ones(self.E, dtype=torch.float32, device=flat_param.device)
        self._flags: Dict[Tuple[bool, ...], torch.Tensor] = {}

    def clip(self, flat_grad: torch.Tensor, max_norm: float) -> torch.Tensor:
        _lib.check(self.lib.pdf_clip_scale_batched(self.E, flat_grad.data_ptr(), self.P, float(max_norm), self._scale.data_ptr(),
                                                   _lib.stream_ptr()), "pdf_clip_scale_batched")
        return self._scale

    def _active_ptr(self, flags: Tuple[bool, ...]):
        if all(flags):
            return None
        if flags not in self._flags:
            self._flags[flags] = torch.tensor(flags, dtype=torch.uint8, device=self.p.device)
        return self._flags[flags].data_ptr()

    def step(self, flat_grad: torch.Tensor, scale: Optional[torch.Tensor] = None, active: Optional[Sequence[bool]] = None):
        """one Adam step of every active member; members whose step counts differ (after an earlier early stop) step in one launch
        per distinct count"""
        act = [True] * self.E if active is None else [bool(a) for a in active]
        for cnt in sorted({self.steps[e] for e in range(self.E) if act[e]}):
            flags = tuple(act[e] and self.steps[e] == cnt for e in range(self.E))
            _lib.check(self.lib.pdf_adam_step_batched(self.E, self.p.data_ptr(), flat_grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                                      self.P, self.lr, self.b1, self.b2, self.eps, self.wd, cnt + 1, _p(scale),
                                                      self._active_ptr(flags), _lib.stream_ptr()), "pdf_adam_step_batched")
            for e in range(self.E):
                if flags[e]:
                    self.steps[e] += 1

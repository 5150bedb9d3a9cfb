"""Host side of K2: ResNet18/50 (torchvision state_dict layout, fc = Identity, eval mode) lowered to a
flat list of NHWC ops executed by libpdfusion_b200.so.

Reference: `_build_resnet_backbone` + the chunked `model(batch)` loop, data/openneuro_features.py:153-164,
257-262.  The state_dict key layout (SURVEY.md A.6) is the weight-interchange format: any torchvision
ResNet18/50 state_dict loads unchanged.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Sequence, Tuple

import torch
import torch.nn as nn

from . import _lib

RESNET_SPECS = {"resnet18": ("basic", [2, 2, 2, 2], 512), "resnet50": ("bottleneck", [3, 4, 6, 3], 2048)}
_PLANES = [64, 128, 256, 512]


# ----------------------------------------------------------------------------------------------------
# state_dict-compatible module (used only to create / hold weights; the forward pass below is for
# completeness of the nn.Module contract, the product path never calls it)
# ----------------------------------------------------------------------------------------------------
class _Basic(nn.Module):
    expansion = 1

    def __init__(self, inp, planes, stride, down):
        super().__init__()
        self.conv1 = nn.Conv2d(inp, planes, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(planes, planes, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = down

    def forward(self, x):
        idn = x if self.downsample is None else self.downsample(x)
        o = self.relu(self.bn1(self.conv1(x)))
        return self.relu(self.bn2(self.conv2(o)) + idn)


class _Bottleneck(nn.Module):
    expansion = 4

    def __init__(self, inp, planes, stride, down):
        super().__init__()
        self.conv1 = nn.Conv2d(inp, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, stride, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = down

    def forward(self, x):
        idn = x if self.downsample is None else self.downsample(x)
        o = self.relu(self.bn1(self.conv1(x)))
        o = self.relu(self.bn2(self.conv2(o)))
        return self.relu(self.bn3(self.conv3(o)) + idn)


class ResNet2D(nn.Module):
    """torchvision.models.resnet.ResNet with identical parameter names, construction order and
    initialisation, so `torch.manual_seed(s); ResNet2D(arch)` reproduces torchvision's random init."""

    def __init__(self, arch: str):
        super().__init__()
        kind, layers, _ = RESNET_SPECS[arch]
        block = _Basic if kind == "basic" else _Bottleneck
        self.inplanes = 64
        self.conv1 = nn.Conv2d(3, 64, 7, 2, 3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, 2, 1)
        for i, (planes, n) in enumerate(zip(_PLANES, layers), start=1):
            setattr(self, f"layer{i}", self._make_layer(block, planes, n, 1 if i == 1 else 2))
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        self.fc = nn.Linear(512 * block.expansion, 1000)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)

    def _make_layer(self, block, planes, blocks, stride):
        down = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            down = nn.Sequential(nn.Conv2d(self.inplanes, planes * block.expansion, 1, stride, bias=False),
                                 nn.BatchNorm2d(planes * block.expansion))
        layers = [block(self.inplanes, planes, stride, down)]
        self.inplanes = planes * block.expansion
        for _ in range(1, blocks):
            layers.append(block(self.inplanes, planes, 1, None))
        return nn.Sequential(*layers)

    def forward(self, x):
        x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        return self.fc(torch.flatten(self.avgpool(x), 1))


def detect_arch(sd: Dict[str, torch.Tensor]) -> str:
    return "resnet50" if "layer1.0.conv3.weight" in sd else "resnet18"


# ----------------------------------------------------------------------------------------------------
# lowering
# ----------------------------------------------------------------------------------------------------
def _bn_affine(sd, prefix: str, eps: float = 1e-5) -> Tuple[torch.Tensor, torch.Tensor]:
    """eval-mode BatchNorm as y = x*scale + shift (float64 maths, SURVEY.md A.5)."""
    g, b = sd[prefix + ".weight"].double(), sd[prefix + ".bias"].double()
    mu, var = sd[prefix + ".running_mean"].double(), sd[prefix + ".running_var"].double()
    scale = g / torch.sqrt(var + eps)
    return scale, b - mu * scale


def conv_list(arch: str) -> List[dict]:
    """Every conv of the network in execution order with its wiring."""
    kind, layers, _ = RESNET_SPECS[arch]
    out = [dict(name="conv1", bn="bn1", cin=3, cout=64, k=7, stride=2, pad=3, role="stem")]
    inp = 64
    for li, (planes, n) in enumerate(zip(_PLANES, layers), start=1):
        for bi in range(n):
            p = f"layer{li}.{bi}"
            stride = 2 if (li > 1 and bi == 0) else 1
            exp = 1 if kind == "basic" else 4
            has_down = bi == 0 and (stride != 1 or inp != planes * exp)
            if kind == "basic":
                out.append(dict(name=p + ".conv1", bn=p + ".bn1", cin=inp, cout=planes, k=3, stride=stride, pad=1, role="a", block=p, down=has_down))
                out.append(dict(name=p + ".conv2", bn=p + ".bn2", cin=planes, cout=planes, k=3, stride=1, pad=1, role="last", block=p))
            else:
                out.append(dict(name=p + ".conv1", bn=p + ".bn1", cin=inp, cout=planes, k=1, stride=1, pad=0, role="a", block=p, down=has_down))
                out.append(dict(name=p + ".conv2", bn=p + ".bn2", cin=planes, cout=planes, k=3, stride=stride, pad=1, role="b", block=p))
                out.append(dict(name=p + ".conv3", bn=p + ".bn3", cin=planes, cout=planes * 4, k=1, stride=1, pad=0, role="last", block=p))
            if has_down:
                out.append(dict(name=p + ".downsample.0", bn=p + ".downsample.1", cin=inp, cout=planes * exp, k=1, stride=stride, pad=0, role="down", block=p))
            inp = planes * exp
    return out


def flops_per_image(arch: str, input_size: int = 224, folded_stem: bool = False) -> float:
    """2*MAC over all convs at 3 x S x S (SURVEY.md 8(d): 3 627 122 688 r18 / 8 174 272 512 r50 at 224)."""
    convs = conv_list(arch)
    ho = (input_size + 6 - 7) // 2 + 1
    total = 2.0 * ho * ho * 64 * 49 * (1 if folded_stem else 3)
    size = (ho + 2 - 3) // 2 + 1
    block_in = t = size
    for cv in convs[1:]:
        if cv["role"] == "a":
            block_in = t = size
        hin = block_in if cv["role"] in ("a", "down") else t
        ho = (hin + 2 * cv["pad"] - cv["k"]) // cv["stride"] + 1
        total += 2.0 * ho * ho * cv["cout"] * cv["k"] ** 2 * cv["cin"]
        if cv["role"] in ("a", "b"):
            t = ho
        elif cv["role"] == "last":
            t = size = ho
    return total


# measured (profiles/r01_op_times_dual.txt): stage 2 -21 us, stage 3 -6 us, stage 4 +15 us (its 128-wide tiles re-read A four times)
DEFAULT_DUAL_STAGES = (2, 3)
# Bottleneck networks, bf16 path: residual stages whose conv3 launch also computes the NEXT block's conv1 (conv_pw.cu) -- the
# chained accumulator needs planes <= 256 TMEM columns, i.e. stages 1..3
DEFAULT_CHAIN_STAGES = (1, 2, 3)
# Bottleneck networks, bf16 path: residual stages whose block-0 conv3 launch also computes the projection shortcut (downsample) as
# more K of the same GEMM (conv_pw.cu, shortcut segment); the downsample launch and its 4x-wide output disappear.  Measured
# (profiles/r03_shortcut_ab.txt, 768 slices, downsample + conv3 -> fused conv3): stage 1 840 -> 516 us, stage 2 597 -> 498 us,
# stage 3 426 -> 404 us, stage 4 290 -> 308 us (its K = 1536 k-loop re-streams the A tile for each of 16 N chunks)
DEFAULT_SHORTCUT_STAGES = (1, 2, 3)


def _parse_stages(env: str, default: Sequence[int]) -> Tuple[int, ...]:
    """Stage list of a tuning hook: unset = default, "" or "none" = no stage, "1,2" = those stages."""
    v = os.environ.get(env)
    if v is None:
        return tuple(default)
    if v.strip().lower() == "none":
        return ()
    return tuple(int(t) for t in v.split(",") if t)


def lower_resnet(arch: str, n: int, S: int, bf16: bool, fused_stem: bool, chunks: List[int], in_bytes: int | None = None,
                 dual_stages: Sequence[int] = (), chain_stages: Sequence[int] = (), cross_stage_chain: bool = True,
                 shortcut_stages: Sequence[int] = ()):
    """The network as a flat, ordered list of ops over symbolic buffers.

    Returns (ops, extents, final_hw): ops = [(name, fields, refs, weight_name)], where refs maps the pointer fields
    d_in / d_out / d_residual to (buffer, byte offset); extents = bytes each buffer must hold.  Buffers: "input",
    "output", o0..o4 (stage outputs of the chunk being consumed), s0..s3 (scratch inside a stage).

    dual_stages: residual stages (2..4) of a BasicBlock network whose first block computes its 1x1 downsample INSIDE the 3x3 conv1
    launch (bf16 path; the conv op then carries `_weight2` = the downsample's weight name and a `d_out2` reference).

    chain_stages: residual stages (1..3) of a Bottleneck network whose conv3 launch also computes the next block's conv1 (the op
    carries `_weight3` and a `d_out3` reference; that conv1 is not emitted).  With cross_stage_chain the LAST conv3 of such a stage
    also computes the first conv1 of the following stage (stride 1 in torchvision's v1.5 Bottleneck; <= 256 output channels), into
    buffer x<k+1>.

    shortcut_stages: residual stages (1..4) of a Bottleneck network whose first block emits no downsample op: its conv3 op reads the
    block input as a shortcut segment (refs d_residual = the block input, fields sc_c / sc_hw, `_shortcut` = the downsample's
    weight name; the weights are [W3 | Wds] and the bias b3 + bds) -- relu(h W3^T + x_s Wds^T + b3 + bds) is one GEMM over K.

    chunks[k] = images per launch of stage k (0 = stem, 1..4 = residual stages).  The op list is depth-first: a
    stage-k chunk is preceded by the stage-(k-1) chunks that produce its input, so the big early tensors are consumed
    while they are still in L2 (SURVEY.md 7.3-1)."""
    kind, _, _ = RESNET_SPECS[arch]
    prec = _lib.PREC_BF16 if bf16 else _lib.PREC_F32
    esz = 2 if bf16 else 4
    exp = 1 if kind == "basic" else 4
    h1 = (S + 6 - 7) // 2 + 1
    h2 = (h1 + 2 - 3) // 2 + 1
    if in_bytes is None:                      # bytes of one input image (the fused stem reads a zero-padded image)
        in_bytes = S * S * 2 if bf16 else S * S * 3 * 4
    # stage geometry: spatial size and channels of each stage's OUTPUT (stage 0 = stem + maxpool)
    hw, ch = [h2], [64]
    for k in range(1, 5):
        hw.append(hw[-1] if k == 1 else (hw[-1] + 2 - 3) // 2 + 1)
        ch.append(_PLANES[k - 1] * exp)

    convs = conv_list(arch)
    stage_blocks: List[List[Dict[str, dict]]] = [[] for _ in range(5)]
    for cv in convs[1:]:
        k, bi = int(cv["block"][5]), int(cv["block"].split(".")[1])
        while len(stage_blocks[k]) <= bi:
            stage_blocks[k].append({})
        stage_blocks[k][bi][cv["role"]] = cv

    extents: Dict[str, int] = {}
    ops: List[tuple] = []
    scratch = ("s0", "s1", "s2", "s3", "s4")

    def ref(buf, off, nbytes):
        extents[buf] = max(extents.get(buf, 0), off + nbytes)
        return (buf, off)

    def add(name, refs, wname=None, **kw):
        ops.append((name, kw, refs, wname))

    def out_bytes(k, count, final=False):
        return count * hw[k] * hw[k] * ch[k] * (4 if (final and bf16) else esz)

    def emit_stem(start, count, dst):
        src = ref("input", start * in_bytes, count * in_bytes)
        if bf16 and fused_stem:
            # conv1 + bn1 + relu + maxpool in one kernel (stem_tc.cu): the patch matrix never leaves shared memory
            add("stem.fused", dict(d_in=src, d_out=dst), "conv1", kind=_lib.OP_STEM_FUSED, precision=prec, n=count, h=S, w=S, c=1,
                k=64, r=7, s=7, stride=2, pad=3, ho=h2, wo=h2, relu=1)
            return
        conv_out = ref("s0", 0, count * h1 * h1 * 64 * esz)
        if bf16:
            col = ref("s1", 0, count * h1 * h1 * 64 * esz)
            add("stem.im2col", dict(d_in=src, d_out=col), None, kind=_lib.OP_STEM_IM2COL, precision=prec, n=count, h=S, w=S, c=1, k=64,
                r=7, s=7, stride=2, pad=3, ho=h1, wo=h1)
            add("conv1", dict(d_in=col, d_out=conv_out), "conv1", kind=_lib.OP_CONV, precision=prec, n=count, h=h1, w=h1, c=64, k=64,
                r=1, s=1, stride=1, pad=0, ho=h1, wo=h1, relu=1)
        else:
            add("conv1", dict(d_in=src, d_out=conv_out), "conv1", kind=_lib.OP_CONV, precision=prec, n=count, h=S, w=S, c=3, k=64, r=7,
                s=7, stride=2, pad=3, ho=h1, wo=h1, relu=1)
        add("maxpool", dict(d_in=conv_out, d_out=dst), None, kind=_lib.OP_MAXPOOL, precision=prec, n=count, h=h1, w=h1, c=64, ho=h2,
            wo=h2)

    def cross_chain(k):
        """conv1 of stage k+1's first block, if the last conv3 launch of stage k may compute it (chained, conv_pw.cu)."""
        if not (bf16 and kind == "bottleneck" and k in chain_stages and 1 <= k < 4 and stage_blocks[k + 1]):
            return None
        nxt = stage_blocks[k + 1][0]["a"]
        if nxt["k"] == 1 and nxt["stride"] == 1 and nxt["cout"] in (64, 128, 256) and ch[k] % 128 == 0 and cross_stage_chain:
            return nxt
        return None

    def emit_stage(k, count, src, dst, chain_out=None, pre_chained=None):
        """All blocks of residual stage k over `count` images: src = stage k-1 output, dst = stage k output.
        chain_out: (ref, conv) -- the stage's last conv3 launch also computes the NEXT stage's first conv1 into ref;
        pre_chained: that tensor, handed to the stage that consumes it."""
        x, x_h, x_c = src, hw[k - 1], ch[k - 1]
        blocks = stage_blocks[k]
        free = list(scratch)
        chained = pre_chained
        for bi, cvs in enumerate(blocks):
            last_block = bi == len(blocks) - 1
            idn, idn_slot = x, None
            fuse_down = sc_down = None
            if "down" in cvs and (bf16 and kind == "bottleneck" and k in shortcut_stages and cvs["down"]["k"] == 1 and x_c % 64 == 0
                                  and not (last_block and k == 4)):
                sc_down = cvs["down"]["name"]              # computed by conv3's launch as more K; x stays alive to the block's end
            elif "down" in cvs:
                cv = cvs["down"]
                idn_slot = free.pop(0)
                idn = ref(idn_slot, 0, out_bytes(k, count))
                a = cvs["a"]
                if (bf16 and kind == "basic" and k in dual_stages and a["k"] == 3 and a["pad"] == 1 and a["stride"] == cv["stride"]
                        and a["cout"] == cv["cout"] and cv["cout"] % 128 == 0):
                    fuse_down = cv["name"]                 # computed by conv1's launch from its centre-tap tiles
                else:
                    add(cv["name"], dict(d_in=x, d_out=idn), cv["name"], kind=_lib.OP_CONV, precision=prec, n=count, h=x_h, w=x_h, c=x_c,
                        k=cv["cout"], r=1, s=1, stride=cv["stride"], pad=0, ho=hw[k], wo=hw[k], relu=0)
            t, t_h, t_c, t_slot = x, x_h, x_c, None
            seq = [cvs["a"]] + ([cvs["b"]] if "b" in cvs else []) + [cvs["last"]]
            if chained is not None:                        # conv1 of this block was computed by the previous block's conv3 launch
                t, t_h, t_c, t_slot = chained
                seq = seq[1:]
                chained = None
            nxt = blocks[bi + 1]["a"] if not last_block else None
            chain_next = (nxt is not None and bf16 and kind == "bottleneck" and k in chain_stages and nxt["k"] == 1 and nxt["stride"] == 1
                          and nxt["cout"] in (64, 128, 256) and cvs["last"]["cout"] % 128 == 0)
            for cv in seq:
                ho = (t_h + 2 * cv["pad"] - cv["k"]) // cv["stride"] + 1
                is_last = cv["role"] == "last"
                final = is_last and last_block and k == 4
                if is_last and last_block:
                    o, o_slot = dst, None
                else:
                    o_slot = free.pop(0)
                    o = ref(o_slot, 0, count * ho * ho * cv["cout"] * esz)
                refs = dict(d_in=t, d_out=o)
                if is_last:
                    refs["d_residual"] = idn
                extra = {}
                if is_last and sc_down is not None:
                    refs["d_residual"] = x
                    extra.update(_shortcut=sc_down, sc_c=x_c, sc_hw=(x_h << 16) | x_h)
                if fuse_down is not None and cv["role"] == "a":
                    refs["d_out2"] = idn
                    extra["_weight2"] = fuse_down
                if is_last and last_block and chain_out is not None:
                    refs["d_out3"] = chain_out[0]
                    extra["_weight3"] = chain_out[1]["name"]
                    extra["k3"] = chain_out[1]["cout"]
                if is_last and chain_next:
                    c_slot = free.pop(0)
                    refs["d_out3"] = ref(c_slot, 0, count * ho * ho * nxt["cout"] * esz)
                    extra["_weight3"] = nxt["name"]
                    extra["k3"] = nxt["cout"]
                    chained = (refs["d_out3"], ho, nxt["cout"], c_slot)
                add(cv["name"], refs, cv["name"], kind=_lib.OP_CONV, precision=prec, n=count, h=t_h, w=t_h, c=t_c, k=cv["cout"],
                    r=cv["k"], s=cv["k"], stride=cv["stride"], pad=cv["pad"], ho=ho, wo=ho, relu=1,
                    out_f32=1 if (final and bf16) else 0, **extra)
                if t_slot is not None:
                    free.append(t_slot)
                t, t_h, t_c, t_slot = o, ho, cv["cout"], o_slot
            if idn_slot is not None:
                free.append(idn_slot)
            if x[0] in scratch:
                free.append(x[0])
            x, x_h, x_c = t, t_h, t_c

    def emit(k, start, count, dst, chain_out=None):
        """Produce the stage-k output of images [start, start+count) at `dst`, depth-first over the earlier stages."""
        if k == 0:
            emit_stem(start, count, dst)
            return
        below = f"o{k - 1}"                       # holds the stage k-1 output of this chunk only
        per = hw[k - 1] * hw[k - 1] * ch[k - 1] * esz
        nxt = cross_chain(k - 1)                  # this stage's first conv1, computed by the stage below (its input never re-read)
        perc = hw[k - 1] * hw[k - 1] * nxt["cout"] * esz if nxt else 0
        for s0 in range(0, count, chunks[k - 1]):
            cnt = min(chunks[k - 1], count - s0)
            emit(k - 1, start + s0, cnt, ref(below, s0 * per, cnt * per),
                 (ref(f"x{k}", s0 * perc, cnt * perc), nxt) if nxt else None)
        emit_stage(k, count, (below, 0), dst, chain_out, ((f"x{k}", 0), hw[k - 1], nxt["cout"], None) if nxt else None)

    per4 = out_bytes(4, 1, final=True)
    for s0 in range(0, n, chunks[4]):
        cnt = min(chunks[4], n - s0)
        emit(4, s0, cnt, ref("o4", s0 * per4, cnt * per4))
    add("avgpool", dict(d_in=("o4", 0), d_out=ref("output", 0, n * ch[4] * 4)), None, kind=_lib.OP_AVGPOOL, precision=prec, n=n,
        h=hw[4], w=hw[4], c=ch[4], out_f32=1 if bf16 else 0)
    return ops, extents, hw[4]


class ResNetEncoder:
    """Runs `n_images` slices [n, S, S] through the backbone and returns [n, D] f32 embeddings.

    precision "bf16": tcgen05/TMEM implicit-GEMM convs, BN folded into bf16 weights + f32 bias, stem as a
        one-channel 7x7 (the 3 identical input channels folded: needs channel-uniform mean/std);
    precision "fp32": CUDA-core FFMA convs on the exact 3-channel input, BN applied as scale/shift in the epilogue.
    """

    def __init__(self, state_dict: Dict[str, torch.Tensor], n_images: int, input_size: int = 224,
                 precision: str = "bf16", arch: str | None = None, device=None, fused_stem: bool = True,
                 front_chunk: int | None = None, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.arch = arch or detect_arch(state_dict)
        self.kind, self.layers, self.emb_dim = RESNET_SPECS[self.arch]
        self.n = int(n_images)
        self.S = int(input_size)
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.bf16 = precision == "bf16"
        self.precision = precision
        self.fused_stem = bool(fused_stem)
        # (x-mean)/std of the reference's 3-channel input.  The bf16 path feeds ONE channel u = (x-mean_avg)/std_avg
        # (`input_mean_std`) and folds the per-channel differences into the stem weights and a border-dependent bias.
        self.mean = [float(m) for m in mean]
        self.std = [float(v) for v in std]
        self.input_mean_std = (sum(self.mean) / 3.0, sum(self.std) / 3.0)
        uniform = len(set(self.mean)) == 1 and len(set(self.std)) == 1
        if self.bf16 and not uniform and not self.fused_stem:
            raise ValueError("per-channel mean/std on the bf16 path needs the fused stem")
        env_chunk = os.environ.get("PDFUSION_B200_CHUNKS")          # "c1" or "c1,c2,c3,c4" (tuning hook)
        if front_chunk is None and env_chunk:
            vals = [int(v) for v in env_chunk.split(",")]
            front_chunk = vals[0] if len(vals) == 1 else vals
        self.front_chunk = front_chunk
        # residual stages whose 1x1 downsample is computed inside conv1's launch (BasicBlock networks, bf16 path)
        self.dual_stages = _parse_stages("PDFUSION_B200_DUAL", DEFAULT_DUAL_STAGES)          # tuning hook: "2,3,4" = those stages
        self.chain_stages = _parse_stages("PDFUSION_B200_CHAIN", DEFAULT_CHAIN_STAGES)       # tuning hook: "1,2" = those stages
        # Bottleneck stages whose downsample is computed inside block 0's conv3 launch (tuning hook: "1,2,3" = those stages)
        self.shortcut_stages = _parse_stages("PDFUSION_B200_SHORTCUT", DEFAULT_SHORTCUT_STAGES)
        sd = {k: v.detach().to("cpu") for k, v in state_dict.items()}
        self._keep: List[torch.Tensor] = []     # device tensors referenced by the plan
        self._build(sd)

    # -- weights ---------------------------------------------------------------------------------
    def _dev(self, t: torch.Tensor) -> torch.Tensor:
        d = t.contiguous().to(self.device)
        self._keep.append(d)
        return d

    def _conv_weights(self, sd, cv):
        w = sd[cv["name"] + ".weight"].double()                      # [K, C, R, S]
        scale, shift = _bn_affine(sd, cv["bn"])
        if self.bf16:
            wf = w * scale.view(-1, 1, 1, 1)
            if cv["role"] == "stem":
                # the three input channels are the same image: xn_c = a_c*u + b_c with u = (x-mean_avg)/std_avg
                m_avg, s_avg = self.input_mean_std
                a = torch.tensor([s_avg / sc_ for sc_ in self.std], dtype=torch.float64)
                bco = torch.tensor([(m_avg - mc) / sc_ for mc, sc_ in zip(self.mean, self.std)], dtype=torch.float64)
                w1 = (wf * a.view(1, 3, 1, 1)).sum(dim=1)               # [64, 7, 7]: channels folded
                border = None
                if bool((bco != 0).any()):
                    # sum_c w[k,c,t] * b_c over the taps INSIDE the image is a bias that depends on the conv pixel's border
                    # class; `shift` takes the interior value, the blob the differences (stem_tc.cu, pdf_op.d_scale)
                    wb = (wf * bco.view(1, 3, 1, 1)).sum(dim=1)         # [64, 7, 7]
                    S = self.S
                    h1 = (S + 6 - 7) // 2 + 1
                    masks, cls = [], []
                    for cy in range(h1):
                        mk = tuple(0 <= 2 * cy - 3 + r < S for r in range(7))
                        if mk not in masks:
                            masks.append(mk)
                        cls.append(masks.index(mk))
                    full = tuple([True] * 7)
                    if masks[0] != full:                               # class 0 must be the interior class
                        j = masks.index(full)
                        masks[0], masks[j] = masks[j], masks[0]
                        cls = [j if c == 0 else (0 if c == j else c) for c in cls]
                    nc = len(masks)
                    mt = torch.tensor(masks, dtype=torch.float64)      # [nc, 7]
                    inside = torch.einsum("krs,ar,bs->abk", wb, mt, mt)  # [nc, nc, 64]
                    delta = inside - inside[0, 0]
                    shift = shift + inside[0, 0]
                    blob = torch.cat([torch.tensor([nc, h1] + cls, dtype=torch.int32).view(torch.uint8),
                                      delta.float().contiguous().view(-1).view(torch.uint8)])
                    border = self._dev(blob)
                if self.fused_stem:
                    # stem_tc.cu: row v*64+c, K index t*8+s holds w[c][t-4v][s] (variant 1 = the filter 4 patch rows lower)
                    mat = torch.zeros(2, 64, 16, 8, dtype=torch.float64)
                    mat[0, :, 0:7, :7] = w1
                    mat[1, :, 4:11, :7] = w1
                    # K slots 88, 89 (t = 11, s = 0, 1) multiply a constant 1 in the kernel's B matrix: the bias rides through the
                    # tensor core as two bf16 terms (hi + lo, relative error 2^-17)
                    hi = shift.to(torch.bfloat16).double()
                    mat[:, :, 11, 0] = hi
                    mat[:, :, 11, 1] = shift - hi
                    mat = mat.reshape(128, 128)
                else:
                    mat = torch.zeros(w1.shape[0], 8, 8, dtype=torch.float64)  # im2col kernel: K index = r*8 + s
                    mat[:, :7, :7] = w1
                    mat = mat.reshape(w1.shape[0], 64)
                return self._dev(mat.to(torch.bfloat16)), border, self._dev(shift.float())
            return self._dev(wf.permute(0, 2, 3, 1).to(torch.bfloat16)), None, self._dev(shift.float())   # [K,R,S,C]
        return self._dev(w.permute(2, 3, 1, 0).float()), self._dev(scale.float()), self._dev(shift.float())  # [R,S,C,K]

    def _shortcut_weights(self, sd, wname, wname_sc, weights):
        """conv3 with its block's projection shortcut as more K: [W3 | Wds] ([K][c + sc_c] bf16, both BN folded), bias b3 + bds
        (summed in float64, then rounded once to f32)."""
        bn = {cv["name"]: cv["bn"] for cv in conv_list(self.arch)}
        w3, wds = weights[wname][0], weights[wname_sc][0]
        w = torch.cat([w3.reshape(w3.shape[0], -1), wds.reshape(wds.shape[0], -1)], dim=1)
        bias = _bn_affine(sd, bn[wname])[1] + _bn_affine(sd, bn[wname_sc])[1]
        return self._dev(w), None, self._dev(bias.float())

    # -- op list ---------------------------------------------------------------------------------
    def _chunk_sizes(self, h2: int, esz: int) -> List[int]:
        """Images per launch for the stem (index 0) and the four residual stages (1..4).

        `front_chunk` (or PDFUSION_B200_CHUNKS) turns on depth-first execution: a stage-k chunk is preceded by the
        stage-(k-1) chunks that produce its input, so early-stage tensors can be consumed from L2.  Measured on B200
        (gpurun_out/sweep_chunks.txt, C2, 768 slices) it LOSES 10-30 %: the 56x56 layers are bound by the
        shared-memory operand feed of the N=64 MMAs, not by HBM, and every extra launch costs a prologue and a tail.
        The default is therefore one launch per layer over the whole batch."""
        if isinstance(self.front_chunk, (list, tuple)):          # explicit per-stage sizes (stages 1..4)
            c = [max(1, min(self.n, int(v))) for v in self.front_chunk]
            c = (c + [self.n] * 4)[:4]
            return [c[0]] + c
        if self.front_chunk is not None:
            c1 = max(1, min(self.n, int(self.front_chunk)))
            c = [c1, c1]
            for _ in range(3):
                c.append(min(self.n, c[-1] * 2))
            c[4] = self.n
            return c
        return [self.n] * 5

    def _build(self, sd):
        n, S = self.n, self.S
        esz = 2 if self.bf16 else 4
        h1 = (S + 6 - 7) // 2 + 1
        h2 = (h1 + 2 - 3) // 2 + 1
        self.input_padded = None
        if self.bf16 and self.fused_stem:
            # zero-padded one-channel images (border written once, here); `input` is the S x S interior view
            pitch, rows = _lib.stem_padded_dims(S)
            self.input_padded = torch.zeros((n, rows, pitch), dtype=torch.bfloat16, device=self.device)
            lo = _lib.STEM_PAD_LO
            self.input = self.input_padded[:, lo:lo + S, lo:lo + S]
            in_bytes = rows * pitch * 2
        elif self.bf16:
            self.input = torch.empty((n, S, S), dtype=torch.bfloat16, device=self.device)
            in_bytes = S * S * 2
        else:
            self.input = torch.empty((n, S, S, 3), dtype=torch.float32, device=self.device)
            in_bytes = S * S * 3 * 4
        self.output = torch.empty((n, self.emb_dim), dtype=torch.float32, device=self.device)
        self.chunks = self._chunk_sizes(h2, esz)
        ops, extents, self.final_hw = lower_resnet(self.arch, n, S, self.bf16, self.fused_stem, self.chunks, in_bytes, self.dual_stages,
                                                     self.chain_stages, os.environ.get("PDFUSION_B200_XCHAIN", "1") != "0",
                                                     self.shortcut_stages)
        weights = {cv["name"]: self._conv_weights(sd, cv) for cv in conv_list(self.arch)}

        self.buffers = {name: torch.empty(nbytes, dtype=torch.uint8, device=self.device) for name, nbytes in extents.items()
                        if name not in ("input", "output")}
        base = {name: t.data_ptr() for name, t in self.buffers.items()}
        base["input"] = (self.input_padded if self.input_padded is not None else self.input).data_ptr()
        base["output"] = self.output.data_ptr()
        cops: List[_lib.Op] = []
        self.op_names: List[str] = []
        for name, kw, refs, wname in ops:
            op = _lib.Op()
            kw = dict(kw)
            wname2 = kw.pop("_weight2", None)
            wname3 = kw.pop("_weight3", None)
            wname_sc = kw.pop("_shortcut", None)
            for key, v in kw.items():
                setattr(op, key, v)
            if wname2 is not None:
                w2, _, b2 = weights[wname2]
                op.d_weight2, op.d_bias2 = w2.data_ptr(), b2.data_ptr()
            if wname3 is not None:
                w3, _, b3 = weights[wname3]
                op.d_weight3, op.d_bias3 = w3.data_ptr(), b3.data_ptr()
            for key, (buf, off) in refs.items():
                setattr(op, key, base[buf] + off)
            if wname is not None:
                w, sc, b = weights[wname] if wname_sc is None else self._shortcut_weights(sd, wname, wname_sc, weights)
                op.d_weight, op.d_scale, op.d_bias = w.data_ptr(), _lib.ptr(sc), b.data_ptr()
            cops.append(op)
            self.op_names.append(name)
        arr = (_lib.Op * len(cops))(*cops)
        plan = C.c_void_p()
        _lib.check(self.lib.pdf_plan_create(C.byref(plan), arr, len(cops)), "pdf_plan_create")
        self.plan = plan
        self.n_ops = len(cops)
        self.ops = cops

    def __del__(self):
        try:
            if getattr(self, "plan", None):
                self.lib.pdf_plan_destroy(self.plan)
                self.plan = None
        except Exception:
            pass

    @property
    def flops(self) -> float:
        """FLOPs actually executed by one run (stem folded to one channel, K padded to 64, on the bf16 path)."""
        return float(self.lib.pdf_plan_flops(self.plan))

    def algorithmic_flops(self) -> float:
        """SURVEY.md 8(d) figure for the work done: reference FLOPs, minus 2/3 of the stem when it is folded."""
        return self.n * flops_per_image(self.arch, self.S, folded_stem=self.bf16)

    def forward(self, x: torch.Tensor | None = None) -> torch.Tensor:
        """x: [n,S,S] bf16 (bf16 path) or [n,S,S,3] f32 (fp32 path); None = data already in self.input.
        Enqueues on the current stream, returns the (reused) output buffer [n, D] f32."""
        if x is not None and x.data_ptr() != self.input.data_ptr():
            self.input.copy_(x.reshape(self.input.shape))      # (into the interior view when the input is padded)
        _lib.check(self.lib.pdf_plan_run(self.plan, _lib.stream_ptr()), "pdf_plan_run")
        return self.output

    def feature_map(self) -> torch.Tensor:
        """The last stage's output of the latest run, [n, hw, hw, D] f32 (the average-pool input: the embedding is its spatial
        mean).  A read-only view of an encoder buffer that the next run overwrites."""
        hw = self.final_hw
        return self.buffers["o4"][: self.n * hw * hw * self.emb_dim * 4].view(torch.float32).view(self.n, hw, hw, self.emb_dim)

    def run_range(self, first: int, count: int) -> None:
        _lib.check(self.lib.pdf_plan_run_range(self.plan, first, count, _lib.stream_ptr()), "pdf_plan_run_range")

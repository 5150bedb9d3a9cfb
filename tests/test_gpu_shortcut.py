"""conv_pw_kernel's shortcut segment: a Bottleneck's projection shortcut (downsample 1x1 conv + BN of the block input x) computed as
more K of block 0's conv3, relu([h | x_s] [W3 | Wds]^T + b3 + bds) -- against an f32 torch computation on the same bf16 operands,
and the whole ResNet50 encoder with the shortcut segments on against the separate downsample launches and the fp32 path."""
import ctypes as C

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from pd_fusion_b200 import _lib
from pd_fusion_b200.backbone import ResNet2D, ResNetEncoder

CASES = [  # n, ho, c (conv3 input), sc_c (block input), cout, sh (block input size: ho = stride 1, else stride 2), k3 (chained conv1)
    (3, 14, 64, 64, 256, 14, 64),         # stage-1 shape: stride-1 shortcut, chained 256 -> 64
    (2, 7, 64, 64, 256, 7, 0),            # M = 98: one partial tile, unchained
    (5, 14, 128, 256, 512, 28, 128),      # stage-2 shape: im2col-mode shortcut 28 -> 14, chained
    (2, 7, 256, 512, 1024, 14, 256),      # stage-3 shape: the chained weight tile takes a whole ring stage
    (4, 4, 512, 1024, 2048, 7, 0),        # stage-4 shape at an odd size: 7 -> 4, 16 chunks per tile, K = 1536
    (3, 9, 64, 64, 256, 9, 0),            # odd stride-1 size
    (2, 18, 128, 256, 512, 35, 0),        # odd stride-2 size (S = 70: 35 -> 18)
    (300, 9, 64, 64, 256, 9, 64),         # > 148 M tiles: persistence, ring phases, buffer reuse
    (400, 9, 128, 256, 512, 17, 128),     # > 148 M tiles through im2col-mode loads (17 -> 9), chained
]


def _run(lib, ops, n_runs=2):
    plan = C.c_void_p()
    _lib.check(lib.pdf_plan_create(C.byref(plan), ops, len(ops)))
    try:
        for _ in range(n_runs):                          # twice: barriers / TMEM must come back clean
            _lib.check(lib.pdf_plan_run(plan, _lib.stream_ptr()))
        torch.cuda.synchronize()
        return lib.pdf_plan_flops(plan)
    finally:
        lib.pdf_plan_destroy(plan)


@pytest.mark.parametrize("n,ho,c,sc_c,cout,sh,k3", CASES)
def test_shortcut_segment_vs_torch(n, ho, c, sc_c, cout, sh, k3):
    lib = _lib.load()
    g = torch.Generator().manual_seed(n * 1000 + c + sc_c + k3)
    stride = 1 if sh == ho else 2
    assert (sh - 1) // stride + 1 == ho
    h = (torch.randn(n, ho, ho, c, generator=g) * 0.5).to(torch.bfloat16)
    x = (torch.randn(n, sh, sh, sc_c, generator=g) * 0.5).to(torch.bfloat16)
    w = (torch.randn(cout, c + sc_c, generator=g) / (c + sc_c) ** 0.5).to(torch.bfloat16)
    bias = torch.randn(cout, generator=g)
    w3 = (torch.randn(k3, cout, generator=g) / cout ** 0.5).to(torch.bfloat16) if k3 else None
    b3 = torch.randn(k3, generator=g) if k3 else None
    hd, xd, wd, bd = h.cuda(), x.cuda(), w.cuda(), bias.cuda()
    outs = []
    for mc in (0, 1):                                    # single CTAs and weight-multicast CTA pairs: bit-identical
        out = torch.full((n, ho, ho, cout), float("nan"), dtype=torch.bfloat16, device="cuda")
        out3 = torch.full((n, ho, ho, k3), float("nan"), dtype=torch.bfloat16, device="cuda") if k3 else None
        op = (_lib.Op * 1)()
        o = op[0]
        o.kind, o.precision = _lib.OP_CONV, _lib.PREC_BF16
        o.n, o.h, o.w, o.c, o.k, o.r, o.s, o.stride, o.pad, o.ho, o.wo, o.relu = n, ho, ho, c, cout, 1, 1, 1, 0, ho, ho, 1
        o.d_in, o.d_weight, o.d_bias, o.d_out, o.d_residual = hd.data_ptr(), wd.data_ptr(), bd.data_ptr(), out.data_ptr(), xd.data_ptr()
        o.sc_c, o.sc_hw = sc_c, (sh << 16) | sh
        if k3:
            w3d, b3d = w3.cuda(), b3.cuda()
            o.d_weight3, o.d_bias3, o.d_out3, o.k3 = w3d.data_ptr(), b3d.data_ptr(), out3.data_ptr(), k3
        try:
            _lib.check(lib.pdf_debug_set_pw_multicast(mc))
            flops = _run(lib, op)
        finally:
            lib.pdf_debug_set_pw_multicast(0)
        assert flops == 2.0 * n * ho * ho * cout * (c + sc_c) + (2.0 * n * ho * ho * k3 * cout if k3 else 0.0)
        outs.append((out.cpu(), out3.cpu() if k3 else None))
    assert torch.equal(outs[0][0], outs[1][0]) and (not k3 or torch.equal(outs[0][1], outs[1][1]))
    got, got3 = outs[0]
    xs = x[:, ::stride, ::stride].float()
    y = (h.float().reshape(-1, c) @ w[:, :c].float().T + xs.reshape(-1, sc_c) @ w[:, c:].float().T + bias).clamp_min(0)
    got = got.float().reshape(-1, cout)
    assert torch.isfinite(got).all()
    err = (got - y).abs().max().item()
    assert err < 1.2e-2 * max(1.0, y.abs().max().item()), err          # one bf16 rounding of the output
    if k3:
        t = (got @ w3.float().T + b3).clamp_min(0)                      # the chained conv reads the rounded output
        got3 = got3.float().reshape(-1, k3)
        assert torch.isfinite(got3).all()
        err3 = (got3 - t).abs().max().item()
        assert err3 < 1.2e-2 * max(1.0, t.abs().max().item()), err3


def test_shortcut_segment_rejects_bad_sizes():
    """The stride follows from the shortcut input's size: anything but (ho, wo) or its stride-2 source is refused."""
    lib = _lib.load()
    n, ho, c, sc_c, cout = 2, 7, 64, 64, 256
    h = torch.zeros(n, ho, ho, c, dtype=torch.bfloat16, device="cuda")
    x = torch.zeros(n, 16, 16, sc_c, dtype=torch.bfloat16, device="cuda")
    w = torch.zeros(cout, c + sc_c, dtype=torch.bfloat16, device="cuda")
    out = torch.empty(n, ho, ho, cout, dtype=torch.bfloat16, device="cuda")
    op = (_lib.Op * 1)()
    o = op[0]
    o.kind, o.precision = _lib.OP_CONV, _lib.PREC_BF16
    o.n, o.h, o.w, o.c, o.k, o.r, o.s, o.stride, o.pad, o.ho, o.wo, o.relu = n, ho, ho, c, cout, 1, 1, 1, 0, ho, ho, 1
    o.d_in, o.d_weight, o.d_out, o.d_residual = h.data_ptr(), w.data_ptr(), out.data_ptr(), x.data_ptr()
    o.sc_c, o.sc_hw = sc_c, (16 << 16) | 16               # 16 -> 8 at stride 2, not 7
    plan = C.c_void_p()
    assert lib.pdf_plan_create(C.byref(plan), op, 1) != 0


def _sd():
    torch.manual_seed(1234)
    return {k: v for k, v in ResNet2D("resnet50").state_dict().items() if not k.startswith("fc.")}


@pytest.mark.parametrize("n,S", [(5, 96), (3, 70), (16, 224)])
def test_shortcut_encoder_equals_separate_downsample(monkeypatch, n, S):
    """ResNet50 with every stage's projection shortcut inside block 0's conv3 against the separate downsample launches.  Not bit
    for bit: the separate path rounds the shortcut to bf16 before the add, the fused one adds it in the f32 accumulator.  That
    removes one bf16 rounding per element of each stage's block-0 output, not a reordering, so the 2e-3 bound of the tests whose
    bf16 intermediates stay the same does not hold: measured on a B200, 3.6e-3 at 96 px and 1.5e-3 at 224 px, where the bf16 path
    itself lies 4.0-4.5e-3 from the fp32 path with or without the fusion (test_shortcut_bf16_within_contract_of_fp32)."""
    sd = _sd()
    x = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(n + S)) * 2 - 1).to(torch.bfloat16).cuda()
    res = {}
    for sc in ("1,2,3,4", "none"):
        monkeypatch.setenv("PDFUSION_B200_SHORTCUT", sc)
        enc = ResNetEncoder(sd, n, S, precision="bf16")
        res[sc] = (enc.forward(x).clone(), enc.op_names, enc.flops)
        torch.cuda.synchronize()
    (a, names_a, fl_a), (b, names_b, fl_b) = res["1,2,3,4"], res["none"]
    assert not any("downsample" in v for v in names_a) and sum("downsample" in v for v in names_b) == 4
    assert len(names_a) == len(names_b) - 4
    assert fl_a == fl_b                                   # the downsample's MACs moved into conv3's K
    assert torch.isfinite(a).all() and float(b.abs().max()) > 0
    rel = ((a - b).norm(dim=1) / b.norm(dim=1)).max().item()
    assert rel < (2e-3 if S >= 224 else 5e-3), rel


def test_shortcut_encoder_default_stages(monkeypatch):
    monkeypatch.delenv("PDFUSION_B200_SHORTCUT", raising=False)
    from pd_fusion_b200.backbone import DEFAULT_SHORTCUT_STAGES
    enc = ResNetEncoder(_sd(), 2, 64, precision="bf16")
    assert enc.shortcut_stages == DEFAULT_SHORTCUT_STAGES
    for k in range(1, 5):
        assert (f"layer{k}.0.downsample.0" in enc.op_names) == (k not in DEFAULT_SHORTCUT_STAGES)


@pytest.mark.parametrize("n,S", [(4, 96), (3, 70)])
def test_shortcut_bf16_within_contract_of_fp32(monkeypatch, n, S):
    """bf16 path with every shortcut fused against the fp32 path on the same (uniformly normalised) input: within 1e-2 per slice."""
    sd = _sd()
    u = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(7 * n + S)) * 2 - 1).to(torch.bfloat16)
    monkeypatch.setenv("PDFUSION_B200_SHORTCUT", "1,2,3,4")
    enc = ResNetEncoder(sd, n, S, precision="bf16")
    got = enc.forward(u.cuda()).clone()
    enc32 = ResNetEncoder(sd, n, S, precision="fp32")
    ref = enc32.forward(u.float().unsqueeze(-1).expand(n, S, S, 3).contiguous().cuda()).clone()
    torch.cuda.synchronize()
    rel = ((got - ref).norm(dim=1) / ref.norm(dim=1)).max().item()
    assert rel < 1e-2, rel

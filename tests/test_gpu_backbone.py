"""K2 parity on the GPU: tcgen05 building block, FP32 and BF16 ResNet encoders vs the oracle / golden."""
import json

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O
from pd_fusion_b200 import _lib
from pd_fusion_b200.backbone import ResNet2D, ResNetEncoder
from pd_fusion_b200.synthetic import synthetic_volume


def _sd(arch):
    torch.manual_seed(1234)
    return {k: v for k, v in ResNet2D(arch).state_dict().items() if not k.startswith("fc.")}


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (300, 128, 192), (1000, 256, 576), (77, 512, 128),
                                   (20480, 256, 192), (19001, 128, 576), (9600, 512, 128), (40000, 256, 64)])   # last four: CTA-pair kernel
def test_umma_selftest(M, N, K):
    """TMA (2D, 128B swizzle) -> tcgen05.mma (TMEM accumulator) -> tcgen05.ld against an f32 matmul of the same bf16 data.
    The large cases also run through the CTA-pair kernel (tcgen05.mma.cta_group::2, multicast commit, remote arrives)."""
    lib = _lib.load()
    lib.pdf_debug_enable_pair(1 if M >= 9600 else 0)
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N)
    a = torch.randn(M, K, generator=g).to(torch.bfloat16).cuda()
    b = torch.randn(N, K, generator=g).to(torch.bfloat16).cuda()
    c = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    _lib.check(lib.pdf_selftest_umma(M, N, K, a.data_ptr(), b.data_ptr(), c.data_ptr(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    lib.pdf_debug_enable_pair(2)
    ref = a.float().cpu().double() @ b.float().cpu().double().T
    err = (c.cpu().double() - ref).abs().max().item()
    assert err < 1e-3 * max(1.0, ref.abs().max().item()), err


def _inputs(case_spec):
    sp = case_spec
    raw = synthetic_volume(sp["index"], tuple(sp["shape"]), bad_fraction=1e-4 if sp["shape"][0] < 100 else 1e-5)
    _, idx, sl = O.preprocess_subject(raw, tuple(sp["target"]), sp["axes"], sp["counts"])
    return O.slices_to_input(sl, sp["input_size"])        # [L,3,S,S] f32


@pytest.mark.parametrize("case", ["r18_small", "r50_small", "r18_c2"])
def test_fp32_encoder_vs_reference(golden, case):
    g = golden("embed")
    sp = json.loads(str(g[f"{case}/spec"]))
    x = _inputs(sp)
    enc = ResNetEncoder(_sd(sp["arch"]), x.shape[0], sp["input_size"], precision="fp32")
    out = enc.forward(torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 3, 1))).cuda())
    torch.cuda.synchronize()
    emb, ref = out.cpu().numpy(), g[f"{case}/emb"]
    rel = np.linalg.norm(emb - ref) / np.linalg.norm(ref)
    assert rel < 1e-5, rel                                  # north_star: fp32 path within 1e-5


@pytest.mark.parametrize("case", ["r18_small", "r50_small", "r18_c2", "r50_c3"])
def test_bf16_encoder_vs_reference(golden, case):
    g = golden("embed")
    sp = json.loads(str(g[f"{case}/spec"]))
    x = _inputs(sp)
    enc = ResNetEncoder(_sd(sp["arch"]), x.shape[0], sp["input_size"], precision="bf16")
    out = enc.forward(torch.from_numpy(np.ascontiguousarray(x[:, 0])).to(torch.bfloat16).cuda())
    torch.cuda.synchronize()
    emb, ref = out.cpu().numpy(), g[f"{case}/emb"]
    rel = np.linalg.norm(emb - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert rel.max() < 1e-2, rel                            # north_star: bf16 path within 1e-2 (norm-wise, per slice)


@pytest.mark.parametrize("S,n", [(224, 4), (64, 6), (70, 3)])
def test_bf16_encoder_with_per_channel_statistics(S, n):
    """ImageNet mean/std (what pretrained torchvision weights bring): the tcgen05 path feeds ONE channel normalised with the
    channel-averaged statistics; per-channel scale goes into the stem weights, the per-channel offset into a bias that
    depends on how much of the 7x7 window is inside the image.  Checked against the oracle on the true 3-channel input."""
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    sd = _sd("resnet18")
    g = torch.Generator().manual_seed(S + n)
    x = torch.rand(n, S, S, generator=g)                                      # slices in [0, 1]
    x[:, : S // 3] *= 0.02                                                    # dark background up to the border
    enc = ResNetEncoder(sd, n, S, precision="bf16", mean=mean, std=std)
    m_avg, s_avg = enc.input_mean_std
    enc.input.copy_(((x - m_avg) / s_avg).to(torch.bfloat16))
    out = enc.forward(None).clone()
    torch.cuda.synchronize()
    x3 = torch.stack([(x - m) / s_ for m, s_ in zip(mean, std)], dim=1)        # [n,3,S,S] f32, the reference's input
    ref = O.resnet_forward(sd, "resnet18", x3).numpy()
    emb = out.cpu().numpy()
    rel = np.linalg.norm(emb - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert rel.max() < 1e-2, rel
    # the correction matters: without the border blob the same weights must be measurably worse at small sizes
    enc32 = ResNetEncoder(sd, n, S, precision="fp32", mean=mean, std=std)
    out32 = enc32.forward(x3.permute(0, 2, 3, 1).contiguous().cuda()).cpu().numpy()
    rel32 = np.linalg.norm(out32 - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert rel32.max() < 1e-5, rel32


def test_bf16_layers_vs_fp32_layers():
    """Layer-by-layer: every bf16 tcgen05 conv (im2col TMA, strides, padding, residual epilogue) against the
    FP32 CUDA-core conv of the same layer fed with the SAME (bf16-rounded) input."""
    lib = _lib.load()
    torch.manual_seed(0)
    cases = [  # n, h, c, k, r, stride, pad, residual
        (3, 14, 64, 64, 3, 1, 1, True), (2, 16, 64, 128, 3, 2, 1, False), (2, 15, 128, 256, 1, 2, 0, False),
        (5, 8, 256, 64, 1, 1, 0, True), (1, 7, 512, 512, 3, 1, 1, True), (4, 9, 128, 128, 3, 2, 1, False),
    ]
    import ctypes as C
    for (n, h, c, k, r, stride, pad, res) in cases:
        ho = (h + 2 * pad - r) // stride + 1
        x = (torch.randn(n, h, h, c) * 0.5).to(torch.bfloat16)
        w = (torch.randn(k, r, r, c) / (r * r * c) ** 0.5).to(torch.bfloat16)
        bias = torch.randn(k)
        resid = (torch.randn(n, ho, ho, k) * 0.5).to(torch.bfloat16) if res else None
        xd, wd, bd = x.cuda(), w.cuda(), bias.cuda()
        rd = resid.cuda() if res else None
        out16 = torch.empty(n, ho, ho, k, dtype=torch.bfloat16, device="cuda")
        out32 = torch.empty(n, ho, ho, k, dtype=torch.float32, device="cuda")
        x32, w32 = xd.float().contiguous(), wd.float().permute(1, 2, 3, 0).contiguous()
        r32 = rd.float().contiguous() if res else None
        ops = (_lib.Op * 2)()
        for o, (prec, xi, wi, ri, oo) in zip(ops, [(_lib.PREC_BF16, xd, wd, rd, out16), (_lib.PREC_F32, x32, w32, r32, out32)]):
            o.kind, o.precision = _lib.OP_CONV, prec
            o.n, o.h, o.w, o.c, o.k, o.r, o.s, o.stride, o.pad, o.ho, o.wo, o.relu = n, h, h, c, k, r, r, stride, pad, ho, ho, 1
            o.d_in, o.d_weight, o.d_bias, o.d_out = xi.data_ptr(), wi.data_ptr(), bd.data_ptr(), oo.data_ptr()
            o.d_residual = ri.data_ptr() if res else None
        plan = C.c_void_p()
        _lib.check(lib.pdf_plan_create(C.byref(plan), ops, 2))
        _lib.check(lib.pdf_plan_run(plan, _lib.stream_ptr()))
        torch.cuda.synchronize()
        lib.pdf_plan_destroy(plan)
        a, b = out16.float().cpu(), out32.cpu()
        err = (a - b).abs().max().item()
        assert err < 2e-2 * max(1.0, b.abs().max().item()), ((n, h, c, k, r, stride, pad, res), err)


@pytest.mark.parametrize("S,n", [(224, 3), (64, 5), (70, 2)])
def test_fused_stem_equals_unfused(S, n):
    """stem_fused_kernel (in-smem im2col + tcgen05 + fused maxpool) must reproduce the three-kernel stem bit for bit."""
    sd = _sd("resnet18")
    x = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(S)) * 2 - 1).to(torch.bfloat16).cuda()
    outs = []
    for fused in (True, False):
        enc = ResNetEncoder(sd, n, S, precision="bf16", fused_stem=fused)
        enc.input.copy_(x)
        n_stem = 1 if fused else 3
        enc.run_range(0, n_stem)
        torch.cuda.synchronize()
        hp = ((S - 1) // 2 + 1 + 2 - 3) // 2 + 1
        first_conv = enc.ops[n_stem]           # the pooled stem output is the input of the first residual conv
        assert first_conv.h == hp
        slot = enc.buffers["o0"]                # stage-0 (stem + maxpool) output of the first chunk
        assert slot.data_ptr() == first_conv.d_in
        outs.append(slot[: n * hp * hp * 64 * 2].view(torch.bfloat16).clone())
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("arch,n,chunks", [("resnet18", 7, [2, 3, 4, 7]), ("resnet50", 5, [1, 2, 2, 4])])
def test_chunked_front_is_bit_identical(arch, n, chunks):
    """Depth-first chunking only changes WHICH images a launch covers, never the arithmetic of an output element."""
    sd = _sd(arch)
    S = 96
    x = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(n)) * 2 - 1).to(torch.bfloat16).cuda()
    outs = []
    for fc in (chunks, [n, n, n, n]):
        enc = ResNetEncoder(sd, n, S, precision="bf16", front_chunk=fc)
        outs.append(enc.forward(x).clone())
        torch.cuda.synchronize()
    assert torch.isfinite(outs[0]).all() and torch.equal(outs[0], outs[1])


def test_pair_kernel_matches_single_cta_kernel():
    """The CTA-pair conv kernel (cta_group::2, M = 256 across two SMs) accumulates the same K steps in the same order as the
    single-CTA kernel: a network large enough to route layers 3-4 through it gives the same embeddings as with pairs off; and
    with programmatic dependent launch off."""
    lib = _lib.load()
    sd = _sd("resnet18")
    n, S = 400, 224
    x = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(5)) * 2 - 1).to(torch.bfloat16).cuda()
    outs = {}
    try:
        for mode, pdl in ((2, 1), (0, 1), (1, 1), (2, 0), (3, 1)):       # 3 = + resident-weight pairs on the 128-channel 3x3 layers
            lib.pdf_debug_enable_pair(mode)
            lib.pdf_debug_enable_pdl(pdl)
            enc = ResNetEncoder(sd, n, S, precision="bf16")
            outs[(mode, pdl)] = enc.forward(x).clone()
            torch.cuda.synchronize()
    finally:
        lib.pdf_debug_enable_pair(2)
        lib.pdf_debug_enable_pdl(1)
    ref = outs[(0, 1)]
    assert torch.isfinite(ref).all()
    for key, o in outs.items():
        err = (o - ref).abs().max().item()
        assert err <= 1e-5 * ref.abs().max().item(), (key, err)


@pytest.mark.parametrize("n,S", [(7, 96), (40, 224), (3, 70)])
def test_fused_downsample_equals_separate_launches(monkeypatch, n, S):
    """resnet18's three 1x1 stride-2 downsample convolutions are computed inside the 3x3 stride-2 conv1 launch of their block
    (same centre-tap A tiles, second TMEM accumulator): the embeddings equal those of the separate launches."""
    sd = _sd("resnet18")
    x = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(n)) * 2 - 1).to(torch.bfloat16).cuda()
    outs = []
    for dual in ("2,3,4", "", "3"):
        monkeypatch.setenv("PDFUSION_B200_DUAL", dual)
        enc = ResNetEncoder(sd, n, S, precision="bf16")
        assert enc.dual_stages == tuple(int(v) for v in dual.split(",") if v)
        assert ("layer2.0.downsample.0" in enc.op_names) == (2 not in enc.dual_stages)
        outs.append(enc.forward(x).clone())
        torch.cuda.synchronize()
    ref = outs[1]
    assert torch.isfinite(ref).all()
    for o in (outs[0], outs[2]):
        assert (o - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()


def test_horizontally_shared_conv_equals_generic():
    """conv3x3_hs.cu: one im2col tile of W+2 positions per filter row serves the three horizontal taps through shifted MMA
    descriptors (A fetched 3x instead of 9x).  Same K order per output element as the generic kernel: the embeddings agree with
    the kernel off, on for the 128-channel layers, and on for every eligible layer."""
    lib = _lib.load()
    sd = _sd("resnet18")
    n, S = 200, 224
    x = (torch.rand(n, S, S, generator=torch.Generator().manual_seed(9)) * 2 - 1).to(torch.bfloat16).cuda()
    outs = {}
    try:
        for mode in (0, 1, 2):
            lib.pdf_debug_set_hs_mode(mode)
            enc = ResNetEncoder(sd, n, S, precision="bf16")
            outs[mode] = enc.forward(x).clone()
            torch.cuda.synchronize()
    finally:
        lib.pdf_debug_set_hs_mode(1)
    ref = outs[0]
    assert torch.isfinite(ref).all()
    for mode in (1, 2):
        # the taps are accumulated in (row, channel chunk, column) order instead of (row, column, channel chunk): f32 sums differ in the
        # last bits and a few bf16 activations round the other way -- far inside the 1e-2 contract, far outside what a wrong tap would do
        rel = ((outs[mode] - ref).norm(dim=1) / ref.norm(dim=1)).max().item()
        assert rel < 2e-3, (mode, rel)


@pytest.mark.parametrize("n,h,c,k,res", [(2, 6, 64, 128, False), (3, 28, 128, 128, True), (7, 14, 256, 256, True), (9, 7, 128, 512, False),
                                         (40, 28, 128, 128, True)])
def test_horizontally_shared_conv_single_layer(n, h, c, k, res):
    """One 3x3 stride-1 layer through conv3x3_hs.cu against an f32 convolution of the same bf16 data (bias, residual, ReLU; one and
    several n-tiles; tiles that run through image rows and images; more tiles than CTAs)."""
    import ctypes as C
    lib = _lib.load()
    g = torch.Generator().manual_seed(n * 100 + h)
    x = (torch.randn(n, h, h, c, generator=g) * 0.5).to(torch.bfloat16).cuda()
    w = (torch.randn(k, 3, 3, c, generator=g) / (3.0 * c ** 0.5)).to(torch.bfloat16).cuda()
    bias = torch.randn(k, generator=g).cuda()
    resid = (torch.randn(n, h, h, k, generator=g) * 0.5).to(torch.bfloat16).cuda() if res else None
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), bias, padding=1).permute(0, 2, 3, 1)
    if res:
        ref = ref + resid.float()
    ref = torch.relu(ref)
    out = torch.full((n, h, h, k), float("nan"), dtype=torch.bfloat16, device="cuda")
    ops = (_lib.Op * 1)()
    o = ops[0]
    o.kind, o.precision = _lib.OP_CONV, _lib.PREC_BF16
    o.n, o.h, o.w, o.c, o.k, o.r, o.s, o.stride, o.pad, o.ho, o.wo, o.relu = n, h, h, c, k, 3, 3, 1, 1, h, h, 1
    o.d_in, o.d_weight, o.d_bias, o.d_out = x.data_ptr(), w.data_ptr(), bias.data_ptr(), out.data_ptr()
    o.d_residual = resid.data_ptr() if res else None
    plan = C.c_void_p()
    lib.pdf_debug_set_hs_mode(3)                       # every eligible layer, whatever its size
    try:
        _lib.check(lib.pdf_plan_create(C.byref(plan), ops, 1))
        _lib.check(lib.pdf_plan_run(plan, _lib.stream_ptr()))
        torch.cuda.synchronize()
    finally:
        lib.pdf_debug_set_hs_mode(1)
    lib.pdf_plan_destroy(plan)
    err = (out.float() - ref).abs().max().item()
    assert not torch.isnan(out.float()).any() and err <= 2e-2 * max(1.0, ref.abs().max().item()), err


def test_umma_shifted_descriptor_probe():
    """Records whether an MMA operand may start at an arbitrary 128-byte row of a resident, 128B-swizzled tile --
    the precondition for halo-resident 3x3 convolutions.  The result is printed (pytest -s shows it)."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(3)
    a = torch.randn(256, 64, generator=g).to(torch.bfloat16).cuda()
    b = torch.randn(64, 64, generator=g).to(torch.bfloat16).cuda()
    res = {}
    for mode in (0, 1):
        for shift in (0, 1, 2, 3, 5, 8, 9, 58, 59, 117, 128):
            c = torch.zeros(128, 64, dtype=torch.float32, device="cuda")
            _lib.check(lib.pdf_selftest_umma_shift(64, shift, mode, a.data_ptr(), b.data_ptr(), c.data_ptr(), _lib.stream_ptr()))
            torch.cuda.synchronize()
            ref = a[shift:shift + 128].float() @ b.float().T
            res[(mode, shift)] = bool((c - ref).abs().max().item() < 1e-2)
    for mode in (0, 1):
        print(f"mode {mode}: " + " ".join(f"{s}:{'ok' if v else 'BAD'}" for (m, s), v in res.items() if m == mode))
    assert res[(0, 0)] and res[(0, 8)] and res[(0, 128)]      # 1024-byte aligned starts must work


@pytest.mark.parametrize("n,h,res", [(3, 56, True), (2, 28, False), (5, 17, True), (1, 9, False), (40, 56, True)])
def test_halo_conv_matches_im2col_conv(n, h, res):
    """conv3x3_c64_kernel (halo loaded once, 9 shifted descriptors, resident weights, persistent CTAs) vs the generic
    im2col-TMA kernel on the same bf16 data."""
    import ctypes as C
    lib = _lib.load()
    g = torch.Generator().manual_seed(n * 100 + h)
    x = (torch.randn(n, h, h, 64, generator=g) * 0.5).to(torch.bfloat16).cuda()
    w = (torch.randn(64, 3, 3, 64, generator=g) / 24.0).to(torch.bfloat16).cuda()
    bias = torch.randn(64, generator=g).cuda()
    resid = (torch.randn(n, h, h, 64, generator=g) * 0.5).to(torch.bfloat16).cuda() if res else None
    outs = []
    for disable in (0, 1):
        lib.pdf_debug_disable_halo(disable)
        out = torch.full((n, h, h, 64), float("nan"), dtype=torch.bfloat16, device="cuda")
        ops = (_lib.Op * 1)()
        o = ops[0]
        o.kind, o.precision = _lib.OP_CONV, _lib.PREC_BF16
        o.n, o.h, o.w, o.c, o.k, o.r, o.s, o.stride, o.pad, o.ho, o.wo, o.relu = n, h, h, 64, 64, 3, 3, 1, 1, h, h, 1
        o.d_in, o.d_weight, o.d_bias, o.d_out = x.data_ptr(), w.data_ptr(), bias.data_ptr(), out.data_ptr()
        o.d_residual = resid.data_ptr() if res else None
        plan = C.c_void_p()
        try:
            _lib.check(lib.pdf_plan_create(C.byref(plan), ops, 1))
            _lib.check(lib.pdf_plan_run(plan, _lib.stream_ptr()))
            torch.cuda.synchronize()
        finally:
            lib.pdf_debug_disable_halo(0)
        lib.pdf_plan_destroy(plan)
        outs.append(out.float().cpu())
    assert not torch.isnan(outs[0]).any()
    err = (outs[0] - outs[1]).abs().max().item()
    assert err <= 1e-2 * max(1.0, outs[1].abs().max().item()), err

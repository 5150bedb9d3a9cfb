"""Explanations on the GPU (pdf_mil_explain, pdf_gradcam, MilAttentionModel.explain, MilAttentionFineTuneModel.explain) against a
float64 torch computation of the same nn.Modules on the same weights: MILAttentionNet in eval mode and backbone.ResNet2D with a
forward hook on layer4, the logit differentiated by autograd."""
import copy

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import torch.nn.functional as F  # noqa: E402

from oracle import oracle as O  # noqa: E402
from pd_fusion_b200.heads import gradcam  # noqa: E402
from pd_fusion_b200.synthetic import synthetic_volume  # noqa: E402


def _head_oracle(net, x):
    """float64 logit, attention, contributions and d logit / d x of one bag x [L, D] through MILAttentionNet `net` (eval)."""
    x = x.detach().double().clone().requires_grad_(True)
    h = net.instance(x)
    s = (net.attn_w(net.attn_v(h) * net.attn_u(h)) if net.gated else net.attn(h)).squeeze(-1)
    a = torch.softmax(s, dim=0)
    lin = net.classifier[0]
    u = h @ lin.weight[0]
    z = lin(a @ h)[0]
    (dx,) = torch.autograd.grad(z, x)
    return z.item(), a.detach(), (a * u).detach(), dx


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ------------------------------------------------------------------------------------------------------ 1. MIL head
@pytest.mark.parametrize("gated", [True, False])
@pytest.mark.parametrize("dims", [(2048, 256, 128), (24, 12, 6)])
def test_mil_head_explain(gated, dims):
    from pd_fusion_b200.models.mil_attention import MilAttentionModel
    D, H, A = dims
    torch.manual_seed(3)
    m = MilAttentionModel(D, {"gated": gated, "hidden_dim": H, "attn_dim": A, "missing_prob": 0.37})
    rng = np.random.default_rng(11)
    lens = [7, None, 48, 1, 5, 48, None, 3]
    bags = [None if L is None else rng.normal(0.0, 1.0, (L, D)).astype(np.float32) for L in lens]
    masks = {"mri": np.array([1, 1, 1, 1, 0, 1, 1, 1])}                    # bag 4 is dropped by the mask
    ex = m.explain(bags, masks)
    prob = m.predict_proba(bags, masks)
    net = copy.deepcopy(m.model).double().eval().cuda()
    b_cls = float(net.classifier[0].bias)
    live = [i for i, L in enumerate(lens) if L is not None and masks["mri"][i]]
    for i in range(len(bags)):
        if i not in live:
            assert ex["attention"][i] is None and ex["contribution"][i] is None and np.isnan(ex["logit"][i])
            assert ex["prob"][i] == prob[i] == 0.37
            continue
        z, a, c, _ = _head_oracle(net, torch.from_numpy(bags[i]).cuda())
        att, con = ex["attention"][i], ex["contribution"][i]
        assert att.shape == con.shape == (lens[i],)
        assert np.abs(att - a.cpu().numpy()).max() <= 1e-6
        assert abs(float(att.astype(np.float64).sum()) - 1.0) <= 1e-6
        assert np.abs(con - c.cpu().numpy()).max() <= 1e-5
        # the per-slice decomposition: sum_l contrib + b_cls = logit, up to the rounding of a sum of terms of this size
        scale = float(np.abs(con).astype(np.float64).sum()) + abs(b_cls)
        assert abs(float(con.astype(np.float64).sum()) + b_cls - ex["logit"][i]) <= 1e-5 * scale
        assert abs(ex["logit"][i] - z) <= 1e-5 * max(1.0, abs(z))
    assert np.abs(ex["prob"] - prob).max() <= 1e-6
    print(f"explain prob vs predict_proba (gated={gated}, dims={dims}): bit-identical={bool(np.array_equal(ex['prob'], prob))}")

    # the head's gradient with respect to every instance
    head, X, lens_d = m._upload(bags, live)
    logit, attn, contrib, dX = head.explain(X, lens_d, need_grad=True)
    assert dX.shape == X.shape
    for j, i in enumerate(live):
        _, _, _, dx = _head_oracle(net, torch.from_numpy(bags[i]).cuda())
        assert _rel(dX[j, :lens[i]].cpu().numpy(), dx.cpu().numpy()) <= 1e-4, i
        assert not dX[j, lens[i]:].any() and not attn[j, lens[i]:].any() and not contrib[j, lens[i]:].any()
    # a missing bag (len 0) inside the call: NaN logit, zero attention and gradient
    lens0 = lens_d.clone()
    lens0[1] = 0
    logit0, attn0, _, dX0 = head.explain(X, lens0, need_grad=True)
    assert torch.isnan(logit0[1]) and not attn0[1].any() and not dX0[1].any()
    assert torch.equal(logit0[0], logit[0]) and torch.equal(dX0[0], dX[0])


# ------------------------------------------------------------------------------------------------------ 2. pdf_gradcam alone
@pytest.mark.parametrize("hw", [3, 7])
@pytest.mark.parametrize("C", [512, 2048])
@pytest.mark.parametrize("out_hw", [(160, 160), (96, 128)])
def test_gradcam_kernel(hw, C, out_hw):
    gen = torch.Generator(device="cuda").manual_seed(hw * 7919 + C)
    n = 5
    fmap = torch.randn((n, hw, hw, C), generator=gen, device="cuda").relu_()
    g = torch.randn((n, C), generator=gen, device="cuda")
    cam, small = gradcam(fmap, g, out_hw, cam_small=True)
    ref_small = torch.relu(torch.einsum("nijc,nc->nij", fmap.double(), g.double()) / (hw * hw))
    ref = F.interpolate(ref_small[:, None], size=out_hw, mode="bilinear", align_corners=False)[:, 0]
    for k in range(n):
        assert _rel(small[k].cpu().numpy(), ref_small[k].cpu().numpy()) <= 1e-5
        assert _rel(cam[k].cpu().numpy(), ref[k].cpu().numpy()) <= 1e-5
    assert (cam >= 0).all()
    # every pixel negative: exact zeros
    cam0, small0 = gradcam(fmap + 0.1, -g.abs() - 0.1, out_hw, cam_small=True)
    assert not cam0.any() and not small0.any()


# ------------------------------------------------------------------------------------------------------ 3-5. fine-tune model
def _ft_model(backbone, input_size, count, target=(64, 64, 64)):
    from pd_fusion_b200.models.mil_attention_finetune import MilAttentionFineTuneModel
    torch.manual_seed(21)
    return MilAttentionFineTuneModel({"backbone": backbone, "pretrained": False, "target_shape": target, "slice_axis": 2,
                                      "slice_count": count, "input_size": input_size, "train_aug": False, "batch_size": 4})


def _ft_oracle(m, slices, autocast=False):
    """Grad-CAM of one bag's slices [L, H, W] through the model's own modules: float64 (or the f32 backbone under
    torch.autocast(bfloat16), head in f32) -> (logit, attention, contributions, cam [L, H, W]) in float64."""
    dt = torch.float32 if autocast else torch.float64
    net = copy.deepcopy(m.backbone).to(dt).eval()
    head = copy.deepcopy(m.attn).to(dt).eval()
    feats = {}
    hook = net.layer4.register_forward_hook(lambda mod, inp, out: feats.__setitem__("a", out))
    x = torch.from_numpy(O.slices_to_input(slices, m.input_size, m.mean_vals, m.std_vals)).to("cuda", dt)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        net(x)
    hook.remove()
    act = feats["a"].detach().requires_grad_(True)
    emb = act.to(dt).mean(dim=(2, 3))                   # the average pool (fc is Identity), differentiated from layer4 on
    h = head.instance(emb)
    s = (head.attn_w(head.attn_v(h) * head.attn_u(h)) if head.gated else head.attn(h)).squeeze(-1)
    a = torch.softmax(s, dim=0)
    lin = head.classifier[0]
    z = lin(a @ h)[0]
    (grad,) = torch.autograd.grad(z, act)
    act, grad = act.detach().double(), grad.double()
    small = torch.relu((grad.mean(dim=(2, 3), keepdim=True) * act).sum(dim=1))
    cam = F.interpolate(small[:, None], size=tuple(slices.shape[1:]), mode="bilinear", align_corners=False)[:, 0]
    return z.item(), a.detach().double().cpu().numpy(), (a * (h @ lin.weight[0])).detach().double().cpu().numpy(), cam.cpu().numpy()


def _bags(m, tmp_path, lens, hw):
    rng = np.random.default_rng(5)
    bags = [rng.random((L, hw, hw), dtype=np.float32) for L in lens]
    p = tmp_path / "vol.npy"
    np.save(p, synthetic_volume(3, (72, 80, 70), 0.0).astype(np.float32))
    return bags + [str(p)]


@pytest.mark.parametrize("cfg", [("resnet18", 64, 6, [6, 3]), ("resnet50", 224, 48, [48, 48])], ids=["resnet18", "resnet50"])
def test_finetune_explain_fp32(tmp_path, monkeypatch, cfg):
    monkeypatch.setenv("PD_FUSION_B200_PRECISION", "fp32")
    backbone, size, count, lens = cfg
    m = _ft_model(backbone, size, count)
    bags = _bags(m, tmp_path, lens, 64)
    bags.insert(1, None)
    ex = m.explain(bags)
    prob = m.predict_proba(bags)
    assert np.abs(ex["prob"] - prob).max() <= 1e-6
    assert ex["cam"][1] is None and ex["slices"][1] is None and np.isnan(ex["logit"][1])
    for i, b in enumerate(bags):
        if b is None:
            continue
        sl = ex["slices"][i]
        assert np.array_equal(sl, m._bag_slices(b))
        assert ex["cam"][i].shape == sl.shape and (ex["cam"][i] >= 0).all()
        z, a, c, cam = _ft_oracle(m, sl)
        assert np.abs(ex["attention"][i] - a).max() <= 1e-4
        assert np.abs(ex["contribution"][i] - c).max() <= 1e-4 * max(1.0, np.abs(c).max())
        err = _rel(ex["cam"][i], cam)
        print(f"fp32 {backbone} bag {i} ({sl.shape[0]} slices): CAM distance to float64 {err:.2e}")
        assert err <= 1e-3, (i, err)


@pytest.mark.parametrize("cfg", [("resnet18", 64, 6, [6, 3]), ("resnet50", 224, 48, [48, 48])], ids=["resnet18", "resnet50"])
def test_finetune_explain_bf16(tmp_path, monkeypatch, cfg):
    """The bf16 encoder's CAMs against float64, with the bar calibrated by torch's own autocast(bfloat16) Grad-CAM of the same
    network: at most 3x its distance, and never held tighter than 2e-2."""
    monkeypatch.delenv("PD_FUSION_B200_PRECISION", raising=False)
    backbone, size, count, lens = cfg
    m = _ft_model(backbone, size, count)
    bags = _bags(m, tmp_path, lens, 64)
    ex = m.explain(bags)
    assert np.abs(ex["prob"] - m.predict_proba(bags)).max() <= 1e-6
    for i in range(len(bags)):
        sl = ex["slices"][i]
        _, _, _, ref = _ft_oracle(m, sl)
        _, _, _, tbf = _ft_oracle(m, sl, autocast=True)
        ours, torch_bf16 = _rel(ex["cam"][i], ref), _rel(tbf, ref)
        print(f"bf16 {backbone} bag {i} ({sl.shape[0]} slices): CAM distance to float64 {ours:.2e}, torch autocast bf16 {torch_bf16:.2e}")
        assert ours <= max(3.0 * torch_bf16, 2e-2), (i, ours, torch_bf16)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_finetune_explain_pass_structure(tmp_path, monkeypatch, precision):
    """One bag per encoder pass gives bit for bit what one pass over all bags gives."""
    from pd_fusion_b200 import backbone as BB
    monkeypatch.setenv("PD_FUSION_B200_PRECISION", precision)
    m = _ft_model("resnet18", 64, 6)
    bags = _bags(m, tmp_path, [6, 4, 6], 64)
    passes = [0]
    real = BB.ResNetEncoder.forward

    def counting(self, *a, **k):
        passes[0] += 1
        return real(self, *a, **k)
    monkeypatch.setattr(BB.ResNetEncoder, "forward", counting)
    one = m.explain(bags)
    assert passes[0] == 1
    longest = max(s.shape[0] for s in one["slices"])
    monkeypatch.setenv("PD_FUSION_B200_FT_IMAGES", str(longest))
    passes[0] = 0
    many = m.explain(bags)
    assert passes[0] == len(bags)
    assert np.array_equal(one["prob"], many["prob"]) and np.array_equal(one["logit"], many["logit"])
    for key in ("attention", "contribution", "slices", "cam"):
        for a, b in zip(one[key], many[key]):
            assert np.array_equal(a, b), key

"""Explanations of the fusion heads on the GPU (pdf_moddrop_explain, pdf_moe_explain, ModalityDropoutModel.explain, MoEModel.explain,
evaluation.evaluate.explain_model) against float64 torch on the same ModalityDropoutNet / MoENet modules in eval mode: Shapley values
by brute-force enumeration of the masked inputs, integrated gradients by autograd at the same midpoints."""
import json
from math import factorial

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402
from pd_fusion_b200.heads import ModDropSweep, MoeSweep  # noqa: E402
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutNet  # noqa: E402
from pd_fusion_b200.models.moe import MoENet  # noqa: E402
from pd_fusion_b200.synthetic import synthetic_table  # noqa: E402

S = 7


def _shapley64(v, mk):
    """brute force: v [2^M, N] float64 coalition values, mk [S, N, M] {0,1} -> phi [S, N, M]"""
    Sn, N, M = mk.shape
    P = (mk.astype(np.int64) << np.arange(M)).sum(-1)                     # [S, N]
    p = np.array([bin(q).count("1") for q in range(1 << M)])[P]
    wt = np.array([[factorial(t) * factorial(q - t - 1) / factorial(q) if t < q else 0.0 for t in range(M + 1)] for q in range(M + 1)])
    phi = np.zeros((Sn, N, M))
    for m in range(M):
        for T in range(1 << M):
            if (T >> m) & 1:
                continue
            on = ((P & T) == T) & (((P >> m) & 1) == 1)
            phi[:, :, m] += np.where(on, wt[p, bin(T).count("1")], 0.0) * (v[T | (1 << m)] - v[T])[None, :]
    return phi


def _cols(sizes, bits):
    """feature-column mask [F] of the modality bit set `bits` (blocks in order)"""
    return np.concatenate([np.full(d, (bits >> j) & 1, np.float64) for j, d in enumerate(sizes)])


def _md_net(dims, hidden, seed):
    torch.manual_seed(seed)
    net = ModalityDropoutNet(dims, hidden, 0.3).eval()
    return net


def _md_oracle_values(net, X, sizes):
    """v [2^M, N] float64 logits of every coalition (net without its final Sigmoid)"""
    f = net.net[:-1].double().cuda()
    Xd = torch.from_numpy(X).double().cuda()
    with torch.no_grad():
        return np.stack([f(Xd * torch.from_numpy(_cols(sizes, c)).cuda())[:, 0].cpu().numpy() for c in range(1 << len(sizes))])


def _forward_margin(layers, x):
    """float64 forward of Linear/ReLU/Dropout(eval) layers without the final Sigmoid -> (logit [n], margin [n], z1 [n, h1]): margin =
    the smallest |z| / (|W||h| + |b|) over the hidden pre-activations, i.e. how far the row is from a ReLU kink relative to the rounding
    scale; z1 = layer 1's pre-activation (its gradient is delta1)"""
    lins = [m for m in layers if isinstance(m, torch.nn.Linear)]
    margin = torch.full((x.shape[0],), float("inf"), dtype=x.dtype, device=x.device)
    h, z1 = x, None
    for i, lin in enumerate(lins):
        z = lin(h)
        z1 = z if z1 is None else z1
        if i < len(lins) - 1:
            bound = h.detach().abs() @ lin.weight.detach().abs().T + lin.bias.detach().abs()
            margin = torch.minimum(margin, (z.detach().abs() / bound).min(1).values)
            h = torch.relu(z)
    return z[:, 0], margin, z1


def _ig_cond(xm, dbar, W1, ig):
    """conditioning of ig = (x (.) m) (.) (dbar W1) per row: || |x m| (.) (|dbar| |W1|) || / || ig ||, all float64 (inf where ig = 0).
    A float32 computation that rounds dbar and sums the h1 products dbar_i W1_if is off by about one float32 ulp times this."""
    num = torch.linalg.norm(xm.abs() * (dbar.abs() @ W1.abs()), dim=-1).cpu().numpy()
    den = np.linalg.norm(ig, axis=-1)
    return np.where(den > 0, num / np.maximum(den, 1e-300), np.inf)


def _md_oracle_ig(net, X, mk, sizes, K):
    """ig [S, N, F] float64, the smallest ReLU margin [S, N] over the K midpoints, and the conditioning [S, N] of ig"""
    f = net.net[:-1].double().cuda()
    W1 = f[0].weight.detach()
    Xd = torch.from_numpy(X).double().cuda()
    out = np.zeros((mk.shape[0],) + X.shape)
    margin, cond = np.zeros(mk.shape[:2]), np.zeros(mk.shape[:2])
    for s in range(mk.shape[0]):
        colm = torch.from_numpy(np.repeat(mk[s].astype(np.float64), sizes, axis=1)).cuda()
        xm = Xd * colm
        g = torch.zeros_like(xm)
        d1 = torch.zeros((X.shape[0], W1.shape[0]), dtype=torch.float64, device=xm.device)
        mg = torch.full((X.shape[0],), float("inf"), dtype=torch.float64, device=xm.device)
        for k in range(K):
            inp = ((k + 0.5) / K * xm).requires_grad_(True)
            z, mk_, z1 = _forward_margin(f, inp)
            gk, dk = torch.autograd.grad(z.sum(), [inp, z1])
            g += gk
            d1 += dk
            mg = torch.minimum(mg, mk_)
        out[s] = (xm * g / K).cpu().numpy()
        margin[s] = mg.cpu().numpy()
        cond[s] = _ig_cond(xm, d1 / K, W1, out[s])
    return out, margin, cond


def _check_ig(got, ref, margin, cond, what):
    """per-subject relative norm error <= max(1e-5, eps32 * cond), i.e. 1e-5 unless the subject's ig is so ill-conditioned that one
    float32 ulp of its summed magnitudes is larger.  The exception: a float64 path passing a ReLU kink closer than float32 rounding
    (margin < 1e-5), where no float32 evaluation can decide the gate; such subjects must stay rare."""
    nr = np.linalg.norm(ref, axis=-1)
    assert np.all(got[nr == 0] == 0), what
    live = nr > 0
    rel = np.linalg.norm(got - ref, axis=-1)[live] / nr[live]
    tol = np.maximum(1e-5, np.finfo(np.float32).eps * cond[live])
    bad = rel > tol
    assert np.median(rel) <= 1e-6, (what, float(np.median(rel)))
    assert np.all(margin[live][bad] < 1e-5), (what, float((rel / tol)[margin[live] >= 1e-5].max()))
    assert bad.mean() <= 0.01, (what, float(bad.mean()))


def _check_shapley(phi, value, base, ref_phi, ref_v, mk, sizes):
    Mm = mk.shape[2]
    P = (mk.astype(np.int64) << np.arange(Mm)).sum(-1)
    scale = np.abs(ref_phi).sum(-1) + abs(ref_v[0, 0])
    err = np.abs(phi - ref_phi).max(-1)
    assert np.all(err <= 1e-5 * scale), float((err / scale).max())
    dead = (mk == 0) | (np.array(sizes)[None, None, :] == 0)
    assert np.all(phi[dead] == 0)                                        # absent and zero-width modalities: exactly 0
    np.testing.assert_allclose(value, np.take_along_axis(ref_v, P, axis=0), rtol=0, atol=2e-5 * (np.abs(ref_v).max() + 1))
    sum_tol = 4 * np.finfo(np.float32).eps * (np.abs(phi).sum(-1) + np.abs(value) + abs(base))
    assert np.all(np.abs(phi.astype(np.float64).sum(-1) - (value.astype(np.float64) - base)) <= sum_tol)   # efficiency


MD_CASES = [({"clinical": 0, "datspect": 0, "mri": 512}, [256, 128, 64]),      # C2 widths
            ({"clinical": 10, "datspect": 5, "mri": 20}, [64, 32]),
            ({"clinical": 7, "datspect": 3, "mri": 33}, [500, 40]),
            ({"clinical": 10, "datspect": 5, "mri": 20}, [])]


@pytest.mark.parametrize("dims,hidden", MD_CASES)
@pytest.mark.parametrize("N", [100_000, 300])
def test_moddrop_shapley_and_value(dims, hidden, N):
    """Exact Shapley values of the logit under 7 random scenario masks; value = the sweep's logit (sigmoid bit-identical to the
    sweep's probability, tiled or warp-per-pair); two calls bit-identical."""
    net = _md_net(dims, hidden, N + len(hidden))
    sw = ModDropSweep(net.state_dict(), dims)
    sizes = [dims[m] for m in sw.mods]
    rng = np.random.default_rng(N)
    X = rng.standard_normal((N, sum(sizes))).astype(np.float32)
    mk = (rng.random((S, N, 3)) < 0.6).astype(np.uint8)
    Xd, md = torch.from_numpy(X).cuda(), torch.from_numpy(mk).cuda()
    value, base, phi, ig = sw.explain(Xd, md, 0)
    assert ig is None
    prob = sw.forward(Xd, md)
    assert torch.equal(torch.sigmoid(value), prob)
    v2, b2, phi2, _ = sw.explain(Xd, md, 0)
    assert torch.equal(v2, value) and torch.equal(b2, base) and torch.equal(phi2, phi)
    ref_v = _md_oracle_values(net, X, sizes)
    _check_shapley(phi.cpu().numpy(), value.cpu().numpy(), float(base.item()), _shapley64(ref_v, mk), ref_v, mk, sizes)
    assert abs(base.item() - ref_v[0, 0]) <= 1e-5 * (abs(ref_v[0, 0]) + 1)


@pytest.mark.parametrize("dims,hidden,K", [(MD_CASES[0][0], MD_CASES[0][1], 32), (MD_CASES[1][0], MD_CASES[1][1], 1),
                                           (MD_CASES[1][0], MD_CASES[1][1], 8), (MD_CASES[1][0], MD_CASES[1][1], 32),
                                           (MD_CASES[1][0], MD_CASES[1][1], 100), (MD_CASES[2][0], MD_CASES[2][1], 32),
                                           (MD_CASES[3][0], MD_CASES[3][1], 8)])
def test_moddrop_integrated_gradients(dims, hidden, K):
    """IG of the logit from 0 with K midpoints against autograd in float64: per-subject relative norm error <= 1e-5, absent
    modalities' features exactly 0, bit-identical across calls.  One-layer net: ig = (x (.) m) (.) w1 and its per-modality sums are the
    Shapley values."""
    N = 3000
    net = _md_net(dims, hidden, K + len(hidden))
    sw = ModDropSweep(net.state_dict(), dims)
    sizes = [dims[m] for m in sw.mods]
    rng = np.random.default_rng(K)
    X = rng.standard_normal((N, sum(sizes))).astype(np.float32)
    mk = (rng.random((S, N, 3)) < 0.6).astype(np.uint8)
    Xd, md = torch.from_numpy(X).cuda(), torch.from_numpy(mk).cuda()
    value, base, phi, ig = sw.explain(Xd, md, K)
    ig = ig.cpu().numpy()
    assert torch.equal(sw.explain(Xd, md, K)[3].cpu(), torch.from_numpy(ig))
    colm = np.repeat(mk, sizes, axis=2)
    assert np.all(ig[colm == 0] == 0)
    ref, margin, cond = _md_oracle_ig(net, X, mk, sizes, K)
    _check_ig(ig, ref, margin, cond, "moddrop")
    if not hidden:
        w1 = net.net[0].weight.detach().cpu().numpy()[0].astype(np.float64)
        np.testing.assert_allclose(ig, X[None].astype(np.float64) * colm * w1, rtol=1e-6, atol=1e-7)
        phi = phi.cpu().numpy()
        off = np.cumsum([0] + sizes)
        per_mod = np.stack([ig[:, :, off[j]:off[j + 1]].sum(-1) for j in range(3)], axis=-1)
        scale = np.abs(phi).sum(-1, keepdims=True) + abs(base.item())
        assert np.all(np.abs(per_mod - phi) <= 1e-6 * scale)


def _moe_net(dims, seed):
    torch.manual_seed(seed)
    return MoENet(dims, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16]}).eval()


def _moe_oracle(net, X, mk, mods, K):
    """v [2^E, N] (coalitions) and, with K, ig {mod: [S, N, d]} float64"""
    n64 = net.double().cuda()
    Xd = {m: torch.from_numpy(X[m]).double().cuda() for m in mods}
    E, N = len(mods), X[mods[0]].shape[0]
    v = []
    with torch.no_grad():
        for c in range(1 << E):
            cm = torch.tensor([(c >> j) & 1 for j in range(E)], dtype=torch.float64).cuda()
            v.append(n64({m: Xd[m] * cm[j] for j, m in enumerate(mods)}, cm.expand(N, E))[:, 0].cpu().numpy())
    v = np.stack(v)
    if not K:
        return v, None
    ig = {m: np.zeros((mk.shape[0], N, X[m].shape[1])) for m in mods}
    margin = {m: np.zeros(mk.shape[:2]) for m in mods}         # per expert, as _md_oracle_ig
    cond = {m: np.zeros(mk.shape[:2]) for m in mods}
    for s in range(mk.shape[0]):
        mask = torch.from_numpy(mk[s].astype(np.float64)).cuda()
        xm = {m: Xd[m] * mask[:, j:j + 1] for j, m in enumerate(mods)}
        g = {m: torch.zeros_like(xm[m]) for m in mods}
        d1 = {m: 0.0 for m in mods}
        mg = {m: torch.full((N,), float("inf"), dtype=torch.float64, device=Xd[m].device) for m in mods}
        w = n64.router(mask).detach()                          # MoENet.forward: router(mask), experts gated in sorted order
        for k in range(K):
            inp = {m: ((k + 0.5) / K * xm[m]).requires_grad_(True) for m in mods}
            out, z1 = 0.0, {}
            for j, m in enumerate(mods):
                z, mk_, z1[m] = _forward_margin(n64.experts[m].net[:-1], inp[m])
                out = out + torch.sigmoid(z) * w[:, j]
                mg[m] = torch.minimum(mg[m], mk_)
            grads = torch.autograd.grad(out.sum(), [inp[m] for m in mods] + [z1[m] for m in mods])
            for j, m in enumerate(mods):
                g[m] += grads[j]
                d1[m] = d1[m] + grads[len(mods) + j]
        for m in mods:
            ig[m][s] = (xm[m] * g[m] / K).cpu().numpy()
            margin[m][s] = mg[m].cpu().numpy()
            cond[m][s] = _ig_cond(xm[m], d1[m] / K, n64.experts[m].net[0].weight.detach(), ig[m][s])
    return v, (ig, margin, cond)


@pytest.mark.parametrize("dims", [{"clinical": 10, "mri": 512}, {"clinical": 10, "datspect": 5, "mri": 20}])
@pytest.mark.parametrize("N,K", [(100_000, 0), (2000, 32), (2000, 8), (2000, 1)])
def test_moe_explain(dims, N, K):
    """MoE: Shapley values of the probability (value bit-identical to pdf_moe_sweep), IG per expert against float64 autograd."""
    net = _moe_net(dims, N + K + len(dims))
    mods = sorted(dims)
    sw = MoeSweep(net.state_dict(), mods)
    rng = np.random.default_rng(N + K)
    X = {m: rng.standard_normal((N, dims[m])).astype(np.float32) for m in mods}
    mk = (rng.random((S, N, len(mods))) < 0.6).astype(np.uint8)
    Xd, md = {m: torch.from_numpy(X[m]).cuda() for m in mods}, torch.from_numpy(mk).cuda()
    value, base, phi, ig = sw.explain(Xd, md, K)
    assert torch.equal(value, sw.forward(Xd, md))
    again = sw.explain(Xd, md, K)
    assert torch.equal(again[0], value) and torch.equal(again[2], phi)
    v, ref = _moe_oracle(net, X, mk, mods, K)
    _check_shapley(phi.cpu().numpy(), value.cpu().numpy(), float(base.item()), _shapley64(v, mk), v, mk, [dims[m] for m in mods])
    if not K:
        assert ig is None
        return
    for j, m in enumerate(mods):
        assert torch.equal(again[3][j], ig[j])
        got = ig[j].cpu().numpy()
        assert np.all(got[mk[:, :, j] == 0] == 0)
        _check_ig(got, ref[0][m], ref[1][m], ref[2][m], m)


def test_model_explain_and_explain_model(golden):
    """ModalityDropoutModel.explain / MoEModel.explain take predict_proba's arguments and return its probabilities; explain_model
    draws evaluate_model's scenario masks (same seed -> the same per-scenario probabilities); the MIL kind is refused."""
    from pd_fusion_b200.data.preprocess import NaNRobustScaler
    from pd_fusion_b200.evaluation.evaluate import _sweep_probs, explain_model
    from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel
    from pd_fusion_b200.models.mil_attention import MilAttentionModel
    from pd_fusion_b200.models.moe import MoEModel
    g = golden("heads")
    dims = json.loads(str(g["table/dims"]))
    df, masks = synthetic_table(int(g["table/n"]), dims, seed=42, mask_seed=7)
    scen = json.loads(str(g["scenarios"]))
    cols = [c for m in O.MODALITIES for c in df.columns if c.startswith(m + "_")]
    md = ModalityDropoutModel(dims, {"hidden_dims": [64, 32], "dropout": 0.2, "lr": 1e-3, "epochs": 1})
    md.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moddrop/sd/")})
    scaler = NaNRobustScaler().fit(df[cols].values)
    np.random.seed(11)
    probs, _ = _sweep_probs(md, df, masks, (None, scaler, cols), scen["scenarios"])
    np.random.seed(11)
    ex = explain_model(md, df, masks, (None, scaler, cols), scen, steps=8)
    assert list(ex) == [sc["name"] for sc in scen["scenarios"]]
    for s, sc in enumerate(scen["scenarios"]):
        e = ex[sc["name"]]
        assert np.array_equal(e["prob"], probs[s].astype(np.float64))
        tot = sum(e["shapley"].values())
        assert np.all(np.abs(tot - (e["logit"] - e["base_logit"])) <= 1e-5 * (np.abs(e["logit"]) + 1))
        assert e["ig"].shape == (len(df), len(cols))
    X = scaler.transform(df[cols].values)
    cur = {m: g["masks_seed11"][2][:, i] for i, m in enumerate(O.MODALITIES)}
    e = md.explain(X, masks=cur, steps=0)
    assert e["prob"].dtype == np.float64 and np.array_equal(e["prob"], md.predict_proba(X, masks=cur).astype(np.float64))
    assert e["ig"] is None and set(e["shapley"]) == set(O.MODALITIES)

    mods = [str(m) for m in g["moe/mods"]]
    moe = MoEModel({m: dims[m] for m in mods}, {"expert_hidden_dims": [32, 16], "router_hidden_dims": [16], "lr": 1e-3, "epochs": 1})
    moe.model.load_state_dict({k.split("/sd/")[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("moe/sd/")})
    prep = {}
    for m in mods:
        cm = [c for c in df.columns if c.startswith(m + "_")]
        prep[m] = (None, NaNRobustScaler().fit(df[cm].values), cm)
    np.random.seed(12)
    probs, _ = _sweep_probs(moe, df, {m: masks[m] for m in mods}, prep, scen["scenarios"])
    np.random.seed(12)
    ex = explain_model(moe, df, {m: masks[m] for m in mods}, prep, scen, steps=4)
    for s, sc in enumerate(scen["scenarios"]):
        e = ex[sc["name"]]
        assert np.array_equal(e["prob"], probs[s].astype(np.float64))
        assert set(e["ig"]) == set(mods)
    mk = g["moe/masks_seed12"][1]
    Xd = {m: torch.FloatTensor(prep[m][1].transform(df[prep[m][2]].values) * mk[:, i:i + 1]) for i, m in enumerate(mods)}
    e = moe.explain(Xd, torch.FloatTensor(mk.astype(np.float32)), steps=8)
    assert np.array_equal(e["prob"], moe.predict_proba(Xd, torch.FloatTensor(mk.astype(np.float32))).astype(np.float64))
    assert np.all(np.abs(sum(e["shapley"].values()) - (e["prob"] - e["base_prob"])) <= 1e-6)
    assert all(e["ig"][m].shape == (len(df), dims[m]) for m in mods)

    mil = MilAttentionModel(8, {"hidden_dim": 8, "attn_dim": 4, "gated": True})
    with pytest.raises(ValueError, match="MilAttentionModel.explain"):
        explain_model(mil, df, masks, ("mil", "bags"), scen)
    with pytest.raises(ValueError, match="MilAttentionModel.explain"):
        explain_model(object(), df, masks, (None, scaler, cols), scen)

"""Deep ensembles on the GPU (csrc/train.cu, training.Batched*, models.ensemble.HeadEnsemble, evaluation.evaluate.ensemble_model):
the batched kernels against the single-model kernels member by member, every member against the single-model training sequence of
its seed, independence of the other members, determinism, launch counts, and the ensemble's inference and evaluation."""
import ctypes as C

import numpy as np
import pandas as pd
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from pd_fusion_b200 import _lib  # noqa: E402
from pd_fusion_b200.models.ensemble import HeadEnsemble  # noqa: E402
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel  # noqa: E402
from pd_fusion_b200.models.mil_attention import MilAttentionModel  # noqa: E402
from pd_fusion_b200.models.moe import MoEModel  # noqa: E402
from test_ensemble_cabi import ensemble_stats_np  # noqa: E402

DIMS = {"clinical": 7, "datspect": 5, "mri": 9}
SEEDS = [11, 23, 5, 42]
# The MIL attention-score bias shifts every score of a bag alike, and the softmax does not see a shift: its gradient is exactly zero, so
# what the kernels compute for it is rounding noise of a zero sum, which depends on the summation order (atomics in the single kernel,
# bag order here).  Adam normalises that noise into full-size steps, so this one scalar follows a different random walk on either path.
SCORE_BIAS = ("attn_w.bias", "attn.2.bias")


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-12))


def _lib_():
    return _lib.load()


def _s():
    return _lib.stream_ptr()


# ------------------------------------------------------------------ kernels against the single-model kernels

GEMM_CASES = [  # (name, E, M, N, K, A layout, B layout, bias, act, acc); layouts are (rs, cs, member stride) in elements
    ("forward", 3, 70, 33, 19, "rowmajor", "weight", True, 1, 0),
    ("shared_input", 4, 130, 64, 40, "shared", "weight", True, 0, 0),
    ("wgrad", 3, 33, 19, 70, "transposed", "rowmajor_k", False, 0, 1),
    ("dgrad", 2, 70, 19, 33, "rowmajor", "weight_t", False, 0, 0),
    ("colsum", 3, 1, 33, 70, "ones", "rowmajor_k", False, 0, 1),
]


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_batched_bit_identical(case):
    name, E, M, N, K, al, bl, has_bias, act, acc = case
    g = torch.Generator(device="cuda").manual_seed(1)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g)
    if al == "rowmajor":
        A, (a_rs, a_cs, a_es) = rnd(E, M, K), (K, 1, M * K)
    elif al == "shared":
        A, (a_rs, a_cs, a_es) = rnd(M, K), (K, 1, 0)
    elif al == "transposed":                     # A(i, k) = d[k, i]: dW = d^T x
        A, (a_rs, a_cs, a_es) = rnd(E, K, M), (1, M, K * M)
    else:
        A, (a_rs, a_cs, a_es) = torch.ones(K, device="cuda"), (0, 1, 0)
    P = 4096 + 8                                  # weights live in rows of a flat [E, P] buffer
    if bl == "weight":                           # B(k, j) = W[j, k], W [N, K]
        Bt, (b_rs, b_cs, b_es) = rnd(E, P), (1, K, P)
    elif bl == "weight_t":                       # B(k, j) = W[k, j], W [K, N]
        Bt, (b_rs, b_cs, b_es) = rnd(E, P), (N, 1, P)
    else:
        Bt, (b_rs, b_cs, b_es) = rnd(E, K, N), (N, 1, K * N)
    bias = rnd(E, P) if has_bias else None
    C0 = rnd(E, M, N)
    Cb, Cs = C0.clone(), C0.clone()
    lib = _lib_()
    _lib.check(lib.pdf_gemm_f32_batched(E, M, N, K, A.data_ptr(), a_rs, a_cs, a_es, Bt.data_ptr(), b_rs, b_cs, b_es, Cb.data_ptr(), N, M * N,
                                        None if bias is None else bias.data_ptr() + 4 * 8, P, act, acc, _s()), "batched")
    for e in range(E):
        _lib.check(lib.pdf_gemm_f32(M, N, K, A.data_ptr() + 4 * e * a_es, a_rs, a_cs, Bt.data_ptr() + 4 * e * b_es, b_rs, b_cs,
                                    Cs[e].data_ptr(), N, None if bias is None else bias.data_ptr() + 4 * (e * P + 8), act, acc, _s()), "single")
    torch.cuda.synchronize()
    assert torch.equal(Cb, Cs)


def test_bce_and_moe_batched_against_single():
    lib, E, n, M = _lib_(), 3, 1037, 3
    g = torch.Generator(device="cuda").manual_seed(2)
    z = torch.randn(E, n, device="cuda", generator=g) * 4
    y = (torch.rand(E, n, device="cuda", generator=g) < 0.4).float()
    pb, dzb, lb = torch.empty_like(z), torch.empty_like(z), torch.empty(E, device="cuda")
    _lib.check(lib.pdf_bce_sigmoid_train_batched(E, n, z.data_ptr(), y.data_ptr(), n, pb.data_ptr(), lb.data_ptr(), dzb.data_ptr(), _s()), "b")
    zm = torch.randn(E, n, M, device="cuda", generator=g) * 3
    rm = torch.randn(E, n, M, device="cuda", generator=g) * 2
    ym = y[0].contiguous()
    ob, lmb, dzm, drm = torch.empty(E, n, device="cuda"), torch.empty(E, device="cuda"), torch.empty_like(zm), torch.empty_like(rm)
    _lib.check(lib.pdf_moe_combine_train_batched(E, n, M, zm.data_ptr(), rm.data_ptr(), ym.data_ptr(), 0, ob.data_ptr(), lmb.data_ptr(),
                                                 dzm.data_ptr(), drm.data_ptr(), _s()), "m")
    for e in range(E):
        p, dz, l = torch.empty(n, device="cuda"), torch.empty(n, device="cuda"), torch.zeros(1, device="cuda")
        _lib.check(lib.pdf_bce_sigmoid_train(n, z[e].data_ptr(), y[e].data_ptr(), p.data_ptr(), l.data_ptr(), dz.data_ptr(), _s()), "s")
        assert torch.equal(p, pb[e]) and torch.equal(dz, dzb[e])
        assert abs(float(l) - float(lb[e])) <= 1e-6 * abs(float(l))
        o, lm, dz2, dr2 = torch.empty(n, device="cuda"), torch.zeros(1, device="cuda"), torch.empty(n, M, device="cuda"), torch.empty(n, M, device="cuda")
        _lib.check(lib.pdf_moe_combine_train(n, M, zm[e].data_ptr(), rm[e].data_ptr(), ym.data_ptr(), o.data_ptr(), lm.data_ptr(), dz2.data_ptr(),
                                             dr2.data_ptr(), _s()), "s")
        assert torch.equal(o, ob[e]) and torch.equal(dz2, dzm[e]) and torch.equal(dr2, drm[e])
        assert abs(float(lm) - float(lmb[e])) <= 1e-6 * abs(float(lm))


@pytest.mark.parametrize("gated", [True, False])
def test_mil_pool_batched_against_single(gated):
    lib, E, B, L, H, A = _lib_(), 3, 6, 9, 40, 12
    NA = 2 * A if gated else A
    g = torch.Generator(device="cuda").manual_seed(3)
    h = torch.relu(torch.randn(E, B * L, H, device="cuda", generator=g))
    vu = torch.randn(E, B * L, NA, device="cuda", generator=g)
    lens = torch.randint(0, L + 1, (E, B), device="cuda", generator=g, dtype=torch.int32)
    lens[:, 0] = 0
    lens[:, 1] = L
    y = (torch.rand(E, B, device="cuda", generator=g) < 0.5).float()
    P = 256                                      # member row: w_w [A] @0, b_w @64, w_cls [H] @128, b_cls @192
    W = torch.randn(E, P, device="cuda", generator=g)
    G = torch.randn(E, P, device="cuda", generator=g)  # gradients accumulate onto what is there
    Gs = G.clone()
    w = _lib.MilWeights()
    w.D, w.H, w.A, w.gated = 16, H, A, int(gated)
    t = _lib.MilTrain()
    t.loss_type, t.pos_weight, t.focal_gamma, t.focal_alpha = 0, 1.7, 2.0, -1.0

    def point(wb, gb, e):
        b = 4 * e * P
        w.w_w, w.b_w, w.w_cls, w.b_cls = (wb + b + 4 * o for o in (0, 64, 128, 192))
        t.d_w_w, t.d_b_w, t.d_w_cls, t.d_b_cls = (gb + b + 4 * o for o in (0, 64, 128, 192))
    point(W.data_ptr(), G.data_ptr(), 0)
    prob, loss, dh, dvu = torch.empty(E, B, device="cuda"), torch.empty(E, device="cuda"), torch.empty_like(h), torch.empty_like(vu)
    ws = torch.empty(int(lib.pdf_mil_pool_train_batched_workspace_bytes(E, C.byref(w), B)), dtype=torch.uint8, device="cuda")
    _lib.check(lib.pdf_mil_pool_train_batched(E, C.byref(w), P, C.byref(t), P, B, L, h.data_ptr(), vu.data_ptr(), lens.data_ptr(), y.data_ptr(),
                                              prob.data_ptr(), loss.data_ptr(), dh.data_ptr(), dvu.data_ptr(), ws.data_ptr(), _s()), "b")
    for e in range(E):
        point(W.data_ptr(), Gs.data_ptr(), e)
        p, l, d1, d2 = torch.empty(B, device="cuda"), torch.zeros(1, device="cuda"), torch.empty_like(h[e]), torch.empty_like(vu[e])
        _lib.check(lib.pdf_mil_pool_train(C.byref(w), C.byref(t), B, L, h[e].data_ptr(), vu[e].data_ptr(), lens[e].data_ptr(), y[e].data_ptr(),
                                          p.data_ptr(), l.data_ptr(), d1.data_ptr(), d2.data_ptr(), _s()), "s")
        assert torch.equal(p, prob[e]) and torch.equal(d1, dh[e]) and torch.equal(d2, dvu[e])
        assert abs(float(l) - float(loss[e])) <= 1e-6 * abs(float(l))
    for lo, hi in ((0, A), (64, 65), (128, 128 + H), (192, 193)):
        assert _rel(G[:, lo:hi], Gs[:, lo:hi]) <= 1e-6


def test_clip_and_adam_batched_against_single():
    lib, E, P = _lib_(), 3, 1000
    g = torch.Generator(device="cuda").manual_seed(4)
    p0, grad = torch.randn(E, P, device="cuda", generator=g), torch.randn(E, P, device="cuda", generator=g)
    grad[1] *= 1e-3                              # member 1 is not clipped
    scale = torch.empty(E, device="cuda")
    _lib.check(lib.pdf_clip_scale_batched(E, grad.data_ptr(), P, 5.0, scale.data_ptr(), _s()), "clip")
    pb, mb, vb = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    active = torch.tensor([1, 1, 0], dtype=torch.uint8, device="cuda")
    for step in (1, 2):
        _lib.check(lib.pdf_adam_step_batched(E, pb.data_ptr(), grad.data_ptr(), mb.data_ptr(), vb.data_ptr(), P, 1e-2, 0.9, 0.999, 1e-8, 0.01,
                                             step, scale.data_ptr(), active.data_ptr(), _s()), "adam")
    for e in range(E):
        acc, sc = torch.zeros(1, device="cuda"), torch.empty(2, device="cuda")
        _lib.check(lib.pdf_sumsq_f32(grad[e].data_ptr(), P, acc.data_ptr(), _s()), "s")
        _lib.check(lib.pdf_clip_scale(acc.data_ptr(), 5.0, sc.data_ptr(), _s()), "s")
        assert abs(float(sc[0]) - float(scale[e])) <= 1e-6 * float(sc[0])
        if e == 2:
            assert torch.equal(pb[e], p0[e]) and not mb[e].any()
            continue
        p, m, v = p0[e].clone(), torch.zeros(P, device="cuda"), torch.zeros(P, device="cuda")
        for step in (1, 2):
            _lib.check(lib.pdf_adam_step(p.data_ptr(), grad[e].data_ptr(), m.data_ptr(), v.data_ptr(), P, 1e-2, 0.9, 0.999, 1e-8, 0.01, step,
                                         scale[e:].data_ptr(), _s()), "s")
        assert torch.equal(p, pb[e]) and torch.equal(m, mb[e]) and torch.equal(v, vb[e])


# ------------------------------------------------------------------ members against the single-model sequence of their seeds

def _moddrop_data(n=300, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, sum(DIMS.values()))).astype(np.float32)
    y = (X[:, 0] + 0.5 * X[:, 8] - 0.3 * X[:, 14] + 0.5 * rng.standard_normal(n) > 0).astype(np.float32)
    return X, y


def _moddrop_args(epochs=2):
    return (DIMS, {"hidden_dims": [32, 16], "dropout": 0.2, "moddrop_rate": 0.3, "lr": 1e-3, "epochs": epochs, "batch_size": 32})


def _moe_data(n=400, seed=1):
    rng = np.random.default_rng(seed)
    dims = {"clinical": 6, "datspect": 4}
    X = {m: rng.standard_normal((n, d)).astype(np.float32) for m, d in dims.items()}
    mask = (rng.random((n, 2)) < 0.8).astype(np.float32)
    y = (X["clinical"][:, 0] + X["datspect"][:, 1] > 0).astype(np.float32)
    return dims, X, y, mask


def _moe_args(dims, epochs=15):
    return (dims, {"expert_hidden_dims": [16, 8], "router_hidden_dims": [8], "lr": 3e-3, "epochs": epochs})


def _mil_data(n, seed, D=16):
    rng = np.random.default_rng(seed)
    bags = [rng.standard_normal((int(rng.integers(2, 9)), D)).astype(np.float32) for _ in range(n)]
    y = np.array([float(b[:, 0].mean() > 0) for b in bags], dtype=np.float32)
    return bags, y


def _mil_args(patience=1, epochs=8):
    return (16, {"hidden_dim": 24, "attn_dim": 8, "gated": True, "dropout": 0.25, "max_grad_norm": 0.5, "class_weight": "balanced",
                 "lr": 3e-3, "epochs": epochs, "batch_size": 16, "early_stopping_patience": patience})


def _rng_state():
    return torch.get_rng_state(), torch.cuda.get_rng_state(), np.random.get_state()


def _assert_rng_same(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert a[2][0] == b[2][0] and np.array_equal(a[2][1], b[2][1]) and a[2][2:] == b[2][2:]


def _single(cls, args, seed, *train_args):
    torch.manual_seed(seed)
    np.random.seed(seed)
    m = cls(*args)
    m.train(*train_args)
    return m


def _check_members(ens, cls, args, train_args):
    torch.manual_seed(1234)
    np.random.seed(99)
    torch.cuda.manual_seed(77)
    before = _rng_state()
    ens.train(*train_args)
    torch.cuda.synchronize()
    _assert_rng_same(before, _rng_state())
    for e, s in enumerate(ens.seeds):
        ref = _single(cls, args, s, *train_args)
        mine = ens.members[e]
        for (k, v), (k2, v2) in zip(ref.model.state_dict().items(), mine.model.state_dict().items()):
            assert k == k2
            if k in SCORE_BIAS:
                continue
            assert _rel(v2.float(), v.float()) < 2e-4, (s, k)
        lr_ = torch.cat(ref.last_losses).cpu().numpy()
        lm = torch.cat(mine.last_losses).cpu().numpy()
        assert lr_.shape == lm.shape, (s, lr_.shape, lm.shape)
        np.testing.assert_allclose(lm, lr_, rtol=2e-5, atol=0)


def test_moddrop_members_equal_single_models():
    X, y = _moddrop_data()
    _check_members(HeadEnsemble(ModalityDropoutModel, _moddrop_args(), SEEDS), ModalityDropoutModel, _moddrop_args(), (X, y))


def test_moe_members_equal_single_models():
    dims, X, y, mask = _moe_data()
    _check_members(HeadEnsemble(MoEModel, _moe_args(dims), SEEDS), MoEModel, _moe_args(dims), (X, y, mask))


def test_mil_members_equal_single_models_with_early_stopping():
    bags, y = _mil_data(160, 5)
    vbags, _ = _mil_data(40, 6)
    vy = np.random.default_rng(7).integers(0, 2, 40).astype(np.float32)      # noisy validation labels: each member stops on its own
    for k in range(6):                           # the first seed set whose members stop at different epochs
        seeds = [s + 4 * k for s in SEEDS]
        ens = HeadEnsemble(MilAttentionModel, _mil_args(), seeds)
        ens.train(bags, y, (vbags, vy))
        if len(set(ens.stopped_epoch)) > 1:
            break
    assert len(set(ens.stopped_epoch)) > 1, ens.stopped_epoch
    _check_members(HeadEnsemble(MilAttentionModel, _mil_args(), seeds), MilAttentionModel, _mil_args(), (bags, y, (vbags, vy)))


# ------------------------------------------------------------------ independence, determinism, launches

def _weights(ens, e):
    return {k: v.detach().clone() for k, v in ens.members[e].model.state_dict().items()}


def test_members_do_not_depend_on_each_other_and_runs_repeat():
    X, y = _moddrop_data()
    bags, yb = _mil_data(64, 8)
    for cls, args, targs in ((ModalityDropoutModel, _moddrop_args(), (X, y)), (MilAttentionModel, _mil_args(0, 3), (bags, yb))):
        runs = []
        for seeds in ([5], [1, 5, 9], [9, 3, 7, 5], [1, 5, 9]):
            ens = HeadEnsemble(cls, args, seeds)
            ens.train(*targs)
            runs.append((seeds, ens))
        ref = _weights(runs[0][1], 0)
        for seeds, ens in runs[1:]:
            w = _weights(ens, seeds.index(5))
            assert all(torch.equal(ref[k], w[k]) for k in ref), (cls.__name__, seeds)
        for e in range(3):                        # two runs of the same ensemble
            a, b = _weights(runs[1][1], e), _weights(runs[3][1], e)
            assert all(torch.equal(a[k], b[k]) for k in a)


def test_launches_per_step_do_not_depend_on_members():
    X, y = _moddrop_data()
    dims, Xm, ym, mask = _moe_data()
    bags, yb = _mil_data(64, 8)
    cases = ((ModalityDropoutModel, _moddrop_args(1), (X, y)), (MoEModel, _moe_args(dims, 3), (Xm, ym, mask)),
             (MilAttentionModel, _mil_args(0, 2), (bags, yb)))
    for cls, args, targs in cases:
        per = []
        for E in (1, 8):
            ens = HeadEnsemble(cls, args, list(range(E)))
            n0 = _lib.launch_count()
            ens.train(*targs)
            per.append((_lib.launch_count() - n0) / len(ens.last_losses))
        assert per[0] == per[1], (cls.__name__, per)


# ------------------------------------------------------------------ inference and evaluation

def _trained_moddrop(seeds):
    X, y = _moddrop_data()
    ens = HeadEnsemble(ModalityDropoutModel, _moddrop_args(), seeds)
    ens.train(X, y)
    return ens


def test_sweep_mean_and_statistics():
    from pd_fusion_b200.data.schema import MODALITIES
    X, _ = _moddrop_data(500, 3)
    rng = np.random.default_rng(4)
    masks = (rng.random((5, 500, len(MODALITIES))) < 0.7).astype(np.uint8)
    ens = _trained_moddrop(SEEDS)
    dims, Xm, ym, mmask = _moe_data()
    moe = HeadEnsemble(MoEModel, _moe_args(dims, 3), SEEDS)
    moe.train(Xm, ym, mmask)
    bags, yb = _mil_data(64, 8)
    mil = HeadEnsemble(MilAttentionModel, _mil_args(0, 2), SEEDS)
    mil.train(bags, yb)
    bags_m = [None if i % 7 == 0 else b for i, b in enumerate(bags)]
    mri = (rng.random((3, 64)) < 0.7).astype(int)
    mods = sorted(dims)
    moe_masks = (rng.random((4, 400, 2)) < 0.7).astype(np.uint8)
    for e_, args in ((ens, (X, masks, list(MODALITIES))), (moe, (Xm, moe_masks, mods)), (mil, (bags_m, mri))):
        own = np.stack([m.predict_proba_sweep(*args) for m in e_.members])
        members, st = e_.predict_ensemble_sweep(*args)
        assert np.array_equal(members, own)
        mean = e_.predict_proba_sweep(*args)
        assert mean.dtype == np.float64
        assert np.abs(mean - own.astype(np.float64).mean(0)).max() <= 1e-12
        ref = ensemble_stats_np(np.asarray(members, dtype=np.float32))
        for s in range(len(st)):
            got = np.stack([st[s][k] for k in ("mean", "std", "entropy", "expected_entropy", "mutual_info")], -1)
            assert np.abs(got - ref[s]).max() <= 1e-12
    # one scenario through predict_proba equals the sweep's first scenario
    assert np.array_equal(ens.predict_proba(X), ens.predict_proba_sweep(X, np.ones((1, 500, 3), np.uint8), list(MODALITIES))[0])
    # E = 1 and identical members: exactly no spread
    one = _trained_moddrop([7])
    same = HeadEnsemble(ModalityDropoutModel, _moddrop_args(), [1, 2, 3])
    for m in same.members:
        m.model.load_state_dict(ens.members[0].model.state_dict())
        m.invalidate()
    for e_ in (one, same):
        _, st = e_.predict_ensemble_sweep(X, masks, list(MODALITIES))
        assert all(np.all(d["std"] == 0) and np.all(d["mutual_info"] == 0) for d in st)


def test_save_and_load(tmp_path):
    ens = _trained_moddrop(SEEDS[:2])
    ens.save(tmp_path / "ens.pt")
    back = HeadEnsemble.load(tmp_path / "ens.pt", ModalityDropoutModel, _moddrop_args())
    assert back.seeds == ens.seeds
    X, _ = _moddrop_data(50, 9)
    assert np.array_equal(back.predict_proba(X), ens.predict_proba(X))


def test_ensemble_model_against_evaluate_model(golden):
    import json
    from oracle import oracle as O
    from pd_fusion_b200.data.preprocess import NaNRobustScaler
    from pd_fusion_b200.evaluation.evaluate import ensemble_model, evaluate_model
    from pd_fusion_b200.synthetic import synthetic_table
    g = golden("heads")
    dims = json.loads(str(g["table/dims"]))
    df, masks = synthetic_table(int(g["table/n"]), dims, seed=42, mask_seed=7)
    cfg = json.loads(str(g["scenarios"]))
    cols = [c for m in O.MODALITIES for c in df.columns if c.startswith(m + "_")]
    prep = (None, NaNRobustScaler().fit(df[cols].values), cols)
    from pd_fusion_b200.data.preprocess import preprocess_features
    from pd_fusion_b200.data.schema import TARGET_COL
    Xtr = preprocess_features(df, cols, None, prep[1])[0]
    ens = HeadEnsemble(ModalityDropoutModel, (dims, {"hidden_dims": [32, 16], "dropout": 0.2, "lr": 1e-3, "epochs": 2}), [3, 4, 5])
    ens.train(Xtr, df[TARGET_COL].values.astype(np.float32))
    rng = np.random.default_rng(5)
    n, D = 200, 16
    bags = [None if i % 5 == 0 else rng.standard_normal((int(rng.integers(1, 6)), D)).astype(np.float32) for i in range(n)]
    dfm = pd.DataFrame({"diagnosis": rng.integers(0, 2, n), "mri_mil": bags, "subject": rng.integers(0, 80, n)})
    mmask = {"clinical": np.ones(n, int), "datspect": np.ones(n, int), "mri": (rng.random(n) < 0.8).astype(int)}
    mcfg = {"scenarios": [{"name": "baseline", "drop_modalities": []}, {"name": "half", "drop_modalities": ["mri"], "drop_rate": 0.5}],
            "group_col": "subject"}
    mil = HeadEnsemble(MilAttentionModel, (D, {"hidden_dim": 8, "attn_dim": 4, "gated": True, "missing_prob": 0.3, "epochs": 2}), [1, 2])
    mil.train([b for b in bags if b is not None], dfm["diagnosis"].values[[b is not None for b in bags]].astype(np.float32))
    for e_, d, mk, pr, c in ((ens, df, masks, prep, cfg), (mil, dfm, mmask, ("mil", "mri_mil"), mcfg)):
        np.random.seed(17)
        ev = evaluate_model(e_, d, mk, pr, c)
        after_eval = np.random.get_state()
        np.random.seed(17)
        res = ensemble_model(e_, d, mk, pr, c)
        after = np.random.get_state()
        assert after_eval[0] == after[0] and np.array_equal(after_eval[1], after[1]) and after_eval[2:] == after[2:]
        per_member = []
        for m in e_.members:
            np.random.seed(17)
            per_member.append(evaluate_model(m, d, mk, pr, c))
        y = d[TARGET_COL].values
        for sc in c["scenarios"]:
            r = res[sc["name"]]
            assert r["metrics"] == ev[sc["name"]] or all(
                (np.isnan(r["metrics"][k]) and np.isnan(v)) or r["metrics"][k] == v for k, v in ev[sc["name"]].items())
            for e in range(len(e_)):
                assert r["members"][e].keys() == per_member[e][sc["name"]].keys()
                for k, v in per_member[e][sc["name"]].items():
                    assert (np.isnan(v) and np.isnan(r["members"][e][k])) or r["members"][e][k] == v, (e, k)
            for k in r["member_mean"]:
                vals = [m[k] for m in r["members"]]
                assert r["member_mean"][k] == pytest.approx(float(np.mean(vals)), nan_ok=True)
            assert all(r[k].shape == (len(d),) and r[k].dtype == np.float64 for k in ("mean", "std", "entropy", "expected_entropy", "mutual_info"))
            order = np.argsort(r["entropy"], kind="stable")
            err = ((r["mean"] >= 0.5).astype(int) != y.astype(int))[order]
            assert np.allclose(r["risk_coverage"]["risk"], np.cumsum(err) / np.arange(1, len(y) + 1), rtol=0, atol=1e-15)
    with pytest.raises(ValueError, match="HeadEnsemble"):
        ensemble_model(ens.members[0], df, masks, prep, cfg)

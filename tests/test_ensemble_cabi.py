"""The deep-ensemble entry points (csrc/train.cu) and models.ensemble.HeadEnsemble without a GPU: prototypes agree with the header,
every bad argument is refused with PDF_ERR_ARG before any device work, the members' private random streams reproduce the seed
contract's global-RNG draws, the class and seed checks, and the ensemble statistics restated in numpy."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from pd_fusion_b200 import _lib
from pd_fusion_b200.models.ensemble import HeadEnsemble
from pd_fusion_b200.models.fusion_moddrop import ModalityDropoutModel
from pd_fusion_b200.models.mil_attention import MilAttentionModel
from pd_fusion_b200.models.moe import MoEModel

ROOT = Path(__file__).resolve().parents[1]
HEADER = (ROOT / "include" / "pdfusion_b200.h").read_text()
NAMES = ("pdf_gemm_f32_batched", "pdf_bce_sigmoid_train_batched", "pdf_moe_combine_train_batched",
         "pdf_mil_pool_train_batched_workspace_bytes", "pdf_mil_pool_train_batched", "pdf_clip_scale_batched", "pdf_adam_step_batched",
         "pdf_ensemble_stats")
FAKE = 1 << 12              # an aligned non-null address: never dereferenced, every call below fails its checks first
ERR_ARG = -1
DIMS = {"clinical": 5, "datspect": 3, "mri": 4}
STATS = ("mean", "std", "entropy", "expected_entropy", "mutual_info")


def _declaration(name):
    m = re.search(r"\b(int|size_t)\s+" + name + r"\s*\(([^;]*)\)\s*;", HEADER)
    assert m, f"{name} not declared in the header"
    args = re.sub(r"/\*.*?\*/", "", m.group(2), flags=re.S)
    return m.group(1), [a.strip() for a in args.split(",")]


def test_prototypes_match_header():
    scalar = {"int": C.c_int, "float": C.c_float, "long": C.c_long, "long long": C.c_longlong}
    for name in NAMES:
        ret, args = _declaration(name)
        restype, argtypes = _lib.PROTOTYPES[name]
        assert restype is {"int": C.c_int, "size_t": C.c_size_t}[ret], name
        assert len(argtypes) == len(args), name
        for decl, t in zip(args, argtypes):
            if "*" in decl or decl.startswith("pdf_stream_t"):
                assert t is _lib._P or issubclass(t, C._Pointer), (name, decl)
            else:
                assert t is scalar[" ".join(decl.split()[:-1])], (name, decl)
    lib = _lib.load()
    for name in NAMES:
        assert hasattr(lib, name)


def _gemm(**kw):
    a = dict(E=2, M=4, N=4, K=4, A=FAKE, a_rs=4, a_cs=1, a_es=16, B=FAKE, b_rs=4, b_cs=1, b_es=16, Cm=FAKE, c_rs=4, c_es=16, bias=None,
             bias_es=0, act=0, acc=0)
    a.update(kw)
    return _lib.load().pdf_gemm_f32_batched(a["E"], a["M"], a["N"], a["K"], a["A"], a["a_rs"], a["a_cs"], a["a_es"], a["B"], a["b_rs"],
                                            a["b_cs"], a["b_es"], a["Cm"], a["c_rs"], a["c_es"], a["bias"], a["bias_es"], a["act"], a["acc"],
                                            None)


@pytest.mark.parametrize("kw", [dict(E=0), dict(E=1025), dict(M=0), dict(N=0), dict(K=0), dict(A=None), dict(B=None), dict(Cm=None),
                                dict(A=FAKE + 2), dict(B=FAKE + 1), dict(Cm=FAKE + 2), dict(bias=FAKE + 2), dict(a_es=-1), dict(b_es=-1),
                                dict(c_es=-16), dict(bias=FAKE, bias_es=-1), dict(c_es=0)])
def test_gemm_refusals(kw):
    assert _gemm(**kw) == ERR_ARG


def _mil(H=8, A=4, w_ptr=FAKE):
    w = _lib.MilWeights()
    w.D, w.H, w.A, w.gated = 16, H, A, 1
    w.w_w = w.b_w = w.w_cls = w.b_cls = w_ptr
    t = _lib.MilTrain()
    t.loss_type, t.pos_weight, t.focal_gamma, t.focal_alpha = 0, 1.0, 2.0, -1.0
    t.d_w_w = t.d_b_w = t.d_w_cls = t.d_b_cls = FAKE
    return w, t


def test_loss_and_optimizer_refusals():
    lib = _lib.load()
    for E, n, z, y, y_es in ((0, 4, FAKE, FAKE, 4), (1025, 4, FAKE, FAKE, 4), (2, 0, FAKE, FAKE, 4), (2, 4, None, FAKE, 4),
                             (2, 4, FAKE + 2, FAKE, 4), (2, 4, FAKE, FAKE, -1)):
        assert lib.pdf_bce_sigmoid_train_batched(E, n, z, y, y_es, FAKE, FAKE, FAKE, None) == ERR_ARG
    for E, n, M, z in ((0, 4, 2, FAKE), (2, 0, 2, FAKE), (2, 4, 0, FAKE), (2, 4, 9, FAKE), (2, 4, 2, None), (2, 4, 2, FAKE + 1)):
        assert lib.pdf_moe_combine_train_batched(E, n, M, z, FAKE, FAKE, 0, FAKE, FAKE, FAKE, FAKE, None) == ERR_ARG
    w, t = _mil()
    assert lib.pdf_mil_pool_train_batched_workspace_bytes(3, C.byref(w), 5) == 3 * 5 * (8 + 4 + 3) * 4
    assert lib.pdf_mil_pool_train_batched_workspace_bytes(0, C.byref(w), 5) == 0
    assert lib.pdf_mil_pool_train_batched_workspace_bytes(3, C.byref(w), 0) == 0
    good = dict(E=2, w_es=64, g_es=64, B=4, L=3, ptrs=[FAKE] * 9)

    def mil(**kw):
        a = dict(good, **kw)
        ww, tt = kw.get("wt", (w, t))
        return lib.pdf_mil_pool_train_batched(a["E"], C.byref(ww), a["w_es"], C.byref(tt), a["g_es"], a["B"], a["L"], *a["ptrs"], None)
    assert mil(E=0) == ERR_ARG and mil(E=1025) == ERR_ARG and mil(B=0) == ERR_ARG and mil(L=0) == ERR_ARG
    assert mil(w_es=-1) == ERR_ARG and mil(g_es=-1) == ERR_ARG and mil(L=60000) == ERR_ARG       # the bag exceeds shared memory
    for i in range(9):
        for bad in (None, FAKE + 2):
            ptrs = [FAKE] * 9
            ptrs[i] = bad
            assert mil(ptrs=ptrs) == ERR_ARG, (i, bad)
    assert mil(wt=_mil(w_ptr=None)) == ERR_ARG and mil(wt=_mil(H=0)) == ERR_ARG
    for E, P, g, s in ((0, 8, FAKE, FAKE), (2, 0, FAKE, FAKE), (2, 8, None, FAKE), (2, 8, FAKE, FAKE + 2)):
        assert lib.pdf_clip_scale_batched(E, g, P, 1.0, s, None) == ERR_ARG
    for E, P, step, p, sc in ((0, 8, 1, FAKE, None), (1025, 8, 1, FAKE, None), (2, 0, 1, FAKE, None), (2, 8, 0, FAKE, None),
                              (2, 8, 1, None, None), (2, 8, 1, FAKE + 2, None), (2, 8, 1, FAKE, FAKE + 2)):
        assert lib.pdf_adam_step_batched(E, p, FAKE, FAKE, FAKE, P, 1e-3, 0.9, 0.999, 1e-8, 0.0, step, sc, None, None) == ERR_ARG
    for E, pairs, pr, st in ((0, 4, FAKE, FAKE), (1025, 4, FAKE, FAKE), (2, 0, FAKE, FAKE), (2, 4, None, FAKE), (2, 4, FAKE, FAKE + 4)):
        assert lib.pdf_ensemble_stats(E, pairs, pr, st, None) == ERR_ARG


def _md_args(dropout=0.2):
    return (DIMS, {"hidden_dims": [16, 8], "dropout": dropout, "lr": 1e-3, "epochs": 2, "batch_size": 8, "moddrop_rate": 0.3})


def _rng_states():
    return torch.get_rng_state(), np.random.get_state()


def _same_rng(a, b):
    return torch.equal(a[0], b[0]) and a[1][0] == b[1][0] and np.array_equal(a[1][1], b[1][1]) and a[1][2:] == b[1][2:]


def test_member_streams_reproduce_the_global_draws():
    """member e's CPU generator continues exactly where torch's global RNG stands after the seed contract's constructor, and its
    RandomState draws what np.random draws after np.random.seed(s_e)"""
    seeds, n = [3, 11, 7], 50
    np.random.seed(1)
    torch.manual_seed(2)
    before = _rng_states()
    ens = HeadEnsemble(ModalityDropoutModel, _md_args(), seeds)
    assert _same_rng(before, _rng_states())                       # building the ensemble leaves the global RNGs alone
    for e, s in enumerate(seeds):
        torch.manual_seed(s)
        np.random.seed(s)
        ref = ModalityDropoutModel(*_md_args())
        for (k, v), (k2, v2) in zip(ref.model.state_dict().items(), ens.members[e].model.state_dict().items()):
            assert k == k2 and torch.equal(v, v2)
        for _ in range(3):                                        # every epoch's permutation
            assert torch.equal(torch.randperm(n), torch.randperm(n, generator=ens._cpu_gens[e]))
        assert np.array_equal(np.array([np.random.rand() for _ in range(12)]), ens._np_rngs[e].rand(12))


def test_member_classes_and_seeds():
    with pytest.raises(ValueError, match="supports"):
        HeadEnsemble(dict, (), [1, 2])

    class Sub(ModalityDropoutModel):
        pass
    with pytest.raises(ValueError, match="supports"):
        HeadEnsemble(Sub, _md_args(), [1, 2])
    with pytest.raises(ValueError, match="distinct"):
        HeadEnsemble(ModalityDropoutModel, _md_args(), [1, 2, 1])
    with pytest.raises(ValueError, match="1..1024"):
        HeadEnsemble(ModalityDropoutModel, _md_args(), [])
    ens = HeadEnsemble(MoEModel, (DIMS, {"expert_hidden_dims": [8], "router_hidden_dims": [4], "lr": 1e-3, "epochs": 1}), [5, 6])
    assert len(ens) == 2 and all(isinstance(m, MoEModel) for m in ens.members)
    assert not hasattr(ens, "mask_dim") and not hasattr(ens, "predict_uncertainty_sweep")
    mil = HeadEnsemble(MilAttentionModel, (16, {"hidden_dim": 8, "attn_dim": 4, "gated": True}), [0, 1])
    assert all(isinstance(m, MilAttentionModel) for m in mil.members)


def _entropy(q):
    with np.errstate(divide="ignore", invalid="ignore"):
        return -(np.where(q > 0, q * np.log(q), 0.0)) - np.where(q < 1, (1 - q) * np.log(1 - q), 0.0)


def ensemble_stats_np(probs):
    """pdf_ensemble_stats restated: probs [E, ...] float32 -> [..., 5] float64, ascending e, sums of differences to member 0"""
    p = probs.astype(np.float64)
    E = p.shape[0]
    p0, h0 = p[0], _entropy(p[0])
    sd, sh = np.zeros_like(p0), np.zeros_like(p0)
    for e in range(E):
        sd = sd + (p[e] - p0)
        sh = sh + (_entropy(p[e]) - h0)
    mean = p0 + sd / E
    v = np.zeros_like(p0)
    for e in range(E):
        v = v + (p[e] - mean) ** 2
    ent, eent = _entropy(mean), h0 + sh / E
    return np.stack([mean, np.sqrt(v / E), ent, eent, np.maximum(0.0, ent - eent)], axis=-1)


def test_statistics_of_equal_members_are_exact():
    rng = np.random.default_rng(0)
    p = rng.random((3, 100)).astype(np.float32)
    p[:, :3] = [0.0, 1.0, 0.5]
    for E in (1, 2, 7):
        st = ensemble_stats_np(np.repeat(p[:1], E, axis=0))
        assert np.all(st[..., 1] == 0) and np.all(st[..., 4] == 0)
        assert np.array_equal(st[..., 0], p[0].astype(np.float64))
    st = ensemble_stats_np(p)
    assert np.allclose(st[..., 0], p.astype(np.float64).mean(0), rtol=0, atol=1e-15)
    assert np.allclose(st[..., 1], p.astype(np.float64).std(0), rtol=0, atol=1e-15)
    assert np.all(st[..., 4] >= 0)

"""The fusion-head explanation entry points (pdf_moddrop_explain, pdf_moe_explain) without a GPU: prototypes agree with the header,
the workspace formulas, and bad arguments refused with PDF_ERR_ARG before any device work."""
import ctypes as C
import re
from pathlib import Path

from pd_fusion_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
HEADER = (ROOT / "include" / "pdfusion_b200.h").read_text()
NAMES = ("pdf_moddrop_explain_workspace_bytes", "pdf_moddrop_explain", "pdf_moe_explain_workspace_bytes", "pdf_moe_explain")
CTYPE = {"int": C.c_int, "size_t": C.c_size_t}
FAKE = 1 << 12              # a 16-byte aligned non-null address: never dereferenced, every call below fails its checks first


def _declaration(name):
    m = re.search(r"\b(int|size_t)\s+" + name + r"\s*\(([^;]*)\)\s*;", HEADER)
    assert m, f"{name} not declared in the header"
    args = re.sub(r"/\*.*?\*/", "", m.group(2), flags=re.S)
    return m.group(1), [a.strip() for a in args.split(",")]


def test_prototypes_match_header():
    for name in NAMES:
        ret, args = _declaration(name)
        restype, argtypes = _lib.PROTOTYPES[name]
        assert restype is CTYPE[ret], name
        assert len(argtypes) == len(args), name
        for decl, t in zip(args, argtypes):
            if "*" in decl:
                assert t is _lib._P or issubclass(t, C._Pointer), (name, decl)
            elif decl.startswith("pdf_stream_t"):
                assert t is _lib._P, (name, decl)
            else:
                assert t is C.c_int, (name, decl)
    lib = _lib.load()
    for name in NAMES:
        assert hasattr(lib, name)


def _mlp(dims, mod_widths=None):
    """pdf_mlp with fake weight pointers; dims = [F, hidden..., 1]"""
    m = _lib.Mlp()
    m.n_layers = len(dims) - 1
    for i, d in enumerate(dims):
        m.dims[i] = d
    for i in range(m.n_layers):
        m.w[i], m.b[i] = FAKE, FAKE
    widths = (mod_widths if mod_widths is not None else [dims[0]])[:_lib.PDF_MAX_MODS]
    m.n_mods = len(widths) if mod_widths is None else len(mod_widths)
    off = 0
    for i, w in enumerate(widths):
        m.mod_off[i] = off
        off += w
    m.mod_off[len(widths)] = off
    return m


def _moe(expert_dims, router_hidden=16):
    net = _lib.Moe()
    net.n_experts = len(expert_dims)
    for e, dims in enumerate(expert_dims[:_lib.PDF_MAX_MODS]):
        net.expert[e] = _mlp(dims)
    net.router_hidden = router_hidden
    net.w_r0 = net.b_r0 = net.w_r1 = net.b_r1 = FAKE
    return net


def _align(n):
    return (n + 63) // 64 * 64


def test_workspace_bytes():
    lib = _lib.load()
    net = _mlp([35, 64, 32, 1], [10, 5, 20])
    N, S = 10, 7
    base = _align(3 * N * 64) + _align(8 * N)                     # partials [M, N, h1] | coalition values [2^M, N]
    assert lib.pdf_moddrop_explain_workspace_bytes(C.byref(net), N, S, 0) == base * 4 + 256
    assert lib.pdf_moddrop_explain_workspace_bytes(C.byref(net), N, S, 32) == (base + _align(S * N * 64)) * 4 + 256   # + mean delta1
    one = _mlp([35, 1], [10, 5, 20])                              # one layer: no delta1, the gradient is w1
    assert lib.pdf_moddrop_explain_workspace_bytes(C.byref(one), N, S, 32) == (_align(3 * N * 1) + _align(8 * N)) * 4 + 256
    for args in ((None, N, S, 0), (C.byref(net), 0, S, 0), (C.byref(net), N, 0, 0), (C.byref(net), N, S, -1)):
        assert lib.pdf_moddrop_explain_workspace_bytes(*args) == 0
    moe = _moe([[10, 32, 16, 1], [512, 32, 16, 1]])
    base = _align(4 * N) + _align(4 * 2)                          # coalition values [2^E, N] | router weights [2^E, E]
    assert lib.pdf_moe_explain_workspace_bytes(C.byref(moe), N, S, 0) == base * 4 + 256
    # + expert partials and mean delta1 [N, max h1], average input gradient [N, max d]
    assert lib.pdf_moe_explain_workspace_bytes(C.byref(moe), N, S, 8) == (base + 2 * _align(N * 32) + _align(N * 512)) * 4 + 256
    assert lib.pdf_moe_explain_workspace_bytes(None, N, S, 0) == 0
    assert lib.pdf_moe_explain_workspace_bytes(C.byref(_moe([[4, 1]] * 9)), N, S, 0) == 0


def test_moddrop_explain_argument_validation_without_gpu():
    lib = _lib.load()
    good = _mlp([35, 64, 32, 1], [10, 5, 20])

    def call(net=good, n=4, s=2, x=FAKE, masks=FAKE, steps=8, ws=FAKE, value=FAKE, base=FAKE, shap=FAKE, ig=FAKE):
        return lib.pdf_moddrop_explain(C.byref(net) if net is not None else None, n, s, x, masks, steps, ws, value, base, shap, ig, None)

    for kw in (dict(net=None), dict(n=0), dict(s=0), dict(n=-1), dict(x=None), dict(masks=None), dict(ws=None), dict(value=None),
               dict(base=None), dict(shap=None)):
        assert call(**kw) == -1, kw
        assert b"bad arguments" in lib.pdf_last_error(), kw
    assert call(steps=257) == -1 and b"steps must be 0..256" in lib.pdf_last_error()
    assert call(steps=-1) == -1 and b"steps must be 0..256" in lib.pdf_last_error()
    assert call(steps=0) == -1 and b"steps >= 1" in lib.pdf_last_error()            # IG requested without steps
    assert call(net=_mlp([9, 8, 1], [1] * 9)) == -1 and b"modalities" in lib.pdf_last_error()
    assert call(net=_mlp([35, 64, 1], [10, 5, 19])) == -1 and b"tile [0, F)" in lib.pdf_last_error()
    assert call(net=_mlp([35, 64, 1], [10, 30, -5])) == -1 and b"tile [0, F)" in lib.pdf_last_error()
    assert call(net=_mlp([35, 64, 2], [35])) == -1 and b"one output" in lib.pdf_last_error()
    wide = _mlp([35, 1024, 1024, 1024, 1024, 1], [10, 5, 20])     # 4 x 1025 activations per row: 16 rows need > 227 KB
    assert call(net=wide) == -1 and b"too wide" in lib.pdf_last_error()


def test_moe_explain_argument_validation_without_gpu():
    lib = _lib.load()
    good = _moe([[10, 32, 16, 1], [512, 32, 16, 1]])
    xs = (C.c_void_p * 9)(*([FAKE] * 9))
    igs = (C.c_void_p * 9)(*([FAKE] * 9))

    def call(net=good, n=4, s=2, x=xs, masks=FAKE, steps=8, ws=FAKE, value=FAKE, base=FAKE, shap=FAKE, ig=igs):
        return lib.pdf_moe_explain(C.byref(net) if net is not None else None, n, s, x, masks, steps, ws, value, base, shap, ig, None)

    for kw in (dict(net=None), dict(n=0), dict(s=0), dict(x=None), dict(masks=None), dict(ws=None), dict(value=None), dict(base=None),
               dict(shap=None)):
        assert call(**kw) == -1, kw
        assert b"bad arguments" in lib.pdf_last_error(), kw
    assert call(steps=257) == -1 and b"steps must be 0..256" in lib.pdf_last_error()
    assert call(steps=0) == -1 and b"steps >= 1" in lib.pdf_last_error()
    assert call(net=_moe([[4, 8, 1]] * 9)) == -1 and b"experts" in lib.pdf_last_error()
    bad_ig = (C.c_void_p * 2)(FAKE, None)
    assert call(ig=bad_ig) == -1 and b"d_ig[1]" in lib.pdf_last_error()
    bad_x = (C.c_void_p * 2)(FAKE, None)
    assert call(x=bad_x) == -1
    assert call(net=_moe([[10, 32, 16, 1], [512, 1024, 1024, 1024, 1024, 1]])) == -1 and b"too wide" in lib.pdf_last_error()
    router = _moe([[10, 32, 1], [12, 8, 1]], router_hidden=0)
    assert call(net=router) == -1 and b"router" in lib.pdf_last_error()

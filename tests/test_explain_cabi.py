"""The explanation entry points (pdf_mil_explain, pdf_gradcam) without a GPU: prototypes agree with the header, and bad
arguments are refused with PDF_ERR_ARG before any device work."""
import ctypes as C
import re
from pathlib import Path

from pd_fusion_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
HEADER = (ROOT / "include" / "pdfusion_b200.h").read_text()
NAMES = ("pdf_mil_explain_workspace_bytes", "pdf_mil_explain", "pdf_gradcam")
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


def _weights(D=64, H=32, A=16, gated=1):
    w = _lib.MilWeights()
    w.D, w.H, w.A, w.gated = D, H, A, gated
    for f in ("w_inst", "b_inst", "w_v", "b_v", "w_u", "b_u", "w_w", "b_w", "w_cls", "b_cls"):
        setattr(w, f, FAKE)
    return w


def test_mil_explain_argument_validation_without_gpu():
    lib = _lib.load()
    w = _weights()
    assert lib.pdf_mil_explain_workspace_bytes(None, 2, 4) == 0
    assert lib.pdf_mil_explain_workspace_bytes(C.byref(w), 0, 4) == 0
    assert lib.pdf_mil_explain_workspace_bytes(C.byref(w), 2, 0) == 0
    # h, vu, dh, dvu for 8 rows (H = 32, NA = 32), each region padded to 64 floats, + 512
    assert lib.pdf_mil_explain_workspace_bytes(C.byref(w), 2, 4) == 4 * 4 * 256 + 512

    def call(w=w, n=2, L=4, bags=FAKE, lens=FAKE, ws=FAKE, logit=FAKE, attn=FAKE, contrib=FAKE, dx=None):
        return lib.pdf_mil_explain(C.byref(w) if w is not None else None, n, L, bags, lens, ws, logit, attn, contrib, dx, None)

    for kw in (dict(w=None), dict(n=0), dict(L=0), dict(n=-3), dict(bags=None), dict(lens=None), dict(ws=None), dict(logit=None),
               dict(attn=None), dict(contrib=None)):
        assert call(**kw) == -1, kw
    assert call(w=_weights(H=4096)) == -1 and b"dims" in lib.pdf_last_error()
    for bad in (_weights(D=0), _weights(A=0), _weights(H=0)):
        assert call(w=bad) == -1
    nw = _weights()
    nw.w_u = None
    assert call(w=nw) == -1 and b"null weight" in lib.pdf_last_error()
    nw.gated = 0                                     # the plain head needs no w_u
    nw.w_cls = None
    assert call(w=nw) == -1
    assert call(L=60000) == -1 and b"shared memory" in lib.pdf_last_error()
    assert call(n=1 << 20, L=1 << 12) == -1


def test_gradcam_argument_validation_without_gpu():
    lib = _lib.load()

    def call(n=2, hw=7, c=512, fmap=FAKE, g=FAKE, oh=32, ow=32, small=None, cam=FAKE):
        return lib.pdf_gradcam(n, hw, c, fmap, g, oh, ow, small, cam, None)

    for kw in (dict(n=0), dict(hw=0), dict(c=0), dict(oh=0), dict(ow=-1), dict(fmap=None), dict(g=None), dict(cam=None)):
        assert call(**kw) == -1, kw
    assert call(c=514) == -1 and b"c % 4" in lib.pdf_last_error()
    assert call(fmap=FAKE + 4) == -1                 # float4 loads need a 16-byte aligned feature map
    assert call(hw=65) == -1
    assert call(oh=1 << 15) == -1
    assert call(c=1 << 16) == -1 and b"shared memory" in lib.pdf_last_error()

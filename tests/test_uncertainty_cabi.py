"""The Monte-Carlo dropout entry points (pdf_moddrop_mc, pdf_mil_mc) without a GPU: prototypes agree with the header, the workspace
formulas, every bad argument refused with PDF_ERR_ARG before any device work, and the restated mask rule of tests/mc_oracle.py."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

import bootstrap_oracle as B
import mc_oracle as O
from pd_fusion_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
HEADER = (ROOT / "include" / "pdfusion_b200.h").read_text()
NAMES = ("pdf_moddrop_mc_workspace_bytes", "pdf_moddrop_mc", "pdf_mil_mc_workspace_bytes", "pdf_mil_mc")
FAKE = 1 << 12              # a 256-byte aligned non-null address: never dereferenced, every call below fails its checks first


def _declaration(name):
    m = re.search(r"\b(int|size_t)\s+" + name + r"\s*\(([^;]*)\)\s*;", HEADER)
    assert m, f"{name} not declared in the header"
    args = re.sub(r"/\*.*?\*/", "", m.group(2), flags=re.S)
    return m.group(1), [a.strip() for a in args.split(",")]


def test_prototypes_match_header():
    scalar = {"int": C.c_int, "float": C.c_float, "uint64_t": C.c_uint64}
    for name in NAMES:
        ret, args = _declaration(name)
        restype, argtypes = _lib.PROTOTYPES[name]
        assert restype is {"int": C.c_int, "size_t": C.c_size_t}[ret], name
        assert len(argtypes) == len(args), name
        for decl, t in zip(args, argtypes):
            if "*" in decl:
                assert t is _lib._P or issubclass(t, C._Pointer), (name, decl)
            elif decl.startswith("pdf_stream_t"):
                assert t is _lib._P, (name, decl)
            else:
                assert t is scalar[decl.split()[0]], (name, decl)
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
    widths = mod_widths if mod_widths is not None else [dims[0]]
    m.n_mods = len(widths)
    off = 0
    for i, w in enumerate(widths[:_lib.PDF_MAX_MODS]):
        m.mod_off[i] = off
        off += w
    m.mod_off[min(len(widths), _lib.PDF_MAX_MODS)] = off
    return m


def _mil(D=64, H=32, A=16, gated=True):
    w = _lib.MilWeights()
    w.D, w.H, w.A, w.gated = D, H, A, int(gated)
    for f in ("w_inst", "b_inst", "w_v", "b_v", "w_u", "b_u", "w_w", "b_w", "w_cls", "b_cls"):
        setattr(w, f, FAKE)
    w.missing_prob = 0.5
    return w


def _align(n):
    return (n + 63) // 64 * 64


def test_workspace_bytes():
    lib = _lib.load()
    net = _mlp([35, 64, 32, 1], [10, 5, 20])
    N, S, T = 10, 7, 32
    # per-modality partials [M, N, h1] | sample probabilities [S, N, T]
    assert lib.pdf_moddrop_mc_workspace_bytes(C.byref(net), N, S, T) == (_align(3 * N * 64) + _align(S * N * T)) * 4 + 256
    for args in ((None, N, S, T), (C.byref(net), 0, S, T), (C.byref(net), N, 0, T), (C.byref(net), N, S, 0), (C.byref(net), N, S, 4097)):
        assert lib.pdf_moddrop_mc_workspace_bytes(*args) == 0
    w = _mil()
    # h [n*Lmax, H] | scores [n*Lmax] | bag sample probabilities [n, T]
    assert lib.pdf_mil_mc_workspace_bytes(C.byref(w), N, 48, T) == (_align(N * 48 * 32) + _align(N * 48) + _align(N * T)) * 4 + 256
    for args in ((None, N, 48, T), (C.byref(w), 0, 48, T), (C.byref(w), N, 0, T), (C.byref(w), N, 48, 0), (C.byref(w), N, 48, 5000)):
        assert lib.pdf_mil_mc_workspace_bytes(*args) == 0


def test_moddrop_mc_argument_validation_without_gpu():
    lib = _lib.load()
    good = _mlp([35, 64, 32, 1], [10, 5, 20])

    def call(net=good, p=0.2, n=4, s=2, x=FAKE, masks=FAKE, T=8, seed=1, ws=FAKE, stats=FAKE, samples=FAKE):
        return lib.pdf_moddrop_mc(C.byref(net) if net is not None else None, p, n, s, x, masks, T, seed, ws, stats, samples, None)

    for kw in (dict(net=None), dict(n=0), dict(s=0), dict(n=-1), dict(x=None), dict(masks=None), dict(ws=None), dict(stats=None)):
        assert call(**kw) == -1, kw
        assert b"bad arguments" in lib.pdf_last_error(), kw
    for p in (-0.1, 1.0, 1.5, float("nan")):
        assert call(p=p) == -1 and b"p_drop" in lib.pdf_last_error(), p
    for T in (0, -1, 4097):
        assert call(T=T) == -1 and b"n_samples must be 1..4096" in lib.pdf_last_error(), T
    for kw in (dict(x=FAKE + 2), dict(stats=FAKE + 4), dict(ws=FAKE + 64), dict(samples=FAKE + 1)):
        assert call(**kw) == -1 and b"misaligned" in lib.pdf_last_error(), kw
    assert call(net=_mlp([9, 8, 1], [1] * 9)) == -1
    assert call(net=_mlp([35, 64, 1], [10, 5, 19])) == -1 and b"tile [0, F)" in lib.pdf_last_error()
    assert call(net=_mlp([35, 64, 1], [10, 30, -5])) == -1 and b"tile [0, F)" in lib.pdf_last_error()
    assert call(net=_mlp([35, 64, 2], [35])) == -1 and b"one output" in lib.pdf_last_error()
    wide = _mlp([35, 1024, 1024, 1024, 1024, 1], [10, 5, 20])     # 4 x 1025 activations per row: 16 rows need > 227 KB
    assert call(net=wide) == -1 and b"too wide" in lib.pdf_last_error()


def test_mil_mc_argument_validation_without_gpu():
    lib = _lib.load()
    good = _mil()

    def call(w=good, p=0.3, n=4, lmax=48, bags=FAKE, lens=FAKE, s=2, live=FAKE, T=8, seed=1, ws=FAKE, stats=FAKE, samples=FAKE):
        return lib.pdf_mil_mc(C.byref(w) if w is not None else None, p, n, lmax, bags, lens, s, live, T, seed, ws, stats, samples, None)

    for kw in (dict(w=None), dict(n=0), dict(lmax=0), dict(s=0), dict(bags=None), dict(lens=None), dict(ws=None), dict(stats=None)):
        assert call(**kw) == -1, kw
        assert b"bad arguments" in lib.pdf_last_error(), kw
    for p in (-1e-3, 1.0, float("inf"), float("nan")):
        assert call(p=p) == -1 and b"p_drop" in lib.pdf_last_error(), p
    for T in (0, 4097):
        assert call(T=T) == -1 and b"n_samples must be 1..4096" in lib.pdf_last_error(), T
    for kw in (dict(bags=FAKE + 2), dict(lens=FAKE + 1), dict(stats=FAKE + 4), dict(ws=FAKE + 16), dict(samples=FAKE + 2)):
        assert call(**kw) == -1 and b"misaligned" in lib.pdf_last_error(), kw
    assert call(lmax=65537) == -1 and b"Lmax" in lib.pdf_last_error()
    assert call(w=_mil(H=4096)) == -1 and b"bad dims" in lib.pdf_last_error()
    assert call(w=_mil(A=0)) == -1 and b"bad dims" in lib.pdf_last_error()
    nu = _mil()
    nu.w_u = None
    assert call(w=nu) == -1 and b"null weight" in lib.pdf_last_error()
    assert call(w=_mil(H=2048, A=2000)) == -1 and b"too wide" in lib.pdf_last_error()     # 16 rows of h and vu need > 227 KB


def test_philox_words_known_answers_and_bootstrap_word():
    """Random123's known-answer vectors for Philox4x32-10, and word 0 equals bootstrap_oracle's generator"""
    def run(c, k):
        return [int(w[0]) for w in O.philox4x32_10_words(*(np.array([v], np.uint64) for v in c), *k)]
    assert run((0, 0, 0, 0), (0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert run((0xffffffff,) * 4, (0xffffffff, 0xffffffff)) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert run((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == [0xd16cfe09, 0x94fdcceb, 0x5001e420,
                                                                                               0x24126ea1]
    rng = np.random.default_rng(0)
    c = [rng.integers(0, 2 ** 32, 1000, dtype=np.uint64) for _ in range(4)]
    assert np.array_equal(O.philox4x32_10_words(*c, 123, 456)[0], B.philox4x32_10(*c, 123, 456))


@pytest.mark.parametrize("p", [0.2, 0.5])
def test_keep_fraction(p):
    """10^6 units over rows, samples, layers and instances keep a fraction 1 - p (+- 0.002), each kept unit scaled by 1 / (1 - p)"""
    m = O.keep_mask(7, p, np.arange(250)[:, None, None], np.arange(8)[None, :, None], (np.arange(5) << 16)[None, None, :] | 3, 100)
    assert m.size == 10 ** 6
    assert abs((m > 0).mean() - (1 - p)) <= 0.002
    assert np.all(m[m > 0] == np.float32(1 / (1 - np.float32(p))))
    assert (O.keep_mask(7, 0.0, np.arange(100), 0, 0, 64) == 1.0).all()


def test_counters_never_equal_bootstrap_counters():
    """the bootstrap's counters are (u, b, 0, 0); every dropout counter has the top bit of word 3 set"""
    c = O.counters(np.arange(300)[:, None, None], np.arange(4096, step=97)[None, :, None],
                   ((np.arange(8) << 16) | 65535)[None, None, :], 4096)
    assert np.all(c[3] & np.uint64(0x80000000))
    assert c[3].max() == 0x80000000 | 1023


def test_risk_coverage_restatement():
    from pd_fusion_b200.evaluation.evaluate import _risk_coverage_by_entropy
    rng = np.random.default_rng(3)
    y, mean = rng.integers(0, 2, 200), rng.random(200)
    ent = np.round(O.entropy(mean), 2)              # ties: the stable order keeps row order
    rc = _risk_coverage_by_entropy(y, mean, ent)
    order = sorted(range(200), key=lambda i: (ent[i], i))
    err = [float((mean[i] >= 0.5) != y[i]) for i in order]
    risk = [sum(err[:k]) / k for k in range(1, 201)]
    assert np.allclose(rc["risk"], risk, rtol=0, atol=1e-15)
    assert np.array_equal(rc["coverage"], np.arange(1, 201) / 200)
    assert rc["aurc"] == pytest.approx(np.mean(risk), abs=1e-15)

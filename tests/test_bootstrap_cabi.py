"""The device bootstrap (pdf_bootstrap_metrics) without a GPU: prototypes agree with the header, the workspace formula, bad arguments
refused with PDF_ERR_ARG before any device work, the Poisson table, the weight restatement's moments, and bootstrap_model's interval
arithmetic on a fixed replicate array."""
import ctypes as C
import re
from fractions import Fraction
from math import factorial
from pathlib import Path

import numpy as np
import pytest

from bootstrap_oracle import POISSON1, bootstrap_weights
from pd_fusion_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
HEADER = (ROOT / "include" / "pdfusion_b200.h").read_text()
NAMES = ("pdf_bootstrap_metrics_workspace_bytes", "pdf_bootstrap_metrics")
CTYPE = {"int": C.c_int, "size_t": C.c_size_t, "uint64_t": C.c_uint64}
FAKE = 1 << 12              # a 256-byte aligned non-null address: never dereferenced, every call below fails its checks first


def _declaration(name):
    m = re.search(r"\b(int|size_t)\s+" + name + r"\s*\(([^;]*)\)\s*;", HEADER)
    assert m, f"{name} not declared in the header"
    args = re.sub(r"/\*.*?\*/", "", m.group(2), flags=re.S)
    return m.group(1), [a.strip() for a in args.split(",")]


def test_prototypes_match_header():
    lib = _lib.load()
    for name in NAMES:
        ret, args = _declaration(name)
        restype, argtypes = _lib.PROTOTYPES[name]
        assert restype is CTYPE[ret], name
        assert len(argtypes) == len(args), name
        for decl, t in zip(args, argtypes):
            if "*" in decl or decl.startswith("pdf_stream_t"):
                assert t is _lib._P, (name, decl)
            else:
                assert t is CTYPE[decl.split()[-2] if len(decl.split()) > 2 else decl.split()[0]], (name, decl)
        assert hasattr(lib, name)


def _align(n):
    return (n + 255) // 256 * 256


@pytest.mark.parametrize("S,N", [(1, 1), (7, 1000), (3, 100003), (7, 10 ** 6)])
def test_workspace_bytes(S, N):
    lib = _lib.load()
    # sorted prob f64 | unit i32 | flags u8 per (scenario, position); two f64 key and two i32 index buffers of one scenario;
    # radix-sort scratch bound 4 N + 64 KiB
    want = _align(8 * S * N) + _align(4 * S * N) + _align(S * N) + 2 * _align(8 * N) + 2 * _align(4 * N) + _align(4 * N + 65536)
    assert lib.pdf_bootstrap_metrics_workspace_bytes(S, N) == want


def test_workspace_bytes_refuses_bad_sizes():
    lib = _lib.load()
    for S, N in ((0, 10), (1, 0), (-1, 10), (1, -5), (1, (1 << 28) + 1)):
        assert lib.pdf_bootstrap_metrics_workspace_bytes(S, N) == 0


def test_argument_validation_without_gpu():
    lib = _lib.load()

    def call(S=2, n=10, B=4, seed=0, prob=FAKE, label=FAKE, unit=FAKE, ws=FAKE, out=FAKE):
        return lib.pdf_bootstrap_metrics(S, n, B, seed, prob, label, unit, ws, out, None)

    for kw in (dict(S=0), dict(S=-1), dict(n=0), dict(n=-3), dict(B=-1), dict(prob=None), dict(label=None), dict(ws=None),
               dict(out=None)):
        assert call(**kw) == -1, kw
        assert b"bad arguments" in lib.pdf_last_error(), kw
    assert call(B=(1 << 20) + 1) == -1 and b"n_boot must be" in lib.pdf_last_error()
    assert call(n=(1 << 28) + 1) == -1 and b"n must be" in lib.pdf_last_error()
    for kw in (dict(prob=FAKE + 4), dict(out=FAKE + 2), dict(unit=FAKE + 1), dict(ws=FAKE + 16)):
        assert call(**kw) == -1, kw
        assert b"misaligned" in lib.pdf_last_error(), kw


def test_poisson_table_is_the_exact_cdf():
    """T_k = floor(2^32 P(X <= k)) from the exact rational partial sums bracketing e^-1, and the kernel's table is the same."""
    # e^-1 lies between consecutive partial sums of sum (-1)^j / j!; 40 terms pin it far below 2^-32 / 13!
    lo = sum(Fraction((-1) ** j, factorial(j)) for j in range(41))
    hi = sum(Fraction((-1) ** j, factorial(j)) for j in range(40))
    lo, hi = min(lo, hi), max(lo, hi)
    want = []
    for k in range(13):
        s = sum(Fraction(1, factorial(i)) for i in range(k + 1))
        a, b = (lo * s * 2 ** 32).__floor__(), (hi * s * 2 ** 32).__floor__()
        assert a == b
        want.append(a)
    assert [int(t) for t in POISSON1] == want
    assert want[-1] == 2 ** 32 - 1
    src = (ROOT / "robust-multimodal-pd_b200" / "csrc" / "metrics.cu").read_text()
    table = re.search(r"kPoisson1\[13\]\s*=\s*\{([^}]*)\}", src).group(1)
    assert [int(v.strip().rstrip("u"), 16) for v in table.split(",")] == want


def test_weight_restatement():
    """Philox4x32-10 known-answer vector (Random123's kat_vectors: counter and key all ones), determinism, and Poisson(1) moments."""
    from bootstrap_oracle import philox4x32_10
    f = np.uint64(0xFFFFFFFF)
    assert int(philox4x32_10(f, f, f, f, 0xFFFFFFFF, 0xFFFFFFFF)) == 0x408f276d
    z = np.uint64(0)
    assert int(philox4x32_10(z, z, z, z, 0, 0)) == 0x6627e8d5
    units = np.arange(10 ** 6)
    w = bootstrap_weights(1234, 7, units)
    assert np.array_equal(w, bootstrap_weights(1234, 7, units))
    assert not np.array_equal(w, bootstrap_weights(1234, 8, units))
    assert not np.array_equal(w, bootstrap_weights(1235, 7, units))
    assert w.min() >= 0 and w.max() <= 13
    assert abs(w.mean() - 1) < 5e-3 and abs(w.var() - 1) < 1e-2
    assert np.array_equal(bootstrap_weights(1234, 7, units[::-1])[::-1], w)


def test_summarize_bootstrap_arithmetic():
    from pd_fusion_b200.evaluation.evaluate import summarize_bootstrap
    rng = np.random.default_rng(0)
    S, B, K = 3, 200, 2
    reps = rng.random((S, B, K))
    reps[1, :50, 0] = np.nan
    reps[2, :, 1] = np.nan
    point = rng.random((S, K))
    res = summarize_bootstrap(["a", "b", "c"], ["m0", "m1"], point, reps, alpha=0.1, ref=1)
    assert list(res) == ["a", "b", "c"] and "delta" not in res["b"] and set(res["a"]["delta"]) == {"m0", "m1"}
    r = res["b"]["m0"]
    ok = reps[1, 50:, 0]
    assert r["value"] == point[1, 0] and r["n_valid"] == 150
    assert (r["lo"], r["hi"]) == tuple(np.percentile(ok, [5, 95]))
    d = res["a"]["delta"]["m0"]
    assert d["value"] == point[0, 0] - point[1, 0] and d["n_valid"] == 150
    assert (d["lo"], d["hi"]) == tuple(np.percentile(reps[0, 50:, 0] - ok, [5, 95]))
    r = res["c"]["m1"]
    assert r["n_valid"] == 0 and np.isnan(r["lo"]) and np.isnan(r["hi"])
    assert res["a"]["m1"]["lo"] == np.percentile(reps[0, :, 1], 5)

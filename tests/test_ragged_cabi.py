"""Ragged batches without a device: the descriptor layout the header declares, the 16-byte packing of volumes, and argument
errors of the ragged entry points (returned before anything touches the device)."""
import ctypes as C
import re
from pathlib import Path

import pytest

from pd_fusion_b200 import _lib
from pd_fusion_b200.preprocess import RaggedBatch, ragged_offsets

HEADER = (Path(__file__).resolve().parents[1] / "include" / "pdfusion_b200.h").read_text()


def _cfg():
    cfg = _lib.PreprocCfg()
    cfg.out_shape[:] = (32, 32, 32)
    cfg.n_axes, cfg.axes[0], cfg.counts[0], cfg.input_size = 1, 2, 4, 64
    cfg.mean[:], cfg.std[:] = (0.5,) * 3, (0.5,) * 3
    return cfg


def _descs(shapes, code=4):
    offs, _ = ragged_offsets(shapes)
    d = (_lib.VolumeDesc * len(shapes))()
    for b, (sh, off) in enumerate(zip(shapes, offs)):
        d[b].shape[:] = sh
        d[b].nifti_datatype, d[b].raw_offset, d[b].src_offset, d[b].slope = code, off, 2 * off, 1.0
    return d


def test_volume_desc_layout_matches_header():
    assert C.sizeof(_lib.VolumeDesc) == 3 * 4 + 3 * 4 + 2 * 8 + 2 * 8
    assert [(n, getattr(_lib.VolumeDesc, n).offset) for n in ("src_offset", "raw_offset", "slope", "inter")] == \
        [("src_offset", 24), ("raw_offset", 32), ("slope", 40), ("inter", 48)]
    assert int(re.search(r"#define PDF_RAGGED_MAX_BATCH (\d+)", HEADER).group(1)) == _lib.PDF_RAGGED_MAX_BATCH


def test_packing_offsets_are_16_byte_aligned():
    shapes = [(5, 7, 3), (4, 4, 4), (33, 27, 31), (2, 2, 2), (160, 160, 161)]
    offs, n = ragged_offsets(shapes)
    assert offs[0] == 0 and all(o % 4 == 0 for o in offs)
    for (a, sa), b in zip(zip(offs, shapes), offs[1:] + [n]):
        vox = sa[0] * sa[1] * sa[2]
        assert a + vox <= b < a + vox + 4          # no overlap, less than 16 bytes of padding


def test_descriptors_round_trip():
    import torch
    vols = [torch.arange(s[0] * s[1] * s[2], dtype=torch.float32).reshape(s) for s in [(3, 5, 7), (4, 4, 2), (2, 3, 9)]]
    rb = RaggedBatch.from_volumes(vols, "cpu")
    assert len(rb) == 3
    for b, v in enumerate(vols):
        assert rb.shape(b) == tuple(v.shape) and int(rb.descs[b].raw_offset) % 4 == 0
        assert torch.equal(rb[b], v)
    copy = (_lib.VolumeDesc * 3).from_buffer_copy(bytes(rb.descs))
    assert [tuple(d.shape) for d in copy] == [tuple(v.shape) for v in vols]
    assert [d.raw_offset for d in copy] == [d.raw_offset for d in rb.descs]


def test_ragged_workspace_and_slice_major_limits():
    lib = _lib.load()
    cfg = _cfg()
    d = _descs([(40, 36, 44)] * (_lib.PDF_RAGGED_MAX_BATCH + 1))
    assert lib.pdf_preproc_ragged_workspace_bytes(C.byref(cfg), 0) == 0
    assert lib.pdf_preproc_ragged_workspace_bytes(C.byref(cfg), _lib.PDF_RAGGED_MAX_BATCH + 1) == 0
    # the uniform workspace of the same batch, then one interpolation table per subject
    assert lib.pdf_preproc_ragged_workspace_bytes(C.byref(cfg), 3) > lib.pdf_preproc_workspace_bytes(C.byref(cfg), 3)
    assert lib.pdf_preproc_slice_major_ok_ragged(C.byref(cfg), 2, d) == 1
    assert lib.pdf_preproc_slice_major_ok_ragged(C.byref(cfg), _lib.PDF_RAGGED_MAX_BATCH + 1, d) == 0
    d[1].shape[2] = 45                                        # Z % 4 != 0: one ineligible subject makes the batch C-order
    assert lib.pdf_preproc_slice_major_ok_ragged(C.byref(cfg), 2, d) == 0


@pytest.mark.parametrize("defect", ["oversized", "empty", "null", "datatype", "raw_offset", "src_offset", "shape"])
def test_malformed_descriptor_sets_are_argument_errors(defect):
    lib = _lib.load()
    cfg = _cfg()
    n = _lib.PDF_RAGGED_MAX_BATCH + 1 if defect == "oversized" else 3
    d = _descs([(20, 24, 16), (33, 27, 30), (40, 36, 44)] * (n // 3 + 1))
    batch = 0 if defect == "empty" else n
    descs = None if defect == "null" else d
    if defect == "datatype":
        d[1].nifti_datatype = 1024
    elif defect == "raw_offset":
        d[2].raw_offset += 2
    elif defect == "src_offset":
        d[2].src_offset += 1                                  # int16 voxels at an odd byte
    elif defect == "shape":
        d[0].shape[1] = 0
    fake = C.c_void_p(16)                                     # never dereferenced: the arguments are refused first
    rc = lib.pdf_decode_volumes(batch, descs, fake, fake, None)
    assert rc == -1 and b"pdf_decode_volumes" in lib.pdf_last_error()
    if defect in ("datatype", "src_offset"):
        return                                                # decode-only fields: the resample does not read them
    assert lib.pdf_resample_stats_ragged(C.byref(cfg), batch, descs, fake, fake, fake, None) == -1
    assert b"preproc" in lib.pdf_last_error()
    assert lib.pdf_preprocess_ragged(C.byref(cfg), batch, descs, fake, fake, fake, fake, fake, fake, fake, _lib.OUT_BF16_C1, None) == -1

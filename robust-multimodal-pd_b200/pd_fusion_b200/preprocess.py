"""Host side of K1: batched volume -> network-input preprocessing on the GPU.

Mirrors, for a whole batch of subjects resident in HBM, the reference's per-subject CPU sequence
`_load_volume` -> `_normalize_volume_for_resnet` -> `_select_slices` -> F.interpolate/normalise
(data/openneuro_features.py:22-32, 121-151, 250-255).  All arithmetic runs in
libpdfusion_b200.so; this class only owns the device buffers.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Sequence

import torch

from . import _lib


@dataclass
class PreprocResult:
    net_input: torch.Tensor   # [B, L, S, S] bf16, [B, L, rows, pitch] bf16 (zero-padded) or [B, L, S, S, 3] f32
    zoomed: torch.Tensor      # [B, T0, T1, T2] f32 (resampled, un-normalised); [B, T2, T0, T1] from a slice-major run()
    lohi: torch.Tensor        # [B, 4] f32: lo, hi, denominator, has_positive
    indices: torch.Tensor     # [B, L] i32 (-1 in unused slots)
    nslices: torch.Tensor     # [B, n_axes] i32
    slice_major: bool = False  # whether `zoomed` came out slice-major


def ragged_offsets(shapes: Sequence[Sequence[int]]):
    """Offsets (float32 elements, multiples of 4: every volume starts 16-byte aligned) of volumes of `shapes` packed one after the
    other, and the packed length."""
    offs, n = [], 0
    for sh in shapes:
        offs.append(n)
        n += (int(sh[0]) * int(sh[1]) * int(sh[2]) + 3) // 4 * 4
    return offs, n


class RaggedBatch:
    """Raw volumes of different shapes in one packed float32 device buffer, C order [X, Y, Z] each at the descriptor's raw_offset,
    plus the host array of `pdf_volume_desc` that places them: the input of the ragged preprocessing entry points.
    batch[b] is subject b's volume as a [X, Y, Z] view."""

    def __init__(self, raw: torch.Tensor, descs):
        self.raw, self.descs = raw, descs

    @classmethod
    def from_volumes(cls, volumes, device) -> "RaggedBatch":
        """Packs float32 [X, Y, Z] arrays or tensors of any shapes."""
        vols = [torch.as_tensor(v, dtype=torch.float32) for v in volumes]
        offs, n = ragged_offsets([v.shape for v in vols])
        descs = (_lib.VolumeDesc * len(vols))()
        host = torch.zeros(max(n, 4), dtype=torch.float32)
        for b, (v, off) in enumerate(zip(vols, offs)):
            descs[b].shape[:] = [int(d) for d in v.shape]
            descs[b].nifti_datatype, descs[b].raw_offset, descs[b].slope = 16, off, 1.0
            host[off:off + v.numel()] = v.reshape(-1)
        return cls(host.to(device), descs)

    def __len__(self) -> int:
        return len(self.descs)

    def shape(self, b: int):
        return tuple(int(v) for v in self.descs[b].shape)

    def __getitem__(self, b: int) -> torch.Tensor:
        X, Y, Z = self.shape(b)
        off = int(self.descs[b].raw_offset)
        return self.raw[off:off + X * Y * Z].view(X, Y, Z)


class VolumePreprocessor:
    def __init__(self, in_shape: Sequence[int] | None, target_shape: Sequence[int] = (160, 160, 160),
                 axes: Sequence[int] = (2,), counts: Sequence[int] = (24,), input_size: int = 224,
                 mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5), out_mode: int = _lib.OUT_BF16_C1,
                 max_batch: int = 1, device=None, slice_major: bool = False):
        """slice_major: `run()` (the fused pipeline) keeps the resampled volume slice-axis-major, [B, T2, T0, T1], when the library
        supports it for this configuration (one axis group on axis 2; `pdf_preproc_slice_major_ok`): the selected planes are then
        contiguous and the plane-gather pass disappears.  `PreprocResult.zoomed` of such a run has that layout
        (`self.run_slice_major`); the stage-level entry points (resample / select / gather / gather_slices) always use the
        reference's C order.

        in_shape None: ragged mode.  run() and resample() then take a `RaggedBatch` of subjects of any raw shapes (at most
        PDF_RAGGED_MAX_BATCH); a run is slice-major when every subject of its batch allows it (`PreprocResult.slice_major`)."""
        _lib.require_cuda()
        self.lib = _lib.load()
        if len(axes) != len(counts) or not 1 <= len(axes) <= _lib.PDF_MAX_AXES:
            raise ValueError("slice-counts must match length of slice-axes")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.ragged = in_shape is None
        self.in_shape = None if self.ragged else tuple(int(v) for v in in_shape)
        self.target_shape = tuple(int(v) for v in target_shape)
        self.axes, self.counts = [int(a) for a in axes], [int(c) for c in counts]
        self.lmax = sum(self.counts)
        self.input_size = int(input_size)
        self.out_mode = out_mode
        self.max_batch = int(max_batch)
        cfg = _lib.PreprocCfg()
        if not self.ragged:
            cfg.in_shape[:] = self.in_shape
        cfg.out_shape[:] = self.target_shape
        cfg.n_axes = len(self.axes)
        for i in range(_lib.PDF_MAX_AXES):
            cfg.axes[i] = self.axes[i] if i < len(self.axes) else 0
            cfg.counts[i] = self.counts[i] if i < len(self.counts) else 0
        cfg.input_size = self.input_size
        cfg.mean[:] = [float(m) for m in mean]
        cfg.std[:] = [float(s) for s in std]
        self.cfg = cfg
        self.cfg_run = cfg                                    # configuration of the fused run(): slice-major where possible
        self.run_slice_major = False
        self.cfg_sm = None                                    # slice-major copy of cfg (ragged mode: used batch by batch)
        if slice_major and (self.ragged or self.lib.pdf_preproc_slice_major_ok(C.byref(cfg))):
            self.cfg_sm = _lib.PreprocCfg.from_buffer_copy(cfg)
            self.cfg_sm.slice_major = 1
            if not self.ragged:
                self.cfg_run = self.cfg_sm
                self.run_slice_major = True
        if self.ragged:
            if not 1 <= self.max_batch <= _lib.PDF_RAGGED_MAX_BATCH:
                raise ValueError(f"a ragged preprocessor takes 1..{_lib.PDF_RAGGED_MAX_BATCH} subjects per batch")
            ws = self.lib.pdf_preproc_ragged_workspace_bytes(C.byref(cfg), self.max_batch)
        else:
            ws = self.lib.pdf_preproc_workspace_bytes(C.byref(cfg), self.max_batch)
        if ws == 0:
            raise _lib.PdfusionError("pdf_preproc_workspace_bytes returned 0 (bad configuration)")
        B, S = self.max_batch, self.input_size
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(ws, dtype=torch.uint8, device=self.device)
            self.zoomed = torch.empty((B,) + self.target_shape, dtype=torch.float32, device=self.device)
            self.lohi = torch.empty((B, 4), dtype=torch.float32, device=self.device)
            self.indices = torch.empty((B, self.lmax), dtype=torch.int32, device=self.device)
            self.nslices = torch.empty((B, len(self.axes)), dtype=torch.int32, device=self.device)
            if out_mode == _lib.OUT_BF16_C1:
                self.net_input = torch.empty((B, self.lmax, S, S), dtype=torch.bfloat16, device=self.device)
            elif out_mode == _lib.OUT_BF16_C1_PAD:
                pitch, rows = _lib.stem_padded_dims(S)       # the border is zeroed here, once; the kernels only write the image
                self.net_input = torch.zeros((B, self.lmax, rows, pitch), dtype=torch.bfloat16, device=self.device)
            else:
                self.net_input = torch.empty((B, self.lmax, S, S, 3), dtype=torch.float32, device=self.device)

    def _check_raw(self, raw) -> int:
        if self.ragged != isinstance(raw, RaggedBatch):
            raise ValueError("a ragged preprocessor (in_shape None) takes a RaggedBatch, a uniform one a [B, X, Y, Z] tensor")
        if self.ragged:
            if not (raw.raw.is_cuda and raw.raw.dtype == torch.float32 and raw.raw.is_contiguous()):
                raise ValueError("the packed raw buffer must be a contiguous float32 CUDA tensor")
            if not 1 <= len(raw) <= self.max_batch:
                raise ValueError(f"ragged batch of {len(raw)} subjects, max_batch {self.max_batch}")
            need = max(int(d.raw_offset) + int(d.shape[0]) * int(d.shape[1]) * int(d.shape[2]) for d in raw.descs)
            if need > raw.raw.numel():
                raise ValueError(f"descriptors reach element {need} of a packed buffer of {raw.raw.numel()}")
            return len(raw)
        if not (raw.is_cuda and raw.dtype == torch.float32 and raw.is_contiguous()):
            raise ValueError("raw volumes must be a contiguous float32 CUDA tensor [B, X, Y, Z]")
        if tuple(raw.shape[1:]) != self.in_shape or raw.shape[0] > self.max_batch:
            raise ValueError(f"raw volumes {tuple(raw.shape)} do not match in_shape {self.in_shape} / max_batch {self.max_batch}")
        return int(raw.shape[0])

    def run(self, raw, net_input: torch.Tensor | None = None) -> PreprocResult:
        """Enqueues resample+stats, select, gather/resize on the current stream (no sync).  raw: [B, X, Y, Z] f32 on the device, or
        a RaggedBatch in ragged mode."""
        B = self._check_raw(raw)
        out = self.net_input if net_input is None else net_input
        args = (self.zoomed.data_ptr(), self.workspace.data_ptr(), self.lohi.data_ptr(), self.indices.data_ptr(),
                self.nslices.data_ptr(), out.data_ptr(), self.out_mode, _lib.stream_ptr())
        if self.ragged:
            slice_major = self.cfg_sm is not None and bool(self.lib.pdf_preproc_slice_major_ok_ragged(C.byref(self.cfg_sm), B, raw.descs))
            cfg = self.cfg_sm if slice_major else self.cfg
            _lib.check(self.lib.pdf_preprocess_ragged(C.byref(cfg), B, raw.descs, raw.raw.data_ptr(), *args), "pdf_preprocess_ragged")
        else:
            slice_major = self.run_slice_major
            _lib.check(self.lib.pdf_preprocess(C.byref(self.cfg_run), B, raw.data_ptr(), *args), "pdf_preprocess")
        zoomed = self.zoomed[:B]
        if slice_major:                                       # same bytes, [B, T2, T0, T1]
            T0, T1, T2 = self.target_shape
            zoomed = zoomed.view(B, T2, T0, T1)
        return PreprocResult(out[:B], zoomed, self.lohi[:B], self.indices[:B], self.nslices[:B], slice_major)

    # stage-level entry points (parity tests, per-kernel timing)
    def resample(self, raw) -> torch.Tensor:
        B = self._check_raw(raw)
        if self.ragged:
            _lib.check(self.lib.pdf_resample_stats_ragged(C.byref(self.cfg), B, raw.descs, raw.raw.data_ptr(), self.zoomed.data_ptr(),
                                                          self.workspace.data_ptr(), _lib.stream_ptr()), "pdf_resample_stats_ragged")
        else:
            _lib.check(self.lib.pdf_resample_stats(C.byref(self.cfg), B, raw.data_ptr(), self.zoomed.data_ptr(),
                                                   self.workspace.data_ptr(), _lib.stream_ptr()), "pdf_resample_stats")
        return self.zoomed[:B]

    def select(self, B: int):
        _lib.check(self.lib.pdf_select_bounds_indices(C.byref(self.cfg), B, self.zoomed.data_ptr(), self.workspace.data_ptr(),
                                                      self.lohi.data_ptr(), self.indices.data_ptr(), self.nslices.data_ptr(),
                                                      _lib.stream_ptr()), "pdf_select_bounds_indices")
        return self.lohi[:B], self.indices[:B], self.nslices[:B]

    def select_raw(self, vol: torch.Tensor):
        """Indices of `_select_slices` on an already-normalised volume: extent test is voxel > 0 (no re-normalisation)."""
        B = self._check_raw(vol)
        self.resample(vol)                      # in_shape == target_shape: identity zoom, gathers plane maxima
        self.cfg.extent_raw = 1
        try:
            _, idx, ns = self.select(B)
        finally:
            self.cfg.extent_raw = 0
        return idx, ns

    def gather(self, B: int) -> torch.Tensor:
        _lib.check(self.lib.pdf_gather_resize_normalize(C.byref(self.cfg), B, self.zoomed.data_ptr(), self.workspace.data_ptr(),
                                                        self.lohi.data_ptr(), self.indices.data_ptr(), self.nslices.data_ptr(),
                                                        self.net_input.data_ptr(), self.out_mode, _lib.stream_ptr()),
                   "pdf_gather_resize_normalize")
        return self.net_input[:B]

    # ---- test-time augmentation (a6): slices -> affine/intensity/noise/clip -> network input
    def slice_shape(self):
        """(H, W) of the selected slices; every axis group must agree (the reference concatenates them)."""
        shapes = set()
        for a in self.axes:
            dims = list(self.target_shape)
            dims.pop(a)
            shapes.add(tuple(dims))
        if len(shapes) != 1:
            raise ValueError("slice groups of different shapes cannot be concatenated (the reference needs a cubic target_shape)")
        return shapes.pop()

    def gather_slices(self, B: int) -> torch.Tensor:
        """`_select_slices` of the normalised volume, all axis groups concatenated: [B, L, H, W] f32 (after select())."""
        H, W = self.slice_shape()
        if getattr(self, "_slices", None) is None:
            self._slices = torch.empty((self.max_batch, self.lmax, H, W), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.pdf_gather_slices(C.byref(self.cfg), B, self.zoomed.data_ptr(), self.lohi.data_ptr(), self.indices.data_ptr(),
                                              self.nslices.data_ptr(), self._slices.data_ptr(), _lib.stream_ptr()), "pdf_gather_slices")
        return self._slices[:B]

    def tta_augment(self, slices: torch.Tensor, params: torch.Tensor, noise: torch.Tensor | None, affine_only: bool = False) -> torch.Tensor:
        """One augmentation pass.  slices [B, L, H, W] f32; params = pdf_tta_params bytes of the B subjects on the device;
        noise [B, L, H, W] f64 on the device or None."""
        B, L, H, W = (int(v) for v in slices.shape)
        out = torch.empty_like(slices)
        _lib.check(self.lib.pdf_tta_augment(B, L, H, W, slices.data_ptr(), params.data_ptr(), _lib.ptr(noise), int(affine_only),
                                            out.data_ptr(), _lib.stream_ptr()), "pdf_tta_augment")
        return out

    def resize_slices(self, slices: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """Bilinear resize + (x-mean)/std of ready-made [0,1] slices into the network-input layout of this preprocessor."""
        B, L, H, W = (int(v) for v in slices.shape)
        out = self.net_input if out is None else out
        mean = (C.c_float * 3)(*[float(v) for v in self.cfg.mean])
        std = (C.c_float * 3)(*[float(v) for v in self.cfg.std])
        _lib.check(self.lib.pdf_resize_slices(B, L, H, W, self.input_size, mean, std, slices.data_ptr(), out.data_ptr(), self.out_mode,
                                              _lib.stream_ptr()), "pdf_resize_slices")
        return out[:B]

    def normalized_volume(self, B: int) -> torch.Tensor:
        """`_normalize_volume_for_resnet` output itself (parity helper)."""
        out = torch.empty_like(self.zoomed[:B])
        vox = self.target_shape[0] * self.target_shape[1] * self.target_shape[2]
        _lib.check(self.lib.pdf_normalize_volume(B, vox, self.zoomed.data_ptr(), self.lohi.data_ptr(), out.data_ptr(),
                                                 _lib.stream_ptr()), "pdf_normalize_volume")
        return out

    def algorithmic_bytes(self, batch: RaggedBatch | None = None) -> int:
        """SURVEY.md 8(d): 4XYZ + 2*4*T^3 + 4*L*T^2 + b_out*L*I^2 per subject.  Ragged mode: the sum over the subjects of `batch`,
        each with its own 4XYZ."""
        if self.ragged:
            if batch is None:
                raise ValueError("a ragged preprocessor counts the bytes of a given RaggedBatch")
            return sum(self._algorithmic_bytes(batch.shape(b)) for b in range(len(batch)))
        return self._algorithmic_bytes(self.in_shape)

    def _algorithmic_bytes(self, in_shape) -> int:
        X, Y, Z = in_shape
        T0, T1, T2 = self.target_shape
        plane = 0
        for a, c in zip(self.axes, self.counts):
            dims = [T0, T1, T2]
            dims.pop(a)
            plane += 4 * c * dims[0] * dims[1]
        b_out = 12 if self.out_mode == _lib.OUT_F32_NHWC3 else 2
        return 4 * X * Y * Z + 8 * T0 * T1 * T2 + plane + b_out * self.lmax * self.input_size ** 2

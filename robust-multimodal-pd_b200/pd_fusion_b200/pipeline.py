"""Volume -> embedding pipeline for a batch of subjects resident in HBM (K1 + K2 + slice mean).

Replaces the serial per-subject loop of `build_resnet2d_embeddings`
(data/openneuro_features.py:226-265) and of scripts/build_resnet2d_mil_embeddings.py:112-158:
every subject of the batch is resampled, normalised, sliced and encoded by the same sequence of launches.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Dict, Sequence

import torch

from . import _lib
from .backbone import ResNetEncoder, detect_arch
from .preprocess import RaggedBatch, VolumePreprocessor


@dataclass
class EmbedResult:
    embeddings: torch.Tensor    # [B, L, D] f32 per-slice embeddings (MIL bag)
    mean: torch.Tensor          # [B, D] f32 mean over the valid slices (non-MIL embedding)
    indices: torch.Tensor       # [B, L] i32
    nslices: torch.Tensor       # [B, n_axes] i32


class EmbeddingPipeline:
    def __init__(self, backbone_state_dict: Dict[str, torch.Tensor], in_shape: Sequence[int] | None,
                 target_shape: Sequence[int] = (160, 160, 160), axes: Sequence[int] = (2,), counts: Sequence[int] = (24,),
                 input_size: int = 224, precision: str = "bf16", max_subjects: int = 8, mean=(0.5, 0.5, 0.5),
                 std=(0.5, 0.5, 0.5), arch: str | None = None, device=None):
        """in_shape None: one pipeline for subjects of every raw shape -- embed() / embed_tta() then take a RaggedBatch
        (see VolumePreprocessor); the end-to-end embed_host / embed_overlapped paths need a fixed in_shape."""
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.max_subjects = int(max_subjects)
        self.precision = precision
        self._ctor = dict(sd=backbone_state_dict, input_size=input_size, arch=arch or detect_arch(backbone_state_dict), mean=mean, std=std)
        self._ov = None
        mode = _lib.OUT_BF16_C1_PAD if precision == "bf16" else _lib.OUT_F32_NHWC3   # the fused stem reads a zero-padded image
        with torch.cuda.device(self.device):
            L = int(sum(counts))
            self.enc = ResNetEncoder(backbone_state_dict, self.max_subjects * L, input_size, precision,
                                     arch or detect_arch(backbone_state_dict), self.device, mean=mean, std=std)
            if precision == "bf16":      # one channel, normalised with the channel-averaged statistics (backbone.py folds the rest)
                m_avg, s_avg = self.enc.input_mean_std
                mean, std = (m_avg,) * 3, (s_avg,) * 3
            # (embed() keeps the resampled volume slice-major where the library can: contiguous planes, no gather pass)
            self.pre = VolumePreprocessor(in_shape, target_shape, axes, counts, input_size, mean, std, mode,
                                          self.max_subjects, self.device,
                                          slice_major=os.environ.get("PDFUSION_B200_SLICE_MAJOR", "1") != "0")
            self.L = self.pre.lmax
            self.D = self.enc.emb_dim
            # preprocessing writes straight into the encoder's input buffer
            enc_in = self.enc.input_padded if self.enc.input_padded is not None else self.enc.input
            self._net_input = enc_in.view(self.pre.net_input.shape)
            self.pre.net_input = self._net_input
            self.mean_out = torch.empty((self.max_subjects, self.D), dtype=torch.float32, device=self.device)
            self.nvalid = torch.empty((self.max_subjects,), dtype=torch.int32, device=self.device)

    def embed(self, raw) -> EmbedResult:
        """raw [B<=max_subjects, X, Y, Z] f32 on the device, or a RaggedBatch of B subjects (in_shape None). Enqueues everything
        on the current stream; results live in reused buffers (copy them out before the next call)."""
        B = len(raw) if isinstance(raw, RaggedBatch) else int(raw.shape[0])
        if B < self.max_subjects:   # the encoder plan is built for max_subjects*L images: clear the unused tail
            self.enc.input[B * self.L:].zero_()
        res = self.pre.run(raw, net_input=self._net_input)
        emb = self.enc.forward(None).view(self.max_subjects, self.L, self.D)
        self.nvalid[:B].copy_(res.nslices.sum(dim=1))
        _lib.check(self.lib.pdf_slice_mean(B, self.L, self.D, emb.data_ptr(), self.nvalid.data_ptr(), self.mean_out.data_ptr(),
                                           _lib.stream_ptr()), "pdf_slice_mean")
        return EmbedResult(emb[:B], self.mean_out[:B], res.indices, res.nslices)

    # ---- cross-batch overlap: preprocessing of batch i+1 (CUDA cores, HBM streaming) runs on its own stream next to the
    #      tensor-core conv stack of batch i.  Two encoder instances alternate so that a batch's network input is never
    #      overwritten while its convolutions still read it.
    def enable_overlap(self):
        if self._ov is not None:
            return
        c = self._ctor
        with torch.cuda.device(self.device):
            enc2 = ResNetEncoder(c["sd"], self.max_subjects * self.L, c["input_size"], self.precision, c["arch"], self.device,
                                 mean=c["mean"], std=c["std"])
            encs = [self.enc, enc2]
            ins = [(e.input_padded if e.input_padded is not None else e.input).view(self.pre.net_input.shape) for e in encs]
            B, L = self.max_subjects, self.L
            prio = os.environ.get("PDFUSION_B200_PRIO", "")          # tuning hook: which of the two streams the block scheduler prefers
            self._ov = dict(
                encs=encs, ins=ins, turn=0,
                pre_stream=torch.cuda.Stream(self.device, priority=-1 if prio == "pre" else 0),
                conv_stream=torch.cuda.Stream(self.device, priority=-1 if prio == "conv" else 0),
                pre_done=[torch.cuda.Event() for _ in range(2)], slot_free=[torch.cuda.Event() for _ in range(2)],
                mean=[torch.empty((B, self.D), dtype=torch.float32, device=self.device) for _ in range(2)],
                nvalid=[torch.empty((B,), dtype=torch.int32, device=self.device) for _ in range(2)],
                indices=[torch.empty((B, L), dtype=torch.int32, device=self.device) for _ in range(2)],
                nslices=[torch.empty((B, len(self.pre.axes)), dtype=torch.int32, device=self.device) for _ in range(2)])
            cur = torch.cuda.current_stream(self.device)
            for ev in self._ov["slot_free"]:
                ev.record(cur)

    @property
    def conv_stream(self):
        return self._ov["conv_stream"]

    def overlap_begin(self):
        """The two worker streams start after everything already enqueued on the current stream."""
        cur = torch.cuda.current_stream(self.device)
        self._ov["pre_stream"].wait_stream(cur)
        self._ov["conv_stream"].wait_stream(cur)

    def overlap_end(self):
        """The current stream continues after everything the worker streams were given."""
        cur = torch.cuda.current_stream(self.device)
        cur.wait_stream(self._ov["pre_stream"])
        cur.wait_stream(self._ov["conv_stream"])

    def hold_slot(self, stream) -> None:
        """Consumers that read the latest embed_overlapped() result on ANOTHER stream call this after enqueueing their reads:
        the result slot (encoder output, slice means, indices) is then not reused before `stream` got there."""
        ov = self._ov
        s = (ov["turn"] - 1) & 1
        ov["slot_free"][s].record(stream)

    def embed_overlapped(self, raw: torch.Tensor) -> EmbedResult:
        """Like embed(), but preprocessing is enqueued on the preprocessing stream and the encoder on the convolution
        stream: consecutive calls overlap.  The returned tensors are produced on `conv_stream` and stay valid until the
        call after next (two result slots); bracket a sequence of calls with overlap_begin() / overlap_end()."""
        self.enable_overlap()
        ov = self._ov
        s = ov["turn"] & 1
        ov["turn"] += 1
        B = int(raw.shape[0])
        enc = ov["encs"][s]
        P, Cs = ov["pre_stream"], ov["conv_stream"]
        with torch.cuda.stream(P):
            P.wait_event(ov["slot_free"][s])                  # the convolutions of the batch before last have consumed this input
            if B < self.max_subjects:
                enc.input[B * self.L:].zero_()
            res = self.pre.run(raw, net_input=ov["ins"][s])
            ov["indices"][s][:B].copy_(res.indices)
            ov["nslices"][s][:B].copy_(res.nslices)
            ov["nvalid"][s][:B].copy_(res.nslices.sum(dim=1))
            ov["pre_done"][s].record(P)
        with torch.cuda.stream(Cs):
            Cs.wait_event(ov["pre_done"][s])
            emb = enc.forward(None).view(self.max_subjects, self.L, self.D)
            _lib.check(self.lib.pdf_slice_mean(B, self.L, self.D, emb.data_ptr(), ov["nvalid"][s].data_ptr(), ov["mean"][s].data_ptr(),
                                               _lib.stream_ptr()), "pdf_slice_mean")
            ov["slot_free"][s].record(Cs)
        return EmbedResult(emb[:B], ov["mean"][s][:B], ov["indices"][s][:B], ov["nslices"][s][:B])

    def embed_tta(self, raw, seeds, n_pass: int, tta_cfg: Dict) -> EmbedResult:
        """`tta > 1` path of the builders (data/openneuro_features.py:235-265): every pass re-augments the selected slices
        (affine, intensity, noise, clip), runs the backbone, and the per-slice / slice-mean embeddings are averaged over the
        passes.  seeds[b] seeds subject b's numpy Generator (the reference: abs(hash(str(subject_id))) % 2**32)."""
        import numpy as np

        from .data.tta import draw_passes, params_bytes

        B = len(raw) if isinstance(raw, RaggedBatch) else int(raw.shape[0])
        self.pre.resample(raw)
        _, indices, nslices = self.pre.select(B)
        slices = self.pre.gather_slices(B)
        H, W = self.pre.slice_shape()
        ns = nslices.cpu().numpy()                          # the noise field's shape depends on the slices actually found
        counts = self.pre.counts
        draws = [draw_passes(int(seeds[b]), n_pass, int(ns[b].sum()), (H, W), tta_cfg) for b in range(B)]
        emb_sum = torch.zeros((B, self.L, self.D), dtype=torch.float32, device=self.device)
        mean_sum = torch.zeros((B, self.D), dtype=torch.float32, device=self.device)
        self.nvalid[:B].copy_(nslices.sum(dim=1))
        if B < self.max_subjects:
            self.enc.input[B * self.L:].zero_()
        for p in range(n_pass):
            params = torch.from_numpy(params_bytes([draws[b][p] for b in range(B)])).to(self.device)
            noise = None
            if draws[0][p].noise is not None:
                host = np.zeros((B, self.L, H, W), dtype=np.float64)
                for b in range(B):
                    k, off = 0, 0
                    for a, c in enumerate(counts):              # valid slices are the first ns[b, a] slots of each axis group
                        n = int(ns[b, a])
                        host[b, off:off + n] = draws[b][p].noise[k:k + n]
                        k, off = k + n, off + c
                noise = torch.from_numpy(host).to(self.device)
            aug = self.pre.tta_augment(slices, params, noise)
            self.pre.resize_slices(aug, out=self._net_input)
            emb = self.enc.forward(None).view(self.max_subjects, self.L, self.D)
            _lib.check(self.lib.pdf_slice_mean(B, self.L, self.D, emb.data_ptr(), self.nvalid.data_ptr(), self.mean_out.data_ptr(),
                                               _lib.stream_ptr()), "pdf_slice_mean")
            emb_sum += emb[:B]
            mean_sum += self.mean_out[:B]
        return EmbedResult(emb_sum / float(n_pass), mean_sum / float(n_pass), indices, nslices)

    def embed_host(self, host_batches, out_bags: bool = False, post=None, stored=None):
        """End-to-end path for volumes that live in (pinned) HOST memory: iterates over `host_batches` (tensors
        [B, X, Y, Z] f32), overlapping the H2D copy of batch i+1 (copy stream, second device buffer) with the kernels
        of batch i, and returns a list of host tensors (slice-mean embeddings [B, D], or the bags [B, L, D]).
        `post(EmbedResult) -> device tensor` (e.g. the fusion head under the scenario masks) runs on each batch before the
        read-back; its result is read back too and the list then holds (embeddings, post result) pairs.
        `stored=(nifti_datatype, fortran_order, slope, inter)`: the batches hold the voxels AS STORED in the image files
        ([B, X*Y*Z] of the file's type, e.g. int16) -- the upload then carries the file's bytes and `pdf_decode_volume` produces
        the float32 volumes on the device (half the PCIe traffic for the usual int16 T1 image)."""
        main = torch.cuda.current_stream(self.device)
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(self.device)
            self._raw = [torch.empty((self.max_subjects,) + self.pre.in_shape, dtype=torch.float32, device=self.device) for _ in range(2)]
            self._ev_copy = [torch.cuda.Event() for _ in range(2)]
            self._ev_free = [torch.cuda.Event() for _ in range(2)]
        cs = self._copy_stream
        batches = list(host_batches)
        outs = []
        staged = None
        if stored is not None and batches:
            nbytes = batches[0][0].numel() * batches[0].element_size()
            if getattr(self, "_stored", None) is None or self._stored[0].shape[1] != nbytes:
                self._stored = [torch.empty((self.max_subjects, nbytes), dtype=torch.uint8, device=self.device) for _ in range(2)]
            staged = self._stored

        def start_copy(i):
            slot = i & 1
            with torch.cuda.stream(cs):
                cs.wait_event(self._ev_free[slot])
                if staged is None:
                    self._raw[slot][: batches[i].shape[0]].copy_(batches[i], non_blocking=True)
                else:
                    hb = batches[i]
                    staged[slot][: hb.shape[0]].copy_(hb.view(torch.uint8).reshape(hb.shape[0], -1), non_blocking=True)
                self._ev_copy[slot].record(cs)

        for ev in self._ev_free:
            ev.record(main)
        if batches:
            start_copy(0)
        for i, hb in enumerate(batches):
            slot, B = i & 1, int(hb.shape[0])
            if i + 1 < len(batches):
                start_copy(i + 1)
            main.wait_event(self._ev_copy[slot])
            if staged is not None:
                code, fortran, slope, inter = stored
                X, Y, Z = self.pre.in_shape
                _lib.check(self.lib.pdf_decode_volume(B, int(code), X, Y, Z, int(bool(fortran)), float(slope), float(inter),
                                                      staged[slot].data_ptr(), self._raw[slot].data_ptr(), _lib.stream_ptr()),
                           "pdf_decode_volume")
            res = self.embed(self._raw[slot][:B])
            self._ev_free[slot].record(main)
            src = res.embeddings if out_bags else res.mean
            host = torch.empty(src.shape, dtype=torch.float32).pin_memory()
            host.copy_(src, non_blocking=True)
            if post is not None:
                extra = post(res)
                hx = torch.empty(extra.shape, dtype=extra.dtype).pin_memory()
                hx.copy_(extra, non_blocking=True)
                outs.append((host, hx))
            else:
                outs.append(host)
        main.synchronize()
        return outs

    def algorithmic_bytes_per_subject(self) -> int:
        return self.pre.algorithmic_bytes()

    def algorithmic_flops_per_subject(self) -> float:
        return self.enc.algorithmic_flops() / self.max_subjects

"""ctypes binding of libpdfusion_b200.so (the C ABI declared in include/pdfusion_b200.h).

There is no CPU fallback: if the shared library is missing, or a compute call is made without a
CUDA device, this module raises.  Build with `python __graft_entry__.py` (or `make -C csrc`).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("PDFUSION_B200_LIB", _HERE / "libpdfusion_b200.so"))

PDF_MAX_AXES = 3
PDF_MAX_LAYERS = 8
PDF_MAX_MODS = 8
PDF_RAGGED_MAX_BATCH = 64

OUT_BF16_C1 = 0
OUT_F32_NHWC3 = 1
OUT_BF16_C1_PAD = 2
STEM_PAD_LO = 5

OP_CONV, OP_MAXPOOL, OP_AVGPOOL, OP_STEM_IM2COL, OP_STEM_FUSED = 0, 1, 2, 3, 4
PREC_F32, PREC_BF16, PREC_TF32 = 0, 1, 2


class PreprocCfg(C.Structure):
    _fields_ = [
        ("in_shape", C.c_int32 * 3),
        ("out_shape", C.c_int32 * 3),
        ("n_axes", C.c_int32),
        ("axes", C.c_int32 * PDF_MAX_AXES),
        ("counts", C.c_int32 * PDF_MAX_AXES),
        ("input_size", C.c_int32),
        ("mean", C.c_float * 3),
        ("std", C.c_float * 3),
        ("extent_raw", C.c_int32),
        ("slice_major", C.c_int32),
    ]


class VolumeDesc(C.Structure):
    """pdf_volume_desc: one subject of a ragged batch (raw geometry, and how its stored voxels decode)."""
    _fields_ = [
        ("shape", C.c_int32 * 3),
        ("nifti_datatype", C.c_int32),
        ("fortran_order", C.c_int32),
        ("pad", C.c_int32),
        ("src_offset", C.c_int64),
        ("raw_offset", C.c_int64),
        ("slope", C.c_double),
        ("inter", C.c_double),
    ]


class TtaParams(C.Structure):
    _fields_ = [("rot", C.c_double * 4), ("offset", C.c_double * 2), ("scale", C.c_float), ("shift", C.c_float)]


class Op(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("precision", C.c_int32),
        ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c", C.c_int32),
        ("k", C.c_int32), ("r", C.c_int32), ("s", C.c_int32),
        ("stride", C.c_int32), ("pad", C.c_int32),
        ("ho", C.c_int32), ("wo", C.c_int32),
        ("relu", C.c_int32), ("out_f32", C.c_int32), ("sc_c", C.c_int32),
        ("d_in", C.c_void_p), ("d_weight", C.c_void_p), ("d_scale", C.c_void_p), ("d_bias", C.c_void_p),
        ("d_residual", C.c_void_p), ("d_out", C.c_void_p),
        ("d_weight2", C.c_void_p), ("d_bias2", C.c_void_p), ("d_out2", C.c_void_p),
        ("d_weight3", C.c_void_p), ("d_bias3", C.c_void_p), ("d_out3", C.c_void_p), ("k3", C.c_int32), ("sc_hw", C.c_int32),
    ]


class MilWeights(C.Structure):
    _fields_ = [
        ("D", C.c_int32), ("H", C.c_int32), ("A", C.c_int32), ("gated", C.c_int32),
        ("w_inst", C.c_void_p), ("b_inst", C.c_void_p), ("w_v", C.c_void_p), ("b_v", C.c_void_p),
        ("w_u", C.c_void_p), ("b_u", C.c_void_p), ("w_w", C.c_void_p), ("b_w", C.c_void_p),
        ("w_cls", C.c_void_p), ("b_cls", C.c_void_p),
        ("missing_prob", C.c_float),
    ]


class MilTrain(C.Structure):
    _fields_ = [
        ("loss_type", C.c_int32), ("pos_weight", C.c_float), ("focal_gamma", C.c_float), ("focal_alpha", C.c_float),
        ("d_w_w", C.c_void_p), ("d_b_w", C.c_void_p), ("d_w_cls", C.c_void_p), ("d_b_cls", C.c_void_p),
    ]


class Mlp(C.Structure):
    _fields_ = [
        ("n_layers", C.c_int32),
        ("dims", C.c_int32 * (PDF_MAX_LAYERS + 1)),
        ("w", C.c_void_p * PDF_MAX_LAYERS),
        ("b", C.c_void_p * PDF_MAX_LAYERS),
        ("n_mods", C.c_int32),
        ("mod_off", C.c_int32 * (PDF_MAX_MODS + 1)),
    ]


class Moe(C.Structure):
    _fields_ = [
        ("n_experts", C.c_int32),
        ("expert", Mlp * PDF_MAX_MODS),
        ("router_hidden", C.c_int32),
        ("w_r0", C.c_void_p), ("b_r0", C.c_void_p), ("w_r1", C.c_void_p), ("b_r1", C.c_void_p),
    ]


# name -> (restype, argtypes); also the list tests/test_cabi.py checks against include/pdfusion_b200.h
_P = C.c_void_p
PROTOTYPES = {
    "pdf_version": (C.c_int, []),
    "pdf_last_error": (C.c_char_p, []),
    "pdf_launch_count": (C.c_uint64, []),
    "pdf_preproc_workspace_bytes": (C.c_size_t, [C.POINTER(PreprocCfg), C.c_int]),
    "pdf_resample_stats": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, _P, _P, _P, _P]),
    "pdf_select_bounds_indices": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, _P, _P, _P, _P, _P, _P]),
    "pdf_gather_resize_normalize": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "pdf_preprocess": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "pdf_gather_slices": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, _P, _P, _P, _P, _P, _P]),
    "pdf_tta_augment": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int, _P, _P]),
    "pdf_resize_slices": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), _P, _P, C.c_int, _P]),
    "pdf_normalize_volume": (C.c_int, [C.c_int, C.c_size_t, _P, _P, _P, _P]),
    "pdf_decode_volume": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, _P, _P, _P]),
    "pdf_decode_volumes": (C.c_int, [C.c_int, C.POINTER(VolumeDesc), _P, _P, _P]),
    "pdf_preproc_ragged_workspace_bytes": (C.c_size_t, [C.POINTER(PreprocCfg), C.c_int]),
    "pdf_preproc_slice_major_ok_ragged": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, C.POINTER(VolumeDesc)]),
    "pdf_resample_stats_ragged": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, C.POINTER(VolumeDesc), _P, _P, _P, _P]),
    "pdf_preprocess_ragged": (C.c_int, [C.POINTER(PreprocCfg), C.c_int, C.POINTER(VolumeDesc), _P, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "pdf_stem_padded_dims": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pdf_plan_create": (C.c_int, [C.POINTER(_P), C.POINTER(Op), C.c_int]),
    "pdf_plan_run": (C.c_int, [_P, _P]),
    "pdf_plan_run_range": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "pdf_plan_destroy": (None, [_P]),
    "pdf_plan_flops": (C.c_double, [_P]),
    "pdf_slice_mean": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_mil_workspace_bytes": (C.c_size_t, [C.POINTER(MilWeights), C.c_int, C.c_int]),
    "pdf_mil_forward": (C.c_int, [C.POINTER(MilWeights), C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "pdf_mil_sweep": (C.c_int, [C.POINTER(MilWeights), C.c_int, C.c_int, _P, _P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "pdf_mil_explain_workspace_bytes": (C.c_size_t, [C.POINTER(MilWeights), C.c_int, C.c_int]),
    "pdf_mil_explain": (C.c_int, [C.POINTER(MilWeights), C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pdf_gradcam": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_moddrop_workspace_bytes": (C.c_size_t, [C.POINTER(Mlp), C.c_int]),
    "pdf_moddrop_sweep": (C.c_int, [C.POINTER(Mlp), C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "pdf_moe_sweep": (C.c_int, [C.POINTER(Moe), C.c_int, C.c_int, C.POINTER(_P), _P, _P, _P]),
    "pdf_moddrop_explain_workspace_bytes": (C.c_size_t, [C.POINTER(Mlp), C.c_int, C.c_int, C.c_int]),
    "pdf_moddrop_explain": (C.c_int, [C.POINTER(Mlp), C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P]),
    "pdf_moe_explain_workspace_bytes": (C.c_size_t, [C.POINTER(Moe), C.c_int, C.c_int, C.c_int]),
    "pdf_moe_explain": (C.c_int, [C.POINTER(Moe), C.c_int, C.c_int, C.POINTER(_P), _P, C.c_int, _P, _P, _P, _P, C.POINTER(_P), _P]),
    "pdf_bootstrap_metrics_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "pdf_bootstrap_metrics": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_uint64, _P, _P, _P, _P, _P, _P]),
    "pdf_moddrop_mc_workspace_bytes": (C.c_size_t, [C.POINTER(Mlp), C.c_int, C.c_int, C.c_int]),
    "pdf_moddrop_mc": (C.c_int, [C.POINTER(Mlp), C.c_float, C.c_int, C.c_int, _P, _P, C.c_int, C.c_uint64, _P, _P, _P, _P]),
    "pdf_mil_mc_workspace_bytes": (C.c_size_t, [C.POINTER(MilWeights), C.c_int, C.c_int, C.c_int]),
    "pdf_mil_mc": (C.c_int, [C.POINTER(MilWeights), C.c_float, C.c_int, C.c_int, _P, _P, C.c_int, _P, C.c_int, C.c_uint64, _P, _P, _P, _P]),
    "pdf_gemm_f32": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_long, C.c_long, _P, C.c_long, C.c_long, _P, C.c_long, _P, C.c_int, C.c_int, _P]),
    "pdf_conv_dgrad_f32": (C.c_int, [C.POINTER(Op), _P, _P, _P, C.c_int, _P]),
    "pdf_conv_wgrad_f32": (C.c_int, [C.POINTER(Op), _P, _P, _P, _P]),
    "pdf_bn_train_forward": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, _P, _P, _P, C.c_float, _P, C.c_int, _P, _P, _P, _P, _P, _P]),
    "pdf_bn_train_backward": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, C.c_int, _P, _P, _P]),
    "pdf_bn_train_forward_bf16": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, _P, _P, _P, C.c_float, _P, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "pdf_bn_train_backward_bf16": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, C.c_int, _P, _P, _P]),
    "pdf_maxpool3d_forward": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_maxpool3d_backward": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_shuffle2_3d": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P]),
    "pdf_unshuffle2_3d": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P]),
    "pdf_relu_f32": (C.c_int, [_P, C.c_size_t, _P]),
    "pdf_mse_train": (C.c_int, [C.c_size_t, _P, _P, _P, _P, _P]),
    "pdf_standardize_volume": (C.c_int, [C.c_int, C.c_size_t, _P, _P, C.c_int, _P, _P]),
    "pdf_debug_set_mil_mt": (C.c_int, [C.c_int]),
    "pdf_debug_set_pw_multicast": (C.c_int, [C.c_int]),
    "pdf_debug_set_pw_prefetch": (C.c_int, [C.c_int]),
    "pdf_debug_set_wgrad_waves": (C.c_int, [C.c_int]),
    "pdf_debug_set_wgrad_rowtile": (C.c_int, [C.c_int]),
    "pdf_preproc_slice_major_ok": (C.c_int, [C.POINTER(PreprocCfg)]),
    "pdf_simple_stats_stride": (C.c_int, []),
    "pdf_simple_stats": (C.c_int, [C.c_int, C.c_size_t, C.c_int, _P, _P, _P]),
    "pdf_maxpool_train_forward_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_maxpool_backward_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_avgpool_backward_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_stem_im2col3_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_dilate2_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_scatter_add2_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_pack_conv_weights": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_bn_update_running": (C.c_int, [C.c_int, C.c_int, _P, _P, C.c_float, _P, _P, _P]),
    "pdf_maxpool_backward_f32": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_avgpool_backward_f32": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_mil_pool_train": (C.c_int, [C.POINTER(MilWeights), C.POINTER(MilTrain), C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pdf_bce_sigmoid_train": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P]),
    "pdf_moe_combine_train": (C.c_int, [C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pdf_conv_wgrad_bf16": (C.c_int, [C.POINTER(Op), _P, _P, _P, _P]),
    "pdf_cast_bf16": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "pdf_add_f32": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "pdf_dilate_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "pdf_colsum_f32": (C.c_int, [C.c_int, C.c_int, _P, _P, C.c_int, _P]),
    "pdf_relu_mask_backward": (C.c_int, [_P, _P, _P, C.c_size_t, _P]),
    "pdf_mul_f32": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "pdf_sumsq_f32": (C.c_int, [_P, C.c_size_t, _P, _P]),
    "pdf_clip_scale": (C.c_int, [_P, C.c_float, _P, _P]),
    "pdf_adam_step": (C.c_int, [_P, _P, _P, _P, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, _P, _P]),
    "pdf_gemm_f32_batched": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_long, C.c_long, C.c_long, _P, C.c_long, C.c_long, C.c_long,
                                       _P, C.c_long, C.c_long, _P, C.c_long, C.c_int, C.c_int, _P]),
    "pdf_bce_sigmoid_train_batched": (C.c_int, [C.c_int, C.c_int, _P, _P, C.c_long, _P, _P, _P, _P]),
    "pdf_moe_combine_train_batched": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_long, _P, _P, _P, _P, _P]),
    "pdf_mil_pool_train_batched_workspace_bytes": (C.c_size_t, [C.c_int, C.POINTER(MilWeights), C.c_int]),
    "pdf_mil_pool_train_batched": (C.c_int, [C.c_int, C.POINTER(MilWeights), C.c_long, C.POINTER(MilTrain), C.c_long, C.c_int, C.c_int, _P, _P,
                                             _P, _P, _P, _P, _P, _P, _P, _P]),
    "pdf_clip_scale_batched": (C.c_int, [C.c_int, _P, C.c_long, C.c_float, _P, _P]),
    "pdf_adam_step_batched": (C.c_int, [C.c_int, _P, _P, _P, _P, C.c_long, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, _P,
                                        _P, _P]),
    "pdf_ensemble_stats": (C.c_int, [C.c_int, C.c_longlong, _P, _P, _P]),
    "pdf_selftest_umma": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_selftest_umma_shift": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "pdf_selftest_umma_rate": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "pdf_debug_set_trace": (C.c_int, [_P]),
    "pdf_debug_enable_pair": (C.c_int, [C.c_int]),
    "pdf_debug_set_pre_chunk": (C.c_int, [C.c_int]),
    "pdf_debug_enable_pdl": (C.c_int, [C.c_int]),
    "pdf_debug_set_conv_probe": (C.c_int, [C.c_int]),
    "pdf_debug_set_hs_mode": (C.c_int, [C.c_int]),
    "pdf_debug_disable_halo": (C.c_int, [C.c_int]),
    "pdf_debug_set_pw": (C.c_int, [C.c_int]),
    "pdf_debug_set_sm_cap": (C.c_int, [C.c_int]),
    "pdf_debug_set_moddrop_tiled": (C.c_int, [C.c_int]),
    "pdf_debug_set_pw_config": (C.c_int, [C.c_int, C.c_int]),
}

_lib = None


class PdfusionError(RuntimeError):
    pass


def load():
    """Loads the shared library (once). Raises if it has not been built -- never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise PdfusionError(
            f"{LIB_PATH} not found: build the CUDA extension first (python __graft_entry__.py). "
            "pd_fusion_b200 has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if os.environ.get("PDFUSION_B200_PAIR"):             # tuning hook: CTA-pair (cta_group::2) kernel for Cout >= 128 layers
        lib.pdf_debug_enable_pair(int(os.environ["PDFUSION_B200_PAIR"]))
    if os.environ.get("PDFUSION_B200_HS") is not None:   # tuning hook: horizontally-shared 3x3 kernel (0 off, 1 Cout == 128, 2 all)
        lib.pdf_debug_set_hs_mode(int(os.environ["PDFUSION_B200_HS"]))
    if os.environ.get("PDFUSION_B200_CONV_PROBE"):       # timing probe (garbage outputs): see pdf_debug_set_conv_probe
        lib.pdf_debug_set_conv_probe(int(os.environ["PDFUSION_B200_CONV_PROBE"]))
    if os.environ.get("PDFUSION_B200_PW_PREFETCH") is not None:   # tuning hook: L2 prefetch of the next row tile's A operand
        lib.pdf_debug_set_pw_prefetch(int(os.environ["PDFUSION_B200_PW_PREFETCH"]))
    if os.environ.get("PDFUSION_B200_PW_MC") is not None:   # tuning hook: weight-multicast CTA pairs in the pointwise kernel (0 off)
        lib.pdf_debug_set_pw_multicast(int(os.environ["PDFUSION_B200_PW_MC"]))
    if os.environ.get("PDFUSION_B200_PW") is not None:   # tuning hook: pointwise kernel (0 off, 1 default policy, 2 every 1x1 conv)
        lib.pdf_debug_set_pw(int(os.environ["PDFUSION_B200_PW"]))
    if os.environ.get("PDFUSION_B200_PW_CFG"):           # tuning hook: "stages,staging_buffers" of the pointwise kernel
        a, b = (int(v) for v in os.environ["PDFUSION_B200_PW_CFG"].split(","))
        check_rc = lib.pdf_debug_set_pw_config(a, b)
        if check_rc != 0:
            raise PdfusionError("PDFUSION_B200_PW_CFG: " + lib.pdf_last_error().decode())
    if os.environ.get("PDFUSION_B200_NO_PDL"):           # tuning hook: plain stream-ordered launches
        lib.pdf_debug_enable_pdl(0)
    if os.environ.get("PDFUSION_B200_PRE_CHUNK"):        # tuning hook: subjects per preprocessing sub-batch (L2 residency)
        lib.pdf_debug_set_pre_chunk(int(os.environ["PDFUSION_B200_PRE_CHUNK"]))
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().pdf_last_error().decode("utf-8", "replace")
        raise PdfusionError(f"{what or 'libpdfusion_b200'} failed (rc={rc}): {msg}")


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise PdfusionError("pd_fusion_b200 needs a CUDA device (sm_100a); there is no CPU fallback.")


def stem_padded_dims(S: int):
    """(pitch, rows) of the zero-padded one-channel stem input of an S x S image (image origin at STEM_PAD_LO)."""
    pitch, rows = C.c_int(), C.c_int()
    check(load().pdf_stem_padded_dims(int(S), C.byref(pitch), C.byref(rows)), "pdf_stem_padded_dims")
    return pitch.value, rows.value


def ptr(t) -> int:
    """device pointer of a torch tensor (or None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(load().pdf_launch_count())

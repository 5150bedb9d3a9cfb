/*
 * pdfusion_b200.h -- C ABI of libpdfusion_b200.so (hand-written sm_100a CUDA kernels).
 *
 * The reference (Ardbiu/robust-multimodal-pd) has NO native/FFI boundary: its hot path is Python
 * calling numpy/scipy/torch (SURVEY.md section 8b).  Each entry point below therefore cites the
 * reference Python call site it replaces (file:line relative to the reference root); the ctypes
 * binding a maintainer would add is shown in INTEGRATION.md and implemented in
 * robust-multimodal-pd_b200/pd_fusion_b200/_lib.py.
 *
 * Conventions
 *   - plain C types only; every pointer named d_* is a DEVICE pointer owned by the caller;
 *   - every call takes the CUDA stream (cudaStream_t as void*) it enqueues on and does not
 *     synchronise (unless stated); no allocation inside except plan objects;
 *   - return value 0 = ok, negative = error; pdf_last_error() returns a thread-local message;
 *   - there is NO CPU fallback: on a machine without a CUDA device every compute call fails with
 *     PDF_ERR_CUDA.
 */
#ifndef PDFUSION_B200_H
#define PDFUSION_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDF_OK 0
#define PDF_ERR_ARG (-1)
#define PDF_ERR_CUDA (-2)
#define PDF_ERR_UNSUPPORTED (-3)

#define PDF_MAX_AXES 3

typedef void* pdf_stream_t; /* cudaStream_t */

int pdf_version(void);
const char* pdf_last_error(void);
/* number of kernel launches issued by this library in this process (bench.py: gpu_launches) */
uint64_t pdf_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * K1 -- volume -> network input.  Replaces, per subject,
 *   _load_volume                   data/openneuro_features.py:22-32   (nan_to_num + ndimage.zoom order 1)
 *   _normalize_volume_for_resnet   data/openneuro_features.py:121-132 (p1/p99 of voxels>0, clip, min-max)
 *   _select_slices                 data/openneuro_features.py:134-151 (non-zero extent, linspace indices, gather)
 *   F.interpolate + repeat + (x-mean)/std   data/openneuro_features.py:250-255
 * for a batch of `batch` raw volumes resident in HBM.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t in_shape[3];          /* raw volume X,Y,Z (C order, Z fastest) */
  int32_t out_shape[3];         /* target_shape T0,T1,T2 */
  int32_t n_axes;               /* 1..3 */
  int32_t axes[PDF_MAX_AXES];   /* slice axis per group (slice_axis / slice_axes) */
  int32_t counts[PDF_MAX_AXES]; /* requested slice_count per group */
  int32_t input_size;           /* network input side (224) */
  float mean[3];                /* per-channel mean/std of (x-mean)/std */
  float std[3];
  int32_t extent_raw;           /* 0: extent = any(normalised voxel > 0) (the fused pipeline); 1: any(voxel > 0) on the
                                   resampled volume itself (stand-alone _select_slices on an already-normalised volume) */
  int32_t slice_major;          /* 1: d_zoomed is written / read slice-axis-major, [B][T2][T0][T1], so that the selected planes of a
                                   single-axis axis-2 configuration are contiguous (no plane-gather pass; the stride-T2 gather of
                                   the C-order volume touches every sector of it).  Only where pdf_preproc_slice_major_ok() says
                                   so; pdf_gather_slices / pdf_normalize_volume take the C-order volume only.  0: [B][T0][T1][T2] */
} pdf_preproc_cfg;

/* 1 when cfg (one axis group on axis 2, bulk-copy resample tiles of eight rows: Z % 4 == 0, T1 % 8 == 0, T2 <= 160) can use
 * slice_major = 1 */
int pdf_preproc_slice_major_ok(const pdf_preproc_cfg* cfg);

/* output layouts of pdf_gather_resize_normalize */
#define PDF_OUT_BF16_C1 0 /* [B, L, S, S]    bf16, one channel (requires channel-uniform mean/std) */
#define PDF_OUT_F32_NHWC3 1 /* [B, L, S, S, 3] f32,  exact 3-channel input of the reference */
#define PDF_OUT_BF16_C1_PAD 2 /* [B, L, rows, pitch] bf16, one channel, image origin at (PDF_STEM_PAD_LO, PDF_STEM_PAD_LO) of a
                                 zero border (pdf_stem_padded_dims); the caller zeroes the buffer ONCE, the kernel only writes
                                 the image (and zeros into border pixels that share an 8-byte group with it).  Input layout of
                                 PDF_OP_STEM_FUSED. */
#define PDF_STEM_PAD_LO 5

/* pitch (elements per row, multiple of 8) and row count of the padded stem input of an S x S image */
int pdf_stem_padded_dims(int S, int* pitch, int* rows);

/* bytes of device workspace pdf_preproc_* needs for `batch` subjects (histograms, plane maxima,
 * per-subject select state, interpolation tables). */
size_t pdf_preproc_workspace_bytes(const pdf_preproc_cfg* cfg, int batch);

/* stage 1 (K1a): nan/inf scrub + trilinear resample in float64 exactly as scipy does, one rounding to
 * f32; fused: level-0 radix histogram of positive voxels and per-plane maxima along each axis.
 * d_raw [B,X,Y,Z] f32 -> d_zoomed [B,T0,T1,T2] f32. Also zeroes/initialises the workspace. */
int pdf_resample_stats(const pdf_preproc_cfg* cfg, int batch, const float* d_raw, float* d_zoomed,
                       void* d_workspace, pdf_stream_t stream);

/* stage 2 (K1b): exact order statistics for numpy.percentile(vals,1|99) by radix select on the float
 * bit patterns (two refinement passes over d_zoomed), then the numpy lerp, then (K1c) the non-zero
 * extent per requested axis from the plane maxima and the np.linspace(...).astype(int) indices.
 * d_lohi [B,4] f32 = {lo, hi, denominator (hi-lo+1e-6 as the reference rounds it), n_positive>0 ? 1 : 0};
 * d_indices [B,Lmax] i32 (Lmax = sum(counts)); d_nslices [B,n_axes] i32. */
int pdf_select_bounds_indices(const pdf_preproc_cfg* cfg, int batch, const float* d_zoomed, void* d_workspace,
                              float* d_lohi, int32_t* d_indices, int32_t* d_nslices, pdf_stream_t stream);

/* stage 3 (K1d): gather the selected planes, clip/min-max with lo/hi, bilinear resize to input_size
 * (align_corners=False), (x-mean)/std, write the network input in `out_mode` layout.  Slots beyond
 * d_nslices are zero-filled.  d_workspace: the same workspace (holds the compact axis-2 plane buffer). */
int pdf_gather_resize_normalize(const pdf_preproc_cfg* cfg, int batch, const float* d_zoomed, void* d_workspace,
                                const float* d_lohi, const int32_t* d_indices, const int32_t* d_nslices, void* d_out,
                                int out_mode, pdf_stream_t stream);

/* the three stages back to back on `stream` */
int pdf_preprocess(const pdf_preproc_cfg* cfg, int batch, const float* d_raw, float* d_zoomed, void* d_workspace,
                   float* d_lohi, int32_t* d_indices, int32_t* d_nslices, void* d_out, int out_mode,
                   pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * f4 -- the "simple" feature mode.  Replaces `_compute_simple_features` (data/openneuro_features.py:34-73): over vals =
 * volume[volume > 0] (all voxels when none is positive) mean / std / min / max, np.median, np.percentile 10 / 90 / 1 / 99 (exact
 * order statistics, numpy's float32 'linear' rule), the counts of np.histogram(np.clip(vals, p1, p99), bins, range=(p1, p99)) with
 * its float32 edges, and the central-moment sums behind scipy.stats.skew / kurtosis.  The grid means of the same function are a
 * second trilinear zoom: pdf_resample_stats with out_shape = grid.  d_vol [batch, voxels] f32 (a resampled volume each);
 * d_out: batch * pdf_simple_stats_stride() doubles, per subject
 *   0 n | 1 sum | 2 min | 3 max | 4..6 sum (v-mean)^2,3,4 | 7 median | 8 p10 | 9 p90 | 10 p1 | 11 p99 | 12 all-voxel fallback flag |
 *   16 .. counts[hist_bins] | 16+hist_bins .. edges[hist_bins+1].
 * ------------------------------------------------------------------------------------------ */
int pdf_simple_stats_stride(void);
int pdf_simple_stats(int batch, size_t voxels, int hist_bins, const float* d_vol, double* d_out, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * f4 -- the "cnn3d" feature mode (scripts/build_cnn3d_embeddings.py:28-88, 132-156): pieces of the 3-D conv auto-encoder that are not
 * a 2-D kernel already.  Channels-last [N, D, H, W, C] f32.  The 3x3x3 convolutions run depth-decomposed through the FP32 2-D
 * kernels (pdf_plan_* with residual accumulation, pdf_conv_dgrad_f32, pdf_conv_wgrad_f32), the 2x2x2 stride-2 transposed
 * convolutions as pdf_gemm_f32 + pixel shuffle.
 * pdf_maxpool3d_forward: MaxPool3d(2) with the winner's position (i*4+j*2+k, first maximum in scan order) -> d_idx u8; backward
 *   scatters through it.  pdf_shuffle2_3d: y[n,2d+i,2h+j,2w+k,co] = act(t[v,(i*4+j*2+k)*cout+co] + bias[co]); pdf_unshuffle2_3d: its
 *   backward (ReLU mask from d_y).  pdf_mse_train: d_loss[0] += mean (p-t)^2, d_dpred (or NULL) = 2(p-t)/n.
 * pdf_standardize_volume: load_volume's (v - mean) / (std + 1e-6) over the positive voxels (statistics rows of pdf_simple_stats;
 *   volumes without a positive voxel pass through).
 * ------------------------------------------------------------------------------------------ */
int pdf_maxpool3d_forward(int n, int d, int h, int w, int c, const float* d_x, float* d_y, uint8_t* d_idx, pdf_stream_t stream);
int pdf_maxpool3d_backward(int n, int d, int h, int w, int c, const uint8_t* d_idx, const float* d_dy, float* d_dx, pdf_stream_t stream);
int pdf_shuffle2_3d(int n, int d, int h, int w, int cout, const float* d_t, const float* d_bias, int relu, float* d_y, pdf_stream_t stream);
int pdf_unshuffle2_3d(int n, int d, int h, int w, int cout, const float* d_dy, const float* d_y, int relu, float* d_dt, pdf_stream_t stream);
int pdf_relu_f32(float* d_x, size_t n, pdf_stream_t stream);
int pdf_mse_train(size_t n, const float* d_pred, const float* d_target, float* d_loss, float* d_dpred, pdf_stream_t stream);
int pdf_standardize_volume(int batch, size_t voxels, const float* d_x, const double* d_stats, int stats_stride, float* d_y,
                           pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a6 -- test-time augmentation (`tta > 1`): data/openneuro_features.py:166-178,235-248 and
 * scripts/build_resnet2d_mil_embeddings.py:124-146.  The random draws (angle, translation, scale, shift and the
 * N(0, sigma) field) are made ON THE HOST with the reference's exact numpy calls and passed in as data; the
 * affine resampling, intensity map, noise add and clip run here.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  double rot[4];    /* row-major 2x2 matrix handed to scipy.ndimage.affine_transform */
  double offset[2]; /* its offset = center - rot @ center + translate */
  float scale;      /* 1 + U(-intensity_scale, intensity_scale), rounded to float32 as numpy does */
  float shift;
} pdf_tta_params;

/* `_select_slices` of the normalised volume for every requested axis group, concatenated: d_slices [B, Lmax, H, W] f32
 * (slots beyond d_nslices are zero).  All groups must share one slice shape. */
int pdf_gather_slices(const pdf_preproc_cfg* cfg, int batch, const float* d_zoomed, const float* d_lohi,
                      const int32_t* d_indices, const int32_t* d_nslices, float* d_slices, pdf_stream_t stream);
/* one augmentation pass: d_params [B]; d_noise [B, L, H, W] f64 or NULL (noise_std == 0); d_out [B, L, H, W] f32.
 * affine_only != 0: stop after the affine resampling (`_apply_affine_2d` itself: no intensity map, noise or clip). */
int pdf_tta_augment(int batch, int L, int H, int W, const float* d_slices, const pdf_tta_params* d_params,
                    const double* d_noise, int affine_only, float* d_out, pdf_stream_t stream);
/* bilinear resize (align_corners=False) + (x-mean)/std of ready-made slices in [0,1] -> network input in `out_mode` layout */
int pdf_resize_slices(int batch, int L, int H, int W, int input_size, const float* mean, const float* std,
                      const float* d_slices, void* d_out, int out_mode, pdf_stream_t stream);

/* Stored NIfTI-1 voxels -> the float32 array `nib.load(p).get_fdata().astype(np.float32)` gives the reference
 * (data/openneuro_features.py:24-25), on the device: float64(raw) [* slope + inter when nibabel would scale] -> float32, written
 * C-order [B, X, Y, Z].  nifti_datatype: 2 u8, 4 i16, 8 i32, 16 f32, 64 f64, 256 i8, 512 u16, 768 u32.  fortran_order != 0: the
 * source is x-fastest as in the file (tiled transpose), else already C-order.  d_src / d_dst must not overlap. */
int pdf_decode_volume(int batch, int nifti_datatype, int X, int Y, int Z, int fortran_order, double slope, double inter,
                      const void* d_src, float* d_dst, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Ragged batches: subjects of any raw shape, stored type, byte order and scaling in one batch.  Every stage after the resample
 * works on the target grid, so only decode and resample need per-subject geometry.  The raw volumes are packed one after the
 * other in one float32 buffer (C order [X][Y][Z] each, starting at 16-byte aligned offsets); the descriptors are a HOST array
 * of `batch` entries and reach the kernels as a by-value kernel parameter, so batch <= PDF_RAGGED_MAX_BATCH.
 * ------------------------------------------------------------------------------------------ */
#define PDF_RAGGED_MAX_BATCH 64
typedef struct {
  int32_t shape[3];       /* X, Y, Z of the raw volume */
  int32_t nifti_datatype; /* decode only: 2, 4, 8, 16, 64, 256, 512, 768 as pdf_decode_volume */
  int32_t fortran_order;  /* decode only */
  int32_t pad;
  int64_t src_offset;     /* decode only: bytes into d_src (a multiple of the stored element size) */
  int64_t raw_offset;     /* float32 elements into the packed raw buffer; multiple of 4 (16-byte aligned rows) */
  double slope, inter;    /* decode only: nibabel's scaling rule, as pdf_decode_volume */
} pdf_volume_desc;

/* stored voxels of mixed type, order and scaling -> the packed float32 buffer, one launch (same arithmetic as pdf_decode_volume) */
int pdf_decode_volumes(int batch, const pdf_volume_desc* descs, const void* d_src, float* d_dst, pdf_stream_t stream);
/* workspace of the ragged entry points: the uniform workspace of `batch` subjects followed by one interpolation table per subject
 * (pdf_select_bounds_indices, pdf_gather_* and pdf_normalize_volume then work on the same workspace unchanged).  cfg->in_shape is
 * not read by the ragged entry points. */
size_t pdf_preproc_ragged_workspace_bytes(const pdf_preproc_cfg* cfg, int batch);
/* 1 when every subject of the batch can be resampled slice-major (see pdf_preproc_slice_major_ok); a batch with one ineligible
 * subject runs C-order as a whole */
int pdf_preproc_slice_major_ok_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs);
/* pdf_resample_stats / pdf_preprocess with per-subject raw geometry: d_raw is the packed buffer, descs[b].shape / raw_offset
 * place subject b.  Same outputs, bit for bit, as the uniform entry points on each subject. */
int pdf_resample_stats_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs, const float* d_raw,
                              float* d_zoomed, void* d_workspace, pdf_stream_t stream);
int pdf_preprocess_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs, const float* d_raw, float* d_zoomed,
                          void* d_workspace, float* d_lohi, int32_t* d_indices, int32_t* d_nslices, void* d_out, int out_mode,
                          pdf_stream_t stream);

/* normalised volume itself (parity helper for _normalize_volume_for_resnet): d_zoomed -> d_norm */
int pdf_normalize_volume(int batch, size_t voxels, const float* d_zoomed, const float* d_lohi, float* d_norm,
                         pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K2 -- ResNet2D encoder.  Replaces `model(batch)` on torchvision resnet18/50 with fc=Identity in
 * eval mode (data/openneuro_features.py:153-164,257-262; scripts/build_resnet2d_mil_embeddings.py:148-156).
 * The host folds BatchNorm (eval) and describes the network as a flat list of ops over NHWC buffers.
 * ------------------------------------------------------------------------------------------ */
#define PDF_OP_CONV 0        /* implicit-GEMM convolution (+bias/scale, +residual, +ReLU) */
#define PDF_OP_MAXPOOL 1     /* 3x3 stride 2 pad 1 */
#define PDF_OP_AVGPOOL 2     /* global average over H*W -> [N, C] f32 */
#define PDF_OP_STEM_IM2COL 3 /* [N,H,W] bf16 one-channel image -> [N*Ho*Wo, kpad] bf16 patch matrix (7x7 s2 p3) */
#define PDF_OP_STEM_FUSED 4  /* zero-padded [N,rows,pitch] bf16 image (PDF_OUT_BF16_C1_PAD; h = w = S) -> conv 7x7 s2 p3 (64 ch) + bias
                                + ReLU + maxpool 3x3 s2 p1 -> [N,ho,wo,64] bf16, one kernel.  d_weight: [128][128] bf16, row v*64+c,
                                column t*8+s = w[c][t-4v][s] (BN folded, 3 input channels summed), columns 88 and 89 = the bias of channel c split
                                into two bf16 terms (they multiply a constant 1; d_bias is not read), zero elsewhere.
                                d_scale: NULL, or a border-correction blob for inputs whose (x-mean)/std is PER CHANNEL (the one
                                channel fed to the kernel is then (x-mean_avg)/std_avg and the per-channel offsets become a bias that
                                depends on how much of the 7x7 window lies inside the image):
                                  int32 n_classes, int32 h1, int32 cls[h1], float delta[n_classes][n_classes][64]
                                delta[cls[row]][cls[col]][k] is added to channel k of conv pixel (row, col); class 0 = interior */

#define PDF_PREC_F32 0  /* CUDA-core FFMA path, 1e-5 parity */
#define PDF_PREC_BF16 1 /* tcgen05/TMEM path, bf16 operands, f32 accumulate */
#define PDF_PREC_TF32 2 /* tcgen05/TMEM path on float32 operands (kind::tf32: 10-bit mantissa products, f32 accumulate): MIL head */

typedef struct {
  int32_t kind;
  int32_t precision;
  int32_t n, h, w, c;  /* input tensor NHWC */
  int32_t k, r, s;     /* output channels, filter height/width */
  int32_t stride, pad;
  int32_t ho, wo;      /* output spatial size */
  int32_t relu;
  int32_t out_f32;     /* bf16 path only: store the output tile as f32 instead of bf16 */
  /* bf16 1x1 stride-1 PDF_OP_CONV only, 0 otherwise: the projection shortcut of a ResNet Bottleneck (downsample conv1x1 + BN of the
   * block input x, torchvision resnet.py Bottleneck.forward) computed as more K of this convolution:
   * d_out = relu?(conv1x1([d_in | x_s], d_weight) + d_bias), x_s = x at stride 1 if (sc_h, sc_w) == (ho, wo), else at stride 2
   * (then ho == (sc_h-1)/2+1, wo == (sc_w-1)/2+1).  With sc_c != 0, d_residual points at x [N, sc_h, sc_w, sc_c] bf16 (nothing is
   * added), d_weight is [K][c + sc_c] bf16 (this conv's columns, then the shortcut's; both BN folded), d_bias the sum of both biases;
   * c % 64 == 0, sc_c % 64 == 0.  sc_hw = (sc_h << 16) | sc_w. */
  int32_t sc_c;
  const void* d_in;
  const void* d_weight;   /* f32 path: [R][S][C][K] f32 ; bf16 path: [K][R][S][C] bf16, BN folded */
  const float* d_scale;   /* f32 path: per-channel BN scale (NULL = 1) */
  const float* d_bias;    /* per-channel bias / BN shift (NULL = 0) */
  const void* d_residual; /* same layout/dtype as the (bf16|f32) output, or NULL */
  void* d_out;
  /* bf16 PDF_OP_CONV only, all three NULL otherwise: a 1x1 convolution of the SAME input with the same stride and Cout (a ResNet
   * BasicBlock's downsample next to its 3x3 pad-1 conv1 -- torchvision resnet.py BasicBlock.forward) computed in the same launch from
   * the centre-tap tiles.  d_weight2 [K][C] bf16 (BN folded), d_bias2 [K] f32 or NULL, d_out2 [N,ho,wo,K] bf16 (no ReLU). */
  const void* d_weight2;
  const float* d_bias2;
  void* d_out2;
  /* bf16 1x1 PDF_OP_CONV only, all NULL / 0 otherwise: the NEXT 1x1 convolution, chained while the output tile is still on chip
   * (a ResNet Bottleneck's conv3 + bn3 + add + relu followed by the next block's conv1 + bn1 + relu -- torchvision resnet.py
   * Bottleneck.forward): d_out3 [N,ho,wo,k3] bf16 = relu(conv1x1(d_out, d_weight3) + d_bias3).  d_weight3 [k3][K] bf16 (BN folded),
   * k3 in {64, 128, 256}, K % 128 == 0.  d_out is still written (it is the next block's residual). */
  const void* d_weight3;
  const float* d_bias3;
  void* d_out3;
  int32_t k3;
  int32_t sc_hw;       /* shortcut input's spatial size (sc_h << 16) | sc_w, see sc_c */
} pdf_op;

typedef struct pdf_plan pdf_plan; /* opaque: validated ops + pre-encoded TMA descriptors */

/* validates shapes, encodes the CUtensorMaps of every bf16 conv (needs a CUDA context). */
/* tuning / A-B hook for the pointwise kernel (conv_pw.cu): 0 = 1x1 convolutions stay on the generic kernel, 1 = default
 * policy, 2 = every eligible 1x1 convolution.  Affects plans created afterwards. */
int pdf_debug_set_pw(int mode);
int pdf_debug_set_pw_prefetch(int enable);    /* pointwise kernel: L2 prefetch of the next row tile's A operand (default 0) */
int pdf_debug_set_pw_multicast(int enable);   /* pointwise kernel: weight-multicast CTA pairs for Cin >= 128 (default 0: measured neutral) */
int pdf_debug_set_wgrad_rowtile(int enable);   /* wgrad_tc: 0 = im2col-mode loads for every filter > 1x1 (default 1: row-tiled) */
int pdf_debug_set_wgrad_waves(int waves);  /* wgrad_tc: CTA waves the pixel range is split into (default 1) */
int pdf_debug_set_mil_mt(int row_tiles);   /* MIL tf32 GEMMs: row tiles per weight pass (0 = by batch size, 1, 2) */
/* persistent kernels size their grids for `cap` SMs instead of the device's (0 = off): two streams can then share the GPU */
int pdf_debug_set_sm_cap(int cap);
/* A/B hook: 0 = warp-per-pair ModDrop kernel at every size, 1 (default) = tiled in-block GEMM kernel from 4096 (scenario, subject) pairs up */
int pdf_debug_set_moddrop_tiled(int enable);
/* ring depth (2..6) and staging-buffer count (2..4) of conv_pw_kernel launches (the ring shrinks to what fits 227 KB) */
int pdf_debug_set_pw_config(int stages, int staging_buffers);
int pdf_plan_create(pdf_plan** out, const pdf_op* ops, int n_ops);
int pdf_plan_run(const pdf_plan* plan, pdf_stream_t stream);
/* runs ops [first, first+count) only (per-layer timing / debugging) */
int pdf_plan_run_range(const pdf_plan* plan, int first, int count, pdf_stream_t stream);
void pdf_plan_destroy(pdf_plan* plan);
/* algorithmic FLOPs (2*MAC over conv ops) of one pdf_plan_run */
double pdf_plan_flops(const pdf_plan* plan);

/* mean over the valid slices of each subject: d_emb [B, L, D] f32 -> d_out [B, D] f32
 * (`torch.cat(feats).mean(dim=0)`, data/openneuro_features.py:262).  d_nslices: valid count per subject
 * (sum over axes), or NULL for L. */
int pdf_slice_mean(int batch, int L, int D, const float* d_emb, const int32_t* d_nvalid, float* d_out, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3 -- MIL attention head.  Replaces MILAttentionNet.forward + the per-bag loop of
 * MilAttentionModel.predict_proba (models/mil_attention.py:40-51,157-178) for ALL bags in one launch.
 * d_bags [n_bags, Lmax, D] f32, d_len [n_bags] i32 (0 = missing bag -> missing_prob).
 * Weights are the state_dict tensors, row-major as torch stores them:
 *   w_inst [H,D], b_inst [H]; gated: w_v [A,H], b_v [A], w_u [A,H], b_u [A], w_w [A], b_w [1]
 *   non-gated: w_v = attn.0.weight, b_v = attn.0.bias, w_w = attn.2.weight, b_w = attn.2.bias, w_u = NULL
 *   w_cls [H], b_cls [1].   d_prob [n_bags] f32.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t D, H, A, gated;
  const float *w_inst, *b_inst, *w_v, *b_v, *w_u, *b_u, *w_w, *b_w, *w_cls, *b_cls;
  float missing_prob;
} pdf_mil_weights;

size_t pdf_mil_workspace_bytes(const pdf_mil_weights* w, int n_bags, int Lmax);
/* The MIL head under EVERY scenario in one call (evaluation/evaluate.py:32-37 sets a bag to None where the scenario drops mri and
 * calls predict_proba once per scenario; the bag's probability itself does not depend on the scenario): instance projection and
 * attention layers ONCE over all bags, softmax-pool + classifier once per bag, then
 *   d_prob[s, b] = (d_live[s, b] && d_len[b] > 0) ? p_b : missing_prob          d_live [n_scenarios, n_bags] u8 or NULL (all live).
 * precision PDF_PREC_F32: FFMA GEMMs (<= 5e-6 vs the reference); PDF_PREC_TF32: both linear layers as tcgen05 kind::tf32 GEMMs on
 * the f32 bags (needs H, (2)A in {64,128,256}, D % 32 == 0, H % 32 == 0, and for the gated head w_u == w_v + A*H, b_u == b_v + A,
 * i.e. [W_v; W_u] packed as one matrix), attention scores computed in the GEMM epilogue. */
int pdf_mil_sweep(const pdf_mil_weights* w, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len, int n_scenarios,
                  const uint8_t* d_live, int precision, void* d_workspace, float* d_prob, pdf_stream_t stream);
int pdf_mil_forward(const pdf_mil_weights* w, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len,
                    void* d_workspace, float* d_prob, pdf_stream_t stream);

/* Explanations of the MIL head (csrc/explain.cu), always with the FP32 arithmetic of pdf_mil_sweep's PDF_PREC_F32 path, also for a
 * model that predicts with PDF_PREC_TF32.  For every bag: d_logit [n_bags] = w_cls . sum_l a_l h_l + b_cls, pooled in the order of
 * the sweep's pooling kernel (sigmoid(logit) is its probability; NaN for a bag with d_len 0); d_attn [n_bags, Lmax] = the attention
 * weights a_l; d_contrib [n_bags, Lmax] = a_l (w_cls . h_l), so sum_l contrib + b_cls = logit (both 0 on the padding).
 * d_dx [n_bags, Lmax, D] or NULL: the gradient of the logit (dz = 1, not of a loss) with respect to every instance, 0 on the padding
 * and for missing bags.  Workspace: pdf_mil_explain_workspace_bytes. */
size_t pdf_mil_explain_workspace_bytes(const pdf_mil_weights* w, int n_bags, int Lmax);
int pdf_mil_explain(const pdf_mil_weights* w, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len, void* d_workspace,
                    float* d_logit, float* d_attn, float* d_contrib, float* d_dx /* [n_bags, Lmax, D] or NULL */, pdf_stream_t stream);
/* Grad-CAM at a feature map whose spatial mean is the embedding: d_fmap [n, hw, hw, c] f32 (c % 4 == 0, 16-byte aligned),
 * d_g [n, c] = the gradient of the logit with respect to the embedding.
 *   cam_small[n, i, j] = ReLU(sum_c g[n, c] fmap[n, i, j, c] / hw^2)      (d_cam_small [n, hw, hw] or NULL)
 *   cam[n, out_h, out_w] = bilinear upsample of cam_small, align_corners=False (ATen's source-index rule).  hw <= 64. */
int pdf_gradcam(int n, int hw, int c, const float* d_fmap, const float* d_g, int out_h, int out_w,
                float* d_cam_small /* [n, hw, hw] or NULL */, float* d_cam /* [n, out_h, out_w] */, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K5 -- training (FP32, NHWC).  Replaces torch autograd under MilAttentionFineTuneModel.train / _forward_bags
 * (models/mil_attention_finetune.py:135-162,164-253: backbone in TRAIN mode, BatchNorm statistics per 16-slice chunk, MIL head,
 * BCE / focal loss, backward, clip_grad_norm_, Adam) and under the heads' train loops (models/mil_attention.py:88-155,
 * fusion_moddrop.py:69-91, moe.py:60-70).  The host walks the layer list in reverse (pd_fusion_b200/training.py).
 * ------------------------------------------------------------------------------------------ */
/* C[M,N] (+)= act(sum_k A(i,k) B(k,j) + bias[j]); A(i,k) = A[i*a_rs + k*a_cs], B(k,j) = B[k*b_rs + j*b_cs]; act 1 = ReLU.
 * One entry point for x W^T (forward), dy W (dgrad) and dy^T x (wgrad) of the linear layers. */
int pdf_gemm_f32(int M, int N, int K, const float* A, long a_rs, long a_cs, const float* B, long b_rs, long b_cs, float* C, long c_rs,
                 const float* bias, int act, int accumulate, pdf_stream_t stream);
/* convolution backward; geometry from `op` (n,h,w,c,k,r,s,stride,pad,ho,wo), weights [R][S][C][K] f32 as the FP32 forward path:
 * dgrad d_dx [n,h,w,c] (+)= conv^T(d_dy [n,ho,wo,k], w);  wgrad d_dw [R][S][C][K] += x^T * dy (accumulates: zero it first). */
int pdf_conv_dgrad_f32(const pdf_op* op, const float* d_dy, const float* d_weight, float* d_dx, int accumulate, pdf_stream_t stream);
int pdf_conv_wgrad_f32(const pdf_op* op, const float* d_x, const float* d_dy, float* d_dw, pdf_stream_t stream);
/* train-mode BatchNorm over row groups of the [M, C] activation matrix: group g = rows [d_goff[g], d_goff[g+1]) (one 16-slice chunk
 * of one bag); max_group_rows = the longest group (sizes the reduction grid).  forward: y = (x - mean_g) * invstd_g * gamma + beta
 * (+ residual) (ReLU); saves mean, invstd (biased variance, eps inside) and the unbiased variance (for the running statistics) per
 * (group, channel).  d_scratch: 3 * n_groups * C doubles (float64 partial sums of the slab-split reductions).
 * backward: g = d_dy * (d_y > 0 if relu); d_dgamma += sum g*xhat, d_dbeta += sum g (accumulate over calls: zero first);
 * d_dx = gamma*invstd*(g - mean_g(g) - xhat*mean_g(g*xhat)); d_dres (or NULL) (+)= g, the gradient of the residual branch.
 * Two storage types: f32 (C % 4 == 0; the FP32 parity path) and bf16 (C % 8 == 0; x, residual, y, dy, dx, dres are bf16, everything
 * computed in f32 / f64 -- the tensor-core path, csrc/train_bf16.cu). */
int pdf_bn_train_forward(int n_groups, const int32_t* d_goff, int max_group_rows, int C, const float* d_x, const float* d_gamma,
                         const float* d_beta, float eps, const float* d_residual, int relu, float* d_y, float* d_mean, float* d_invstd,
                         float* d_var_unbiased, double* d_scratch, pdf_stream_t stream);
int pdf_bn_train_backward(int n_groups, const int32_t* d_goff, int max_group_rows, int C, const float* d_dy, const float* d_y,
                          const float* d_x, const float* d_gamma, const float* d_mean, const float* d_invstd, int relu, double* d_scratch,
                          float* d_dx, float* d_dres, int dres_accumulate, float* d_dgamma, float* d_dbeta, pdf_stream_t stream);
/* (bf16 storage: the forward also writes the ReLU mask as ONE BIT per element, d_relu_mask [M*C/8] bytes, bit j of byte i = element
 *  8i+j survived; the backward reads it instead of y -- 1/16 of the bytes) */
int pdf_bn_train_forward_bf16(int n_groups, const int32_t* d_goff, int max_group_rows, int C, const void* d_x, const float* d_gamma,
                              const float* d_beta, float eps, const void* d_residual, int relu, void* d_y, uint8_t* d_relu_mask,
                              float* d_mean, float* d_invstd, float* d_var_unbiased, double* d_scratch, pdf_stream_t stream);
int pdf_bn_train_backward_bf16(int n_groups, const int32_t* d_goff, int max_group_rows, int C, const void* d_dy,
                               const uint8_t* d_relu_mask, const void* d_x, const float* d_gamma, const float* d_mean, const float* d_invstd, int relu,
                               double* d_scratch, void* d_dx, void* d_dres, int dres_accumulate, float* d_dgamma, float* d_dbeta,
                               pdf_stream_t stream);
/* running = (1-momentum)*running + momentum*batch, group after group (the reference forwards its chunks one at a time) */
int pdf_bn_update_running(int n_groups, int C, const float* d_mean, const float* d_var_unbiased, float momentum, float* d_running_mean,
                          float* d_running_var, pdf_stream_t stream);
int pdf_maxpool_backward_f32(int n, int h, int w, int c, const float* d_x, const float* d_dy, float* d_dx, pdf_stream_t stream);
int pdf_avgpool_backward_f32(int n, int hw, int c, const float* d_demb, float* d_dx, pdf_stream_t stream);
/* bf16 storage (c % 8 == 0): x, y, dy, dx bf16; the training-mode max pool records the winning window position (r*3+s of the first
 * maximum, u8 [n,ho,wo,c]) and its backward gathers through it; the average pool's incoming gradient d_demb stays f32 */
int pdf_maxpool_train_forward_bf16(int n, int h, int w, int c, const void* d_x, void* d_y, uint8_t* d_idx, pdf_stream_t stream);
int pdf_maxpool_backward_bf16(int n, int h, int w, int c, const uint8_t* d_idx, const void* d_dy, void* d_dx, pdf_stream_t stream);
int pdf_avgpool_backward_bf16(int n, int hw, int c, const float* d_demb, void* d_dx, pdf_stream_t stream);
/* MIL head, training: everything after the linear layers, forward AND backward, in one kernel (one block per bag).
 * d_h [n_bags*Lmax, H] = dropout(relu(instance(x))); d_vu [n_bags*Lmax, NA] = attention pre-activations incl. bias (NA = 2A gated: v|u).
 * Writes d_prob [n_bags], adds the batch-mean loss to d_loss[0], writes d_dh (pooling path only) and d_dvu, and ACCUMULATES the
 * gradients of attn_w / classifier into the pdf_mil_train pointers.  loss_type 0: BCE * (pos_weight for y >= 0.5), 1: focal. */
typedef struct {
  int32_t loss_type;
  float pos_weight, focal_gamma, focal_alpha; /* focal_alpha < 0: no alpha term */
  float *d_w_w, *d_b_w, *d_w_cls, *d_b_cls;   /* gradient accumulators [A], [1], [H], [1] */
} pdf_mil_train;
int pdf_mil_pool_train(const pdf_mil_weights* w, const pdf_mil_train* t, int n_bags, int Lmax, const float* d_h, const float* d_vu,
                       const int32_t* d_len, const float* d_target, float* d_prob, float* d_loss, float* d_dh, float* d_dvu,
                       pdf_stream_t stream);
/* heads (models/fusion_moddrop.py:69-91, models/moe.py:60-70): Sigmoid + nn.BCELoss (mean) forward and d loss / d logit in one launch;
 * MoE: out = sum_e sigmoid(z[:,e]) * softmax(r)[:,e], BCE(out, y), gradients of the expert logits z and the router logits r */
int pdf_bce_sigmoid_train(int n, const float* d_z, const float* d_y, float* d_prob, float* d_loss, float* d_dz, pdf_stream_t stream);
int pdf_moe_combine_train(int n, int n_experts, const float* d_z, const float* d_r, const float* d_y, float* d_out, float* d_loss,
                          float* d_dz, float* d_dr, pdf_stream_t stream);
/* tensor-core training path (bf16 operands, f32 accumulation and f32 results):
 * pdf_conv_wgrad_bf16: weight gradient as a tcgen05 GEMM over pixels with MN-major operands (csrc/wgrad_tc.cu); d_x [n,h,w,c] bf16,
 *   d_dy [n,ho,wo,k] bf16, d_dw [k][r][s][c] f32 ACCUMULATED into; c % 64 == 0, k % 64 == 0.
 * data gradients run through pdf_plan_* (the forward implicit-GEMM kernels on rotated weights); for strided convolutions the host
 *   first builds pdf_dilate_bf16's zero-dilated copy of dY ([n,hd,wd,k] bf16, dY[p,q] at (offset + p*stride, offset + q*stride)). */
int pdf_conv_wgrad_bf16(const pdf_op* op, const void* d_x, const void* d_dy, float* d_dw, pdf_stream_t stream);
int pdf_cast_bf16(const float* d_x, void* d_y, size_t n, pdf_stream_t stream);
int pdf_add_f32(float* d_x, const float* d_y, size_t n, pdf_stream_t stream);
int pdf_dilate_bf16(int n, int ho, int wo, int k, int hd, int wd, int stride, int offset, const float* d_dy, void* d_out, pdf_stream_t stream);
/* tensor-core path helpers (csrc/train_bf16.cu):
 * pdf_stem_im2col3_bf16: f32 NHWC3 network input [n,h,w,3] -> bf16 patch matrix [n*ho*wo, 192] of the 7x7 s2 p3 stem (column
 *   (r*7+s)*3+ch, columns 147..191 zero): conv1's forward and weight gradient become 1x1 tensor-core GEMMs (c = 192, k = 64);
 * pdf_dilate2_bf16: zero-dilated copy [n,hd,wd,k] of a bf16 dY [n,ho,wo,k] (dY[p,q] at (2p,2q)): data gradient of a stride-2 3x3 conv;
 * pdf_scatter_add2_bf16: d_dx[n,2p,2q,:] += d_t[n,p,q,:] (bf16): data gradient of a stride-2 1x1 conv after its GEMM on dY;
 * pdf_pack_conv_weights: f32 [K,C,R,S] (torchvision) -> bf16 [K][R][S][C] and (d_wrot may be NULL) bf16 [C][R][S][K] with the taps
 *   rotated by 180 degrees, the operand of the data-gradient convolution. */
int pdf_stem_im2col3_bf16(int n, int h, int w, const float* d_x, void* d_out, pdf_stream_t stream);
int pdf_dilate2_bf16(int n, int ho, int wo, int k, int hd, int wd, const void* d_src, void* d_out, pdf_stream_t stream);
int pdf_scatter_add2_bf16(int n, int ho, int wo, int c, int h, int w, const void* d_t, void* d_dx, pdf_stream_t stream);
int pdf_pack_conv_weights(int k, int c, int r, int s, const float* d_w, void* d_wk, void* d_wrot, pdf_stream_t stream);
int pdf_colsum_f32(int M, int N, const float* d_x, float* d_out, int accumulate, pdf_stream_t stream);
/* in place: grad *= (act > 0) * mask   (ReLU + inverted-dropout backward; mask NULL = no dropout) */
int pdf_relu_mask_backward(float* d_grad, const float* d_act, const float* d_mask, size_t n, pdf_stream_t stream);
int pdf_mul_f32(float* d_x, const float* d_m, size_t n, pdf_stream_t stream);
/* clip_grad_norm_ + Adam (torch.optim.Adam, L2-style weight decay): d_acc[0] += sum x^2; scale = min(1, max_norm/(norm+1e-6)) */
int pdf_sumsq_f32(const float* d_x, size_t n, float* d_acc, pdf_stream_t stream);
int pdf_clip_scale(const float* d_sumsq, float max_norm, float* d_out2, pdf_stream_t stream);
int pdf_adam_step(float* d_param, const float* d_grad, float* d_m, float* d_v, size_t n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int step, const float* d_grad_scale, pdf_stream_t stream);

/* Deep ensembles: the training kernels above for n_members (1..1024) heads of one architecture in one launch (the statistics:
 * csrc/uncertainty.cu).
 * Member e of an operand starts e * (its member stride, in elements) after member 0; stride 0 = shared by every member.  Per member
 * the results are those of the single kernels: pdf_gemm_f32_batched bit for bit; the loss kernels' elementwise outputs (prob, dz, dr,
 * dh, dvu) bit for bit, their losses and parameter gradients reduced in a fixed order (no atomics), so calls are bit-identical and a
 * member's results do not depend on the other members.  Null or misaligned pointers and bad sizes return PDF_ERR_ARG before any
 * device work.
 * pdf_bce_sigmoid_train_batched: d_z, d_prob, d_dz [E, n], d_y member stride y_es; d_loss [E] WRITTEN (the member's mean BCE).
 * pdf_moe_combine_train_batched: d_z, d_r, d_dz, d_dr [E, n, n_experts], d_out [E, n], d_y member stride y_es, d_loss [E] written.
 * pdf_mil_pool_train_batched: w / t hold member 0's head weights and gradient accumulators, member e's are w_es / g_es floats further;
 *   d_h [E, n_bags*Lmax, H], d_vu [E, n_bags*Lmax, NA], d_len, d_target, d_prob [E, n_bags]; gradients ACCUMULATED (each the sum over
 *   bags in bag order), d_loss [E] written; workspace pdf_mil_pool_train_batched_workspace_bytes.
 * pdf_clip_scale_batched: d_scale[e] = min(1, max_norm / (||row e of d_grad [E, n_params]|| + 1e-6)), clip_grad_norm_ per member.
 * pdf_adam_step_batched: pdf_adam_step over [E, n_params] with member e's gradient scaled by d_grad_scale[e] (NULL = 1); a member
 *   whose d_active[e] is 0 keeps its parameters and moments (d_active NULL = all active). */
int pdf_gemm_f32_batched(int n_members, int M, int N, int K, const float* A, long a_rs, long a_cs, long a_es, const float* B, long b_rs,
                         long b_cs, long b_es, float* C, long c_rs, long c_es, const float* bias, long bias_es, int act, int accumulate,
                         pdf_stream_t stream);
int pdf_bce_sigmoid_train_batched(int n_members, int n, const float* d_z, const float* d_y, long y_es, float* d_prob, float* d_loss,
                                  float* d_dz, pdf_stream_t stream);
int pdf_moe_combine_train_batched(int n_members, int n, int n_experts, const float* d_z, const float* d_r, const float* d_y, long y_es,
                                  float* d_out, float* d_loss, float* d_dz, float* d_dr, pdf_stream_t stream);
size_t pdf_mil_pool_train_batched_workspace_bytes(int n_members, const pdf_mil_weights* w, int n_bags);
int pdf_mil_pool_train_batched(int n_members, const pdf_mil_weights* w, long w_es, const pdf_mil_train* t, long g_es, int n_bags, int Lmax,
                               const float* d_h, const float* d_vu, const int32_t* d_len, const float* d_target, float* d_prob,
                               float* d_loss, float* d_dh, float* d_dvu, void* d_workspace, pdf_stream_t stream);
int pdf_clip_scale_batched(int n_members, const float* d_grad, long n_params, float max_norm, float* d_scale, pdf_stream_t stream);
int pdf_adam_step_batched(int n_members, float* d_param, const float* d_grad, float* d_m, float* d_v, long n_params, float lr, float beta1,
                          float beta2, float eps, float weight_decay, int step, const float* d_grad_scale, const uint8_t* d_active,
                          pdf_stream_t stream);
/* the ensemble statistics of every (scenario, subject) pair: d_probs [E, pairs] f32 -> d_stats [pairs, 5] float64 = mean, std
 * (population), entropy of the mean, mean member entropy, mutual information; pdf_moddrop_mc's formulas with members in place of
 * samples (ascending e), so equal members give exactly std = mutual information = 0 */
int pdf_ensemble_stats(int n_members, long long pairs, const float* d_probs, double* d_stats, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4a -- Fusion-ModDrop under every scenario mask in one launch.  Replaces the per-scenario
 * apply_masks_to_matrix + ModalityDropoutModel.predict_proba (data/feature_utils.py:49-61,
 * models/fusion_moddrop.py:93-114; loop at evaluation/evaluate.py:18-97).
 * d_x [N,F] f32; feature block of modality m = [mod_off[m], mod_off[m+1]); d_masks [S,N,M] u8;
 * MLP layers: n_layers linear layers (ReLU between, sigmoid last), weights [out,in] row-major.
 * d_prob [S,N] f32.
 * ------------------------------------------------------------------------------------------ */
#define PDF_MAX_LAYERS 8
#define PDF_MAX_MODS 8
typedef struct {
  int32_t n_layers;
  int32_t dims[PDF_MAX_LAYERS + 1]; /* dims[0]=F ... dims[n_layers]=1 */
  const float* w[PDF_MAX_LAYERS];
  const float* b[PDF_MAX_LAYERS];
  int32_t n_mods;
  int32_t mod_off[PDF_MAX_MODS + 1];
} pdf_mlp;

size_t pdf_moddrop_workspace_bytes(const pdf_mlp* net, int n_subjects);
int pdf_moddrop_sweep(const pdf_mlp* net, int n_subjects, int n_scenarios, const float* d_x, const uint8_t* d_masks,
                      void* d_workspace, float* d_prob, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4b -- MoE head under every scenario mask.  Replaces evaluate.py:52-63 (x_m * mask_m) +
 * MoENet.forward (models/moe.py:37-47): router MLP(mask)+softmax, per-modality expert MLP+sigmoid,
 * gated sum.  Experts listed in sorted(modality) order; expert e reads d_x[e] [N, dims[0]].
 * router: w_r0 [R,M], b_r0 [R], w_r1 [M,R], b_r1 [M].
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t n_experts;
  pdf_mlp expert[PDF_MAX_MODS];
  int32_t router_hidden;
  const float *w_r0, *b_r0, *w_r1, *b_r1;
} pdf_moe;

int pdf_moe_sweep(const pdf_moe* net, int n_subjects, int n_scenarios, const float* const* d_x /* host array of device ptrs */,
                  const uint8_t* d_masks, float* d_prob, pdf_stream_t stream);

/* Explanations of the fusion heads (csrc/fusion_explain.cu): exact modality Shapley values and integrated gradients, for every
 * (scenario, subject) pair of the sweep's inputs.  A missing modality is a zeroed one, so the all-zero input is the baseline.  Modality
 * (expert) m is bit m of a coalition, in the sweep's order (sorted(modality)).  The value v of a coalition is the logit (the value before
 * net's final sigmoid) for ModDrop and the output probability for MoE; the sweep kernel evaluates all 2^M coalitions once per subject.
 *   d_value [S,N] = v(P), P = the modalities present under scenario s: for ModDrop the logit of pdf_moddrop_sweep's probability (same
 *     kernel, same arithmetic), for MoE pdf_moe_sweep's probability bit for bit;
 *   d_base [1] = v(empty set), the same for every subject;
 *   d_shap [S,N,M] = phi_m = sum over T subset P\{m} of |T|!(|P|-|T|-1)!/|P|! (v(T+m) - v(T)), summed in float64, so that
 *     sum_m phi_m = value - base.  An absent or zero-width modality gets exactly 0;
 *   integrated gradients from 0 with `steps` midpoints alpha_k = (k + 1/2)/steps (1..256; 0 only with d_ig NULL):
 *     ModDrop d_ig [S,N,F] = (x (.) m_s) (.) mean_k d logit / d x at alpha_k (x (.) m_s);
 *     MoE d_ig[e] [S,N,d_e] (host array of E device pointers) = the same for the probability: (x_e m_e) (.) w_e(m_s) (.)
 *       mean_k d sigmoid(z_e) / d x_e at alpha_k x_e, w_e = the router weight; 0 where expert e is absent.
 * Two calls return bit-identical results (no atomics).  The IG kernel keeps every hidden layer's activations of 64, 32 or 16 rows in
 * shared memory; a net whose hidden widths do not fit 227 KB even at 16 rows is refused (PDF_ERR_ARG), as are bad arguments, before
 * any device work.  Workspace: pdf_moddrop_explain_workspace_bytes / pdf_moe_explain_workspace_bytes. */
size_t pdf_moddrop_explain_workspace_bytes(const pdf_mlp* net, int n_subjects, int n_scenarios, int steps);
int pdf_moddrop_explain(const pdf_mlp* net, int n_subjects, int n_scenarios, const float* d_x, const uint8_t* d_masks, int steps,
                        void* d_workspace, float* d_value /* [S,N] logit */, float* d_base /* [1] */, float* d_shap /* [S,N,M] */,
                        float* d_ig /* [S,N,F] or NULL */, pdf_stream_t stream);
size_t pdf_moe_explain_workspace_bytes(const pdf_moe* net, int n_subjects, int n_scenarios, int steps);
int pdf_moe_explain(const pdf_moe* net, int n_subjects, int n_scenarios, const float* const* d_x, const uint8_t* d_masks, int steps,
                    void* d_workspace, float* d_value /* [S,N] prob */, float* d_base /* [1] */, float* d_shap /* [S,N,E] */,
                    float* const* d_ig /* host array of E device ptrs [S,N,d_e], or NULL */, pdf_stream_t stream);

/* Bootstrap replicates of the scenario metrics (csrc/metrics.cu), for every scenario in one call.  A Poisson(1) bootstrap: replicate b
 * gives sampling unit u the integer weight w = Poisson1(philox4x32_10(key = seed, counter = (u, b, 0, 0)).x), Poisson1 = inversion of
 * the 32-bit word against T_k = floor(2^32 P(X <= k)), k = 0..12 (w <= 13).  Weights are stateless in (seed, b, u): replicate b is the
 * same whatever n_boot, n_scenarios or the unit count, and pairs across scenarios.
 *   d_prob [S,N] float64 probabilities in [0, 1]; d_label [N], != 0 positive; d_unit [N] non-negative unit ids or NULL (unit = row);
 *   d_out [S, 1+B, 6] float64: row 0 is the point estimate (every weight 1), row 1+b replicate b.  The six metrics are those of
 *     utils.metrics.compute_metrics in its order (roc_auc, pr_auc, balanced_accuracy, f1, brier_score, ece), each equal to the
 *     sklearn / numpy function with sample_weight = w: roc_auc NaN without both classes, pr_auc 0 without positives, balanced accuracy
 *     the recall of the one class present, F1 0 on zero division; every metric NaN when the total weight is 0.
 * AUC, balanced accuracy and F1 are exact integer rationals divided once; the float64 sums are in a fixed order, so calls are
 * bit-identical.  n_boot = 0 computes the point estimate only.  Bad arguments (S < 1, N < 1 or N > 2^28, B < 0 or B > 2^20, NULL
 * d_prob / d_label / d_workspace / d_out, d_prob or d_out not 8-byte, d_unit not 4-byte or d_workspace not 256-byte aligned) return
 * PDF_ERR_ARG before any device work.  Workspace: pdf_bootstrap_metrics_workspace_bytes (0 for bad sizes). */
size_t pdf_bootstrap_metrics_workspace_bytes(int n_scenarios, int n);
int pdf_bootstrap_metrics(int n_scenarios, int n, int n_boot, uint64_t seed, const double* d_prob /* [S,N] */,
                          const uint8_t* d_label /* [N], != 0 positive */, const int32_t* d_unit /* [N] or NULL = row index */,
                          void* d_workspace, double* d_out /* [S, 1+B, 6] */, pdf_stream_t stream);

/* Monte-Carlo (MC) dropout uncertainty of the ModDrop and MIL heads (csrc/uncertainty.cu), for every scenario in one call: T = n_samples
 * stochastic forward passes with the heads' nn.Dropout layers active (and nothing else: the scenario masks play the part of the
 * training-time modality dropout).  Dropout probability p = p_drop in [0, 1) (a float, widened to double): unit j of row n, sample t
 * is dropped iff
 *   philox4x32_10(key = seed, counter = (n, t, (l << 16) | i, 0x80000000 | (j >> 2))).word[j & 3] < floor(p 2^32)   (float64),
 * and a kept unit is multiplied by the float (float)(1 / (1 - p)).  ModDrop: n = subject row of d_x, l = hidden-layer index (0: the
 * first hidden layer's output), i = 0.  MIL: n = bag index, l = 0, i = instance index within the bag.  The top bit of counter word 3
 * keeps these streams apart from pdf_bootstrap_metrics' counters (u, b, 0, 0).  The masks are stateless: sample t of row n has the
 * same masks under every scenario, and nothing depends on S, N, T or the launch shape.
 *   d_stats [S,N,5] float64, per (scenario, subject) over the T sample probabilities p_t, in ascending t:
 *     0 mean = mean_t p_t;  1 std = sqrt(mean_t (p_t - mean)^2) (population);  2 entropy = H(mean),
 *     H(q) = -q ln q - (1-q) ln(1-q) with 0 ln 0 = 0 (nats);  3 expected_entropy = mean_t H(p_t);
 *     4 mutual_info = max(0, entropy - expected_entropy).  T equal samples give exactly mean = p_t, std = mutual_info = 0.
 *   d_samples [S,N,T] float32 sample probabilities, or NULL.
 * ModDrop: d_x [N,F] and d_masks [S,N,M] as pdf_moddrop_sweep.  Layer 1 comes from the sweep's per-modality partials, layers 2.. run
 *   on the shared-memory tile of pdf_moddrop_explain (a net too wide for it is refused the same way); with p = 0 every sample is the
 *   sweep's probability up to float32 rounding.
 * MIL: d_bags, d_len, d_live [S,n_bags] (NULL: live everywhere) as pdf_mil_sweep, FP32 arithmetic whatever the sweep's precision;
 *   live[s, b] && len[b] > 0 selects the bag's samples (which do not depend on s), anything else is missing_prob for every sample.
 *   Lmax <= 65536.
 * Bad arguments (p outside [0, 1), T outside 1..4096, S < 1, N < 1, NULL inputs, workspace or d_stats, d_stats not 8-byte, the float
 * and int arrays not 4-byte or d_workspace not 256-byte aligned, a net the tile does not fit) return PDF_ERR_ARG before any device
 * work.  No atomics: two calls are bit-identical.  Workspace: pdf_moddrop_mc_workspace_bytes / pdf_mil_mc_workspace_bytes (0 for bad
 * sizes). */
size_t pdf_moddrop_mc_workspace_bytes(const pdf_mlp* net, int n_subjects, int n_scenarios, int n_samples);
int pdf_moddrop_mc(const pdf_mlp* net, float p_drop, int n_subjects, int n_scenarios, const float* d_x, const uint8_t* d_masks,
                   int n_samples, uint64_t seed, void* d_workspace, double* d_stats /* [S,N,5] */,
                   float* d_samples /* [S,N,T] or NULL */, pdf_stream_t stream);
size_t pdf_mil_mc_workspace_bytes(const pdf_mil_weights* w, int n_bags, int Lmax, int n_samples);
int pdf_mil_mc(const pdf_mil_weights* w, float p_drop, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len,
               int n_scenarios, const uint8_t* d_live /* [S,n_bags] or NULL */, int n_samples, uint64_t seed,
               void* d_workspace, double* d_stats /* [S,n_bags,5] */, float* d_samples /* [S,n_bags,T] or NULL */, pdf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Self-tests of the tensor-core building blocks (used by tests/ and smoke on the GPU box).
 * pdf_selftest_umma: C[M,N] = A[M,K] * B[N,K]^T through TMA(2D tiled) + tcgen05.mma, bf16 in / f32 out.
 * ------------------------------------------------------------------------------------------ */
int pdf_selftest_umma(int M, int N, int K, const void* d_a_bf16, const void* d_b_bf16, float* d_c, pdf_stream_t stream);
/* C[128,N] = A[shift:shift+128, 0:64] * B[N,64]^T where A (256 x 64) is loaded ONCE into shared memory and the MMA
 * reads it through a descriptor whose start address is advanced by `shift` rows (shift*128 bytes).
 * mode 0: descriptor base_offset = 0; mode 1: base_offset = (start_address >> 7) & 7.  Probes the shifted-window
 * operand reuse a halo-resident 3x3 convolution needs. */
int pdf_selftest_umma_shift(int N, int shift, int mode, const void* d_a_bf16, const void* d_b_bf16, float* d_c, pdf_stream_t stream);

/* Probe: tensor-pipe rate of back-to-back shared-memory-operand MMAs (M=128, N in {64,128,256}, K=16) with resident
 * operands; `iters` x 36 MMAs per CTA, `grid` CTAs; mode bit 0 = walk the halo conv's 9 row-shifted A windows.
 * d_cycles[grid] receives the SM-clock cycles each CTA took (profiles/r01_umma_rate.txt). */
int pdf_selftest_umma_rate(int N, int iters, int mode, int grid, unsigned long long* d_cycles, pdf_stream_t stream);

/* Tuning / test hook for the CTA-pair kernel (tcgen05.mma.cta_group::2, csrc/conv_tc2.cu): 0 = never, 1 = every eligible
 * Cout >= 128 layer, 2 (default) = only 3x3 layers with 256-wide tiles, where it wins under the power cap (DESIGN.md section 4),
 * 3 = 2 plus the resident-weights variant on 128-channel 3x3 layers (measured slower). */
int pdf_debug_enable_pair(int enable);

/* Tuning / test hook: enable == 0 launches the tcgen05 kernels without programmatic dependent launch (default: on -- the prologue
 * of each convolution kernel overlaps the tail of its predecessor; results are identical). */
int pdf_debug_enable_pdl(int enable);

/* Tuning / test hook for the horizontally-shared 3x3 stride-1 kernel (csrc/conv3x3_hs.cu: one activation tile per filter row serves its
 * three taps): 0 = off, 1 (default) = eligible layers with Cout == 128 and enough tiles for every SM, 2 = every such layer with
 * Cout % 128 == 0, 3 = 2 whatever the size (tests).  Read when a plan is created. */
int pdf_debug_set_hs_mode(int mode);

/* Timing probe for the generic tcgen05 conv kernel -- outputs are garbage while it is set.  bit 0: the epilogue only hands the
 * accumulator back (no TMEM read, no stores); bit 1: the MMA issuer skips the MMAs (TMA ring and commits still run); bit 2: the
 * epilogue runs without its global stores; 0 = normal. */
int pdf_debug_set_conv_probe(int mode);

/* Tuning hook: pdf_preprocess works through the batch in sub-batches of `subjects` volumes (0 = the whole batch at once) so that
 * one sub-batch's resampled volumes stay L2-resident across the histogram passes and the plane gather.  Results are identical. */
int pdf_debug_set_pre_chunk(int subjects);

/* Debug hook: CTA 0 of the following PDF_OP_STEM_FUSED launches records clock64 stamps of its warp roles,
 * [64 tiles][16 events] u64, into d_buf (NULL switches it off).  The stamps are compiled in only when the library is built with
 * -DPDF_STEM_TRACE (they cost 15 % of the kernel's run time); otherwise the call is accepted and nothing is recorded. */
int pdf_debug_set_trace(unsigned long long* d_buf);

/* Test hook: disable != 0 makes later pdf_plan_create calls route 3x3/s1 64->64 convolutions through the generic
 * im2col kernel instead of the halo-resident kernel (A/B parity of the two tensor-core kernels). */
int pdf_debug_disable_halo(int disable);

#ifdef __cplusplus
}
#endif
#endif /* PDFUSION_B200_H */

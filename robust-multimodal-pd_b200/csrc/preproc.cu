// K1: raw T1 volume -> network input, batched over subjects, HBM-bound.
//
//   decode_*_kernel        stored NIfTI voxels (any type, x-fastest) -> float32 C-order, nibabel's float64 scaling rule
//   resample_tma_kernel    nan/inf scrub + trilinear zoom in float64 (scipy order, one f32 rounding), input rows streamed by
//   (resample_kernel)      cp.async.bulk; + level-0 radix histogram of positive voxels + per-plane maxima (3 axes) + global min
//   scan_kernel<0|1|2>     per subject: locate the bucket of each of the 4 order statistics numpy.percentile needs
//   hist_kernel<1>         11-bit refinement histograms over the resampled volume + compaction of the candidate voxels
//   hist_kernel<2>         8-bit refinement from the candidate list (full scan only when the list overflowed)
//   finalize (in scan<2>)  numpy lerp -> lo/hi, extents from plane maxima, np.linspace(...).astype(int) indices
//   extract_planes_kernel  axis-2 planes (stride-T2 gather), clipped to [lo, hi] -> compact [L2][T0][T1]
//   resize_band_kernel     (clip) + bilinear (align_corners=False) + min-max + (x-mean)/std -> bf16 one channel (padded for the stem)
//   resize_kernel          the same for the f32 NHWC3 layout and odd sizes
//   gather_slices / tta    slices themselves and their test-time augmentation (a6)
//
// Reference call sites: data/openneuro_features.py:22-32, 121-151, 250-255 (see include/pdfusion_b200.h).
#include "common.cuh"
#include "tc_common.cuh"

namespace pdf {

constexpr int kPlaneMax = 1024;   // max target dim
constexpr int kH0 = 4096, kH1 = 2048, kH2 = 256;
constexpr int kNQ = 4;            // sorted[f0], sorted[f1] for q=1 and q=99
constexpr int kResStages = 4;     // bulk-copy ring depth of resample_tma_kernel

struct SubjState {
  uint32_t hist0[kH0];
  uint32_t hist1[kNQ][kH1];
  uint32_t hist2[kNQ][kH2];
  uint32_t plane_max[3][kPlaneMax];  // ordered keys; 0 = "no voxel seen"
  uint32_t gmin_key;                 // ordered key of the global minimum (init 0xffffffff)
  uint32_t n_pos;
  uint32_t prefix[kNQ];              // high bits of the answer found so far (0xffffffff = no query)
  uint32_t rank[kNQ];                // residual rank inside the current bucket
  float gamma[2];                    // numpy gamma for q=1 / q=99
  uint32_t n_cand;                   // voxels sharing a level-0 bucket with a query (appended to the candidate list by hist<1>)
  uint32_t pad[2];
};

struct ZoomTables {                  // lives at the head of the workspace
  int i0[3][kPlaneMax];
  int i1[3][kPlaneMax];
  double w0[3][kPlaneMax];
  double w1[3][kPlaneMax];
};

// Raw geometry of the subjects of one resample launch, passed by value (__grid_constant__: read from the parameter bank, no copy).
// A uniform batch has one entry and subject b's volume at b * X*Y*Z; a ragged batch has one entry per subject of the launch, and
// `subj` is the subject's index in the batch (the launch may cover a subset: the bulk-copy kernel takes the subjects whose rows fit
// its ring, resample_kernel the rest).  NR = input rows a tile touches at the launch's TJ; plane_max = the largest per-subject
// staging plane of the launch (NR * Z; resample_kernel: rounded up to even), which sizes the shared-memory layout.
struct ResampleSubj {
  int X, Y, Z, NR;
  int subj, pad;
  long long raw_off;   // float32 elements into the packed raw buffer (ragged)
  ZoomTables* tabs;
};
struct ResampleGeom {
  int uniform, n, plane_max, pad;
  ResampleSubj s[PDF_RAGGED_MAX_BATCH];
};

__device__ __forceinline__ const ResampleSubj& geom_entry(const ResampleGeom& g) { return g.s[g.uniform ? 0 : blockIdx.y]; }
__device__ __forceinline__ int geom_subject(const ResampleGeom& g) { return g.uniform ? (int)blockIdx.y : g.s[blockIdx.y].subj; }
__device__ __forceinline__ const float* geom_raw(const ResampleGeom& g, const float* raw, const ResampleSubj& e) {
  return raw + (g.uniform ? (size_t)blockIdx.y * e.X * e.Y * e.Z : (size_t)e.raw_off);
}

struct Workspace {
  ZoomTables* tabs;
  SubjState* st;
  float* planes;   // [B][L2z][T0][T1]
  uint32_t* cand;  // [B][cand_cap] bit patterns of the level-2 candidates
  size_t cand_cap;
};

// candidate list capacity per subject: a quarter of the volume; denser buckets fall back to a full second scan
static size_t cand_capacity(const pdf_preproc_cfg* cfg) {
  return ((size_t)cfg->out_shape[0] * cfg->out_shape[1] * cfg->out_shape[2] / 4 + 63) & ~(size_t)63;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static int count_axis2(const pdf_preproc_cfg* cfg) {
  int n = 0;
  for (int a = 0; a < cfg->n_axes; ++a)
    if (cfg->axes[a] == 2) n += cfg->counts[a];
  return n;
}

static Workspace carve(const pdf_preproc_cfg* cfg, int batch, void* ws) {
  Workspace w;
  char* p = reinterpret_cast<char*>(ws);
  w.tabs = reinterpret_cast<ZoomTables*>(p);
  p += align_up(sizeof(ZoomTables), 256);
  w.st = reinterpret_cast<SubjState*>(p);
  p += align_up(sizeof(SubjState) * (size_t)batch, 256);
  w.planes = reinterpret_cast<float*>(p);
  p += align_up((size_t)batch * count_axis2(cfg) * cfg->out_shape[0] * cfg->out_shape[1] * sizeof(float), 256);
  w.cand = reinterpret_cast<uint32_t*>(p);
  w.cand_cap = cand_capacity(cfg);
  return w;
}

// everything but cfg->in_shape (which the ragged entry points take per subject from their descriptors)
static int validate_target(const pdf_preproc_cfg* cfg, int batch) {
  PDF_REQUIRE(cfg != nullptr && batch > 0, "preproc: null cfg or batch <= 0");
  for (int i = 0; i < 3; ++i) {
    PDF_REQUIRE(cfg->out_shape[i] >= 2 && cfg->out_shape[i] <= kPlaneMax, "preproc: shapes must be >=2 and target dims <= %d", kPlaneMax);
  }
  PDF_REQUIRE(cfg->n_axes >= 1 && cfg->n_axes <= PDF_MAX_AXES, "preproc: n_axes must be 1..3");
  for (int a = 0; a < cfg->n_axes; ++a) {
    PDF_REQUIRE(cfg->axes[a] >= 0 && cfg->axes[a] <= 2, "preproc: axis must be 0..2");
    PDF_REQUIRE(cfg->counts[a] >= 1 && cfg->counts[a] <= kPlaneMax, "preproc: slice count out of range");
  }
  PDF_REQUIRE(cfg->input_size >= 1, "preproc: input_size must be positive");
  if (cfg->slice_major)
    PDF_REQUIRE(cfg->n_axes == 1 && cfg->axes[0] == 2, "preproc: slice_major is the layout of single-axis axis-2 configurations");
  return PDF_OK;
}

static int validate(const pdf_preproc_cfg* cfg, int batch) {
  if (int rc = validate_target(cfg, batch)) return rc;
  for (int i = 0; i < 3; ++i) PDF_REQUIRE(cfg->in_shape[i] >= 2, "preproc: shapes must be >=2 and target dims <= %d", kPlaneMax);
  return PDF_OK;
}

static int validate_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs) {
  if (int rc = validate_target(cfg, batch)) return rc;
  PDF_REQUIRE(batch <= PDF_RAGGED_MAX_BATCH && descs, "preproc (ragged): batch must be 1..%d with a descriptor per subject",
              PDF_RAGGED_MAX_BATCH);
  for (int b = 0; b < batch; ++b) {
    const pdf_volume_desc& v = descs[b];
    PDF_REQUIRE(v.shape[0] >= 2 && v.shape[1] >= 2 && v.shape[2] >= 2, "preproc (ragged): subject %d: raw dims must be >= 2", b);
    PDF_REQUIRE(v.raw_offset >= 0 && v.raw_offset % 4 == 0, "preproc (ragged): subject %d: raw_offset must be a non-negative "
                "multiple of 4", b);
  }
  return PDF_OK;
}

// the resample kernel writes slice-major only from its 8-row bulk-copy tiles (see resample_tma_kernel / pdf_resample_stats)
static bool slice_major_ok_shape(const pdf_preproc_cfg* cfg, int Y, int Z) {
  if (!cfg || cfg->n_axes != 1 || cfg->axes[0] != 2) return false;
  const int T0 = cfg->out_shape[0], T1 = cfg->out_shape[1], T2 = cfg->out_shape[2];
  if (Z % 4 != 0 || (T2 + 31) / 32 * 32 > 160 || T1 < 8 || T1 % 8 != 0) return false;
  const double ystep = (double)(Y - 1) / (double)(T1 - 1);
  const int NR = (int)(7 * ystep) + 3;
  const size_t smem = (size_t)kResStages * 2 * NR * Z * 4 + (size_t)(kH0 + T0 + T1) * 4 + 16 + (size_t)T1 * 32 + 2 * kResStages * 8 + 128;
  return smem <= 110 * 1024;
}
static bool slice_major_ok(const pdf_preproc_cfg* cfg) { return cfg && slice_major_ok_shape(cfg, cfg->in_shape[1], cfg->in_shape[2]); }

// ------------------------------------------------------------------------------------------------------
// grid (.., entries of g): one table per geometry entry
__global__ void init_tables_kernel(const __grid_constant__ ResampleGeom g, SubjState* st, int batch, int T0, int T1, int T2) {
  const ResampleSubj& e = geom_entry(g);
  ZoomTables* tabs = e.tabs;
  const int src[3] = {e.X, e.Y, e.Z};
  const int dst[3] = {T0, T1, T2};
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  for (int a = 0; a < 3; ++a) {
    if (t < dst[a]) {
      // ndimage.zoom(grid_mode=False): coordinate = i * (src-1)/(dst-1) in float64
      double step = __ddiv_rn((double)(src[a] - 1), (double)(dst[a] - 1));
      double c = __dmul_rn((double)t, step);
      double f = floor(c);
      double w1 = __dsub_rn(c, f);
      int i0 = (int)f;
      tabs->i0[a][t] = i0;
      tabs->i1[a][t] = min(i0 + 1, src[a] - 1);
      tabs->w0[a][t] = __dsub_rn(1.0, w1);
      tabs->w1[a][t] = w1;
    }
  }
  if (blockIdx.y == 0 && t < batch) st[t].gmin_key = 0xffffffffu;
}

__device__ __forceinline__ double scrub(float v) {  // np.nan_to_num(nan=0, posinf=0, neginf=0)
  return isfinite(v) ? (double)v : 0.0;
}

// One tile = output plane i, TJ consecutive output rows j, all k.  The 2 x nr input rows the tile touches
// ([x0|x1][ylo..yhi][0..Z)) are contiguous in HBM per plane: they are streamed in once with 16-byte loads,
// scrubbed, widened to float64 and parked in shared memory; every output voxel then reads its 8 taps from
// shared memory.  Blocks are persistent over tiles so the histogram / plane-maximum partials are flushed once.
__global__ void __launch_bounds__(256)
resample_kernel(const float* __restrict__ raw, float* __restrict__ zoomed, SubjState* __restrict__ states,
                const __grid_constant__ ResampleGeom g, int T0, int T1, int T2, int TJ) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const ResampleSubj& ge = geom_entry(g);
  const ZoomTables* __restrict__ tabs = ge.tabs;
  const int Y = ge.Y, Z = ge.Z, NR = ge.NR;
  double* s_in = reinterpret_cast<double*>(sm_raw);                      // [2][NR][Z]
  uint32_t* s_hist = reinterpret_cast<uint32_t*>(s_in + 2 * (size_t)g.plane_max);
  uint32_t* s_imax = s_hist + kH0;
  uint32_t* s_jmax = s_imax + T0;
  const int b = geom_subject(g);
  const int tid = threadIdx.x, nthr = blockDim.x;
  for (int i = tid; i < kH0 + T0 + T1; i += nthr) s_hist[i] = 0;        // hist, imax, jmax are contiguous
  __syncthreads();

  SubjState* st = states + b;
  const float* rb = geom_raw(g, raw, ge);
  float* zb = zoomed + (size_t)b * T0 * T1 * T2;
  const int tiles_per_i = (T1 + TJ - 1) / TJ;
  const int ntiles = T0 * tiles_per_i;
  const int kchunks = (T2 + nthr - 1) / nthr;
  const size_t plane = ((size_t)NR * Z + 1) & ~(size_t)1;   // even: keeps plane 1 16-byte aligned for double2 stores
  uint32_t tmin = 0xffffffffu, kmax0 = 0;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int i = tile / tiles_per_i;
    const int j0 = (tile - i * tiles_per_i) * TJ, j1 = min(j0 + TJ, T1);
    const int ylo = tabs->i0[1][j0], yhi = tabs->i1[1][j1 - 1];
    const int n = (yhi - ylo + 1) * Z;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int xa = a ? tabs->i1[0][i] : tabs->i0[0][i];
      const float* src = rb + ((size_t)xa * Y + ylo) * Z;
      double* dst = s_in + a * plane;
      if (((reinterpret_cast<uintptr_t>(src) & 15) == 0) && (n & 3) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(src);
        for (int q = tid; q < (n >> 2); q += nthr) {
          const float4 v = __ldg(s4 + q);
          reinterpret_cast<double2*>(dst)[2 * q] = make_double2(scrub(v.x), scrub(v.y));
          reinterpret_cast<double2*>(dst)[2 * q + 1] = make_double2(scrub(v.z), scrub(v.w));
        }
      } else {
        for (int q = tid; q < n; q += nthr) dst[q] = scrub(__ldg(src + q));
      }
    }
    __syncthreads();
    const double wx0 = tabs->w0[0][i], wx1 = tabs->w1[0][i];
    for (int kc = 0; kc < kchunks; ++kc) {
      const int k = kc * nthr + tid;
      const bool act = k < T2;
      int z0 = 0, z1 = 0;
      double wz0 = 0.0, wz1 = 0.0;
      if (act) { z0 = tabs->i0[2][k]; z1 = tabs->i1[2][k]; wz0 = tabs->w0[2][k]; wz1 = tabs->w1[2][k]; }
      uint32_t tile_max = 0;
      for (int j = j0; j < j1; ++j) {
        uint32_t key = 0;
        if (act) {
          const int y0 = tabs->i0[1][j] - ylo, y1 = tabs->i1[1][j] - ylo;
          const double wy0 = tabs->w0[1][j], wy1 = tabs->w1[1][j];
          const double* r00 = s_in + (size_t)y0 * Z;
          const double* r01 = s_in + (size_t)y1 * Z;
          const double* r10 = r00 + plane;
          const double* r11 = r01 + plane;
          // scipy NI_ZoomShift order: t += ((v*wx)*wy)*wz, taps in (x,y,z) lexicographic order, no FMA contraction
          double t = 0.0;
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r00[z0], wx0), wy0), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r00[z1], wx0), wy0), wz1));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r01[z0], wx0), wy1), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r01[z1], wx0), wy1), wz1));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r10[z0], wx1), wy0), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r10[z1], wx1), wy0), wz1));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r11[z0], wx1), wy1), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(r11[z1], wx1), wy1), wz1));
          const float out = __double2float_rn(t);
          zb[((size_t)i * T1 + j) * T2 + k] = out;
          key = float_to_ordered(out);
          tile_max = max(tile_max, key);
          tmin = min(tmin, key);
          if (out > 0.0f) atomicAdd(&s_hist[__float_as_uint(out) >> 19], 1u);
        }
        const uint32_t wmax = __reduce_max_sync(0xffffffffu, key);
        if ((tid & 31) == 0 && wmax != 0) atomicMax(&s_jmax[j], wmax);
      }
      if (kchunks == 1) kmax0 = max(kmax0, tile_max);
      else if (act && tile_max != 0) atomicMax(&st->plane_max[2][k], tile_max);
      const uint32_t imx = __reduce_max_sync(0xffffffffu, tile_max);
      if ((tid & 31) == 0 && imx != 0) atomicMax(&s_imax[i], imx);
    }
    __syncthreads();
  }
  if (kchunks == 1 && tid < T2 && kmax0 != 0) atomicMax(&st->plane_max[2][tid], kmax0);
  const uint32_t wmin = __reduce_min_sync(0xffffffffu, tmin);
  if ((tid & 31) == 0 && wmin != 0xffffffffu) atomicMin(&st->gmin_key, wmin);
  __syncthreads();
  for (int i = tid; i < kH0; i += nthr) {
    const uint32_t c = s_hist[i];
    if (c) atomicAdd(&st->hist0[i], c);
  }
  for (int i = tid; i < T0; i += nthr) if (s_imax[i]) atomicMax(&st->plane_max[0][i], s_imax[i]);
  for (int i = tid; i < T1; i += nthr) if (s_jmax[i]) atomicMax(&st->plane_max[1][i], s_jmax[i]);
}

// Same tile decomposition, but the input rows are streamed by the bulk-copy engine (cp.async.bulk, the 1-D TMA
// path) into a ring of shared-memory stages while the compute warps work on earlier tiles: warp 0 is the producer
// (one lane issues two bulk copies per tile and arms the stage's mbarrier with the byte count), the other warps
// consume.  Needs 16-byte aligned rows (Z % 4 == 0).  Compute threads: [half][k], half = row parity inside the tile.

__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// (Widening float32 -> float64 and narrowing the sum back with integer instructions instead of F2F was measured 23 % SLOWER:
// 671 vs 543 us for 32 subjects, profiles/r01_pre_times.txt.  The conversions are not the bound.)
__device__ __forceinline__ double scrub_bits(float v) {   // nan/inf -> 0, else widen
  return (fabsf(v) < INFINITY) ? (double)v : 0.0;
}

// Per-row constants of the y axis, staged in shared memory once per block: two 16-byte loads per output row instead of
// four table loads from global memory plus the address arithmetic around them.
struct __align__(16) JEntry {
  int y0b, y1b;        // byte offset (y * Z * 4) of the two input rows
  int pad0, pad1;
  double w0, w1;
};

__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t key_of(float f) { return float_to_ordered(f); }

// NEED_JMAX: plane maxima along axis 1 are only needed when axis 1 is one of the slicing axes; they cost a warp
// reduction + shared atomic per output row, so the common axis-2 / axis-0 configurations skip them.
// ZMAJOR: the resampled volume is written slice-axis-major, [T2][T0][T1] (pdf_preproc_cfg.slice_major: single-axis axis-2
// configurations, whose selected planes are then CONTIGUOUS -- the stride-T2 plane gather touched every sector of the volume to
// deliver L of T2 planes).  The two row halves then own rows [j0, j0+4) and [j0+4, j0+8) of a tile instead of alternating rows, a
// thread keeps its four results in registers and stores them as ONE 16-byte vector at (k, i, j0 + 4*half): no shared-memory
// transpose, no extra barrier, and half a sector per lane and store (the other half comes from the other row half; L2 merges).
template <bool NEED_JMAX, bool ZMAJOR>
__global__ void __launch_bounds__(352, 2)
resample_tma_kernel(const float* __restrict__ raw, float* __restrict__ zoomed, SubjState* __restrict__ states,
                    const __grid_constant__ ResampleGeom g, int T0, int T1, int T2, int TJ, int KT) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const ResampleSubj& ge = geom_entry(g);
  const ZoomTables* __restrict__ tabs = ge.tabs;
  const int Y = ge.Y, Z = ge.Z, NR = ge.NR;
  const uint32_t stage_bytes = (uint32_t)(2 * g.plane_max * 4);
  float* s_stage = reinterpret_cast<float*>(sm_raw);
  uint32_t* s_hist = reinterpret_cast<uint32_t*>(sm_raw + (size_t)kResStages * stage_bytes);
  uint32_t* s_imax = s_hist + kH0;
  uint32_t* s_jmax = s_imax + T0;
  size_t off = ((size_t)kResStages * stage_bytes + (size_t)(kH0 + T0 + T1) * 4 + 15) & ~(size_t)15;
  JEntry* s_jtab = reinterpret_cast<JEntry*>(sm_raw + off);
  off += (size_t)T1 * sizeof(JEntry);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(sm_raw + off);
  const uint32_t bar_full = smem_u32(s_bar), bar_empty = bar_full + kResStages * 8;
  const int b = geom_subject(g);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int n_cwarps = (nthr - 32) / 32;
  for (int i = tid; i < kH0 + T0 + T1; i += nthr) s_hist[i] = 0;
  for (int j = tid; j < T1; j += nthr) {
    JEntry e;
    e.y0b = tabs->i0[1][j] * Z * 4; e.y1b = tabs->i1[1][j] * Z * 4; e.pad0 = e.pad1 = 0;
    e.w0 = tabs->w0[1][j]; e.w1 = tabs->w1[1][j];
    s_jtab[j] = e;
  }
  if (tid == 0) {
    for (int s = 0; s < kResStages; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, n_cwarps); }
    fence_barrier_init();
  }
  __syncthreads();

  SubjState* st = states + b;
  const float* rb = geom_raw(g, raw, ge);
  float* zb = zoomed + (size_t)b * T0 * T1 * T2;
  const int tiles_per_i = (T1 + TJ - 1) / TJ;
  const int ntiles = T0 * tiles_per_i;
  const int plane = NR * Z;
  // warp-uniform role / row bookkeeping (the shuffle tells the compiler so: it can live in uniform registers)
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int lane = tid & 31;

  if (warp == 0) {
    if (elect_one()) {
      int it = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int stage = it % kResStages;
        const uint32_t phase = (uint32_t)(it / kResStages) & 1u;
        const int i = tile / tiles_per_i;
        const int j0 = (tile - i * tiles_per_i) * TJ, j1 = min(j0 + TJ, T1);
        const int ylo = tabs->i0[1][j0], yhi = tabs->i1[1][j1 - 1];
        const uint32_t bytes = (uint32_t)((yhi - ylo + 1) * Z * 4);
        mbar_wait(bar_empty + stage * 8, phase ^ 1u);
        mbar_expect_tx(bar_full + stage * 8, 2 * bytes);
        const uint32_t dst = smem_u32(s_stage) + stage * stage_bytes;
        bulk_load(dst, rb + ((size_t)tabs->i0[0][i] * Y + ylo) * Z, bytes, bar_full + stage * 8);
        bulk_load(dst + plane * 4, rb + ((size_t)tabs->i1[0][i] * Y + ylo) * Z, bytes, bar_full + stage * 8);
      }
    }
  } else {
    const int wph = KT >> 5;                       // compute warps per row half
    const int cw = warp - 1;
    const int half = cw / wph;
    const int k = (cw - half * wph) * 32 + lane;
    const bool act = k < T2;
    uint32_t z0b = 0, z1b = 0;
    double wz0 = 0.0, wz1 = 0.0;
    if (act) { z0b = (uint32_t)tabs->i0[2][k] * 4u; z1b = (uint32_t)tabs->i1[2][k] * 4u; wz0 = tabs->w0[2][k]; wz1 = tabs->w1[2][k]; }
    const uint32_t planeb = (uint32_t)plane * 4u;
    const uint32_t stage0 = smem_u32(s_stage);
    float vmin = INFINITY, kmaxf = -INFINITY;
    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int stage = it % kResStages;
      const uint32_t phase = (uint32_t)(it / kResStages) & 1u;
      const int i = tile / tiles_per_i;
      const int j0 = (tile - i * tiles_per_i) * TJ, j1 = min(j0 + TJ, T1);
      const double wx0 = tabs->w0[0][i], wx1 = tabs->w1[0][i];
      const uint32_t sbase = stage0 + (uint32_t)stage * stage_bytes - (uint32_t)s_jtab[j0].y0b;
      float* op = zb + ((size_t)i * T1 + (j0 + half)) * T2 + k;
      mbar_wait(bar_full + stage * 8, phase);
      float tmaxf = -INFINITY;
      float acc4[4] = {0.f, 0.f, 0.f, 0.f};
      auto do_row = [&](const int j, const int r) {
        const JEntry e = s_jtab[j];
        const uint32_t r0 = sbase + (uint32_t)e.y0b, r1 = sbase + (uint32_t)e.y1b;
        const float f000 = lds_f32(r0 + z0b), f001 = lds_f32(r0 + z1b), f010 = lds_f32(r1 + z0b), f011 = lds_f32(r1 + z1b);
        const float f100 = lds_f32(r0 + planeb + z0b), f101 = lds_f32(r0 + planeb + z1b);
        const float f110 = lds_f32(r1 + planeb + z0b), f111 = lds_f32(r1 + planeb + z1b);
        const uint32_t orall = __float_as_uint(f000) | __float_as_uint(f001) | __float_as_uint(f010) | __float_as_uint(f011) |
                               __float_as_uint(f100) | __float_as_uint(f101) | __float_as_uint(f110) | __float_as_uint(f111);
        // background fast path: eight (+-)0 taps give exactly +0.0 in scipy's sum, no float64 work (and no conversion) needed
        float out = 0.0f;
        if ((orall & 0x7fffffffu) != 0u) {
          double t = 0.0;
          double d000, d001, d010, d011, d100, d101, d110, d111;
          if ((orall & 0x7f800000u) != 0x7f800000u) {     // no tap can be NaN/Inf (their exponent bits would survive the OR)
            d000 = (double)f000; d001 = (double)f001; d010 = (double)f010; d011 = (double)f011;
            d100 = (double)f100; d101 = (double)f101; d110 = (double)f110; d111 = (double)f111;
          } else {
            d000 = scrub_bits(f000); d001 = scrub_bits(f001); d010 = scrub_bits(f010); d011 = scrub_bits(f011);
            d100 = scrub_bits(f100); d101 = scrub_bits(f101); d110 = scrub_bits(f110); d111 = scrub_bits(f111);
          }
          // scipy NI_ZoomShift order: t += ((v*wx)*wy)*wz, taps in (x,y,z) lexicographic order, no FMA contraction
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d000, wx0), e.w0), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d001, wx0), e.w0), wz1));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d010, wx0), e.w1), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d011, wx0), e.w1), wz1));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d100, wx1), e.w0), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d101, wx1), e.w0), wz1));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d110, wx1), e.w1), wz0));
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(__dmul_rn(d111, wx1), e.w1), wz1));
          out = __double2float_rn(t);
        }
        if (act) {
          if (ZMAJOR) acc4[r] = out;
          else *op = out;
          tmaxf = fmaxf(tmaxf, out);
          vmin = fminf(vmin, out);
          if (out > 0.0f) atomicAdd(&s_hist[__float_as_uint(out) >> 19], 1u);
        }
        if (NEED_JMAX) {
          const uint32_t wmax = __reduce_max_sync(0xffffffffu, act ? key_of(out) : 0u);
          if (lane == 0 && wmax != 0) atomicMax(&s_jmax[j], wmax);
        }
            };
      const int jbeg = ZMAJOR ? j0 + 4 * half : j0 + half;
      if (ZMAJOR) {
#pragma unroll
        for (int r = 0; r < 4; ++r) do_row(jbeg + r, r);       // (T1 % 8 == 0: every tile has its eight rows)
      } else {
#pragma unroll 2
        for (int j = jbeg; j < j1; j += 2, op += 2 * (size_t)T2) do_row(j, 0);
      }
      if (ZMAJOR && act)
        *reinterpret_cast<float4*>(zb + ((size_t)k * T0 + i) * T1 + jbeg) = make_float4(acc4[0], acc4[1], acc4[2], acc4[3]);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_empty + stage * 8);    // this warp is done reading the stage
      kmaxf = fmaxf(kmaxf, tmaxf);
      const uint32_t imx = __reduce_max_sync(0xffffffffu, tmaxf == -INFINITY ? 0u : key_of(tmaxf));
      if (lane == 0 && imx != 0) atomicMax(&s_imax[i], imx);
    }
    if (act && kmaxf != -INFINITY) atomicMax(&st->plane_max[2][k], key_of(kmaxf));
    const uint32_t wmin = __reduce_min_sync(0xffffffffu, vmin == INFINITY ? 0xffffffffu : key_of(vmin));
    if (lane == 0 && wmin != 0xffffffffu) atomicMin(&st->gmin_key, wmin);
  }
  __syncthreads();
  for (int i = tid; i < kH0; i += nthr) {
    const uint32_t c = s_hist[i];
    if (c) atomicAdd(&st->hist0[i], c);
  }
  for (int i = tid; i < T0; i += nthr) if (s_imax[i]) atomicMax(&st->plane_max[0][i], s_imax[i]);
  if (NEED_JMAX)
    for (int i = tid; i < T1; i += nthr) if (s_jmax[i]) atomicMax(&st->plane_max[1][i], s_jmax[i]);
}

// ------------------------------------------------------------------------------------------------------
// Block-wide bucket search: smallest bin with cumulative count > rank. 256 threads, NB % 256 == 0.
template <int NB>
__device__ void find_bucket(const uint32_t* __restrict__ hist, uint32_t rank, uint32_t* s_scan, uint32_t* out_bin,
                            uint32_t* out_residual) {
  constexpr int PER = NB / 256;
  const int tid = threadIdx.x;
  uint32_t local = 0;
#pragma unroll
  for (int i = 0; i < PER; ++i) local += hist[tid * PER + i];
  // inclusive scan of 256 partials
  uint32_t v = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t n = __shfl_up_sync(0xffffffffu, v, o);
    if ((tid & 31) >= o) v += n;
  }
  if ((tid & 31) == 31) s_scan[tid >> 5] = v;
  __syncthreads();
  if (tid < 8) {
    uint32_t w = s_scan[tid];
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      uint32_t n = __shfl_up_sync(0xffu, w, o);
      if (tid >= o) w += n;
    }
    s_scan[tid] = w;
  }
  __syncthreads();
  const uint32_t incl = v + ((tid >> 5) ? s_scan[(tid >> 5) - 1] : 0u);
  const uint32_t excl = incl - local;
  if (rank >= excl && rank < incl) {
    uint32_t acc = excl;
    for (int i = 0; i < PER; ++i) {
      const uint32_t c = hist[tid * PER + i];
      if (rank < acc + c) { *out_bin = tid * PER + i; *out_residual = rank - acc; break; }
      acc += c;
    }
  }
  __syncthreads();
}

struct FinalizeArgs {
  int T[3];
  int n_axes;
  int axes[PDF_MAX_AXES];
  int counts[PDF_MAX_AXES];
  int lmax;
  int extent_raw;
};

__device__ __forceinline__ float normalise(float v, float lo, float hi, float den) {
  // np.clip(v, lo, hi) = minimum(maximum(v, lo), hi); then (v - lo) / den, all float32
  const float c = fminf(fmaxf(v, lo), hi);
  return __fdiv_rn(__fsub_rn(c, lo), den);
}

template <int LEVEL>
__global__ void __launch_bounds__(256)
scan_kernel(SubjState* __restrict__ states, FinalizeArgs fa, float* __restrict__ lohi, int32_t* __restrict__ indices,
            int32_t* __restrict__ nslices) {
  pdl_launch_dependents();   // programmatic dependent launch (common.cuh): scheduled under the predecessor's tail,
  pdl_wait();                // nothing is read before the predecessor has completed
  __shared__ uint32_t s_scan[8];
  __shared__ uint32_t s_bin[kNQ], s_res[kNQ];
  __shared__ float s_lohi[3];
  __shared__ int s_first, s_last;
  SubjState* st = states + blockIdx.x;
  const int tid = threadIdx.x;

  if (LEVEL == 0) {
    // n_pos and the numpy 'linear' virtual indices, evaluated in float32 as numpy 2.x does (NEP 50)
    __shared__ uint32_t s_n;
    uint32_t local = 0;
    for (int i = tid; i < kH0; i += 256) local += st->hist0[i];
    for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if (tid == 0) s_n = 0;
    __syncthreads();
    if ((tid & 31) == 0) atomicAdd(&s_n, local);
    __syncthreads();
    const uint32_t n = s_n;
    if (tid == 0) {
      st->n_pos = n;
      for (int qi = 0; qi < 2; ++qi) {
        if (n == 0) { st->prefix[2 * qi] = st->prefix[2 * qi + 1] = 0xffffffffu; continue; }
        const float q32 = __fdiv_rn(qi == 0 ? 1.0f : 99.0f, 100.0f);
        const float virt = __fmul_rn((float)(n - 1), q32);
        const float prev = floorf(virt);
        st->gamma[qi] = __fsub_rn(virt, prev);
        uint32_t f0, f1;
        if (virt >= (float)(n - 1)) { f0 = f1 = n - 1; }   // numpy: indexes above bounds -> last element
        else { f0 = (uint32_t)prev; f1 = f0 + 1; }
        st->rank[2 * qi] = f0;
        st->rank[2 * qi + 1] = f1;
        st->prefix[2 * qi] = st->prefix[2 * qi + 1] = 0;
      }
    }
    __syncthreads();
    if (n == 0) return;
    for (int q = 0; q < kNQ; ++q) {
      find_bucket<kH0>(st->hist0, st->rank[q], s_scan, &s_bin[q], &s_res[q]);
    }
    if (tid < kNQ) { st->prefix[tid] = s_bin[tid]; st->rank[tid] = s_res[tid]; }
    return;
  }
  if (LEVEL == 1) {
    if (st->n_pos == 0) return;
    for (int q = 0; q < kNQ; ++q) find_bucket<kH1>(st->hist1[q], st->rank[q], s_scan, &s_bin[q], &s_res[q]);
    if (tid < kNQ) { st->prefix[tid] = (st->prefix[tid] << 11) | s_bin[tid]; st->rank[tid] = s_res[tid]; }
    return;
  }
  // LEVEL == 2: final order statistics, lerp, extents, indices
  const bool has_pos = st->n_pos != 0;
  if (has_pos) {
    for (int q = 0; q < kNQ; ++q) find_bucket<kH2>(st->hist2[q], st->rank[q], s_scan, &s_bin[q], &s_res[q]);
  }
  __syncthreads();
  // global max (needed for the no-positive branch) from the axis-0 plane maxima
  if (tid == 0) { s_first = 0; s_last = 0; }
  __syncthreads();
  {
    uint32_t m = 0;
    for (int i = tid; i < fa.T[0]; i += 256) m = max(m, st->plane_max[0][i]);
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(&s_last), m);
  }
  __syncthreads();
  if (tid == 0) {
    float lo, hi, den;
    if (has_pos) {
      float os[kNQ];
      for (int q = 0; q < kNQ; ++q) os[q] = __uint_as_float((st->prefix[q] << 8) | s_bin[q]);
      float r[2];
      for (int qi = 0; qi < 2; ++qi) {  // numpy _lerp in float32
        const float a = os[2 * qi], b = os[2 * qi + 1], g = st->gamma[qi];
        const float d = __fsub_rn(b, a);
        r[qi] = (g >= 0.5f) ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, g))) : __fadd_rn(a, __fmul_rn(d, g));
      }
      lo = r[0]; hi = r[1];
      den = __fadd_rn(__fsub_rn(hi, lo), 1e-6f);      // np.float32 scalars: stays float32
    } else {
      lo = ordered_to_float(st->gmin_key);            // float(np.min(volume)), float(np.max(volume))
      hi = ordered_to_float((uint32_t)s_last);
      den = __double2float_rn(__dadd_rn(__dsub_rn((double)hi, (double)lo), 1e-6));  // python floats: float64 then cast
    }
    s_lohi[0] = lo; s_lohi[1] = hi; s_lohi[2] = den;
    float* o = lohi + 4 * (size_t)blockIdx.x;
    o[0] = lo; o[1] = hi; o[2] = den; o[3] = has_pos ? 1.0f : 0.0f;
  }
  __syncthreads();
  const float lo = s_lohi[0], hi = s_lohi[1], den = s_lohi[2];
  int off = 0;
  for (int a = 0; a < fa.n_axes; ++a) {
    const int axis = fa.axes[a], T = fa.T[axis], count = fa.counts[a];
    if (tid == 0) { s_first = T; s_last = -1; }
    __syncthreads();
    int lf = T, ll = -1;
    for (int k = tid; k < T; k += 256) {
      const uint32_t key = st->plane_max[axis][k];
      if (key != 0) {
        const float pv = ordered_to_float(key);
        if ((fa.extent_raw ? pv : normalise(pv, lo, hi, den)) > 0.0f) { lf = min(lf, k); ll = max(ll, k); }
      }
    }
    for (int o = 16; o; o >>= 1) {
      lf = min(lf, __shfl_xor_sync(0xffffffffu, lf, o));
      ll = max(ll, __shfl_xor_sync(0xffffffffu, ll, o));
    }
    if ((tid & 31) == 0) { atomicMin(&s_first, lf); atomicMax(&s_last, ll); }
    __syncthreads();
    int first = s_first, last = s_last;
    if (last < 0) { first = 0; last = T - 1; }        // idxs = np.arange(axis_len)
    const int n = min(count, last - first + 1);
    if (tid == 0) nslices[(size_t)blockIdx.x * fa.n_axes + a] = n;
    // np.linspace(first, last, n).astype(int): float64 i*step + first, endpoint forced, truncation
    const double step = (n > 1) ? __ddiv_rn(__dsub_rn((double)last, (double)first), (double)(n - 1)) : 0.0;
    for (int t = tid; t < count; t += 256) {
      int v = -1;
      if (t < n) {
        if (n == 1) v = first;
        else if (t == n - 1) v = last;
        else v = (int)__dadd_rn(__dmul_rn((double)t, step), (double)first);
      }
      indices[(size_t)blockIdx.x * fa.lmax + off + t] = v;
    }
    off += count;
    __syncthreads();
  }
}

// LEVEL 1 scans the resampled volume: 11-bit histograms inside the four level-0 buckets, and every voxel of those buckets is
// appended to the subject's candidate list (one global atomic per warp and 512 voxels).  LEVEL 2 then builds the 8-bit
// histograms from the list -- a few per cent of the volume -- instead of streaming the volume from HBM a third time; a list that
// overflowed its capacity (a quarter of the volume: near-constant images) falls back to the full scan.
constexpr uint32_t kCandChunk = 512;   // = candidates one warp can find per iteration (32 lanes x 16 voxels)

template <int LEVEL>
__global__ void __launch_bounds__(256)
hist_kernel(const float* __restrict__ zoomed, SubjState* __restrict__ states, size_t voxels, uint32_t* __restrict__ cand, size_t cand_cap) {
  constexpr int NB = (LEVEL == 1) ? kH1 : kH2;
  __shared__ uint32_t s_hist[kNQ][NB];
  __shared__ uint32_t s_prefix[kNQ];
  pdl_launch_dependents();   // programmatic dependent launch (common.cuh): scheduled under the predecessor's tail,
  pdl_wait();                // nothing is read before the predecessor has completed
  SubjState* st = states + blockIdx.y;
  if (st->n_pos == 0) return;
  const int tid = threadIdx.x;
  for (int i = tid; i < kNQ * NB; i += 256) (&s_hist[0][0])[i] = 0;
  if (tid < kNQ) s_prefix[tid] = st->prefix[tid];
  __syncthreads();
  const uint32_t p0 = s_prefix[0], p1 = s_prefix[1], p2 = s_prefix[2], p3 = s_prefix[3];
  const float* zb = zoomed + (size_t)blockIdx.y * voxels;
  uint32_t* cb = cand + (size_t)blockIdx.y * cand_cap;
  // returns true when the voxel lies in one of the four queried buckets
  auto visit_bits = [&](uint32_t bits) -> bool {
    const uint32_t hi = (LEVEL == 1) ? (bits >> 19) : (bits >> 8);
    const uint32_t bin = (LEVEL == 1) ? ((bits >> 8) & 0x7ffu) : (bits & 0xffu);
    const bool m0 = hi == p0, m1 = hi == p1, m2 = hi == p2, m3 = hi == p3;
    if (m0) atomicAdd(&s_hist[0][bin], 1u);
    if (m1) atomicAdd(&s_hist[1][bin], 1u);
    if (m2) atomicAdd(&s_hist[2][bin], 1u);
    if (m3) atomicAdd(&s_hist[3][bin], 1u);
    return m0 | m1 | m2 | m3;
  };
  // LEVEL 1 hot path: two unsigned range checks per voxel instead of a sign test, a shift, four compares and four predicated
  // atomics.  Ranks f0 and f0+1 are consecutive order statistics, so every bucket strictly between p0 and p1 (p2 and p3) is
  // empty and "hi in {p0,p1}" is the range [p0 << 19, (p1 << 19) | 0x7ffff]; zero and negative bit patterns fall outside both.
  const uint32_t loA = max(p0 << 19, 1u), spanA = ((p1 << 19) | 0x7ffffu) - loA;
  const uint32_t loB = max(p2 << 19, 1u), spanB = ((p3 << 19) | 0x7ffffu) - loB;
  auto visit = [&](float v) -> bool {
    const uint32_t bits = __float_as_uint(v);
    if (LEVEL == 1) return ((bits - loA <= spanA) || (bits - loB <= spanB)) ? visit_bits(bits) : false;
    return v > 0.0f ? visit_bits(bits) : false;
  };
  bool from_list = false;
  if (LEVEL == 2) {
    const size_t n_list = st->n_cand;
    from_list = n_list <= cand_cap;
    if (from_list)
      for (size_t i = (size_t)blockIdx.x * 256 + tid; i < n_list; i += (size_t)gridDim.x * 256) visit_bits(__ldcs(cb + i));
  }
  if (!from_list) {
    const size_t n4 = voxels / 4;
    const float4* z4 = reinterpret_cast<const float4*>(zb);
    const bool aligned = ((reinterpret_cast<uintptr_t>(zb) & 15) == 0);
    const int lane = tid & 31;
    uint32_t cur = 0, left = 0;                                             // this warp's current chunk of the candidate list
    if (aligned) {
      // four independent 16-byte loads in flight per thread: the pass is latency-bound otherwise (one load per iteration)
      const size_t stride = (size_t)gridDim.x * 256;
      const size_t n_iter = (n4 + 4 * stride - 1) / (4 * stride);           // uniform trip count: the warp scan below needs all lanes
      size_t i = (size_t)blockIdx.x * 256 + tid;
      for (size_t it = 0; it < n_iter; ++it, i += 4 * stride) {
        float4 q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q[u] = (i + u * stride < n4) ? __ldcs(z4 + i + u * stride) : make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t mine = 0;                                                   // bit u*4+e: element e of load u is a candidate
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          // background (three quarters of a head volume) is skipped four voxels at a time, mostly by whole warps
          if (fmaxf(fmaxf(q[u].x, q[u].y), fmaxf(q[u].z, q[u].w)) > 0.0f) {
            if (visit(q[u].x)) mine |= 1u << (u * 4);
            if (visit(q[u].y)) mine |= 2u << (u * 4);
            if (visit(q[u].z)) mine |= 4u << (u * 4);
            if (visit(q[u].w)) mine |= 8u << (u * 4);
          }
        }
        if (LEVEL == 1 && __any_sync(0xffffffffu, mine != 0u)) {
          const uint32_t cnt = __popc(mine);
          uint32_t incl = cnt;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += nb;
          }
          const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);       // <= 512 = kCandChunk
          if (total) {
            // list space is reserved a chunk at a time per warp (one same-address atomic per 512 entries, not per iteration);
            // an iteration's candidates fill the rest of the current chunk and spill into the new one
            uint32_t fresh = 0;
            if (total > left) {
              if (lane == 0) fresh = atomicAdd(&st->n_cand, kCandChunk);
              fresh = __shfl_sync(0xffffffffu, fresh, 0);
            }
            uint32_t r = incl - cnt;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float e[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (mine & (1u << (u * 4 + k))) {
                  const size_t pos = (r < left) ? (size_t)cur + r : (size_t)fresh + (r - left);
                  if (pos < cand_cap) cb[pos] = __float_as_uint(e[k]);
                  ++r;
                }
            }
            if (total > left) { cur = fresh + (total - left); left = kCandChunk - (total - left); }
            else { cur += total; left -= total; }
          }
        }
      }
      if (LEVEL == 1) {                                                    // unused rest of the warp's last chunk: sentinels
        for (uint32_t k = lane; k < left; k += 32)
          if ((size_t)cur + k < cand_cap) cb[cur + k] = 0xffffffffu;       // sign bit set: never equals a (positive) prefix
      }
      // scalar tail (voxels % 4): too few to matter, appended one by one
      for (size_t t = n4 * 4 + (size_t)blockIdx.x * 256 + tid; t < voxels; t += (size_t)gridDim.x * 256) {
        if (visit(zb[t]) && LEVEL == 1) { const uint32_t pos = atomicAdd(&st->n_cand, 1u); if (pos < cand_cap) cb[pos] = __float_as_uint(zb[t]); }
      }
    } else {
      for (size_t t = (size_t)blockIdx.x * 256 + tid; t < voxels; t += (size_t)gridDim.x * 256) {
        if (visit(zb[t]) && LEVEL == 1) { const uint32_t pos = atomicAdd(&st->n_cand, 1u); if (pos < cand_cap) cb[pos] = __float_as_uint(zb[t]); }
      }
    }
  }
  __syncthreads();
  for (int i = tid; i < kNQ * NB; i += 256) {
    const uint32_t c = (&s_hist[0][0])[i];
    if (c) {
      if (LEVEL == 1) atomicAdd(&st->hist1[i / NB][i % NB], c);
      else atomicAdd(&st->hist2[i / NB][i % NB], c);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
__global__ void normalize_kernel(const float* __restrict__ zoomed, const float* __restrict__ lohi, float* __restrict__ out,
                                 size_t voxels) {
  const float* l = lohi + 4 * (size_t)blockIdx.y;
  const float lo = l[0], hi = l[1], den = l[2];
  const size_t base = (size_t)blockIdx.y * voxels;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < voxels; i += (size_t)gridDim.x * blockDim.x)
    out[base + i] = normalise(zoomed[base + i], lo, hi, den);
}

// axis-2 planes: vol[:, :, idx] has stride T2 between neighbours; copy the selected planes into a compact
// [B][L2][T0*T1] buffer (coalesced writes) so the resize kernel reads rows.
__global__ void extract_planes_kernel(const float* __restrict__ zoomed, const int32_t* __restrict__ indices, int lmax,
                                      int off2, int cnt2, float* __restrict__ planes, int T0, int T1, int T2,
                                      const float* __restrict__ lohi) {
  pdl_launch_dependents();   // programmatic dependent launch (common.cuh): scheduled under the predecessor's tail,
  pdl_wait();                // nothing is read before the predecessor has completed
  const int b = blockIdx.z, l = blockIdx.y;
  const int idx = indices[(size_t)b * lmax + off2 + l];
  if (idx < 0) return;
  const size_t n = (size_t)T0 * T1;
  const float* zb = zoomed + (size_t)b * n * T2 + idx;
  float* pb = planes + ((size_t)b * cnt2 + l) * n;
  // the p1/p99 clip of `_normalize_volume_for_resnet` is applied here, once per voxel: the resize kernel would otherwise clip each
  // voxel once per output pixel that taps it (~8x); this kernel is HBM-bound and does it for free
  const float lo = lohi[4 * (size_t)b], hi = lohi[4 * (size_t)b + 1];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    pb[i] = fminf(fmaxf(__ldg(zb + i * T2), lo), hi);
}

struct ResizeArgs {
  int zmajor;       // 1: zoomed is slice-major [T2][T0][T1] (axis-2 planes contiguous, un-clipped); `planes` is not used
  int T[3];
  int n_axes;
  int axes[PDF_MAX_AXES];
  int counts[PDF_MAX_AXES];
  int lmax, S, cnt2;
  int pitch, rows;  // PDF_OUT_BF16_C1_PAD geometry
  int ready;        // 1: `planes` holds ready-made normalised slices [B, lmax, T0, T1] (pdf_resize_slices): no clip / min-max
  float mean[3], inv_std[3];
  float scale_sq;   // T/S when the slice is square (the usual cubic target), hoisted out of the kernel
};

// Each thread produces 4 horizontally adjacent output pixels of one slice (shares the row geometry, 8-byte bf16 store).
// The min-max affine map is applied AFTER the interpolation (bilinear weights sum to 1, so only rounding differs,
// ~1e-7, against a 1e-5 contract); the clip is applied per tap as in the reference.
template <int MODE>
__global__ void __launch_bounds__(256)
resize_kernel(const float* __restrict__ zoomed, const float* __restrict__ planes, const float* __restrict__ lohi,
              const int32_t* __restrict__ indices, const int32_t* __restrict__ nslices, void* __restrict__ out, ResizeArgs ra) {
  const int b = blockIdx.z, l = blockIdx.y;
  const int S = ra.S;
  constexpr bool PAD = MODE == PDF_OUT_BF16_C1_PAD;
  const int gpr = PAD ? (ra.pitch >> 2) : ((S + 3) >> 2);   // 4-pixel groups per output row
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= gpr * S) return;
  const int oy = g / gpr;
  const int ox0 = (g - oy * gpr) * 4 - (PAD ? PDF_STEM_PAD_LO : 0);   // first image column of the group (may be < 0 when padded)
  const int npx = PAD ? 4 : min(4, S - ox0);
  // locate the axis group of slot l
  int a = 0, t = l, off2 = 0;
  while (a < ra.n_axes - 1 && t >= ra.counts[a]) { if (ra.axes[a] == 2) off2 += ra.counts[a]; t -= ra.counts[a]; ++a; }
  const int axis = ra.axes[a];
  const bool valid = ra.ready ? true : t < nslices[(size_t)b * ra.n_axes + a];
  const size_t opix = PAD ? (((size_t)b * ra.lmax + l) * ra.rows + oy + PDF_STEM_PAD_LO) * ra.pitch + (size_t)(ox0 + PDF_STEM_PAD_LO)
                          : ((size_t)b * ra.lmax + l) * S * S + (size_t)oy * S + ox0;
  float r[4] = {0.f, 0.f, 0.f, 0.f};
  if (valid) {
    const int idx = ra.ready ? 0 : indices[(size_t)b * ra.lmax + l];
    const int T0 = ra.T[0], T1 = ra.T[1], T2 = ra.T[2];
    const float* src;
    int H, W;
    size_t rs;
    if (axis == 0) { src = zoomed + ((size_t)b * T0 + idx) * T1 * T2; H = T1; W = T2; rs = T2; }
    else if (axis == 1) { src = zoomed + (size_t)b * T0 * T1 * T2 + (size_t)idx * T2; H = T0; W = T2; rs = (size_t)T1 * T2; }
    else if (ra.zmajor) { src = zoomed + ((size_t)b * T2 + idx) * T0 * T1; H = T0; W = T1; rs = T1; }
    else { src = planes + ((size_t)b * ra.cnt2 + off2 + t) * T0 * T1; H = T0; W = T1; rs = T1; }
    const float* l4 = lohi + 4 * (size_t)b;
    const float lo = ra.ready ? 0.0f : l4[0], hi = ra.ready ? 1.0f : l4[1];       // ready slices already lie in [0, 1]
    const float inv_den = ra.ready ? 1.0f : __frcp_rn(l4[2]);
    // ATen area_pixel_compute_source_index(align_corners=False): (dst + 0.5) * (in/out) - 0.5, clamped at 0
    const float sh = (H == W) ? ra.scale_sq : __fdiv_rn((float)H, (float)S);
    const float sw = (H == W) ? ra.scale_sq : __fdiv_rn((float)W, (float)S);
    const float fy = fmaxf(__fsub_rn(__fmul_rn(__fadd_rn((float)oy, 0.5f), sh), 0.5f), 0.0f);
    const int y0 = min((int)fy, H - 1), y1 = min(y0 + 1, H - 1);
    const float wy1 = __fsub_rn(fy, (float)y0), wy0 = __fsub_rn(1.0f, wy1);
    const float* row0 = src + y0 * rs;
    const float* row1 = src + y1 * rs;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ox = min(max(ox0 + j, 0), S - 1);
      const float fx = fmaxf(__fsub_rn(__fmul_rn(__fadd_rn((float)ox, 0.5f), sw), 0.5f), 0.0f);
      const int x0 = min((int)fx, W - 1), x1 = min(x0 + 1, W - 1);
      const float wx1 = __fsub_rn(fx, (float)x0), wx0 = __fsub_rn(1.0f, wx1);
      const float v00 = fminf(fmaxf(__ldg(row0 + x0), lo), hi), v01 = fminf(fmaxf(__ldg(row0 + x1), lo), hi);
      const float v10 = fminf(fmaxf(__ldg(row1 + x0), lo), hi), v11 = fminf(fmaxf(__ldg(row1 + x1), lo), hi);
      const float top = __fadd_rn(__fmul_rn(wx0, v00), __fmul_rn(wx1, v01));
      const float bot = __fadd_rn(__fmul_rn(wx0, v10), __fmul_rn(wx1, v11));
      r[j] = (__fadd_rn(__fmul_rn(wy0, top), __fmul_rn(wy1, bot)) - lo) * inv_den;
    }
  }
  if (MODE == PDF_OUT_BF16_C1 || PAD) {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out) + opix;
    __nv_bfloat16 h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool inb = !PAD || (ox0 + j >= 0 && ox0 + j < S);      // border pixels of a padded group stay exactly 0
      h[j] = __float2bfloat16((valid && inb) ? (r[j] - ra.mean[0]) * ra.inv_std[0] : 0.0f);
    }
    if (npx == 4 && ((reinterpret_cast<uintptr_t>(o) & 7) == 0)) {
      uint2 pk;
      pk.x = (uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16);
      pk.y = (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16);
      *reinterpret_cast<uint2*>(o) = pk;
    } else {
      for (int j = 0; j < npx; ++j) o[j] = h[j];
    }
  } else {
    float* o = reinterpret_cast<float*>(out) + opix * 3;
    for (int j = 0; j < npx; ++j) {
#pragma unroll
      for (int c = 0; c < 3; ++c) o[j * 3 + c] = valid ? (r[j] - ra.mean[c]) * ra.inv_std[c] : 0.0f;
    }
  }
}

// bf16 outputs: a thread owns four adjacent output columns for a band of rows, so the horizontal source indices and
// weights are computed once and stay in registers; per pixel only the four loads, the clips and the blend remain
// (the generic kernel above spends ~110 instructions per pixel, mostly on index arithmetic).
// block (64, 4): x = column group (4 pixels), y = row lane; grid (row bands of kBandRows, slices, subjects).
constexpr int kBandRows = 32;
// PRECLIP: every slot reads pre-clipped axis-2 planes (extract_planes_kernel), so the four taps need no clip here.
template <int MODE, bool PRECLIP>
__global__ void __launch_bounds__(256)
resize_band_kernel(const float* __restrict__ zoomed, const float* __restrict__ planes, const float* __restrict__ lohi,
                   const int32_t* __restrict__ indices, const int32_t* __restrict__ nslices, __nv_bfloat16* __restrict__ out, ResizeArgs ra) {
  constexpr bool PAD = MODE == PDF_OUT_BF16_C1_PAD;
  pdl_launch_dependents();   // programmatic dependent launch (common.cuh): scheduled under the predecessor's tail,
  pdl_wait();                // nothing is read before the predecessor has completed
  const int b = blockIdx.z, l = blockIdx.y;
  const int S = ra.S;
  const int gpr = PAD ? (ra.pitch >> 2) : ((S + 3) >> 2);
  const int cg = threadIdx.x;
  if (cg >= gpr) return;
  const int ox0 = cg * 4 - (PAD ? PDF_STEM_PAD_LO : 0);
  int a = 0, t = l, off2 = 0;
  while (a < ra.n_axes - 1 && t >= ra.counts[a]) { if (ra.axes[a] == 2) off2 += ra.counts[a]; t -= ra.counts[a]; ++a; }
  const int axis = ra.axes[a];
  const bool valid = ra.ready ? true : t < nslices[(size_t)b * ra.n_axes + a];
  const int idx = (ra.ready || !valid) ? 0 : indices[(size_t)b * ra.lmax + l];
  const int T0 = ra.T[0], T1 = ra.T[1], T2 = ra.T[2];
  const float* src;
  int H, W;
  size_t rs;
  if (axis == 0) { src = zoomed + ((size_t)b * T0 + idx) * T1 * T2; H = T1; W = T2; rs = T2; }
  else if (axis == 1) { src = zoomed + (size_t)b * T0 * T1 * T2 + (size_t)idx * T2; H = T0; W = T2; rs = (size_t)T1 * T2; }
  else if (ra.zmajor) { src = zoomed + ((size_t)b * T2 + idx) * T0 * T1; H = T0; W = T1; rs = T1; }
  else { src = planes + ((size_t)b * ra.cnt2 + off2 + t) * T0 * T1; H = T0; W = T1; rs = T1; }
  float lo = 0.0f, hi = 1.0f, inv_den = 1.0f;                 // ready slices already lie in [0, 1]
  if (!ra.ready && valid) { const float* l4 = lohi + 4 * (size_t)b; lo = l4[0]; hi = l4[1]; inv_den = __frcp_rn(l4[2]); }
  // ATen area_pixel_compute_source_index(align_corners=False): (dst + 0.5) * (in/out) - 0.5, clamped at 0
  const float sh = (H == W) ? ra.scale_sq : __fdiv_rn((float)H, (float)S);
  const float sw = (H == W) ? ra.scale_sq : __fdiv_rn((float)W, (float)S);
  int x0[4], x1[4];
  float wx0[4], wx1[4];
  bool inb[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    inb[j] = ox0 + j >= 0 && ox0 + j < S;
    const int ox = min(max(ox0 + j, 0), S - 1);
    const float fx = fmaxf(__fsub_rn(__fmul_rn(__fadd_rn((float)ox, 0.5f), sw), 0.5f), 0.0f);
    x0[j] = min((int)fx, W - 1);
    x1[j] = min(x0[j] + 1, W - 1);
    wx1[j] = __fsub_rn(fx, (float)x0[j]);
    wx0[j] = __fsub_rn(1.0f, wx1[j]);
  }
  const float m0 = ra.mean[0], is0 = ra.inv_std[0];
  // A thread owns kBandRows / 4 CONSECUTIVE output rows: their source rows advance by H/S < 1 per step, so consecutive output rows
  // share source rows -- the horizontally blended values of a source row (wx0*v[x0] + wx1*v[x1], the same expression whichever
  // output row uses it) are kept in registers and reused: ~2.6 source rows are loaded and blended per 4 output rows instead of 8.
  constexpr int kRowsPerThread = kBandRows / 4;
  const int oy_beg = blockIdx.x * kBandRows + threadIdx.y * kRowsPerThread;
  const int oy_end = min(S, oy_beg + kRowsPerThread);
  float top[4] = {0.f, 0.f, 0.f, 0.f}, bot[4] = {0.f, 0.f, 0.f, 0.f};
  int cur0 = -1, cur1 = -1;                                   // source rows held in top[] / bot[]
  auto hblend = [&](const int y, float* dst) {
    const float* row = src + (size_t)y * rs;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a = 0.0f, c = 0.0f;
      if (valid && inb[j]) { a = __ldg(row + x0[j]); c = __ldg(row + x1[j]); }
      if (!PRECLIP) { a = fminf(fmaxf(a, lo), hi); c = fminf(fmaxf(c, lo), hi); }
      dst[j] = __fadd_rn(__fmul_rn(wx0[j], a), __fmul_rn(wx1[j], c));
    }
  };
#pragma unroll 1
  for (int oy = oy_beg; oy < oy_end; ++oy) {
    const float fy = fmaxf(__fsub_rn(__fmul_rn(__fadd_rn((float)oy, 0.5f), sh), 0.5f), 0.0f);
    const int y0 = min((int)fy, H - 1), y1 = min(y0 + 1, H - 1);
    const float wy1 = __fsub_rn(fy, (float)y0), wy0 = __fsub_rn(1.0f, wy1);
    if (y0 != cur0) {                                          // (warp-uniform: a warp shares threadIdx.y)
      if (y0 == cur1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) top[j] = bot[j];
      } else {
        hblend(y0, top);
      }
      cur0 = y0;
    }
    if (y1 != cur1) {
      if (y1 == cur0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) bot[j] = top[j];
      } else {
        hblend(y1, bot);
      }
      cur1 = y1;
    }
    uint32_t h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float r = 0.0f;
      if (valid && inb[j]) {
        const float nrm = __fmul_rn(__fsub_rn(__fadd_rn(__fmul_rn(wy0, top[j]), __fmul_rn(wy1, bot[j])), lo), inv_den);
        r = __fmul_rn(__fsub_rn(nrm, m0), is0);     // same roundings as the f32 layout: no fused multiply-add
      }
      h[j] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16(r));
    }
    const size_t opix = PAD ? (((size_t)b * ra.lmax + l) * ra.rows + oy + PDF_STEM_PAD_LO) * ra.pitch + (size_t)(cg * 4)
                            : ((size_t)b * ra.lmax + l) * S * S + (size_t)oy * S + ox0;
    __nv_bfloat16* o = out + opix;
    if ((PAD || ox0 + 4 <= S) && ((reinterpret_cast<uintptr_t>(o) & 7) == 0)) {
      *reinterpret_cast<uint2*>(o) = make_uint2(h[0] | (h[1] << 16), h[2] | (h[3] << 16));
    } else {
      for (int j = 0; j < 4 && ox0 + j < S; ++j) o[j] = __ushort_as_bfloat16((unsigned short)h[j]);
    }
  }
}

// normalised selected slices themselves ([B, Lmax, H, W] f32, `_select_slices` of the normalised volume): the input of
// the test-time-augmentation path.  Axis 0 -> [n, Y, Z], axis 1 -> [n, X, Z], axis 2 -> [n, X, Y].
__global__ void gather_slices_kernel(const float* __restrict__ zoomed, const float* __restrict__ lohi, const int32_t* __restrict__ indices,
                                     const int32_t* __restrict__ nslices, float* __restrict__ out, FinalizeArgs fa, int H, int W) {
  const int b = blockIdx.z, l = blockIdx.y;
  int a = 0, t = l;
  while (a < fa.n_axes - 1 && t >= fa.counts[a]) { t -= fa.counts[a]; ++a; }
  const int axis = fa.axes[a];
  const bool valid = t < nslices[(size_t)b * fa.n_axes + a];
  const int idx = valid ? indices[(size_t)b * fa.lmax + l] : 0;
  const int T1 = fa.T[1], T2 = fa.T[2];
  const float* zb = zoomed + (size_t)b * fa.T[0] * T1 * T2;
  const float* l4 = lohi + 4 * (size_t)b;
  const float lo = l4[0], hi = l4[1], den = l4[2];
  float* ob = out + ((size_t)b * fa.lmax + l) * H * W;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += gridDim.x * blockDim.x) {
    float v = 0.0f;
    if (valid) {
      const int y = i / W, x = i - y * W;
      const size_t src = axis == 0 ? ((size_t)idx * T1 + y) * T2 + x : axis == 1 ? ((size_t)y * T1 + idx) * T2 + x : ((size_t)y * T1 + x) * T2 + idx;
      v = normalise(__ldg(zb + src), lo, hi, den);
    }
    ob[i] = v;
  }
}

// a6, one augmentation pass: scipy.ndimage.affine_transform(order=1, mode="constant", cval=0) of every slice with the
// subject's matrix/offset (float64 coordinates and weights, taps accumulated as ((v*wy)*wx) row-major, one rounding to
// f32), then x*scale+shift in float32, + noise in float64 (when given), clip to [0,1], float32
// (data/openneuro_features.py:166-178, 237-248; scripts/build_resnet2d_mil_embeddings.py:126-139).
__global__ void tta_kernel(const float* __restrict__ slices, const pdf_tta_params* __restrict__ params, const double* __restrict__ noise,
                           float* __restrict__ out, int L, int H, int W, int affine_only) {
  const int b = blockIdx.z, l = blockIdx.y;
  const pdf_tta_params pr = params[b];
  const size_t base = ((size_t)b * L + l) * H * W;
  const float* img = slices + base;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += gridDim.x * blockDim.x) {
    const int oy = i / W, ox = i - oy * W;
    const double c0 = __dadd_rn(__dadd_rn(pr.offset[0], __dmul_rn((double)oy, pr.rot[0])), __dmul_rn((double)ox, pr.rot[1]));
    const double c1 = __dadd_rn(__dadd_rn(pr.offset[1], __dmul_rn((double)oy, pr.rot[2])), __dmul_rn((double)ox, pr.rot[3]));
    float a = 0.0f;
    if (c0 >= 0.0 && c0 <= (double)(H - 1) && c1 >= 0.0 && c1 <= (double)(W - 1)) {
      const double f0 = floor(c0), f1 = floor(c1);
      const double y = __dsub_rn(c0, f0), x = __dsub_rn(c1, f1);
      const int i0 = (int)f0, j0 = (int)f1;
      const bool i1ok = i0 + 1 < H, j1ok = j0 + 1 < W;
      const double wy0 = __dsub_rn(1.0, y), wx0 = __dsub_rn(1.0, x);
      const double v00 = (double)img[i0 * W + j0];
      const double v01 = j1ok ? (double)img[i0 * W + j0 + 1] : 0.0;
      const double v10 = i1ok ? (double)img[(i0 + 1) * W + j0] : 0.0;
      const double v11 = (i1ok && j1ok) ? (double)img[(i0 + 1) * W + j0 + 1] : 0.0;
      double t = 0.0;
      t = __dadd_rn(t, __dmul_rn(__dmul_rn(v00, wy0), wx0));
      t = __dadd_rn(t, __dmul_rn(__dmul_rn(v01, wy0), x));
      t = __dadd_rn(t, __dmul_rn(__dmul_rn(v10, y), wx0));
      t = __dadd_rn(t, __dmul_rn(__dmul_rn(v11, y), x));
      a = __double2float_rn(t);
    }
    if (affine_only) { out[base + i] = a; continue; }      // `_apply_affine_2d` alone
    a = __fadd_rn(__fmul_rn(a, pr.scale), pr.shift);
    float r;
    if (noise) {
      const double d = __dadd_rn((double)a, noise[base + i]);
      r = __double2float_rn(fmin(fmax(d, 0.0), 1.0));
    } else {
      r = fminf(fmaxf(a, 0.0f), 1.0f);
    }
    out[base + i] = r;
  }
}

// ------------------------------------------------------------------------------------------------------
// Voxel decode on the device (SURVEY.md 8f rank 1): the stored voxels of a NIfTI-1 image (any integer or float type, Fortran
// order: x fastest) -> what `nib.load(p).get_fdata().astype(np.float32)` hands the reference (data/openneuro_features.py:24-25):
// float64(raw) [* scl_slope + scl_inter, two roundings, no FMA] -> float32, laid out C-order [X][Y][Z] as the resample kernel
// reads it.  An int16 volume then crosses PCIe at half the bytes of the float32 array the reference would upload.
template <typename T>
__device__ __forceinline__ float decode_one(T v, bool scale, double slope, double inter) {
  double d = (double)v;
  if (scale) d = __dadd_rn(__dmul_rn(d, slope), inter);
  return __double2float_rn(d);
}

// Fortran-order source: a 32 (x) by 32 (z) tile is transposed through shared memory so that both the reads (x fastest) and the
// writes (z fastest) are coalesced.  grid (ceil(X/32), ceil(Z/32), Y * batch), block (32, 8).
template <typename T>
__device__ __forceinline__ void decode_fortran_tile(const T* __restrict__ sb, float* __restrict__ db, int X, int Y, int Z, int x0, int y,
                                                    int z0, bool scale, double slope, double inter, float (*tile)[33]) {
#pragma unroll
  for (int k = 0; k < 32; k += 8) {
    const int x = x0 + threadIdx.x, z = z0 + threadIdx.y + k;
    if (x < X && z < Z) tile[threadIdx.y + k][threadIdx.x] = decode_one(sb[(size_t)x + (size_t)X * (y + (size_t)Y * z)], scale, slope, inter);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 32; k += 8) {
    const int x = x0 + threadIdx.y + k, z = z0 + threadIdx.x;
    if (x < X && z < Z) db[((size_t)x * Y + y) * Z + z] = tile[threadIdx.x][threadIdx.y + k];
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
decode_fortran_kernel(const T* __restrict__ src, float* __restrict__ dst, int X, int Y, int Z, bool scale, double slope, double inter) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z / Y, y = blockIdx.z - b * Y;
  decode_fortran_tile<T>(src + (size_t)b * X * Y * Z, dst + (size_t)b * X * Y * Z, X, Y, Z, blockIdx.x * 32, y, blockIdx.y * 32, scale,
                         slope, inter, tile);
}

template <typename T>
__global__ void __launch_bounds__(256)
decode_linear_kernel(const T* __restrict__ src, float* __restrict__ dst, size_t n, bool scale, double slope, double inter) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dst[i] = decode_one(src[i], scale, slope, inter);
}

template <typename T>
static int launch_decode(int batch, int X, int Y, int Z, int fortran, bool scale, double slope, double inter, const void* src,
                         float* dst, cudaStream_t s) {
  if (fortran) {
    const dim3 grid(ceil_div(X, 32), ceil_div(Z, 32), Y * batch);
    decode_fortran_kernel<T><<<grid, dim3(32, 8), 0, s>>>(reinterpret_cast<const T*>(src), dst, X, Y, Z, scale, slope, inter);
  } else {
    const size_t n = (size_t)batch * X * Y * Z;
    const int blocks = (int)min((size_t)num_sms() * 16, (n + 255) / 256);
    decode_linear_kernel<T><<<max(1, blocks), 256, 0, s>>>(reinterpret_cast<const T*>(src), dst, n, scale, slope, inter);
  }
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

// Ragged decode: one launch over subjects of mixed type, order and scaling.  Blocks are numbered through the subjects (blk_start:
// first block of each subject); a Fortran-order subject gets one block per 32 x 32 (x, z) tile and y, as decode_fortran_kernel, a
// C-order subject one block per kDecodeChunk voxels.  The datatype is a per-block switch: every block decodes one subject.
constexpr int kDecodeChunk = 4096;
struct DecodeSubj {
  long long src_off, raw_off;   // bytes into d_src; float32 elements into d_dst
  int X, Y, Z, code, fortran, scale;
  double slope, inter;
};
struct DecodeGeom {
  int n, pad;
  int blk_start[PDF_RAGGED_MAX_BATCH + 1];
  DecodeSubj s[PDF_RAGGED_MAX_BATCH];
};

template <typename T>
__device__ __forceinline__ void decode_ragged_block(const unsigned char* __restrict__ src, float* __restrict__ dst, const DecodeSubj& d,
                                                    int blk, float (*tile)[33]) {
  const T* sb = reinterpret_cast<const T*>(src + d.src_off);
  float* db = dst + d.raw_off;
  if (d.fortran) {
    const int gx = (d.X + 31) / 32, gxz = gx * ((d.Z + 31) / 32);
    const int y = blk / gxz, r = blk - y * gxz, zt = r / gx, xt = r - zt * gx;
    decode_fortran_tile<T>(sb, db, d.X, d.Y, d.Z, xt * 32, y, zt * 32, d.scale != 0, d.slope, d.inter, tile);
  } else {
    const size_t n = (size_t)d.X * d.Y * d.Z, end = min(n, (size_t)(blk + 1) * kDecodeChunk);
    for (size_t i = (size_t)blk * kDecodeChunk + threadIdx.y * 32 + threadIdx.x; i < end; i += 256)
      db[i] = decode_one(sb[i], d.scale != 0, d.slope, d.inter);
  }
}

__global__ void __launch_bounds__(256)
decode_ragged_kernel(const unsigned char* __restrict__ src, float* __restrict__ dst, const __grid_constant__ DecodeGeom g) {
  __shared__ float tile[32][33];
  int lo = 0, hi = g.n - 1;                     // last subject whose first block is <= blockIdx.x
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (g.blk_start[mid] <= (int)blockIdx.x) lo = mid;
    else hi = mid - 1;
  }
  const DecodeSubj& d = g.s[lo];
  const int blk = (int)blockIdx.x - g.blk_start[lo];
  switch (d.code) {
    case 2: decode_ragged_block<uint8_t>(src, dst, d, blk, tile); break;
    case 4: decode_ragged_block<int16_t>(src, dst, d, blk, tile); break;
    case 8: decode_ragged_block<int32_t>(src, dst, d, blk, tile); break;
    case 16: decode_ragged_block<float>(src, dst, d, blk, tile); break;
    case 64: decode_ragged_block<double>(src, dst, d, blk, tile); break;
    case 256: decode_ragged_block<int8_t>(src, dst, d, blk, tile); break;
    case 512: decode_ragged_block<uint16_t>(src, dst, d, blk, tile); break;
    default: decode_ragged_block<uint32_t>(src, dst, d, blk, tile); break;   // 768 (the host admits no other code)
  }
}

static int nifti_elem_bytes(int code) {
  switch (code) {
    case 2: case 256: return 1;
    case 4: case 512: return 2;
    case 8: case 16: case 768: return 4;
    case 64: return 8;
    default: return 0;
  }
}

// nibabel applies the scaling only when scl_slope is finite and non-zero and (slope, inter) != (1, 0); a non-finite inter counts as 0
static bool nifti_scales(double slope, double inter) { return slope != 0.0 && isfinite(slope) && !(slope == 1.0 && inter == 0.0); }

}  // namespace pdf

using namespace pdf;

extern "C" int pdf_decode_volumes(int batch, const pdf_volume_desc* descs, const void* d_src, float* d_dst, pdf_stream_t stream) {
  PDF_REQUIRE(batch > 0 && batch <= PDF_RAGGED_MAX_BATCH && descs && d_src && d_dst,
              "pdf_decode_volumes: bad arguments (batch must be 1..%d)", PDF_RAGGED_MAX_BATCH);
  DecodeGeom g;
  memset(&g, 0, sizeof(g));
  g.n = batch;
  long long blocks = 0;
  for (int b = 0; b < batch; ++b) {
    const pdf_volume_desc& v = descs[b];
    const int eb = nifti_elem_bytes(v.nifti_datatype);
    PDF_REQUIRE(eb > 0, "pdf_decode_volumes: subject %d: unsupported NIfTI datatype %d", b, v.nifti_datatype);
    PDF_REQUIRE(v.shape[0] > 0 && v.shape[1] > 0 && v.shape[2] > 0, "pdf_decode_volumes: subject %d: bad shape", b);
    PDF_REQUIRE(v.src_offset >= 0 && v.src_offset % eb == 0, "pdf_decode_volumes: subject %d: src_offset must be a non-negative "
                "multiple of the element size", b);
    PDF_REQUIRE(v.raw_offset >= 0 && v.raw_offset % 4 == 0, "pdf_decode_volumes: subject %d: raw_offset must be a non-negative "
                "multiple of 4", b);
    DecodeSubj& d = g.s[b];
    d.src_off = v.src_offset; d.raw_off = v.raw_offset;
    d.X = v.shape[0]; d.Y = v.shape[1]; d.Z = v.shape[2];
    d.code = v.nifti_datatype; d.fortran = v.fortran_order ? 1 : 0;
    d.scale = nifti_scales(v.slope, v.inter) ? 1 : 0;
    d.slope = v.slope; d.inter = isfinite(v.inter) ? v.inter : 0.0;
    g.blk_start[b] = (int)blocks;
    blocks += d.fortran ? (long long)ceil_div(d.X, 32) * ceil_div(d.Z, 32) * d.Y
                        : ((long long)d.X * d.Y * d.Z + kDecodeChunk - 1) / kDecodeChunk;
    PDF_REQUIRE(blocks < (1LL << 31), "pdf_decode_volumes: batch too large for one launch");
  }
  g.blk_start[batch] = (int)blocks;
  decode_ragged_kernel<<<(unsigned)blocks, dim3(32, 8), 0, as_stream(stream)>>>(reinterpret_cast<const unsigned char*>(d_src), d_dst, g);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_decode_volume(int batch, int nifti_datatype, int X, int Y, int Z, int fortran_order, double slope, double inter,
                                 const void* d_src, float* d_dst, pdf_stream_t stream) {
  PDF_REQUIRE(batch > 0 && X > 0 && Y > 0 && Z > 0 && d_src && d_dst, "pdf_decode_volume: bad arguments");
  PDF_REQUIRE((long long)Y * batch <= 65535, "pdf_decode_volume: Y * batch exceeds the grid limit");
  const bool scale = nifti_scales(slope, inter);
  if (!isfinite(inter)) inter = 0.0;
  cudaStream_t s = as_stream(stream);
  switch (nifti_datatype) {
    case 2: return launch_decode<uint8_t>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 4: return launch_decode<int16_t>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 8: return launch_decode<int32_t>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 16: return launch_decode<float>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 64: return launch_decode<double>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 256: return launch_decode<int8_t>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 512: return launch_decode<uint16_t>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    case 768: return launch_decode<uint32_t>(batch, X, Y, Z, fortran_order, scale, slope, inter, d_src, d_dst, s);
    default: break;
  }
  PDF_REQUIRE(false, "pdf_decode_volume: unsupported NIfTI datatype %d", nifti_datatype);
}

namespace pdf {
}  // namespace pdf

using namespace pdf;

static int g_pre_chunk = 0;   // subjects per pdf_preprocess sub-batch (0 = whole batch); pdf_debug_set_pre_chunk

static size_t uniform_workspace_bytes(const pdf_preproc_cfg* cfg, int batch) {
  size_t n = align_up(sizeof(ZoomTables), 256) + align_up(sizeof(SubjState) * (size_t)batch, 256);
  n += align_up((size_t)batch * count_axis2(cfg) * cfg->out_shape[0] * cfg->out_shape[1] * sizeof(float), 256);
  n += (size_t)batch * cand_capacity(cfg) * sizeof(uint32_t);
  return n + 256;
}

// per-subject interpolation tables of a ragged call: after the uniform regions, which keep their places
static ZoomTables* ragged_tables(const pdf_preproc_cfg* cfg, int batch, void* ws) {
  return reinterpret_cast<ZoomTables*>(reinterpret_cast<char*>(ws) + align_up(uniform_workspace_bytes(cfg, batch), 256));
}

extern "C" int pdf_preproc_slice_major_ok(const pdf_preproc_cfg* cfg) { return slice_major_ok(cfg) ? 1 : 0; }

extern "C" int pdf_preproc_slice_major_ok_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs) {
  if (!cfg || !descs || batch <= 0 || batch > PDF_RAGGED_MAX_BATCH) return 0;
  for (int b = 0; b < batch; ++b)
    if (!slice_major_ok_shape(cfg, descs[b].shape[1], descs[b].shape[2])) return 0;
  return 1;
}

extern "C" size_t pdf_preproc_workspace_bytes(const pdf_preproc_cfg* cfg, int batch) {
  if (!cfg || batch <= 0) return 0;
  return uniform_workspace_bytes(cfg, batch);
}

extern "C" size_t pdf_preproc_ragged_workspace_bytes(const pdf_preproc_cfg* cfg, int batch) {
  if (!cfg || batch <= 0 || batch > PDF_RAGGED_MAX_BATCH) return 0;
  return align_up(uniform_workspace_bytes(cfg, batch), 256) + (size_t)batch * sizeof(ZoomTables);
}

// K1a for a uniform batch (descs == nullptr: geometry from cfg->in_shape, subject b at b * X*Y*Z) or a ragged one.  Every subject
// goes through the bulk-copy kernel when its rows fit the staging ring at two rows per tile (Z % 4 == 0, <= 110 KB), the others
// through resample_kernel in a second launch.  The tile height TJ of each launch is chosen once, for its largest subject.
static int resample_impl(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs, const float* d_raw, float* d_zoomed,
                         void* d_workspace, cudaStream_t s) {
  Workspace w = carve(cfg, batch, d_workspace);
  const int T0 = cfg->out_shape[0], T1 = cfg->out_shape[1], T2 = cfg->out_shape[2];
  const int n = descs ? batch : 1;                      // geometry entries
  ZoomTables* rtabs = descs ? ragged_tables(cfg, batch, d_workspace) : nullptr;
  ResampleGeom gi;                                      // all entries: interpolation tables
  memset(&gi, 0, sizeof(gi));
  gi.uniform = descs ? 0 : 1;
  gi.n = n;
  for (int e = 0; e < n; ++e) {
    ResampleSubj& r = gi.s[e];
    const int32_t* sh = descs ? descs[e].shape : cfg->in_shape;
    r.X = sh[0]; r.Y = sh[1]; r.Z = sh[2];
    r.subj = e;
    r.raw_off = descs ? descs[e].raw_offset : 0;
    r.tabs = descs ? rtabs + e : w.tabs;
  }
  const size_t fixed = (size_t)(kH0 + T0 + T1) * sizeof(uint32_t);
  const int KT = (T2 + 31) / 32 * 32;
  const bool tma_batch = ((reinterpret_cast<uintptr_t>(d_raw) & 15) == 0) && KT <= 160 && T1 >= 2;
  auto rows = [&](const ResampleSubj& r, int TJ) { return (int)((TJ - 1) * ((double)(r.Y - 1) / (double)(T1 - 1))) + 3; };
  // bulk-copy pipeline: TJ output rows per tile, kResStages stages of 2 x NR x Z floats
  auto tma_smem = [&](size_t plane) { return (size_t)kResStages * 2 * plane * 4 + fixed + 16 + (size_t)T1 * 32 + 2 * kResStages * 8 + 128; };
  auto res_smem = [&](size_t plane_even) { return 2 * plane_even * sizeof(double) + fixed; };
  bool tma[PDF_RAGGED_MAX_BATCH];
  int n_tma = 0;
  for (int e = 0; e < n; ++e) {
    const ResampleSubj& r = gi.s[e];
    tma[e] = tma_batch && r.Z % 4 == 0 && tma_smem((size_t)rows(r, 2) * r.Z) <= 110 * 1024;
    n_tma += tma[e];
  }
  bool need_jmax = false;
  for (int a = 0; a < cfg->n_axes; ++a) need_jmax |= cfg->axes[a] == 1;
  ResampleGeom gt, gr;                                   // the two launches
  int TJt = 8, TJr = 8;
  size_t smem_t = 0, smem_r = 0;
  if (n_tma) {
    for (; TJt >= 2; TJt >>= 1) {
      size_t plane = 0;
      for (int e = 0; e < n; ++e) if (tma[e]) plane = max(plane, (size_t)rows(gi.s[e], TJt) * gi.s[e].Z);
      smem_t = tma_smem(plane);
      if (smem_t <= 110 * 1024) break;
    }
    memset(&gt, 0, sizeof(gt));
    gt.uniform = gi.uniform;
    for (int e = 0; e < n; ++e) {
      if (!tma[e]) continue;
      ResampleSubj r = gi.s[e];
      r.NR = rows(r, TJt);
      gt.plane_max = max(gt.plane_max, r.NR * r.Z);
      gt.s[gt.n++] = r;
    }
    if (cfg->slice_major)
      PDF_REQUIRE(n_tma == n && TJt == 8 && T1 % 8 == 0 && !need_jmax, "pdf_resample_stats: slice_major needs 8-row tiles (T1 %% 8 == 0, "
                  "rows that fit the staging ring) -- check pdf_preproc_slice_major_ok first");
  }
  if (n_tma < n) {
    PDF_REQUIRE(!cfg->slice_major, "pdf_resample_stats: slice_major needs the bulk-copy resample kernel (Z %% 4 == 0, T2 <= 160): check "
                "pdf_preproc_slice_major_ok first");
    // rows per tile: as many as fit the shared-memory staging buffer (2 planes x NR input rows x Z doubles)
    size_t plane = 0;
    for (; TJr >= 1; TJr >>= 1) {
      plane = 0;
      for (int e = 0; e < n; ++e) if (!tma[e]) plane = max(plane, ((size_t)rows(gi.s[e], TJr) * gi.s[e].Z + 1) & ~(size_t)1);
      smem_r = res_smem(plane);
      if (smem_r <= 72 * 1024 || TJr == 1) break;
    }
    PDF_REQUIRE(smem_r <= 200 * 1024, "pdf_resample_stats: volume rows too long for the shared-memory staging buffer");
    memset(&gr, 0, sizeof(gr));
    gr.uniform = gi.uniform;
    gr.plane_max = (int)plane;
    for (int e = 0; e < n; ++e) {
      if (tma[e]) continue;
      ResampleSubj r = gi.s[e];
      r.NR = rows(r, TJr);
      gr.s[gr.n++] = r;
    }
  }

  PDF_CHECK_CUDA(cudaMemsetAsync(w.st, 0, sizeof(SubjState) * (size_t)batch, s));
  const int tmax = max(max(T0, T1), max(T2, batch));
  init_tables_kernel<<<dim3(ceil_div(tmax, 256), n), 256, 0, s>>>(gi, w.st, batch, T0, T1, T2);
  PDF_CHECK_LAUNCH();
  // subjects per launch: all of a uniform batch (one geometry entry), else the launch's entries
  const int sub_t = descs ? gt.n : batch, sub_r = descs ? gr.n : batch;
  if (n_tma) {
    const int variant = cfg->slice_major ? 2 : (need_jmax ? 1 : 0);
    static size_t configured[3] = {0, 0, 0};
    if (smem_t > configured[variant]) {
      if (variant == 2) PDF_CHECK_CUDA(cudaFuncSetAttribute(resample_tma_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t));
      else if (need_jmax) PDF_CHECK_CUDA(cudaFuncSetAttribute(resample_tma_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t));
      else PDF_CHECK_CUDA(cudaFuncSetAttribute(resample_tma_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t));
      configured[variant] = smem_t;
    }
    const int ntiles = T0 * ceil_div(T1, TJt);
    const int per_sm = max(1, min(4, (int)((220 * 1024) / (smem_t + 1024))));
    // one resident wave: never more blocks than the chip holds at once (a second partial wave would double the time)
    const dim3 grid(max(1, min(ntiles, (num_sms() * per_sm) / sub_t)), sub_t);
    if (variant == 2) resample_tma_kernel<false, true><<<grid, 32 + 2 * KT, smem_t, s>>>(d_raw, d_zoomed, w.st, gt, T0, T1, T2, TJt, KT);
    else if (need_jmax) resample_tma_kernel<true, false><<<grid, 32 + 2 * KT, smem_t, s>>>(d_raw, d_zoomed, w.st, gt, T0, T1, T2, TJt, KT);
    else resample_tma_kernel<false, false><<<grid, 32 + 2 * KT, smem_t, s>>>(d_raw, d_zoomed, w.st, gt, T0, T1, T2, TJt, KT);
    PDF_CHECK_LAUNCH();
  }
  if (n_tma < n) {
    static size_t configured = 0;
    if (smem_r > configured) {
      PDF_CHECK_CUDA(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_r));
      configured = smem_r;
    }
    const int threads = min(256, (T2 + 31) / 32 * 32);
    const int ntiles = T0 * ceil_div(T1, TJr);
    const int per_sm = max(1, min(8, (int)((220 * 1024) / (smem_r + 1024))));
    const dim3 grid(max(1, min(ntiles, ceil_div(num_sms() * per_sm, sub_r))), sub_r);
    resample_kernel<<<grid, threads, smem_r, s>>>(d_raw, d_zoomed, w.st, gr, T0, T1, T2, TJr);
    PDF_CHECK_LAUNCH();
  }
  return PDF_OK;
}

extern "C" int pdf_resample_stats(const pdf_preproc_cfg* cfg, int batch, const float* d_raw, float* d_zoomed,
                                  void* d_workspace, pdf_stream_t stream) {
  if (int rc = validate(cfg, batch)) return rc;
  PDF_REQUIRE(d_raw && d_zoomed && d_workspace, "pdf_resample_stats: null device pointer");
  return resample_impl(cfg, batch, nullptr, d_raw, d_zoomed, d_workspace, as_stream(stream));
}

extern "C" int pdf_resample_stats_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs, const float* d_raw,
                                         float* d_zoomed, void* d_workspace, pdf_stream_t stream) {
  if (int rc = validate_ragged(cfg, batch, descs)) return rc;
  PDF_REQUIRE(d_raw && d_zoomed && d_workspace, "pdf_resample_stats_ragged: null device pointer");
  return resample_impl(cfg, batch, descs, d_raw, d_zoomed, d_workspace, as_stream(stream));
}

extern "C" int pdf_select_bounds_indices(const pdf_preproc_cfg* cfg, int batch, const float* d_zoomed, void* d_workspace,
                                         float* d_lohi, int32_t* d_indices, int32_t* d_nslices, pdf_stream_t stream) {
  if (int rc = validate_target(cfg, batch)) return rc;     // in_shape is not read here (ragged batches leave it unset)
  PDF_REQUIRE(d_zoomed && d_workspace && d_lohi && d_indices && d_nslices, "pdf_select_bounds_indices: null device pointer");
  cudaStream_t s = as_stream(stream);
  Workspace w = carve(cfg, batch, d_workspace);
  FinalizeArgs fa;
  fa.lmax = 0;
  fa.n_axes = cfg->n_axes;
  fa.extent_raw = cfg->extent_raw;
  for (int i = 0; i < 3; ++i) fa.T[i] = cfg->out_shape[i];
  for (int a = 0; a < PDF_MAX_AXES; ++a) {
    fa.axes[a] = a < cfg->n_axes ? cfg->axes[a] : 0;
    fa.counts[a] = a < cfg->n_axes ? cfg->counts[a] : 0;
    fa.lmax += fa.counts[a];
  }
  const size_t voxels = (size_t)cfg->out_shape[0] * cfg->out_shape[1] * cfg->out_shape[2];
  const int hblocks = max(1, min((int)(voxels / 4 / 256 / 4) + 1, ceil_div(num_sms() * 8, batch)));
  PDF_CHECK_CUDA(launch_pdl(scan_kernel<0>, dim3(batch), dim3(256), 0, s, w.st, fa, d_lohi, d_indices, d_nslices));
  PDF_CHECK_LAUNCH();
  PDF_CHECK_CUDA(launch_pdl(hist_kernel<1>, dim3(hblocks, batch), dim3(256), 0, s, d_zoomed, w.st, voxels, w.cand, w.cand_cap));
  PDF_CHECK_LAUNCH();
  PDF_CHECK_CUDA(launch_pdl(scan_kernel<1>, dim3(batch), dim3(256), 0, s, w.st, fa, d_lohi, d_indices, d_nslices));
  PDF_CHECK_LAUNCH();
  PDF_CHECK_CUDA(launch_pdl(hist_kernel<2>, dim3(hblocks, batch), dim3(256), 0, s, d_zoomed, w.st, voxels, w.cand, w.cand_cap));
  PDF_CHECK_LAUNCH();
  PDF_CHECK_CUDA(launch_pdl(scan_kernel<2>, dim3(batch), dim3(256), 0, s, w.st, fa, d_lohi, d_indices, d_nslices));
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

namespace pdf {
// bf16 layouts go through the banded kernel when a row of column groups fits one block row (64 groups = 256 pixels)
static bool launch_resize_band(const ResizeArgs& ra, int out_mode, int batch, const float* d_zoomed, const float* planes, const float* d_lohi,
                               const int32_t* d_indices, const int32_t* d_nslices, void* d_out, cudaStream_t s) {
  const int groups = out_mode == PDF_OUT_BF16_C1_PAD ? ra.pitch / 4 : (ra.S + 3) / 4;
  if (out_mode == PDF_OUT_F32_NHWC3 || groups > 64) return false;
  const dim3 grid(ceil_div(ra.S, kBandRows), ra.lmax, batch), block(64, 4);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(d_out);
  bool preclip = !ra.ready && !ra.zmajor;        // all slots on axis 2: their planes were clipped by extract_planes_kernel
  for (int a = 0; a < ra.n_axes; ++a) preclip = preclip && ra.axes[a] == 2;
  if (out_mode == PDF_OUT_BF16_C1_PAD) {
    if (preclip) resize_band_kernel<PDF_OUT_BF16_C1_PAD, true><<<grid, block, 0, s>>>(d_zoomed, planes, d_lohi, d_indices, d_nslices, o, ra);
    else resize_band_kernel<PDF_OUT_BF16_C1_PAD, false><<<grid, block, 0, s>>>(d_zoomed, planes, d_lohi, d_indices, d_nslices, o, ra);
  } else {
    if (preclip) resize_band_kernel<PDF_OUT_BF16_C1, true><<<grid, block, 0, s>>>(d_zoomed, planes, d_lohi, d_indices, d_nslices, o, ra);
    else resize_band_kernel<PDF_OUT_BF16_C1, false><<<grid, block, 0, s>>>(d_zoomed, planes, d_lohi, d_indices, d_nslices, o, ra);
  }
  return true;
}
}  // namespace pdf

extern "C" int pdf_gather_resize_normalize(const pdf_preproc_cfg* cfg, int batch, const float* d_zoomed, void* d_workspace,
                                              const float* d_lohi, const int32_t* d_indices, const int32_t* d_nslices,
                                              void* d_out, int out_mode, pdf_stream_t stream) {
  if (int rc = validate_target(cfg, batch)) return rc;     // in_shape is not read here (ragged batches leave it unset)
  PDF_REQUIRE(d_zoomed && d_workspace && d_lohi && d_indices && d_nslices && d_out, "pdf_gather_resize_normalize: null device pointer");
  PDF_REQUIRE(out_mode == PDF_OUT_BF16_C1 || out_mode == PDF_OUT_F32_NHWC3 || out_mode == PDF_OUT_BF16_C1_PAD,
              "pdf_gather_resize_normalize: bad out_mode");
  if (out_mode != PDF_OUT_F32_NHWC3) {
    PDF_REQUIRE(cfg->mean[0] == cfg->mean[1] && cfg->mean[1] == cfg->mean[2] && cfg->std[0] == cfg->std[1] && cfg->std[1] == cfg->std[2],
                "PDF_OUT_BF16_C1 needs channel-uniform mean/std");
  }
  cudaStream_t s = as_stream(stream);
  Workspace w = carve(cfg, batch, d_workspace);
  ResizeArgs ra;
  ra.zmajor = cfg->slice_major ? 1 : 0;
  ra.lmax = 0;
  ra.n_axes = cfg->n_axes;
  ra.S = cfg->input_size;
  ra.cnt2 = count_axis2(cfg);
  for (int i = 0; i < 3; ++i) { ra.T[i] = cfg->out_shape[i]; ra.mean[i] = cfg->mean[i]; ra.inv_std[i] = 1.0f / cfg->std[i]; }
  ra.scale_sq = (float)cfg->out_shape[0] / (float)ra.S;
  for (int a = 0; a < PDF_MAX_AXES; ++a) {
    ra.axes[a] = a < cfg->n_axes ? cfg->axes[a] : 0;
    ra.counts[a] = a < cfg->n_axes ? cfg->counts[a] : 0;
    ra.lmax += ra.counts[a];
  }
  const int T0 = cfg->out_shape[0], T1 = cfg->out_shape[1], T2 = cfg->out_shape[2];
  int off = 0, off2 = 0;
  for (int a = 0; a < cfg->n_axes; ++a) {
    if (cfg->axes[a] == 2 && !cfg->slice_major) {
      const int xb = max(1, min(ceil_div((long long)T0 * T1, 256 * 4), 64));
      // (plain launch: with programmatic dependent launch the next kernel's blocks would sit on the SMs waiting while this
      //  multi-wave grid still has blocks to place -- measured 220 -> 403 us for gather + resize)
      extract_planes_kernel<<<dim3(xb, cfg->counts[a], batch), 256, 0, s>>>(d_zoomed, d_indices, ra.lmax, off, ra.cnt2,
                                                                            w.planes + (size_t)off2 * T0 * T1, T0, T1, T2, d_lohi);
      PDF_CHECK_LAUNCH();
      off2 += cfg->counts[a];
    }
    off += cfg->counts[a];
  }
  ra.pitch = ra.rows = 0;
  ra.ready = 0;
  if (out_mode == PDF_OUT_BF16_C1_PAD) {
    if (int rc = pdf_stem_padded_dims(ra.S, &ra.pitch, &ra.rows)) return rc;
  }
  if (launch_resize_band(ra, out_mode, batch, d_zoomed, w.planes, d_lohi, d_indices, d_nslices, d_out, s)) {
    PDF_CHECK_LAUNCH();
    return PDF_OK;
  }
  const int groups = out_mode == PDF_OUT_BF16_C1_PAD ? ra.pitch / 4 : (ra.S + 3) / 4;
  const dim3 grid(ceil_div((long long)ra.S * groups, 256), ra.lmax, batch);
  if (out_mode == PDF_OUT_BF16_C1_PAD)
    resize_kernel<PDF_OUT_BF16_C1_PAD><<<grid, 256, 0, s>>>(d_zoomed, w.planes, d_lohi, d_indices, d_nslices, d_out, ra);
  else if (out_mode == PDF_OUT_BF16_C1)
    resize_kernel<PDF_OUT_BF16_C1><<<grid, 256, 0, s>>>(d_zoomed, w.planes, d_lohi, d_indices, d_nslices, d_out, ra);
  else
    resize_kernel<PDF_OUT_F32_NHWC3><<<grid, 256, 0, s>>>(d_zoomed, w.planes, d_lohi, d_indices, d_nslices, d_out, ra);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

// descs == nullptr: uniform batch of cfg->in_shape volumes; else the ragged batch the descriptors place in d_raw
static int preprocess_impl(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs, const float* d_raw, float* d_zoomed,
                           void* d_workspace, float* d_lohi, int32_t* d_indices, int32_t* d_nslices, void* d_out, int out_mode,
                           pdf_stream_t stream) {
  // Sub-batches: the resampled volumes of one sub-batch (8.4 MB each at 128^3) stay L2-resident between the resample kernel,
  // the two refinement-histogram passes and the plane gather, instead of streaming B x 8.4 MB through HBM four times.
  const int chunk = (g_pre_chunk > 0 && g_pre_chunk < batch) ? g_pre_chunk : batch;
  int lmax = 0;
  for (int a = 0; a < cfg->n_axes; ++a) lmax += cfg->counts[a];
  const size_t S = (size_t)cfg->input_size;
  size_t out_bytes = (size_t)lmax * S * S * (out_mode == PDF_OUT_F32_NHWC3 ? 12 : 2);
  if (out_mode == PDF_OUT_BF16_C1_PAD) {
    int pitch = 0, rows = 0;
    if (int rc = pdf_stem_padded_dims(cfg->input_size, &pitch, &rows)) return rc;
    out_bytes = (size_t)lmax * rows * pitch * 2;
  }
  const size_t vin = (size_t)cfg->in_shape[0] * cfg->in_shape[1] * cfg->in_shape[2];
  const size_t vout = (size_t)cfg->out_shape[0] * cfg->out_shape[1] * cfg->out_shape[2];
  for (int b0 = 0; b0 < batch; b0 += chunk) {
    const int nb = min(chunk, batch - b0);
    const float* raw = descs ? d_raw : d_raw + (size_t)b0 * vin;
    float* zoomed = d_zoomed + (size_t)b0 * vout;
    float* lohi = d_lohi + 4 * (size_t)b0;
    int32_t* indices = d_indices + (size_t)b0 * lmax;
    int32_t* nslices = d_nslices + (size_t)b0 * cfg->n_axes;
    void* out = reinterpret_cast<char*>(d_out) + (size_t)b0 * out_bytes;
    if (int rc = descs ? pdf_resample_stats_ragged(cfg, nb, descs + b0, raw, zoomed, d_workspace, stream)
                       : pdf_resample_stats(cfg, nb, raw, zoomed, d_workspace, stream)) return rc;
    if (int rc = pdf_select_bounds_indices(cfg, nb, zoomed, d_workspace, lohi, indices, nslices, stream)) return rc;
    if (int rc = pdf_gather_resize_normalize(cfg, nb, zoomed, d_workspace, lohi, indices, nslices, out, out_mode, stream)) return rc;
  }
  return PDF_OK;
}

extern "C" int pdf_preprocess(const pdf_preproc_cfg* cfg, int batch, const float* d_raw, float* d_zoomed, void* d_workspace,
                              float* d_lohi, int32_t* d_indices, int32_t* d_nslices, void* d_out, int out_mode,
                              pdf_stream_t stream) {
  if (int rc = validate(cfg, batch)) return rc;
  return preprocess_impl(cfg, batch, nullptr, d_raw, d_zoomed, d_workspace, d_lohi, d_indices, d_nslices, d_out, out_mode, stream);
}

extern "C" int pdf_preprocess_ragged(const pdf_preproc_cfg* cfg, int batch, const pdf_volume_desc* descs, const float* d_raw,
                                     float* d_zoomed, void* d_workspace, float* d_lohi, int32_t* d_indices, int32_t* d_nslices,
                                     void* d_out, int out_mode, pdf_stream_t stream) {
  if (int rc = validate_ragged(cfg, batch, descs)) return rc;
  return preprocess_impl(cfg, batch, descs, d_raw, d_zoomed, d_workspace, d_lohi, d_indices, d_nslices, d_out, out_mode, stream);
}

extern "C" int pdf_debug_set_pre_chunk(int subjects) {
  g_pre_chunk = subjects > 0 ? subjects : 0;
  return PDF_OK;
}

extern "C" int pdf_normalize_volume(int batch, size_t voxels, const float* d_zoomed, const float* d_lohi, float* d_norm,
                                    pdf_stream_t stream) {
  PDF_REQUIRE(batch > 0 && voxels > 0 && d_zoomed && d_lohi && d_norm, "pdf_normalize_volume: bad arguments");
  const int blocks = max(1, min((int)((voxels + 255) / 256), 2048));
  normalize_kernel<<<dim3(blocks, batch), 256, 0, as_stream(stream)>>>(d_zoomed, d_lohi, d_norm, voxels);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_gather_slices(const pdf_preproc_cfg* cfg, int batch, const float* d_zoomed, const float* d_lohi,
                                 const int32_t* d_indices, const int32_t* d_nslices, float* d_slices, pdf_stream_t stream) {
  if (int rc = validate_target(cfg, batch)) return rc;     // in_shape is not read here (ragged batches leave it unset)
  PDF_REQUIRE(d_zoomed && d_lohi && d_indices && d_nslices && d_slices, "pdf_gather_slices: null device pointer");
  PDF_REQUIRE(!cfg->slice_major, "pdf_gather_slices reads the C-order resampled volume (slice_major = 0)");
  FinalizeArgs fa;
  fa.lmax = 0; fa.n_axes = cfg->n_axes; fa.extent_raw = 0;
  for (int i = 0; i < 3; ++i) fa.T[i] = cfg->out_shape[i];
  int H = -1, W = -1;
  for (int a = 0; a < PDF_MAX_AXES; ++a) {
    fa.axes[a] = a < cfg->n_axes ? cfg->axes[a] : 0;
    fa.counts[a] = a < cfg->n_axes ? cfg->counts[a] : 0;
    fa.lmax += fa.counts[a];
    if (a < cfg->n_axes) {
      const int h = cfg->out_shape[fa.axes[a] == 0 ? 1 : 0], w = cfg->out_shape[fa.axes[a] == 2 ? 1 : 2];
      PDF_REQUIRE(H < 0 || (H == h && W == w), "pdf_gather_slices: all slice groups must share one slice shape (the reference concatenates them)");
      H = h; W = w;
    }
  }
  const int xb = max(1, min(ceil_div((long long)H * W, 256 * 4), 64));
  gather_slices_kernel<<<dim3(xb, fa.lmax, batch), 256, 0, as_stream(stream)>>>(d_zoomed, d_lohi, d_indices, d_nslices, d_slices, fa, H, W);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_tta_augment(int batch, int L, int H, int W, const float* d_slices, const pdf_tta_params* d_params,
                               const double* d_noise, int affine_only, float* d_out, pdf_stream_t stream) {
  PDF_REQUIRE(batch > 0 && L > 0 && H > 0 && W > 0 && d_slices && d_params && d_out, "pdf_tta_augment: bad arguments");
  const int xb = max(1, min(ceil_div((long long)H * W, 256 * 2), 64));
  tta_kernel<<<dim3(xb, L, batch), 256, 0, as_stream(stream)>>>(d_slices, d_params, d_noise, d_out, L, H, W, affine_only);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_resize_slices(int batch, int L, int H, int W, int input_size, const float* mean, const float* std,
                                 const float* d_slices, void* d_out, int out_mode, pdf_stream_t stream) {
  PDF_REQUIRE(batch > 0 && L > 0 && H >= 2 && W >= 2 && input_size >= 1 && mean && std && d_slices && d_out, "pdf_resize_slices: bad arguments");
  PDF_REQUIRE(out_mode == PDF_OUT_BF16_C1 || out_mode == PDF_OUT_F32_NHWC3 || out_mode == PDF_OUT_BF16_C1_PAD, "pdf_resize_slices: bad out_mode");
  if (out_mode != PDF_OUT_F32_NHWC3)
    PDF_REQUIRE(mean[0] == mean[1] && mean[1] == mean[2] && std[0] == std[1] && std[1] == std[2], "one-channel output needs channel-uniform mean/std");
  ResizeArgs ra;
  memset(&ra, 0, sizeof(ra));
  ra.ready = 1; ra.n_axes = 1; ra.axes[0] = 2; ra.counts[0] = L; ra.lmax = L; ra.cnt2 = L; ra.S = input_size;
  ra.T[0] = H; ra.T[1] = W; ra.T[2] = 1;
  for (int i = 0; i < 3; ++i) { ra.mean[i] = mean[i]; ra.inv_std[i] = 1.0f / std[i]; }
  ra.scale_sq = (float)H / (float)ra.S;
  if (out_mode == PDF_OUT_BF16_C1_PAD) {
    if (int rc = pdf_stem_padded_dims(ra.S, &ra.pitch, &ra.rows)) return rc;
  }
  cudaStream_t s = as_stream(stream);
  if (launch_resize_band(ra, out_mode, batch, nullptr, d_slices, nullptr, nullptr, nullptr, d_out, s)) {
    PDF_CHECK_LAUNCH();
    return PDF_OK;
  }
  const int groups = out_mode == PDF_OUT_BF16_C1_PAD ? ra.pitch / 4 : (ra.S + 3) / 4;
  const dim3 grid(ceil_div((long long)ra.S * groups, 256), L, batch);
  if (out_mode == PDF_OUT_BF16_C1_PAD)
    resize_kernel<PDF_OUT_BF16_C1_PAD><<<grid, 256, 0, s>>>(nullptr, d_slices, nullptr, nullptr, nullptr, d_out, ra);
  else if (out_mode == PDF_OUT_BF16_C1)
    resize_kernel<PDF_OUT_BF16_C1><<<grid, 256, 0, s>>>(nullptr, d_slices, nullptr, nullptr, nullptr, d_out, ra);
  else
    resize_kernel<PDF_OUT_F32_NHWC3><<<grid, 256, 0, s>>>(nullptr, d_slices, nullptr, nullptr, nullptr, d_out, ra);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

// Bootstrap replicates of the six scenario metrics (utils/metrics.compute_metrics) on the device.
//
// Resampling is a Poisson(1) bootstrap: replicate b gives sampling unit u the integer weight
//   w = Poisson1(philox4x32_10(key = seed, counter = (u, b, 0, 0)).x),
// Poisson1 being inversion of the 32-bit word against kPoisson1 (T_k = floor(2^32 P(X <= k)); w = the least k with word < T_k, so
// w <= 13).  Every weight is a stateless function of (seed, b, u): replicates are paired across scenarios and across the row- and
// subject-level metrics, replicate b does not depend on B, S or the launch shape, and no B x N weight array exists.  Row 0 of every
// scenario is the point estimate: the same computation with every weight 1.
//
// Each scenario's probabilities are sorted once, descending (CUB onesweep radix sort: stable, so deterministic), and (prob, label,
// unit) are gathered into sorted order with one flag byte per position.  bootstrap_metrics_kernel then runs one warp per (scenario,
// replicate); the warps of a block share a scenario and read each staged tile of the sorted arrays from shared memory.  A warp walks
// the tiles in order, regenerates its weights, and takes one warp inclusive scan of the packed (positive, negative) weights per 32
// positions.  At each tie-group end (last position of a run of equal probabilities), with TPp/FPp the running sums at the previous
// group end and TPe/FPe those at this one:
//   2 AUC Wpos Wneg += (FPe - FPp)(TPp + TPe)        exact, int64
//   AP Wpos         += (TPe - TPp) TPe / (TPe + FPe)  float64
// which is sklearn's trapezoid ROC area and step-wise average precision with sample_weight = w.  TP/FP at the 0.5 threshold are
// integers, so AUC, balanced accuracy and F1 are rationals of exact integers divided once.  Brier and the ECE bin sums are float64
// per lane, reduced across the warp in a fixed order: calls are bit-identical and independent of B and S.
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace pdf {

constexpr int kBootWarps = 8;        // replicates of one scenario per block
constexpr int kBootTile = 512;       // sorted positions staged per tile
constexpr int kEceBins = 10;
constexpr int kNoBin = 15;
constexpr uint8_t kFlagPos = 1, kFlagEnd = 2, kFlagPred = 4;   // bits 4..7: ECE bin (kNoBin: p == 0, in no bin)

__device__ __forceinline__ uint32_t boot_weight(uint2 key, uint32_t unit, uint32_t b) {
  // floor(2^32 P(X <= k)), X ~ Poisson(1), k = 0..12 (T_12 = 2^32 - 1)
  constexpr uint32_t kPoisson1[13] = {0x5e2d58d8u, 0xbc5ab1b1u, 0xeb715e1du, 0xfb239797u, 0xff1025f5u, 0xffd90f3bu, 0xfffa8b71u,
                                      0xffff540cu, 0xffffed1fu, 0xfffffe21u, 0xffffffd4u, 0xfffffffcu, 0xffffffffu};
  const uint32_t u = philox4x32_10(make_uint4(unit, b, 0u, 0u), key).x;
  uint32_t w = 0;
#pragma unroll
  for (int k = 0; k < 13; ++k) w += u >= kPoisson1[k];
  return w;
}

// numpy.linspace(0, 1, 11)[k]: k * 0.1 (k < 10), exactly 1.0 at k = 10
__device__ __forceinline__ double ece_edge(int k) { return k == kEceBins ? 1.0 : (double)k * 0.1; }

// the (lo, hi] bin of compute_ece that holds p, kNoBin for p == 0
__device__ __forceinline__ int ece_bin(double p) {
  if (!(p > 0.0)) return kNoBin;
  int k = min(kEceBins - 1, (int)(p * 10.0));
  while (k > 0 && p <= ece_edge(k)) --k;
  while (k < kEceBins - 1 && p > ece_edge(k + 1)) ++k;
  return k;
}

__global__ void boot_copy_keys_kernel(const double* __restrict__ prob, int n, double* __restrict__ keys, int32_t* __restrict__ idx) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    keys[i] = prob[i];
    idx[i] = i;
  }
}

// sorted position i of one scenario: probability, unit and flags (label, tie-group end, p >= 0.5, ECE bin)
__global__ void boot_gather_kernel(const double* __restrict__ prob, const uint8_t* __restrict__ label, const int32_t* __restrict__ unit,
                                   const int32_t* __restrict__ order, int n, double* __restrict__ sp, int32_t* __restrict__ su,
                                   uint8_t* __restrict__ sf) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int j = order[i];
    const double p = prob[j];
    const bool end = i == n - 1 || p != prob[order[i + 1]];
    sp[i] = p;
    su[i] = unit ? unit[j] : j;
    sf[i] = (uint8_t)((label[j] ? kFlagPos : 0) | (end ? kFlagEnd : 0) | (p >= 0.5 ? kFlagPred : 0) | (ece_bin(p) << 4));
  }
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// grid.x = S * ceil((B + 1) / kBootWarps); warp r of scenario s computes row r of out[s] (r = 0: point estimate, r >= 1: replicate
// r - 1).  out [S, 1 + B, 6] = roc_auc, pr_auc, balanced_accuracy, f1, brier_score, ece.
__global__ void __launch_bounds__(kBootWarps * 32)
bootstrap_metrics_kernel(const double* __restrict__ sp, const int32_t* __restrict__ su, const uint8_t* __restrict__ sf, int N, int n_boot,
                         int blocks_per_scenario, uint2 key, double* __restrict__ out) {
  __shared__ double t_p[kBootTile];
  __shared__ int32_t t_u[kBootTile];
  __shared__ uint8_t t_f[kBootTile];
  __shared__ double e_p[kBootWarps][kEceBins][32];     // per lane and ECE bin: sum w p, sum w, sum w [label == pred]
  __shared__ uint32_t e_w[kBootWarps][kEceBins][32];
  __shared__ uint32_t e_a[kBootWarps][kEceBins][32];

  const int s = blockIdx.x / blocks_per_scenario;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = (blockIdx.x - s * blocks_per_scenario) * kBootWarps + warp;
  const bool active = r <= n_boot;
  const uint32_t b = (uint32_t)(r - 1);
  sp += (size_t)s * N;
  su += (size_t)s * N;
  sf += (size_t)s * N;
  for (int k = 0; k < kEceBins; ++k) {
    e_p[warp][k][lane] = 0.0;
    e_w[warp][k][lane] = 0u;
    e_a[warp][k][lane] = 0u;
  }

  long long cTP = 0, cFP = 0;      // running weight sums before the current 32 positions
  long long lTP = 0, lFP = 0;      // running sums at the last tie-group end
  long long auc2 = 0;
  double ap = 0.0, brier = 0.0;
  uint32_t tp_thr = 0, fp_thr = 0;
  int cur_bin = kNoBin;            // a lane meets its bins in one contiguous run each (descending p): accumulate, store at the change
  uint32_t cur_w = 0, cur_a = 0;
  double cur_p = 0.0;
  const uint32_t lt_mask = (1u << lane) - 1u;

  for (int base = 0; base < N; base += kBootTile) {
    const int len = min(kBootTile, N - base);
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
      t_p[i] = sp[base + i];
      t_u[i] = su[base + i];
      t_f[i] = sf[base + i];
    }
    __syncthreads();
    if (!active) continue;
#pragma unroll 1
    for (int w0 = 0; w0 < len; w0 += 32) {
      const int li = w0 + lane;
      const bool valid = li < len;
      const uint8_t f = valid ? t_f[li] : (uint8_t)(kNoBin << 4);
      const double p = valid ? t_p[li] : 0.0;
      uint32_t w = 0;
      if (valid) w = r == 0 ? 1u : boot_weight(key, (uint32_t)t_u[li], b);
      const uint32_t pos = (f & kFlagPos) ? w : 0u, neg = w - pos;
      uint32_t v = pos | (neg << 16);                 // at most 13 * 32 of either per window
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
      }
      const bool end = f & kFlagEnd;
      const uint32_t ends = __ballot_sync(0xffffffffu, end);
      const uint32_t lower = ends & lt_mask;
      const uint32_t vp = __shfl_sync(0xffffffffu, v, lower ? 31 - __clz(lower) : lane);
      if (end) {
        const long long TPe = cTP + (v & 0xffffu), FPe = cFP + (v >> 16);
        const long long TPp = lower ? cTP + (vp & 0xffffu) : lTP, FPp = lower ? cFP + (vp >> 16) : lFP;
        auc2 += (FPe - FPp) * (TPp + TPe);
        if (TPe > TPp) ap += (double)(TPe - TPp) * ((double)TPe / (double)(TPe + FPe));
      }
      if (ends) {
        const uint32_t vl = __shfl_sync(0xffffffffu, v, 31 - __clz(ends));
        lTP = cTP + (vl & 0xffffu);
        lFP = cFP + (vl >> 16);
      }
      const uint32_t vt = __shfl_sync(0xffffffffu, v, 31);
      cTP += vt & 0xffffu;
      cFP += vt >> 16;

      const bool pred = f & kFlagPred;
      if (pred) {
        tp_thr += pos;
        fp_thr += neg;
      }
      const double d = p - ((f & kFlagPos) ? 1.0 : 0.0);
      brier += (double)w * d * d;
      const int bin = f >> 4;
      if (bin != cur_bin) {
        if (cur_bin != kNoBin) {
          e_p[warp][cur_bin][lane] = cur_p;
          e_w[warp][cur_bin][lane] = cur_w;
          e_a[warp][cur_bin][lane] = cur_a;
        }
        cur_bin = bin;
        cur_w = cur_a = 0u;
        cur_p = 0.0;
      }
      cur_w += w;
      cur_a += ((f & kFlagPos) != 0) == pred ? w : 0u;
      cur_p += (double)w * p;
    }
  }
  if (!active) return;
  if (cur_bin != kNoBin) {
    e_p[warp][cur_bin][lane] = cur_p;
    e_w[warp][cur_bin][lane] = cur_w;
    e_a[warp][cur_bin][lane] = cur_a;
  }
  auc2 = warp_sum_i64(auc2);
  ap = warp_sum_f64(ap);
  brier = warp_sum_f64(brier);
  const long long TP = warp_sum_i64(tp_thr), FP = warp_sum_i64(fp_thr);
  __syncwarp();
  if (lane != 0) return;

  const long long Wp = lTP, Wn = lFP, W = Wp + Wn;
  double* o = out + ((size_t)s * (n_boot + 1) + r) * 6;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  if (W == 0) {
    for (int k = 0; k < 6; ++k) o[k] = nan;
    return;
  }
  const long long FN = Wp - TP, TN = Wn - FP;
  o[0] = (Wp > 0 && Wn > 0) ? (double)auc2 / (double)(2 * Wp * Wn) : nan;
  o[1] = Wp > 0 ? ap / (double)Wp : 0.0;
  if (Wp > 0 && Wn > 0)
    o[2] = (double)(TP * Wn + TN * Wp) / (double)(2 * Wp * Wn);
  else
    o[2] = Wp > 0 ? (double)TP / (double)Wp : (double)TN / (double)Wn;   // the recall of the one class present
  const long long f1d = 2 * TP + FP + FN;
  o[3] = f1d > 0 ? (double)(2 * TP) / (double)f1d : 0.0;
  o[4] = brier / (double)W;
  double ece = 0.0;
#pragma unroll 1
  for (int k = 0; k < kEceBins; ++k) {              // compute_ece's loop: frac * |acc - mean p| over the non-empty bins
    double sp_k = 0.0;
    long long sw = 0, sa = 0;
#pragma unroll 4
    for (int l = 0; l < 32; ++l) {
      sp_k += e_p[warp][k][l];
      sw += e_w[warp][k][l];
      sa += e_a[warp][k][l];
    }
    if (sw > 0) ece += ((double)sw / (double)W) * fabs((double)sa / (double)sw - sp_k / (double)sw);
  }
  o[5] = ece;
}

constexpr int kMaxBoot = 1 << 20;
constexpr int kMaxBootN = 1 << 28;       // keeps 2 Wpos Wneg (weights <= 13) inside int64

static size_t boot_align(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// CUB onesweep with caller-provided double buffers: 8 pass histograms, a look-back array of (tiles of >= 256 keys) x 256 digits and
// counters, each region 256-byte aligned.  pdf_bootstrap_metrics checks the real size against this bound before it sorts.
static size_t boot_sort_temp_bound(size_t n) { return 4 * n + 65536; }

struct BootLayout {
  size_t sp, su, sf, keys0, keys1, idx0, idx1, temp, total;
};

static BootLayout boot_layout(size_t S, size_t N) {
  BootLayout L;
  size_t off = 0;
  L.sp = off;    off += boot_align(S * N * sizeof(double));
  L.su = off;    off += boot_align(S * N * sizeof(int32_t));
  L.sf = off;    off += boot_align(S * N);
  L.keys0 = off; off += boot_align(N * sizeof(double));
  L.keys1 = off; off += boot_align(N * sizeof(double));
  L.idx0 = off;  off += boot_align(N * sizeof(int32_t));
  L.idx1 = off;  off += boot_align(N * sizeof(int32_t));
  L.temp = off;  off += boot_align(boot_sort_temp_bound(N));
  L.total = off;
  return L;
}

static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

}  // namespace pdf

using namespace pdf;

extern "C" size_t pdf_bootstrap_metrics_workspace_bytes(int n_scenarios, int n) {
  if (n_scenarios < 1 || n < 1 || n > kMaxBootN) return 0;
  return boot_layout((size_t)n_scenarios, (size_t)n).total;
}

extern "C" int pdf_bootstrap_metrics(int n_scenarios, int n, int n_boot, uint64_t seed, const double* d_prob, const uint8_t* d_label,
                                     const int32_t* d_unit, void* d_workspace, double* d_out, pdf_stream_t stream) {
  PDF_REQUIRE(n_scenarios >= 1 && n >= 1 && n_boot >= 0 && d_prob && d_label && d_workspace && d_out,
              "pdf_bootstrap_metrics: bad arguments");
  PDF_REQUIRE(n_boot <= kMaxBoot, "pdf_bootstrap_metrics: n_boot must be 0..%d (got %d)", kMaxBoot, n_boot);
  PDF_REQUIRE(n <= kMaxBootN, "pdf_bootstrap_metrics: n must be 1..%d (got %d)", kMaxBootN, n);
  PDF_REQUIRE((long long)n_scenarios * ((n_boot + kBootWarps) / kBootWarps) <= 0x7fffffffll,
              "pdf_bootstrap_metrics: n_scenarios * (n_boot + 1) too large");
  PDF_REQUIRE(aligned(d_prob, 8) && aligned(d_out, 8) && aligned(d_workspace, 256) && (!d_unit || aligned(d_unit, 4)),
              "pdf_bootstrap_metrics: misaligned pointer (d_prob, d_out: 8 bytes; d_unit: 4; d_workspace: 256)");
  const size_t S = (size_t)n_scenarios, N = (size_t)n;
  const BootLayout L = boot_layout(S, N);
  char* ws = reinterpret_cast<char*>(d_workspace);
  double* sp = reinterpret_cast<double*>(ws + L.sp);
  int32_t* su = reinterpret_cast<int32_t*>(ws + L.su);
  uint8_t* sf = reinterpret_cast<uint8_t*>(ws + L.sf);
  cub::DoubleBuffer<double> keys(reinterpret_cast<double*>(ws + L.keys0), reinterpret_cast<double*>(ws + L.keys1));
  cub::DoubleBuffer<int32_t> idx(reinterpret_cast<int32_t*>(ws + L.idx0), reinterpret_cast<int32_t*>(ws + L.idx1));
  size_t temp_bytes = 0;
  PDF_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, temp_bytes, keys, idx, n, 0, 64, as_stream(stream)));
  if (temp_bytes > boot_sort_temp_bound(N)) {
    set_error("pdf_bootstrap_metrics: the radix sort needs %zu bytes of scratch, the workspace reserves %zu", temp_bytes,
              boot_sort_temp_bound(N));
    return PDF_ERR_UNSUPPORTED;
  }
  cudaStream_t st = as_stream(stream);
  const int eg = (int)std::min<size_t>((N + 255) / 256, 4096);
  for (size_t s = 0; s < S; ++s) {
    keys.selector = idx.selector = 0;
    boot_copy_keys_kernel<<<eg, 256, 0, st>>>(d_prob + s * N, n, keys.Current(), idx.Current());
    PDF_CHECK_LAUNCH();
    PDF_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(ws + L.temp, temp_bytes, keys, idx, n, 0, 64, st));
    boot_gather_kernel<<<eg, 256, 0, st>>>(d_prob + s * N, d_label, d_unit, idx.Current(), n, sp + s * N, su + s * N, sf + s * N);
    PDF_CHECK_LAUNCH();
  }
  const int per = (n_boot + kBootWarps) / kBootWarps;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  bootstrap_metrics_kernel<<<(unsigned)(S * per), kBootWarps * 32, 0, st>>>(sp, su, sf, n, n_boot, per, key, d_out);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

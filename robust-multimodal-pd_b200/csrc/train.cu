// Training kernels (FP32, NHWC): config 5's fine-tune forward/backward and the device-native training of the fusion heads.
//
// Reference: MilAttentionFineTuneModel._forward_bags / .train (models/mil_attention_finetune.py:135-162, 164-253) -- backbone in
// TRAIN mode (BatchNorm batch statistics per 16-slice chunk of one bag, running statistics updated), MIL attention head, BCE /
// focal loss, loss.backward(), clip_grad_norm_, Adam with two parameter groups -- and the heads' own train loops
// (models/mil_attention.py:88-155, fusion_moddrop.py:69-91, moe.py:60-70).  There torch autograd records the graph and replays
// it through cuDNN/ATen; here every forward op has a hand-written backward kernel and the host (pd_fusion_b200/training.py)
// walks the layer list in reverse.  FP32 throughout: this is the 1e-5-class parity path of training (gradients are compared
// with torch autograd in tests/test_gpu_training.py).
//
//   convolution backward   dgrad and wgrad as CUDA-core implicit GEMMs (the same 64x64x16 tiling as conv_f32_kernel)
//   BatchNorm (train)      per-(group, channel) statistics over a row range of the [M, C] activation matrix, apply (+ residual,
//                          ReLU) and the matching backward (ReLU mask, d_gamma, d_beta, d_x, gradient of the residual branch)
//   pooling backward       3x3/2 max pool (recomputed arg-max, first maximum in window order), global average pool
//   MIL head               ONE kernel per step for everything after the three linear layers: gated attention scores, masked
//                          softmax, pooling, classifier, BCE / focal loss AND their backward (d_h, d_v, d_u, head parameter grads)
//   optimiser              global gradient norm, clip scale, Adam (L2-style weight decay, per-call learning rate)
#include <algorithm>

#include "common.cuh"
#include "ops.cuh"

namespace pdf {

constexpr int TBM = 64, TBN = 64, TBK = 16;

// ------------------------------------------------------------------------------------------------------
// C[M,N] (+)= act( sum_k A(i,k) B(k,j) + bias[j] ) ; A(i,k) = A[i*a_rs + k*a_cs], B(k,j) = B[k*b_rs + j*b_cs], C row stride c_rs
// blockIdx.z = e runs member e of an ensemble: every operand moved by e times its member stride (*_es, 0 = shared)
__global__ void __launch_bounds__(256)
gemm_strided_kernel(const float* __restrict__ A, long a_rs, long a_cs, const float* __restrict__ B, long b_rs, long b_cs,
                    float* __restrict__ C, long c_rs, const float* __restrict__ bias, int M, int N, int K, int act, int accumulate,
                    long a_es, long b_es, long c_es, long bias_es) {
  const long e = blockIdx.z;
  A += e * a_es;
  B += e * b_es;
  C += e * c_es;
  if (bias) bias += e * bias_es;
  __shared__ float As[TBK][TBM + 4];
  __shared__ float Bs[TBK][TBN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * TBM, n0 = blockIdx.y * TBN;
  const int lr = tid >> 2, lk = (tid & 3) * 4;       // A/B loader: row (0..63), 4 consecutive k
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += TBK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = k0 + lk + e;
      As[lk + e][lr] = (m0 + lr < M && k < K) ? __ldg(A + (long)(m0 + lr) * a_rs + (long)k * a_cs) : 0.f;
      Bs[lk + e][lr] = (n0 + lr < N && k < K) ? __ldg(B + (long)k * b_rs + (long)(n0 + lr) * b_cs) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TBK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      if (bias) v += __ldg(bias + n);
      if (act == 1) v = fmaxf(v, 0.f);
      float* c = C + (long)m * c_rs + n;
      *c = accumulate ? *c + v : v;
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// dgrad: dx[n,ih,iw,c] (+)= sum_{r,s,k} dy[n,p,q,k] w[r][s][c][k],  p*stride = ih + pad - r, q*stride = iw + pad - s
__global__ void __launch_bounds__(256)
conv_dgrad_f32_kernel(const float* __restrict__ dy, const float* __restrict__ wgt, float* __restrict__ dx, int N, int H, int W, int C,
                      int K, int R, int S, int stride, int pad, int Ho, int Wo, int accumulate) {
  __shared__ float As[TBK][TBM + 4];
  __shared__ float Bs[TBK][TBN + 4];
  const int tid = threadIdx.x;
  const int M = N * H * W;
  const int Kg = R * S * K;
  const int m0 = blockIdx.x * TBM, n0 = blockIdx.y * TBN;
  const int am = tid >> 2, ak = (tid & 3) * 4;
  const int m = m0 + am;
  int pn = 0, ih = 0, iw = 0;
  const bool mvalid = m < M;
  if (mvalid) {
    pn = m / (H * W);
    const int rem = m - pn * H * W;
    ih = rem / W; iw = rem - ih * W;
  }
  const int bk = tid >> 4, bn = (tid & 15) * 4;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4] = {};
  for (int kg0 = 0; kg0 < Kg; kg0 += TBK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int kg = kg0 + ak + e;
      float v = 0.f;
      if (mvalid && kg < Kg) {
        const int k = kg % K;
        const int rs = kg / K;
        const int s = rs % S, r = rs / S;
        const int ph = ih + pad - r, qw = iw + pad - s;
        if (ph >= 0 && qw >= 0 && ph % stride == 0 && qw % stride == 0) {
          const int p = ph / stride, q = qw / stride;
          if (p < Ho && q < Wo) v = __ldg(dy + (((size_t)pn * Ho + p) * Wo + q) * K + k);
        }
      }
      As[ak + e][am] = v;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int kg = kg0 + bk, col = n0 + bn + e;      // B(kg=(r,s,k), c) = w[((r*S+s)*C + c)*K + k]
      float v = 0.f;
      if (kg < Kg && col < C) {
        const int k = kg % K, rs = kg / K;
        v = __ldg(wgt + ((size_t)rs * C + col) * K + k);
      }
      Bs[bk][bn + e] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TBK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int mm = m0 + ty * 4 + i;
    if (mm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = n0 + tx * 4 + j;
      if (col >= C) continue;
      float* o = dx + (size_t)mm * C + col;
      *o = accumulate ? *o + acc[i][j] : acc[i][j];
    }
  }
}

// wgrad: dw[r][s][c][k] += sum_m x[n, p*stride + r - pad, q*stride + s - pad, c] dy[m, k]   (m = (n,p,q)); the pixel range is
// split over blockIdx.z, partial sums meet in dw through atomicAdd
__global__ void __launch_bounds__(256)
conv_wgrad_f32_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dw, int N, int H, int W, int C,
                      int K, int R, int S, int stride, int pad, int Ho, int Wo, int slab) {
  __shared__ float As[TBK][TBM + 4];
  __shared__ float Bs[TBK][TBN + 4];
  const int tid = threadIdx.x;
  const int M = N * Ho * Wo;
  const int Rows = R * S * C;
  const int i0 = blockIdx.x * TBM, n0 = blockIdx.y * TBN;
  const int mlo = blockIdx.z * slab, mhi = min(M, mlo + slab);
  // A loader: thread -> row i (tid>>2), 4 consecutive pixels;  B loader: thread -> pixel (tid>>4), 4 consecutive k
  const int ai = tid >> 2, ap = (tid & 3) * 4;
  const int row = i0 + ai;
  int ar = 0, as_ = 0, ac = 0;
  const bool rvalid = row < Rows;
  if (rvalid) { ac = row % C; const int rs = row / C; as_ = rs % S; ar = rs / S; }
  const int bp = tid >> 4, bn = (tid & 15) * 4;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4] = {};
  for (int mm0 = mlo; mm0 < mhi; mm0 += TBK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int m = mm0 + ap + e;
      float v = 0.f;
      if (rvalid && m < mhi) {
        const int pn = m / (Ho * Wo);
        const int rem = m - pn * Ho * Wo;
        const int p = rem / Wo, q = rem - p * Wo;
        const int ih = p * stride + ar - pad, iw = q * stride + as_ - pad;
        if (ih >= 0 && ih < H && iw >= 0 && iw < W) v = __ldg(x + (((size_t)pn * H + ih) * W + iw) * C + ac);
      }
      As[ap + e][ai] = v;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int m = mm0 + bp, col = n0 + bn + e;
      Bs[bp][bn + e] = (m < mhi && col < K) ? __ldg(dy + (size_t)m * K + col) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TBK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rr = i0 + ty * 4 + i;
    if (rr >= Rows) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = n0 + tx * 4 + j;
      if (col >= K) continue;
      atomicAdd(dw + (size_t)rr * K + col, acc[i][j]);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// BatchNorm, train mode.  x is the [M, C] matrix of one layer's conv output (rows = pixels in NHWC order); group g covers rows
// [goff[g], goff[g+1]) -- one 16-slice chunk of one bag, the unit the reference pushes through the backbone at a time.
//
// Reductions: grid (C/32, groups, row slabs) -- a (group, channel-block) pair alone would put 32 blocks on the machine for the
// 64-channel layers.  Every block sums its slab in float64 (these per-(group, channel) sums feed (x - mean) * invstd, whose
// cancellation amplifies every ulp of the statistics into the gradients, and Adam's sign-like first steps amplify THAT) and adds
// its partial sums into a float64 scratch with atomicAdd(double); a tiny finalize kernel turns them into mean / invstd.
// With float64 sums the one-pass form var = E[x^2] - mean^2 is exact to ~1e-16 * mean^2 / var.
constexpr int kBnRowsPerBlock = 2048;     // rows of a slab (8 row lanes x 256 iterations)

__global__ void __launch_bounds__(256)
bn_stats_kernel(const float* __restrict__ x, const int* __restrict__ goff, int C, double* __restrict__ acc) {
  __shared__ double red0[8][33], red1[8][33];
  const int g = blockIdx.y;
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const int r0 = goff[g] + blockIdx.z * kBnRowsPerBlock;
  const int r1 = min(goff[g + 1], r0 + kBnRowsPerBlock);
  if (r0 >= r1) return;
  double s = 0.0, q = 0.0;
  if (c < C) {
    int r = r0 + ry;
    for (; r + 24 < r1; r += 32) {                      // four independent loads in flight per thread
      const float a0 = x[(size_t)r * C + c], a1 = x[(size_t)(r + 8) * C + c], a2 = x[(size_t)(r + 16) * C + c], a3 = x[(size_t)(r + 24) * C + c];
      s += ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
      q += ((double)a0 * (double)a0 + (double)a1 * (double)a1) + ((double)a2 * (double)a2 + (double)a3 * (double)a3);
    }
    for (; r < r1; r += 8) { const double a = (double)x[(size_t)r * C + c]; s += a; q += a * a; }
  }
  red0[ry][threadIdx.x & 31] = s; red1[ry][threadIdx.x & 31] = q;
  __syncthreads();
  if (ry == 0 && c < C) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < 8; ++i) { a += red0[i][threadIdx.x & 31]; b += red1[i][threadIdx.x & 31]; }
    atomicAdd(acc + ((size_t)g * C + c) * 2, a);
    atomicAdd(acc + ((size_t)g * C + c) * 2 + 1, b);
  }
}

__global__ void bn_stats_finalize_kernel(const double* __restrict__ acc, const int* __restrict__ goff, int G, int C, float eps,
                                         float* __restrict__ mean, float* __restrict__ invstd, float* __restrict__ var_unbiased) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= G * C) return;
  const int g = i / C;
  const int rows = goff[g + 1] - goff[g];
  const double m = (double)max(rows, 1);
  const double mu = acc[(size_t)i * 2] / m;
  const double v = fmax(acc[(size_t)i * 2 + 1] - m * mu * mu, 0.0);   // sum of squared deviations
  const double var = v / m;
  mean[i] = (float)mu;
  invstd[i] = (float)(1.0 / sqrt(var + (double)eps));
  var_unbiased[i] = (float)(rows > 1 ? v / (double)(rows - 1) : var);
}

__device__ __forceinline__ void store_bf16x4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 o;
  o.x = *reinterpret_cast<uint32_t*>(&lo); o.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = o;
}

// y = (x - mean) * invstd * gamma + beta (+ residual) (ReLU); four channels per thread (C % 4 == 0); optional bf16 copy of y (the
// operand of the next tensor-core convolution)
__global__ void __launch_bounds__(256)
bn_apply_kernel(const float* __restrict__ x, const int* __restrict__ goff, int C, const float* __restrict__ mean,
                const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                const float* __restrict__ residual, int relu, float* __restrict__ y, __nv_bfloat16* __restrict__ y16) {
  const int g = blockIdx.y;
  const size_t lo = (size_t)goff[g] * C / 4, hi = (size_t)goff[g + 1] * C / 4;
  const int C4 = C / 4;
  const float4* mu4 = reinterpret_cast<const float4*>(mean + (size_t)g * C);
  const float4* is4 = reinterpret_cast<const float4*>(invstd + (size_t)g * C);
  for (size_t i = lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (size_t)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4);
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 mu = mu4[c4], is = is4[c4];
    const float4 ga = reinterpret_cast<const float4*>(gamma)[c4], be = reinterpret_cast<const float4*>(beta)[c4];
    float4 v;
    v.x = (xv.x - mu.x) * is.x * ga.x + be.x; v.y = (xv.y - mu.y) * is.y * ga.y + be.y;
    v.z = (xv.z - mu.z) * is.z * ga.z + be.z; v.w = (xv.w - mu.w) * is.w * ga.w + be.w;
    if (residual) { const float4 r = reinterpret_cast<const float4*>(residual)[i]; v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w; }
    if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    reinterpret_cast<float4*>(y)[i] = v;
    if (y16) store_bf16x4(y16 + i * 4, v);
  }
}

// backward, pass 1: per (group, channel) sums of g = dy * relu'(y) and g * xhat (same grid / float64 scheme as bn_stats_kernel)
__global__ void __launch_bounds__(256)
bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ x, const int* __restrict__ goff,
                     int C, const float* __restrict__ mean, const float* __restrict__ invstd, int relu, double* __restrict__ acc) {
  __shared__ double red0[8][33], red1[8][33];
  const int g = blockIdx.y;
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const int r0 = goff[g] + blockIdx.z * kBnRowsPerBlock;
  const int r1 = min(goff[g + 1], r0 + kBnRowsPerBlock);
  if (r0 >= r1) return;
  double s0 = 0.0, s1 = 0.0;
  if (c < C) {
    const float mu = mean[(size_t)g * C + c], is = invstd[(size_t)g * C + c];
    int r = r0 + ry;
    for (; r + 8 < r1; r += 16) {
      const size_t i0 = (size_t)r * C + c, i1 = (size_t)(r + 8) * C + c;
      float g0 = dy[i0], g1 = dy[i1];
      const float x0 = x[i0], x1 = x[i1];
      if (relu) { const float y0 = y[i0], y1 = y[i1]; if (!(y0 > 0.f)) g0 = 0.f; if (!(y1 > 0.f)) g1 = 0.f; }
      s0 += (double)g0 + (double)g1;
      s1 += (double)g0 * (double)((x0 - mu) * is) + (double)g1 * (double)((x1 - mu) * is);
    }
    for (; r < r1; r += 8) {
      const size_t i = (size_t)r * C + c;
      float gr = dy[i];
      if (relu && !(y[i] > 0.f)) gr = 0.f;
      s0 += (double)gr;
      s1 += (double)gr * (double)((x[i] - mu) * is);
    }
  }
  red0[ry][threadIdx.x & 31] = s0; red1[ry][threadIdx.x & 31] = s1;
  __syncthreads();
  if (ry == 0 && c < C) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < 8; ++i) { a += red0[i][threadIdx.x & 31]; b += red1[i][threadIdx.x & 31]; }
    atomicAdd(acc + ((size_t)g * C + c) * 2, a);
    atomicAdd(acc + ((size_t)g * C + c) * 2 + 1, b);
  }
}

// d_gamma / d_beta accumulate over the groups (and over calls); sums[g][c] = (sum g, sum g*xhat) as floats for the apply pass
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ acc, int G, int C, float* __restrict__ sums, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double a = 0.0, b = 0.0;
  for (int g = 0; g < G; ++g) {
    const double s0 = acc[((size_t)g * C + c) * 2], s1 = acc[((size_t)g * C + c) * 2 + 1];
    sums[(size_t)g * C + c] = (float)s0;
    sums[(size_t)(G + g) * C + c] = (float)s1;
    a += s0; b += s1;
  }
  dbeta[c] += (float)a;
  dgamma[c] += (float)b;
}

// backward, pass 2: dx = gamma * invstd * (g - sum_g/m - xhat * sum_gx/m);  dres (+)= g  (the residual branch sees the masked gradient);
// optional bf16 copy of dx (the operand of the tensor-core dgrad / wgrad)
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ x, const int* __restrict__ goff,
                    int C, const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma, int relu,
                    const float* __restrict__ sum_g, const float* __restrict__ sum_gx, float* __restrict__ dx, __nv_bfloat16* __restrict__ dx16,
                    float* __restrict__ dres, int dres_accumulate) {
  const int g = blockIdx.y;
  const float inv_m = 1.0f / (float)max(goff[g + 1] - goff[g], 1);
  const size_t lo = (size_t)goff[g] * C / 4, hi = (size_t)goff[g + 1] * C / 4;
  const int C4 = C / 4;
  const float4* mu4 = reinterpret_cast<const float4*>(mean + (size_t)g * C);
  const float4* is4 = reinterpret_cast<const float4*>(invstd + (size_t)g * C);
  const float4* sg4 = reinterpret_cast<const float4*>(sum_g + (size_t)g * C);
  const float4* sx4 = reinterpret_cast<const float4*>(sum_gx + (size_t)g * C);
  for (size_t i = lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (size_t)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4);
    float4 gr = reinterpret_cast<const float4*>(dy)[i];
    if (relu) {
      const float4 yv = reinterpret_cast<const float4*>(y)[i];
      if (!(yv.x > 0.f)) gr.x = 0.f;
      if (!(yv.y > 0.f)) gr.y = 0.f;
      if (!(yv.z > 0.f)) gr.z = 0.f;
      if (!(yv.w > 0.f)) gr.w = 0.f;
    }
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 mu = mu4[c4], is = is4[c4], ga = reinterpret_cast<const float4*>(gamma)[c4], sg = sg4[c4], sx = sx4[c4];
    float4 o;
    o.x = ga.x * is.x * (gr.x - sg.x * inv_m - (xv.x - mu.x) * is.x * sx.x * inv_m);
    o.y = ga.y * is.y * (gr.y - sg.y * inv_m - (xv.y - mu.y) * is.y * sx.y * inv_m);
    o.z = ga.z * is.z * (gr.z - sg.z * inv_m - (xv.z - mu.z) * is.z * sx.z * inv_m);
    o.w = ga.w * is.w * (gr.w - sg.w * inv_m - (xv.w - mu.w) * is.w * sx.w * inv_m);
    reinterpret_cast<float4*>(dx)[i] = o;
    if (dx16) store_bf16x4(dx16 + i * 4, o);
    if (dres) {
      float4* dr = reinterpret_cast<float4*>(dres) + i;
      if (dres_accumulate) { const float4 d = *dr; gr.x += d.x; gr.y += d.y; gr.z += d.z; gr.w += d.w; }
      *dr = gr;
    }
  }
}

// running statistics: r = (1 - mom) * r + mom * batch, group after group in order (the reference forwards the chunks one by one)
__global__ void bn_running_kernel(const float* __restrict__ mean, const float* __restrict__ var_unbiased, int G, int C, float mom,
                                  float* __restrict__ run_mean, float* __restrict__ run_var) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float m = run_mean[c], v = run_var[c];
  for (int g = 0; g < G; ++g) {
    m = (1.f - mom) * m + mom * mean[(size_t)g * C + c];
    v = (1.f - mom) * v + mom * var_unbiased[(size_t)g * C + c];
  }
  run_mean[c] = m; run_var[c] = v;
}

// ------------------------------------------------------------------------------------------------------
// 3x3 stride-2 pad-1 max pool backward: the gradient of each pooled pixel goes to the FIRST maximum of its window (row-major scan)
__global__ void maxpool_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx, int N, int H, int W,
                                   int C, int Ho, int Wo) {
  const size_t total = (size_t)N * Ho * Wo * C;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    size_t t = i / C;
    const int q = (int)(t % Wo); t /= Wo;
    const int p = (int)(t % Ho);
    const int n = (int)(t / Ho);
    float best = -INFINITY;
    size_t arg = 0;
    bool found = false;
    for (int r = 0; r < 3; ++r) {
      const int ih = p * 2 - 1 + r;
      if (ih < 0 || ih >= H) continue;
      for (int s = 0; s < 3; ++s) {
        const int iw = q * 2 - 1 + s;
        if (iw < 0 || iw >= W) continue;
        const size_t j = (((size_t)n * H + ih) * W + iw) * C + c;
        const float v = x[j];
        if (!found || v > best) { best = v; arg = j; found = true; }
      }
    }
    if (found) atomicAdd(dx + arg, dy[i]);
  }
}

// global average pool backward: dx[n, hw, c] = demb[n, c] / HW
__global__ void avgpool_bwd_kernel(const float* __restrict__ demb, float* __restrict__ dx, int HW, int C, size_t total) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const size_t n = i / ((size_t)HW * C);
    dx[i] = demb[n * C + c] / (float)HW;
  }
}

// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum_t(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ float block_sum(float v, float* red) {     // 256 threads; red[8]
  v = warp_sum_t(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  for (int i = 0; i < 8; ++i) t += red[i];
  return t;
}
__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }

// MIL head, training: everything after the linear layers, forward AND backward, one block per bag.
//   h [n_bags*Lmax, H]   = dropout(relu(instance(x)))     (computed by the GEMM + mask kernels)
//   vu [n_bags*Lmax, NA] = pre-activations of attn_v | attn_u (gated) or attn.0 (plain), bias included
// forward : s_l = w_w . (tanh(v_l) (.) sigmoid(u_l)) + b_w ; a = softmax_l(s) over the bag's len ; pooled = sum_l a_l h_l ;
//           p = sigmoid(w_c . pooled + b_c) ; per-bag loss (BCE, optionally pos-weighted or focal), mean over the batch
// backward: d_h (the pooling path: a_l * d_pooled), d_vu, and the head's small parameter gradients, handed to the sink with the loss:
//           d_w_cls [H], d_b_cls, d_w_w [A], d_b_w.   (models/mil_attention.py:40-51, mil_attention_finetune.py:211-224)
// The single model accumulates them with atomicAdd (MilAtomicSink).  An ensemble runs member e on blockIdx.y (its weights w_es floats,
// its bags one batch further) and stores each bag's terms in a row of its own (MilPartialSink), reduced in bag order afterwards.
struct MilTrainArgs {
  int H, A, gated, Lmax, n_bags;
  int loss_type;          // 0 BCE (x sample weight), 1 focal
  float pos_weight;       // BCE: weight of positive samples (1 = none)
  float focal_gamma, focal_alpha;   // focal_alpha < 0: no alpha term
  const float *w_w, *b_w, *w_cls, *b_cls;
  float *d_w_w, *d_b_w, *d_w_cls, *d_b_cls;
};

struct MilAtomicSink {
  float *loss_sum, *d_w_w, *d_b_w, *d_w_cls, *d_b_cls;
  __device__ void loss(float v) { atomicAdd(loss_sum, v); }
  __device__ void b_cls(float v) { atomicAdd(d_b_cls, v); }
  __device__ void w_cls(int i, float v) { atomicAdd(d_w_cls + i, v); }
  __device__ void b_w(float v) { atomicAdd(d_b_w, v); }
  __device__ void w_w(int j, float v) { atomicAdd(d_w_w + j, v); }
};
// row (member, bag) of partial [E, n_bags, H + A + 3]: d w_cls [H] | d w_w [A] | d b_cls | d b_w | loss / n_bags (zeroed before the launch)
struct MilPartialSink {
  float* partial;
  int H, A;
  __device__ float* row() const { return partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (H + A + 3); }
  __device__ void w_cls(int i, float v) { row()[i] = v; }
  __device__ void w_w(int j, float v) { row()[H + j] = v; }
  __device__ void b_cls(float v) { row()[H + A] = v; }
  __device__ void b_w(float v) { row()[H + A + 1] = v; }
  __device__ void loss(float v) { row()[H + A + 2] = v; }
};

template <class Sink>
__global__ void __launch_bounds__(256)
mil_pool_train_kernel(MilTrainArgs a, long w_es, const float* __restrict__ h, const float* __restrict__ vu, const int32_t* __restrict__ lens,
                      const float* __restrict__ target, float* __restrict__ prob, float* __restrict__ dh, float* __restrict__ dvu, Sink sink) {
  extern __shared__ float sm[];
  const long member = blockIdx.y;
  const size_t mrows = (size_t)a.n_bags * a.Lmax;
  a.w_w += member * w_es; a.b_w += member * w_es; a.w_cls += member * w_es; a.b_cls += member * w_es;
  h += member * mrows * a.H; dh += member * mrows * a.H;
  vu += member * mrows * (a.gated ? 2 * a.A : a.A); dvu += member * mrows * (a.gated ? 2 * a.A : a.A);
  lens += member * a.n_bags; target += member * a.n_bags; prob += member * a.n_bags;
  float* s_a = sm;                     // [Lmax] scores -> attention weights
  float* s_da = sm + a.Lmax;           // [Lmax] d loss / d a_l -> d s_l
  float* s_pool = sm + 2 * a.Lmax;     // [H]
  __shared__ float red[8];
  const int bag = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int len = min(lens[bag], a.Lmax);
  const int H = a.H, A = a.A, NA = a.gated ? 2 * A : A;
  const float* hb = h + (size_t)bag * a.Lmax * H;
  const float* vb = vu + (size_t)bag * a.Lmax * NA;
  float* dhb = dh + (size_t)bag * a.Lmax * H;
  float* dvb = dvu + (size_t)bag * a.Lmax * NA;
  for (size_t i = tid; i < (size_t)a.Lmax * H; i += 256) dhb[i] = 0.f;        // padded rows carry no gradient
  for (size_t i = tid; i < (size_t)a.Lmax * NA; i += 256) dvb[i] = 0.f;
  if (len <= 0) { if (tid == 0) prob[bag] = 0.5f; return; }
  // scores
  for (int l = warp; l < len; l += 8) {
    float sc = 0.f;
    for (int j = lane; j < A; j += 32) {
      float t = tanhf(vb[(size_t)l * NA + j]);
      if (a.gated) t *= sigm(vb[(size_t)l * NA + A + j]);
      sc = fmaf(__ldg(a.w_w + j), t, sc);
    }
    sc = warp_sum_t(sc);
    if (lane == 0) s_a[l] = sc + __ldg(a.b_w);
  }
  __syncthreads();
  float mx = -INFINITY;
  for (int l = tid; l < len; l += 256) mx = fmaxf(mx, s_a[l]);
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  __syncthreads();
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, red[i]);
  float se = 0.f;
  for (int l = tid; l < len; l += 256) { const float e = expf(s_a[l] - mx); s_a[l] = e; se += e; }
  se = block_sum(se, red);
  for (int l = tid; l < len; l += 256) s_a[l] /= se;
  __syncthreads();
  // pooled, logit
  float z = 0.f;
  for (int i = tid; i < H; i += 256) {
    float pl = 0.f;
    for (int l = 0; l < len; ++l) pl = fmaf(s_a[l], hb[(size_t)l * H + i], pl);
    s_pool[i] = pl;
    z = fmaf(__ldg(a.w_cls + i), pl, z);
  }
  z = block_sum(z, red) + __ldg(a.b_cls);
  const float p = sigm(z);
  // loss and d loss / d z  (torch.nn.functional.binary_cross_entropy clamps the logs at -100)
  const float y = target[bag];
  const bool pos = y >= 0.5f;
  const float lp = fmaxf(logf(p), -100.f), l1p = fmaxf(logf(1.f - p), -100.f);
  const float bce = -(y * lp + (1.f - y) * l1p);
  const float dbce_dp = -(y / fmaxf(p, 1e-44f)) * (lp > -100.f ? 1.f : 0.f) + ((1.f - y) / fmaxf(1.f - p, 1e-44f)) * (l1p > -100.f ? 1.f : 0.f);
  float loss, dl_dp;
  if (a.loss_type == 1) {
    const float pt = pos ? p : 1.f - p;
    const float om = 1.f - pt;
    float w = powf(om, a.focal_gamma);
    float dw_dp = (a.focal_gamma == 0.f ? 0.f : -a.focal_gamma * powf(om, a.focal_gamma - 1.f)) * (pos ? 1.f : -1.f);
    const float al = a.focal_alpha < 0.f ? 1.f : (pos ? a.focal_alpha : 1.f - a.focal_alpha);
    w *= al; dw_dp *= al;
    loss = w * bce;
    dl_dp = dw_dp * bce + w * dbce_dp;
  } else {
    const float w = pos ? a.pos_weight : 1.f;
    loss = w * bce;
    dl_dp = w * dbce_dp;
  }
  const float inv_b = 1.f / (float)a.n_bags;                   // mean over the batch
  const float dz = dl_dp * p * (1.f - p) * inv_b;
  if (tid == 0) { prob[bag] = p; sink.loss(loss * inv_b); sink.b_cls(dz); }
  // classifier grads, d pooled
  for (int i = tid; i < H; i += 256) sink.w_cls(i, dz * s_pool[i]);
  // d a_l = d pooled . h_l ;  d h_l = a_l * d pooled   (d pooled_i = dz * w_cls_i)
  for (int l = warp; l < len; l += 8) {
    float da = 0.f;
    for (int i = lane; i < H; i += 32) {
      const float dp = dz * __ldg(a.w_cls + i);
      da = fmaf(dp, hb[(size_t)l * H + i], da);
      dhb[(size_t)l * H + i] = s_a[l] * dp;
    }
    da = warp_sum_t(da);
    if (lane == 0) s_da[l] = da;
  }
  __syncthreads();
  float dot = 0.f;
  for (int l = tid; l < len; l += 256) dot = fmaf(s_a[l], s_da[l], dot);
  dot = block_sum(dot, red);
  for (int l = tid; l < len; l += 256) s_da[l] = s_a[l] * (s_da[l] - dot);       // d s_l (softmax backward)
  __syncthreads();
  float dbw = 0.f;
  for (int l = tid; l < len; l += 256) dbw += s_da[l];
  dbw = block_sum(dbw, red);
  if (tid == 0) sink.b_w(dbw);
  // attention layer: d w_w, d v_pre, d u_pre
  for (int j = tid; j < A; j += 256) {
    const float ww = __ldg(a.w_w + j);
    float dww = 0.f;
    for (int l = 0; l < len; ++l) {
      const float ds = s_da[l];
      const float tv = tanhf(vb[(size_t)l * NA + j]);
      if (a.gated) {
        const float su = sigm(vb[(size_t)l * NA + A + j]);
        dww = fmaf(ds, tv * su, dww);
        dvb[(size_t)l * NA + j] = ds * ww * su * (1.f - tv * tv);
        dvb[(size_t)l * NA + A + j] = ds * ww * tv * su * (1.f - su);
      } else {
        dww = fmaf(ds, tv, dww);
        dvb[(size_t)l * NA + j] = ds * ww * (1.f - tv * tv);
      }
    }
    sink.w_w(j, dww);
  }
}

// ------------------------------------------------------------------------------------------------------
// small elementwise / reduction helpers
__global__ void colsum_kernel(const float* __restrict__ x, int M, int N, float* __restrict__ out, int accumulate) {   // out[j] (+)= sum_i x[i, j]
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  float s = 0.f;
  for (int i = 0; i < M; ++i) s += x[(size_t)i * N + j];
  out[j] = accumulate ? out[j] + s : s;
}
// relu / dropout backward in place: g *= (act > 0) * mask_scale (mask: 0 or 1/(1-p) per element, NULL = no dropout)
__global__ void relu_mask_bwd_kernel(float* __restrict__ g, const float* __restrict__ act, const float* __restrict__ mask, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float v = act[i] > 0.f ? g[i] : 0.f;
    if (mask) v *= mask[i];
    g[i] = v;
  }
}
__global__ void mul_kernel(float* __restrict__ x, const float* __restrict__ m, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) x[i] *= m[i];
}
__global__ void sumsq_kernel(const float* __restrict__ x, size_t n, float* __restrict__ acc) {
  __shared__ float red[8];
  float s = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) s = fmaf(x[i], x[i], s);
  s = block_sum(s, red);
  if (threadIdx.x == 0) atomicAdd(acc, s);
}
// clip_grad_norm_: scale = min(1, max_norm / (sqrt(sumsq) + 1e-6)); writes scale and the norm
__global__ void clip_scale_kernel(const float* __restrict__ sumsq, float max_norm, float* __restrict__ out2) {
  const float norm = sqrtf(sumsq[0]);
  out2[0] = max_norm > 0.f ? fminf(1.f, max_norm / (norm + 1e-6f)) : 1.f;
  out2[1] = norm;
}
// torch.optim.Adam (no amsgrad), L2-style weight decay: g' = g*scale + wd*p; m, v EMAs; p -= lr * mhat / (sqrt(vhat) + eps)
// blockIdx.y = e: member e of an ensemble's flat [E, n] buffers, its gradient scaled by scale[e]; skipped when active[e] == 0
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t n,
                            float lr, float b1, float b2, float eps, float wd, float bc1, float bc2, const float* __restrict__ scale,
                            const uint8_t* __restrict__ active) {
  const size_t e = blockIdx.y;
  if (active && !active[e]) return;
  const float sc = scale ? scale[e] : 1.f;
  p += e * n; g += e * n; m += e * n; v += e * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float gr = g[i] * sc;
    if (wd != 0.f) gr = fmaf(wd, p[i], gr);
    const float mi = b1 * m[i] + (1.f - b1) * gr;
    const float vi = b2 * v[i] + (1.f - b2) * gr * gr;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// p = sigmoid(z); loss += mean_i BCE(p_i, y_i); dz_i = d loss / d z_i   (nn.BCELoss on a Sigmoid output, logs clamped at -100 as torch)
// One element: writes p and dz, returns t log p + (1-t) log(1-p) (the caller subtracts it from its loss sum)
__device__ __forceinline__ float bce_sigmoid_elem(float z, float t, float inv_n, float& p_out, float& dz) {
  const float p = sigm(z);
  const float lp = fmaxf(logf(p), -100.f), l1p = fmaxf(logf(1.f - p), -100.f);
  const float dl_dp = -(t / fmaxf(p, 1e-44f)) * (lp > -100.f ? 1.f : 0.f) + ((1.f - t) / fmaxf(1.f - p, 1e-44f)) * (l1p > -100.f ? 1.f : 0.f);
  p_out = p;
  dz = dl_dp * p * (1.f - p) * inv_n;
  return t * lp + (1.f - t) * l1p;
}
__global__ void bce_sigmoid_kernel(const float* __restrict__ z, const float* __restrict__ y, int n, float* __restrict__ p_out,
                                   float* __restrict__ loss_sum, float* __restrict__ dz) {
  __shared__ float red[8];
  float ls = 0.f;
  const float inv_n = 1.f / (float)n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) ls -= bce_sigmoid_elem(z[i], y[i], inv_n, p_out[i], dz[i]);
  ls = block_sum(ls, red);
  if (threadIdx.x == 0) atomicAdd(loss_sum, ls * inv_n);
}

// MoE combine (models/moe.py:37-47) + BCE, forward and backward: out_i = sum_e sigmoid(z[i,e]) * softmax_e(r[i,:]);
// loss = mean BCE(out, y); dz [n,E] (expert logits), dr [n,E] (router logits).  One row (its E logits z, r): writes out, dz, dr and
// returns t log o + (1-t) log(1-o)
__device__ __forceinline__ float moe_combine_elem(const float* __restrict__ z, const float* __restrict__ r, float t, int E, float inv_n,
                                                  float& out, float* __restrict__ dz, float* __restrict__ dr) {
  float mx = -INFINITY;
  for (int e = 0; e < E; ++e) mx = fmaxf(mx, r[e]);
  float se = 0.f;
  for (int e = 0; e < E; ++e) se += expf(r[e] - mx);
  float o = 0.f;
  for (int e = 0; e < E; ++e) o += sigm(z[e]) * (expf(r[e] - mx) / se);
  const float lp = fmaxf(logf(o), -100.f), l1p = fmaxf(logf(1.f - o), -100.f);
  const float dl_do = (-(t / fmaxf(o, 1e-44f)) * (lp > -100.f ? 1.f : 0.f) + ((1.f - t) / fmaxf(1.f - o, 1e-44f)) * (l1p > -100.f ? 1.f : 0.f)) * inv_n;
  out = o;
  for (int e = 0; e < E; ++e) {
    const float pe = sigm(z[e]);
    const float we = expf(r[e] - mx) / se;
    dz[e] = dl_do * we * pe * (1.f - pe);
    dr[e] = dl_do * we * (pe - o);               // softmax backward: w_e * (d_w_e - sum_j w_j d_w_j), d_w_e = dl_do * p_e
  }
  return t * lp + (1.f - t) * l1p;
}
__global__ void moe_combine_train_kernel(const float* __restrict__ z, const float* __restrict__ r, const float* __restrict__ y, int n, int E,
                                         float* __restrict__ out, float* __restrict__ loss_sum, float* __restrict__ dz, float* __restrict__ dr) {
  __shared__ float red[8];
  float ls = 0.f;
  const float inv_n = 1.f / (float)n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    ls -= moe_combine_elem(z + (size_t)i * E, r + (size_t)i * E, y[i], E, inv_n, out[i], dz + (size_t)i * E, dr + (size_t)i * E);
  ls = block_sum(ls, red);
  if (threadIdx.x == 0) atomicAdd(loss_sum, ls * inv_n);
}

// f32 -> bf16 (round to nearest even): operands of the tensor-core training path
__global__ void cast_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) y[i] = __float2bfloat16(x[i]);
}
__global__ void add_kernel(float* __restrict__ x, const float* __restrict__ y, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) x[i] += y[i];
}
// dY [n, ho, wo, k] -> zero-dilated, zero-bordered copy [n, hd, wd, k] with dY[p, q] at (off + p*stride, off + q*stride): the input
// of the stride-1 convolution that computes the data gradient of a strided convolution (transposed convolution)
__global__ void dilate_bf16_kernel(const float* __restrict__ dy, __nv_bfloat16* __restrict__ out, int N, int Ho, int Wo, int K, int Hd, int Wd,
                                   int stride, int off) {
  const size_t total = (size_t)N * Hd * Wd * K;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    size_t t = i / K;
    const int x = (int)(t % Wd); t /= Wd;
    const int y = (int)(t % Hd);
    const int n = (int)(t / Hd);
    const int py = y - off, px = x - off;
    float v = 0.f;
    if (py >= 0 && px >= 0 && py % stride == 0 && px % stride == 0) {
      const int p = py / stride, q = px / stride;
      if (p < Ho && q < Wo) v = dy[(((size_t)n * Ho + p) * Wo + q) * K + k];
    }
    out[i] = __float2bfloat16(v);
  }
}

// ------------------------------------------------------------------------------------------------------
// Deep ensembles: E members of one head trained in lockstep, every launch covering all members (flat [E, P] parameter and gradient
// buffers, member e's operands e times their member stride further, stride 0 = shared).  Per member the arithmetic is the single
// kernels' (the GEMM tile, bce_sigmoid_elem, moe_combine_elem, the MIL bag, Adam's element); losses, MIL's parameter gradients and the
// clip norms are reduced in a fixed order without atomics, so results repeat bit for bit and do not depend on the other members.
// One block per member: loss[e] = the member's mean BCE (or MoE BCE); y member stride y_es
__global__ void __launch_bounds__(256)
bce_sigmoid_batched_kernel(const float* __restrict__ z, const float* __restrict__ y, long y_es, int n, float* __restrict__ p_out,
                           float* __restrict__ loss, float* __restrict__ dz) {
  __shared__ float red[8];
  const long e = blockIdx.x, off = e * n;
  const float inv_n = 1.f / (float)n;
  float ls = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) ls -= bce_sigmoid_elem(z[off + i], y[e * y_es + i], inv_n, p_out[off + i], dz[off + i]);
  ls = block_sum(ls, red);
  if (threadIdx.x == 0) loss[e] = ls * inv_n;
}
__global__ void __launch_bounds__(256)
moe_combine_batched_kernel(const float* __restrict__ z, const float* __restrict__ r, const float* __restrict__ y, long y_es, int n, int M,
                           float* __restrict__ out, float* __restrict__ loss, float* __restrict__ dz, float* __restrict__ dr) {
  __shared__ float red[8];
  const size_t e = blockIdx.x, off = e * n * M;
  z += off; r += off; dz += off; dr += off; out += e * n; y += e * y_es;
  const float inv_n = 1.f / (float)n;
  float ls = 0.f;
  for (int i = threadIdx.x; i < n; i += 256)
    ls -= moe_combine_elem(z + (size_t)i * M, r + (size_t)i * M, y[i], M, inv_n, out[i], dz + (size_t)i * M, dr + (size_t)i * M);
  ls = block_sum(ls, red);
  if (threadIdx.x == 0) loss[e] = ls * inv_n;
}
// MIL: column c of member e's MilPartialSink rows summed over the bags in ascending order, added to the member's gradient (loss: written)
__global__ void __launch_bounds__(256)
mil_partial_reduce_kernel(const float* __restrict__ partial, int E, int B, int H, int A, float* __restrict__ d_w_cls, float* __restrict__ d_w_w,
                          float* __restrict__ d_b_cls, float* __restrict__ d_b_w, long g_es, float* __restrict__ loss) {
  const int W = H + A + 3;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < (long)E * W; i += (long)gridDim.x * blockDim.x) {
    const long e = i / W;
    const int c = (int)(i - e * W);
    const float* p = partial + (size_t)e * B * W + c;
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += p[(size_t)b * W];
    if (c < H) d_w_cls[e * g_es + c] += s;
    else if (c < H + A) d_w_w[e * g_es + c - H] += s;
    else if (c == H + A) d_b_cls[e * g_es] += s;
    else if (c == H + A + 1) d_b_w[e * g_es] += s;
    else loss[e] = s;
  }
}
// clip_grad_norm_ per member: one block per row of g [E, P]; scale[e] = min(1, max_norm / (norm + 1e-6))
__global__ void __launch_bounds__(256)
clip_scale_batched_kernel(const float* __restrict__ g, long P, float max_norm, float* __restrict__ scale) {
  __shared__ float red[8];
  const float* x = g + (long)blockIdx.x * P;
  float s = 0.f;
  for (long i = threadIdx.x; i < P; i += 256) s = fmaf(x[i], x[i], s);
  s = block_sum(s, red);
  if (threadIdx.x == 0) scale[blockIdx.x] = max_norm > 0.f ? fminf(1.f, max_norm / (sqrtf(s) + 1e-6f)) : 1.f;
}

static inline int ew_blocks(size_t n) { return (int)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)num_sms() * 16)); }

}  // namespace pdf

using namespace pdf;

extern "C" int pdf_gemm_f32(int M, int N, int K, const float* A, long a_rs, long a_cs, const float* B, long b_rs, long b_cs, float* C,
                            long c_rs, const float* bias, int act, int accumulate, pdf_stream_t stream) {
  PDF_REQUIRE(M > 0 && N > 0 && K > 0 && A && B && C, "pdf_gemm_f32: bad arguments");
  dim3 grid(ceil_div(M, TBM), ceil_div(N, TBN));
  gemm_strided_kernel<<<grid, 256, 0, as_stream(stream)>>>(A, a_rs, a_cs, B, b_rs, b_cs, C, c_rs, bias, M, N, K, act, accumulate, 0, 0, 0, 0);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

static int check_conv(const pdf_op* op, const char* what) {
  PDF_REQUIRE(op && op->n > 0 && op->h > 0 && op->w > 0 && op->c > 0 && op->k > 0 && op->r > 0 && op->s > 0 && op->stride > 0 && op->pad >= 0,
              "%s: bad conv description", what);
  PDF_REQUIRE(op->ho == (op->h + 2 * op->pad - op->r) / op->stride + 1 && op->wo == (op->w + 2 * op->pad - op->s) / op->stride + 1,
              "%s: inconsistent conv output size", what);
  return PDF_OK;
}

/* geometry from `op` (n,h,w,c,k,r,s,stride,pad,ho,wo); pointers passed explicitly */
extern "C" int pdf_conv_dgrad_f32(const pdf_op* op, const float* d_dy, const float* d_weight, float* d_dx, int accumulate, pdf_stream_t stream) {
  if (int rc = check_conv(op, "pdf_conv_dgrad_f32")) return rc;
  PDF_REQUIRE(d_dy && d_weight && d_dx, "pdf_conv_dgrad_f32: null pointer");
  dim3 grid(ceil_div((long long)op->n * op->h * op->w, TBM), ceil_div(op->c, TBN));
  conv_dgrad_f32_kernel<<<grid, 256, 0, as_stream(stream)>>>(d_dy, d_weight, d_dx, op->n, op->h, op->w, op->c, op->k, op->r, op->s,
                                                             op->stride, op->pad, op->ho, op->wo, accumulate);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_conv_wgrad_f32(const pdf_op* op, const float* d_x, const float* d_dy, float* d_dw, pdf_stream_t stream) {
  if (int rc = check_conv(op, "pdf_conv_wgrad_f32")) return rc;
  PDF_REQUIRE(d_x && d_dy && d_dw, "pdf_conv_wgrad_f32: null pointer");
  const long long M = (long long)op->n * op->ho * op->wo;
  const int rows = op->r * op->s * op->c;
  const int tiles = ceil_div(rows, TBM) * ceil_div(op->k, TBN);
  // enough pixel slabs to fill the machine ~4x over, each at least 512 pixels
  int nz = (int)std::max<long long>(1, std::min<long long>((M + 511) / 512, (4LL * num_sms() + tiles - 1) / tiles));
  int slab = (int)((M + nz - 1) / nz);
  slab = (slab + TBK - 1) / TBK * TBK;
  nz = (int)((M + slab - 1) / slab);
  dim3 grid(ceil_div(rows, TBM), ceil_div(op->k, TBN), nz);
  conv_wgrad_f32_kernel<<<grid, 256, 0, as_stream(stream)>>>(d_x, d_dy, d_dw, op->n, op->h, op->w, op->c, op->k, op->r, op->s, op->stride,
                                                             op->pad, op->ho, op->wo, slab);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_bn_train_forward(int n_groups, const int32_t* d_goff, int max_group_rows, int C, const float* d_x, const float* d_gamma,
                                    const float* d_beta, float eps, const float* d_residual, int relu, float* d_y, float* d_mean,
                                    float* d_invstd, float* d_var_unbiased, double* d_scratch, pdf_stream_t stream) {
  PDF_REQUIRE(n_groups > 0 && d_goff && max_group_rows > 0 && C > 0 && C % 4 == 0 && d_x && d_gamma && d_beta && d_y && d_mean && d_invstd &&
              d_var_unbiased && d_scratch, "pdf_bn_train_forward: bad arguments (C %% 4 == 0, scratch of 2*groups*C doubles)");
  cudaStream_t s = as_stream(stream);
  PDF_CHECK_CUDA(cudaMemsetAsync(d_scratch, 0, (size_t)2 * n_groups * C * sizeof(double), s));
  bn_stats_kernel<<<dim3(ceil_div(C, 32), n_groups, ceil_div(max_group_rows, kBnRowsPerBlock)), 256, 0, s>>>(d_x, d_goff, C, d_scratch);
  PDF_CHECK_LAUNCH();
  bn_stats_finalize_kernel<<<ceil_div(n_groups * C, 256), 256, 0, s>>>(d_scratch, d_goff, n_groups, C, eps, d_mean, d_invstd, d_var_unbiased);
  PDF_CHECK_LAUNCH();
  bn_apply_kernel<<<dim3(std::max(1, 8 * num_sms() / n_groups), n_groups), 256, 0, s>>>(d_x, d_goff, C, d_mean, d_invstd, d_gamma, d_beta,
                                                                                       d_residual, relu, d_y, nullptr);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_bn_train_backward(int n_groups, const int32_t* d_goff, int max_group_rows, int C, const float* d_dy, const float* d_y,
                                     const float* d_x, const float* d_gamma, const float* d_mean, const float* d_invstd, int relu,
                                     double* d_scratch, float* d_dx, float* d_dres, int dres_accumulate, float* d_dgamma,
                                     float* d_dbeta, pdf_stream_t stream) {
  PDF_REQUIRE(n_groups > 0 && d_goff && max_group_rows > 0 && C > 0 && C % 4 == 0 && d_dy && d_y && d_x && d_gamma && d_mean && d_invstd &&
              d_scratch && d_dx && d_dgamma && d_dbeta, "pdf_bn_train_backward: bad arguments (C %% 4 == 0, scratch of 3*groups*C doubles)");
  cudaStream_t s = as_stream(stream);
  double* acc = d_scratch;                                                // [G][C][2] float64 partial sums
  float* sums = reinterpret_cast<float*>(d_scratch + (size_t)2 * n_groups * C);   // [2][G][C] f32: sum g | sum g*xhat
  PDF_CHECK_CUDA(cudaMemsetAsync(acc, 0, (size_t)2 * n_groups * C * sizeof(double), s));
  bn_bwd_reduce_kernel<<<dim3(ceil_div(C, 32), n_groups, ceil_div(max_group_rows, kBnRowsPerBlock)), 256, 0, s>>>(d_dy, d_y, d_x, d_goff, C, d_mean,
                                                                                                             d_invstd, relu, acc);
  PDF_CHECK_LAUNCH();
  bn_bwd_finalize_kernel<<<ceil_div(C, 128), 128, 0, s>>>(acc, n_groups, C, sums, d_dgamma, d_dbeta);
  PDF_CHECK_LAUNCH();
  bn_bwd_apply_kernel<<<dim3(std::max(1, 8 * num_sms() / n_groups), n_groups), 256, 0, s>>>(
      d_dy, d_y, d_x, d_goff, C, d_mean, d_invstd, d_gamma, relu, sums, sums + (size_t)n_groups * C, d_dx, nullptr, d_dres,
      dres_accumulate);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_bn_update_running(int n_groups, int C, const float* d_mean, const float* d_var_unbiased, float momentum,
                                     float* d_running_mean, float* d_running_var, pdf_stream_t stream) {
  PDF_REQUIRE(n_groups > 0 && C > 0 && d_mean && d_var_unbiased && d_running_mean && d_running_var, "pdf_bn_update_running: bad arguments");
  bn_running_kernel<<<ceil_div(C, 128), 128, 0, as_stream(stream)>>>(d_mean, d_var_unbiased, n_groups, C, momentum, d_running_mean, d_running_var);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_maxpool_backward_f32(int n, int h, int w, int c, const float* d_x, const float* d_dy, float* d_dx, pdf_stream_t stream) {
  PDF_REQUIRE(n > 0 && h > 0 && w > 0 && c > 0 && d_x && d_dy && d_dx, "pdf_maxpool_backward_f32: bad arguments");
  const int ho = (h + 2 - 3) / 2 + 1, wo = (w + 2 - 3) / 2 + 1;
  PDF_CHECK_CUDA(cudaMemsetAsync(d_dx, 0, (size_t)n * h * w * c * sizeof(float), as_stream(stream)));
  maxpool_bwd_kernel<<<ew_blocks((size_t)n * ho * wo * c), 256, 0, as_stream(stream)>>>(d_x, d_dy, d_dx, n, h, w, c, ho, wo);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_avgpool_backward_f32(int n, int hw, int c, const float* d_demb, float* d_dx, pdf_stream_t stream) {
  PDF_REQUIRE(n > 0 && hw > 0 && c > 0 && d_demb && d_dx, "pdf_avgpool_backward_f32: bad arguments");
  const size_t total = (size_t)n * hw * c;
  avgpool_bwd_kernel<<<ew_blocks(total), 256, 0, as_stream(stream)>>>(d_demb, d_dx, hw, c, total);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_mil_pool_train(const pdf_mil_weights* w, const pdf_mil_train* t, int n_bags, int Lmax, const float* d_h, const float* d_vu,
                                  const int32_t* d_len, const float* d_target, float* d_prob, float* d_loss, float* d_dh, float* d_dvu,
                                  pdf_stream_t stream) {
  PDF_REQUIRE(w && t && n_bags > 0 && Lmax > 0 && d_h && d_vu && d_len && d_target && d_prob && d_loss && d_dh && d_dvu,
              "pdf_mil_pool_train: bad arguments");
  PDF_REQUIRE(w->w_w && w->b_w && w->w_cls && w->b_cls && t->d_w_w && t->d_b_w && t->d_w_cls && t->d_b_cls, "pdf_mil_pool_train: null pointer");
  MilTrainArgs a;
  a.H = w->H; a.A = w->A; a.gated = w->gated; a.Lmax = Lmax; a.n_bags = n_bags;
  a.loss_type = t->loss_type; a.pos_weight = t->pos_weight; a.focal_gamma = t->focal_gamma; a.focal_alpha = t->focal_alpha;
  a.w_w = w->w_w; a.b_w = w->b_w; a.w_cls = w->w_cls; a.b_cls = w->b_cls;
  a.d_w_w = t->d_w_w; a.d_b_w = t->d_b_w; a.d_w_cls = t->d_w_cls; a.d_b_cls = t->d_b_cls;
  const size_t smem = ((size_t)2 * Lmax + w->H) * sizeof(float);
  PDF_REQUIRE(smem <= 200 * 1024, "pdf_mil_pool_train: bag too large for shared memory");
  if (smem > 48 * 1024)
    PDF_CHECK_CUDA(cudaFuncSetAttribute(mil_pool_train_kernel<MilAtomicSink>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const MilAtomicSink sink{d_loss, a.d_w_w, a.d_b_w, a.d_w_cls, a.d_b_cls};
  mil_pool_train_kernel<<<n_bags, 256, smem, as_stream(stream)>>>(a, 0L, d_h, d_vu, d_len, d_target, d_prob, d_dh, d_dvu, sink);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_colsum_f32(int M, int N, const float* d_x, float* d_out, int accumulate, pdf_stream_t stream) {
  PDF_REQUIRE(M > 0 && N > 0 && d_x && d_out, "pdf_colsum_f32: bad arguments");
  colsum_kernel<<<ceil_div(N, 128), 128, 0, as_stream(stream)>>>(d_x, M, N, d_out, accumulate);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_relu_mask_backward(float* d_grad, const float* d_act, const float* d_mask, size_t n, pdf_stream_t stream) {
  PDF_REQUIRE(d_grad && d_act && n > 0, "pdf_relu_mask_backward: bad arguments");
  relu_mask_bwd_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(d_grad, d_act, d_mask, n);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_mul_f32(float* d_x, const float* d_m, size_t n, pdf_stream_t stream) {
  PDF_REQUIRE(d_x && d_m && n > 0, "pdf_mul_f32: bad arguments");
  mul_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(d_x, d_m, n);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

/* d_acc[0] += sum x^2 (zero it before the first tensor of a parameter set) */
extern "C" int pdf_sumsq_f32(const float* d_x, size_t n, float* d_acc, pdf_stream_t stream) {
  PDF_REQUIRE(d_x && d_acc && n > 0, "pdf_sumsq_f32: bad arguments");
  sumsq_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(d_x, n, d_acc);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

/* d_out2[0] = min(1, max_norm / (sqrt(d_sumsq[0]) + 1e-6)), d_out2[1] = the norm  (torch.nn.utils.clip_grad_norm_) */
extern "C" int pdf_clip_scale(const float* d_sumsq, float max_norm, float* d_out2, pdf_stream_t stream) {
  PDF_REQUIRE(d_sumsq && d_out2, "pdf_clip_scale: bad arguments");
  clip_scale_kernel<<<1, 1, 0, as_stream(stream)>>>(d_sumsq, max_norm, d_out2);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_adam_step(float* d_param, const float* d_grad, float* d_m, float* d_v, size_t n, float lr, float beta1, float beta2,
                             float eps, float weight_decay, int step, const float* d_grad_scale, pdf_stream_t stream) {
  PDF_REQUIRE(d_param && d_grad && d_m && d_v && n > 0 && step >= 1, "pdf_adam_step: bad arguments");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(d_param, d_grad, d_m, d_v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2, d_grad_scale,
                                                                  nullptr);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_bce_sigmoid_train(int n, const float* d_z, const float* d_y, float* d_prob, float* d_loss, float* d_dz, pdf_stream_t stream) {
  PDF_REQUIRE(n > 0 && d_z && d_y && d_prob && d_loss && d_dz, "pdf_bce_sigmoid_train: bad arguments");
  bce_sigmoid_kernel<<<ew_blocks((size_t)n), 256, 0, as_stream(stream)>>>(d_z, d_y, n, d_prob, d_loss, d_dz);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_moe_combine_train(int n, int n_experts, const float* d_z, const float* d_r, const float* d_y, float* d_out, float* d_loss,
                                     float* d_dz, float* d_dr, pdf_stream_t stream) {
  PDF_REQUIRE(n > 0 && n_experts > 0 && n_experts <= PDF_MAX_MODS && d_z && d_r && d_y && d_out && d_loss && d_dz && d_dr,
              "pdf_moe_combine_train: bad arguments");
  moe_combine_train_kernel<<<ew_blocks((size_t)n), 256, 0, as_stream(stream)>>>(d_z, d_r, d_y, n, n_experts, d_out, d_loss, d_dz, d_dr);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_cast_bf16(const float* d_x, void* d_y, size_t n, pdf_stream_t stream) {
  PDF_REQUIRE(d_x && d_y && n > 0, "pdf_cast_bf16: bad arguments");
  cast_bf16_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(d_x, reinterpret_cast<__nv_bfloat16*>(d_y), n);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_add_f32(float* d_x, const float* d_y, size_t n, pdf_stream_t stream) {
  PDF_REQUIRE(d_x && d_y && n > 0, "pdf_add_f32: bad arguments");
  add_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(d_x, d_y, n);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_dilate_bf16(int n, int ho, int wo, int k, int hd, int wd, int stride, int offset, const float* d_dy, void* d_out,
                               pdf_stream_t stream) {
  PDF_REQUIRE(n > 0 && ho > 0 && wo > 0 && k > 0 && hd >= offset + (ho - 1) * stride + 1 && wd >= offset + (wo - 1) * stride + 1 && stride >= 1 &&
              offset >= 0 && d_dy && d_out, "pdf_dilate_bf16: bad arguments");
  dilate_bf16_kernel<<<ew_blocks((size_t)n * hd * wd * k), 256, 0, as_stream(stream)>>>(d_dy, reinterpret_cast<__nv_bfloat16*>(d_out), n, ho, wo, k,
                                                                                        hd, wd, stride, offset);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

// ------------------------------------------------------------------------------------------------------ deep ensembles
static constexpr int kMaxMembers = 1024;
static bool ens_ok(const void* p) { return p && (reinterpret_cast<uintptr_t>(p) & 3) == 0; }      // non-null, 4-byte aligned
static bool ens_members_ok(int E) { return E >= 1 && E <= kMaxMembers; }

extern "C" int pdf_gemm_f32_batched(int n_members, int M, int N, int K, const float* A, long a_rs, long a_cs, long a_es, const float* B, long b_rs,
                                    long b_cs, long b_es, float* C, long c_rs, long c_es, const float* bias, long bias_es, int act, int accumulate,
                                    pdf_stream_t stream) {
  PDF_REQUIRE(ens_members_ok(n_members) && M > 0 && N > 0 && K > 0, "pdf_gemm_f32_batched: bad sizes (1 <= members <= %d)", kMaxMembers);
  PDF_REQUIRE(ens_ok(A) && ens_ok(B) && ens_ok(C) && (!bias || ens_ok(bias)), "pdf_gemm_f32_batched: null or misaligned pointer");
  PDF_REQUIRE(a_es >= 0 && b_es >= 0 && c_es >= 0 && bias_es >= 0, "pdf_gemm_f32_batched: negative member stride");
  PDF_REQUIRE(n_members == 1 || c_es > 0, "pdf_gemm_f32_batched: members may not share the output");
  dim3 grid(ceil_div(M, TBM), ceil_div(N, TBN), n_members);
  gemm_strided_kernel<<<grid, 256, 0, as_stream(stream)>>>(A, a_rs, a_cs, B, b_rs, b_cs, C, c_rs, bias, M, N, K, act, accumulate, a_es, b_es, c_es,
                                                           bias_es);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_bce_sigmoid_train_batched(int n_members, int n, const float* d_z, const float* d_y, long y_es, float* d_prob, float* d_loss,
                                             float* d_dz, pdf_stream_t stream) {
  PDF_REQUIRE(ens_members_ok(n_members) && n > 0 && y_es >= 0, "pdf_bce_sigmoid_train_batched: bad sizes");
  PDF_REQUIRE(ens_ok(d_z) && ens_ok(d_y) && ens_ok(d_prob) && ens_ok(d_loss) && ens_ok(d_dz), "pdf_bce_sigmoid_train_batched: null or misaligned pointer");
  bce_sigmoid_batched_kernel<<<n_members, 256, 0, as_stream(stream)>>>(d_z, d_y, y_es, n, d_prob, d_loss, d_dz);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_moe_combine_train_batched(int n_members, int n, int n_experts, const float* d_z, const float* d_r, const float* d_y, long y_es,
                                             float* d_out, float* d_loss, float* d_dz, float* d_dr, pdf_stream_t stream) {
  PDF_REQUIRE(ens_members_ok(n_members) && n > 0 && n_experts > 0 && n_experts <= PDF_MAX_MODS && y_es >= 0,
              "pdf_moe_combine_train_batched: bad sizes");
  PDF_REQUIRE(ens_ok(d_z) && ens_ok(d_r) && ens_ok(d_y) && ens_ok(d_out) && ens_ok(d_loss) && ens_ok(d_dz) && ens_ok(d_dr),
              "pdf_moe_combine_train_batched: null or misaligned pointer");
  moe_combine_batched_kernel<<<n_members, 256, 0, as_stream(stream)>>>(d_z, d_r, d_y, y_es, n, n_experts, d_out, d_loss, d_dz, d_dr);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" size_t pdf_mil_pool_train_batched_workspace_bytes(int n_members, const pdf_mil_weights* w, int n_bags) {
  if (!ens_members_ok(n_members) || !w || n_bags <= 0 || w->H <= 0 || w->A <= 0) return 0;
  return (size_t)n_members * n_bags * (w->H + w->A + 3) * sizeof(float);
}

extern "C" int pdf_mil_pool_train_batched(int n_members, const pdf_mil_weights* w, long w_es, const pdf_mil_train* t, long g_es, int n_bags,
                                          int Lmax, const float* d_h, const float* d_vu, const int32_t* d_len, const float* d_target,
                                          float* d_prob, float* d_loss, float* d_dh, float* d_dvu, void* d_workspace, pdf_stream_t stream) {
  PDF_REQUIRE(ens_members_ok(n_members) && w && t && n_bags > 0 && Lmax > 0 && w_es >= 0 && g_es >= 0 && w->H > 0 && w->A > 0,
              "pdf_mil_pool_train_batched: bad arguments");
  PDF_REQUIRE(ens_ok(w->w_w) && ens_ok(w->b_w) && ens_ok(w->w_cls) && ens_ok(w->b_cls) && ens_ok(t->d_w_w) && ens_ok(t->d_b_w) &&
              ens_ok(t->d_w_cls) && ens_ok(t->d_b_cls), "pdf_mil_pool_train_batched: null or misaligned parameter pointer");
  PDF_REQUIRE(ens_ok(d_h) && ens_ok(d_vu) && ens_ok(d_len) && ens_ok(d_target) && ens_ok(d_prob) && ens_ok(d_loss) && ens_ok(d_dh) &&
              ens_ok(d_dvu) && ens_ok(d_workspace), "pdf_mil_pool_train_batched: null or misaligned pointer");
  const size_t smem = ((size_t)2 * Lmax + w->H) * sizeof(float);
  PDF_REQUIRE(smem <= 200 * 1024, "pdf_mil_pool_train_batched: bag too large for shared memory");
  MilTrainArgs a;
  a.H = w->H; a.A = w->A; a.gated = w->gated; a.Lmax = Lmax; a.n_bags = n_bags;
  a.loss_type = t->loss_type; a.pos_weight = t->pos_weight; a.focal_gamma = t->focal_gamma; a.focal_alpha = t->focal_alpha;
  a.w_w = w->w_w; a.b_w = w->b_w; a.w_cls = w->w_cls; a.b_cls = w->b_cls;
  a.d_w_w = t->d_w_w; a.d_b_w = t->d_b_w; a.d_w_cls = t->d_w_cls; a.d_b_cls = t->d_b_cls;
  cudaStream_t s = as_stream(stream);
  float* partial = static_cast<float*>(d_workspace);
  PDF_CHECK_CUDA(cudaMemsetAsync(partial, 0, pdf_mil_pool_train_batched_workspace_bytes(n_members, w, n_bags), s));    // empty bags add 0
  if (smem > 48 * 1024)
    PDF_CHECK_CUDA(cudaFuncSetAttribute(mil_pool_train_kernel<MilPartialSink>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const MilPartialSink sink{partial, w->H, w->A};
  mil_pool_train_kernel<<<dim3(n_bags, n_members), 256, smem, s>>>(a, w_es, d_h, d_vu, d_len, d_target, d_prob, d_dh, d_dvu, sink);
  PDF_CHECK_LAUNCH();
  mil_partial_reduce_kernel<<<ew_blocks((size_t)n_members * (w->H + w->A + 3)), 256, 0, s>>>(partial, n_members, n_bags, w->H, w->A, t->d_w_cls,
                                                                                            t->d_w_w, t->d_b_cls, t->d_b_w, g_es, d_loss);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_clip_scale_batched(int n_members, const float* d_grad, long n_params, float max_norm, float* d_scale, pdf_stream_t stream) {
  PDF_REQUIRE(ens_members_ok(n_members) && n_params > 0, "pdf_clip_scale_batched: bad sizes");
  PDF_REQUIRE(ens_ok(d_grad) && ens_ok(d_scale), "pdf_clip_scale_batched: null or misaligned pointer");
  clip_scale_batched_kernel<<<n_members, 256, 0, as_stream(stream)>>>(d_grad, n_params, max_norm, d_scale);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_adam_step_batched(int n_members, float* d_param, const float* d_grad, float* d_m, float* d_v, long n_params, float lr,
                                     float beta1, float beta2, float eps, float weight_decay, int step, const float* d_grad_scale,
                                     const uint8_t* d_active, pdf_stream_t stream) {
  PDF_REQUIRE(ens_members_ok(n_members) && n_params > 0 && step >= 1, "pdf_adam_step_batched: bad arguments");
  PDF_REQUIRE(ens_ok(d_param) && ens_ok(d_grad) && ens_ok(d_m) && ens_ok(d_v) && (!d_grad_scale || ens_ok(d_grad_scale)),
              "pdf_adam_step_batched: null or misaligned pointer");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  const int per = std::max(1, ew_blocks((size_t)n_params * n_members) / n_members);
  adam_kernel<<<dim3(per, n_members), 256, 0, as_stream(stream)>>>(d_param, d_grad, d_m, d_v, (size_t)n_params, lr, beta1, beta2, eps, weight_decay,
                                                                   bc1, bc2, d_grad_scale, d_active);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

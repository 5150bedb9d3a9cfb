// Explanations of MIL predictions: per-slice attention, per-slice logit contributions, the gradient of the logit with respect to
// every slice embedding, and Grad-CAM maps at the backbone's last stage.  FP32 throughout.
//
// The logit of a bag is exactly decomposable per slice:  z = w_c . sum_l a_l h_l + b_c = sum_l a_l (w_c . h_l) + b_c.
// Its gradient is seeded with dz = 1 (the gradient of z itself, not of a loss) and goes back through the softmax and the
// attention layer(s) with the algebra of mil_pool_train_kernel (train.cu); the linear layers' backward is pdf_gemm_f32.
// The backbone embeds a slice as the spatial mean of its last feature map o4 [hw, hw, C], so dz/do4[i, j, c] = g[c] / hw^2 with
// g = dz/dx the embedding gradient: Grad-CAM at that layer is ReLU(sum_c g[c] o4[i, j, c] / hw^2), one pass over o4, no conv backward.
#include <climits>

#include "common.cuh"
#include "ops.cuh"

namespace pdf {

__device__ __forceinline__ float ex_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float ex_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

// sum over a 256-thread block; every thread gets the total (red[8] is free again on return)
__device__ __forceinline__ float ex_block_sum(float v, float* red) {
  v = ex_warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  for (int i = 0; i < 8; ++i) t += red[i];
  __syncthreads();
  return t;
}

// ------------------------------------------------------------------------------------------------------
// One block per bag, the shape of mil_pool_kernel (heads.cu) on its FP32 inputs: h = ReLU(X W_i^T + b_i) [n_bags*Lmax, H] and the
// attention pre-activations without bias vu [n_bags*Lmax, NA] (NA = 2A gated: v | u), both from gemm_nt_f32_kernel.  The scores,
// the softmax and the pooled logit repeat mil_pool_kernel's arithmetic in its order, so sigmoid(logit) is the sweep's probability.
// Writes attn / contrib [n_bags, Lmax] (0 on the padding) and logit [n_bags] (NaN for a missing bag).  With dh != NULL it also
// writes the backward seeds of dz = 1 over every row of the bag (0 on the padding):
//   dh_l = a_l w_c ;  ds_l = a_l (u_l - sum_k a_k u_k), u_l = w_c . h_l ;  dvu_l = ds_l through w_w and tanh (x sigmoid, gated).
__global__ void __launch_bounds__(256)
mil_explain_kernel(const float* __restrict__ hbuf, const float* __restrict__ vu, const int32_t* __restrict__ lens, int Lmax,
                   pdf_mil_weights w, float* __restrict__ logit, float* __restrict__ attn, float* __restrict__ contrib,
                   float* __restrict__ dh, float* __restrict__ dvu) {
  extern __shared__ float sm[];
  float* s_a = sm;                     // [Lmax] scores -> attention weights
  float* s_u = sm + Lmax;              // [Lmax] u_l = w_c . h_l -> ds_l
  __shared__ float s_red[8];
  const int bag = blockIdx.x;
  const int len = max(0, min(lens[bag], Lmax));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = w.H, A = w.A, NA = w.gated ? 2 * A : A;
  const float* hb = hbuf + (size_t)bag * Lmax * H;
  const float* vb = vu + (size_t)bag * Lmax * NA;
  for (int l = len + tid; l < Lmax; l += 256) {
    attn[(size_t)bag * Lmax + l] = 0.f;
    contrib[(size_t)bag * Lmax + l] = 0.f;
  }
  if (dh) {                            // padded rows (every row of a missing bag) carry no gradient
    for (size_t i = (size_t)len * H + tid; i < (size_t)Lmax * H; i += 256) dh[(size_t)bag * Lmax * H + i] = 0.f;
    for (size_t i = (size_t)len * NA + tid; i < (size_t)Lmax * NA; i += 256) dvu[(size_t)bag * Lmax * NA + i] = 0.f;
  }
  if (len == 0) {
    if (tid == 0) logit[bag] = __int_as_float(0x7fc00000);
    return;
  }
  // scores (mil_pool_kernel's FP32 branch) and u_l
  for (int l = warp; l < len; l += 8) {
    const float* r = vb + (size_t)l * NA;
    float sc = 0.f;
    for (int a = lane; a < A; a += 32) {
      float t = tanhf(r[a] + __ldg(w.b_v + a));
      if (w.gated) t *= ex_sigmoid(r[A + a] + __ldg(w.b_u + a));
      sc = fmaf(__ldg(w.w_w + a), t, sc);
    }
    sc = ex_warp_sum(sc);
    float u = 0.f;
    for (int i = lane; i < H; i += 32) u = fmaf(__ldg(w.w_cls + i), hb[(size_t)l * H + i], u);
    u = ex_warp_sum(u);
    if (lane == 0) { s_a[l] = sc + __ldg(w.b_w); s_u[l] = u; }
  }
  __syncthreads();
  // softmax over the valid instances, as mil_pool_kernel
  float mx = -INFINITY;
  for (int l = tid; l < len; l += 256) mx = fmaxf(mx, s_a[l]);
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = s_red[0];
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, s_red[i]);
  __syncthreads();
  float se = 0.f;
  for (int l = tid; l < len; l += 256) { const float e = expf(s_a[l] - mx); s_a[l] = e; se += e; }
  se = ex_warp_sum(se);
  if (lane == 0) s_red[warp] = se;
  __syncthreads();
  se = 0.f;
  for (int i = 0; i < 8; ++i) se += s_red[i];
  for (int l = tid; l < len; l += 256) s_a[l] = s_a[l] / se;
  __syncthreads();
  // pooled and logit with mil_pool_kernel's four accumulators per column and its reduction order
  float z = 0.f;
  for (int i = tid; i < H; i += 256) {
    float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
    int l = 0;
    for (; l + 4 <= len; l += 4) {
      p0 = fmaf(s_a[l], hb[(size_t)l * H + i], p0);
      p1 = fmaf(s_a[l + 1], hb[(size_t)(l + 1) * H + i], p1);
      p2 = fmaf(s_a[l + 2], hb[(size_t)(l + 2) * H + i], p2);
      p3 = fmaf(s_a[l + 3], hb[(size_t)(l + 3) * H + i], p3);
    }
    for (; l < len; ++l) p0 = fmaf(s_a[l], hb[(size_t)l * H + i], p0);
    z = fmaf(__ldg(w.w_cls + i), (p0 + p1) + (p2 + p3), z);
  }
  z = ex_warp_sum(z);
  __syncthreads();                     // everyone has read s_red (the softmax denominator)
  if (lane == 0) s_red[warp] = z;
  __syncthreads();
  float t = 0.f;
  for (int i = 0; i < 8; ++i) t += s_red[i];
  __syncthreads();
  if (tid == 0) logit[bag] = t + __ldg(w.b_cls);
  float dot = 0.f;
  for (int l = tid; l < len; l += 256) {
    const float a = s_a[l], u = s_u[l];
    attn[(size_t)bag * Lmax + l] = a;
    contrib[(size_t)bag * Lmax + l] = a * u;
    dot = fmaf(a, u, dot);
  }
  if (!dh) return;
  dot = ex_block_sum(dot, s_red);
  for (int l = tid; l < len; l += 256) s_u[l] = s_a[l] * (s_u[l] - dot);     // ds_l (softmax backward of dz/da_l = u_l)
  __syncthreads();
  float* dhb = dh + (size_t)bag * Lmax * H;
  for (size_t i = tid; i < (size_t)len * H; i += 256) {
    const int l = (int)(i / H), c = (int)(i - (size_t)l * H);
    dhb[i] = s_a[l] * __ldg(w.w_cls + c);
  }
  float* dvb = dvu + (size_t)bag * Lmax * NA;
  for (size_t i = tid; i < (size_t)len * A; i += 256) {
    const int l = (int)(i / A), j = (int)(i - (size_t)l * A);
    const float g = s_u[l] * __ldg(w.w_w + j);
    const float tv = tanhf(vb[(size_t)l * NA + j] + __ldg(w.b_v + j));
    if (w.gated) {
      const float su = ex_sigmoid(vb[(size_t)l * NA + A + j] + __ldg(w.b_u + j));
      dvb[(size_t)l * NA + j] = g * su * (1.f - tv * tv);
      dvb[(size_t)l * NA + A + j] = g * tv * su * (1.f - su);
    } else {
      dvb[(size_t)l * NA + j] = g * (1.f - tv * tv);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// Grad-CAM of one slice per block: cam_small[p] = ReLU(sum_c g[c] fmap[p, c] / hw^2) over the hw x hw pixels (a warp per pixel,
// float4 streaming loads: the feature map is read once), then the bilinear upsample (align_corners=False) to out_h x out_w.
// The source index is ATen's area_pixel_compute_source_index rule with the rounding of preproc.cu's resize kernels:
// src = max((dst + 0.5) * (in / out) - 0.5, 0), taps min(floor(src), in - 1) and one further, clamped.
__device__ __forceinline__ void src_taps(int d, float scale, int in, int& i0, int& i1, float& w0, float& w1) {
  const float f = fmaxf(__fsub_rn(__fmul_rn(__fadd_rn((float)d, 0.5f), scale), 0.5f), 0.0f);
  i0 = min((int)f, in - 1);
  i1 = min(i0 + 1, in - 1);
  w1 = __fsub_rn(f, (float)i0);
  w0 = __fsub_rn(1.0f, w1);
}

__global__ void __launch_bounds__(256)
gradcam_kernel(const float* __restrict__ fmap, const float* __restrict__ g, int hw, int C, int out_h, int out_w,
               float* __restrict__ cam_small, float* __restrict__ cam) {
  extern __shared__ float sm[];
  float* s_g = sm;                     // [C]
  float* s_cam = sm + C;               // [hw * hw]
  const int n = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int P = hw * hw, C4 = C >> 2;
  for (int c = tid; c < C; c += 256) s_g[c] = __ldg(g + (size_t)n * C + c);
  __syncthreads();
  const float4* f4 = reinterpret_cast<const float4*>(fmap + (size_t)n * P * C);
  const float4* g4 = reinterpret_cast<const float4*>(s_g);
  const float inv = 1.0f / (float)P;
  for (int p = warp; p < P; p += 8) {
    const float4* row = f4 + (size_t)p * C4;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int k = lane;
    for (; k + 96 < C4; k += 128) {    // four independent 16-byte loads in flight per lane
      const float4 v0 = __ldcs(row + k), v1 = __ldcs(row + k + 32), v2 = __ldcs(row + k + 64), v3 = __ldcs(row + k + 96);
      const float4 q0 = g4[k], q1 = g4[k + 32], q2 = g4[k + 64], q3 = g4[k + 96];
      a0 = fmaf(v0.x, q0.x, fmaf(v0.y, q0.y, fmaf(v0.z, q0.z, fmaf(v0.w, q0.w, a0))));
      a1 = fmaf(v1.x, q1.x, fmaf(v1.y, q1.y, fmaf(v1.z, q1.z, fmaf(v1.w, q1.w, a1))));
      a2 = fmaf(v2.x, q2.x, fmaf(v2.y, q2.y, fmaf(v2.z, q2.z, fmaf(v2.w, q2.w, a2))));
      a3 = fmaf(v3.x, q3.x, fmaf(v3.y, q3.y, fmaf(v3.z, q3.z, fmaf(v3.w, q3.w, a3))));
    }
    for (; k < C4; k += 32) {
      const float4 v = __ldcs(row + k), q = g4[k];
      a0 = fmaf(v.x, q.x, fmaf(v.y, q.y, fmaf(v.z, q.z, fmaf(v.w, q.w, a0))));
    }
    const float s = ex_warp_sum((a0 + a1) + (a2 + a3));
    if (lane == 0) {
      const float v = fmaxf(s * inv, 0.f);
      s_cam[p] = v;
      if (cam_small) cam_small[(size_t)n * P + p] = v;
    }
  }
  __syncthreads();
  const float sh = __fdiv_rn((float)hw, (float)out_h), sw = __fdiv_rn((float)hw, (float)out_w);
  float* o = cam + (size_t)n * out_h * out_w;
  for (int idx = tid; idx < out_h * out_w; idx += 256) {
    const int oy = idx / out_w, ox = idx - oy * out_w;
    int y0, y1, x0, x1;
    float wy0, wy1, wx0, wx1;
    src_taps(oy, sh, hw, y0, y1, wy0, wy1);
    src_taps(ox, sw, hw, x0, x1, wx0, wx1);
    const float top = __fadd_rn(__fmul_rn(wx0, s_cam[y0 * hw + x0]), __fmul_rn(wx1, s_cam[y0 * hw + x1]));
    const float bot = __fadd_rn(__fmul_rn(wx0, s_cam[y1 * hw + x0]), __fmul_rn(wx1, s_cam[y1 * hw + x1]));
    __stcs(o + idx, __fadd_rn(__fmul_rn(wy0, top), __fmul_rn(wy1, bot)));
  }
}

static size_t align64(size_t n) { return (n + 63) & ~(size_t)63; }

}  // namespace pdf

using namespace pdf;

extern "C" size_t pdf_mil_explain_workspace_bytes(const pdf_mil_weights* w, int n_bags, int Lmax) {
  if (!w || n_bags <= 0 || Lmax <= 0 || w->H <= 0 || w->A <= 0) return 0;
  const size_t rows = (size_t)n_bags * Lmax;
  const size_t na = (size_t)(w->gated ? 2 * w->A : w->A);
  // h [rows, H] | vu [rows, NA] | dh [rows, H] | dvu [rows, NA], each region 256-byte aligned
  return (2 * align64(rows * w->H) + 2 * align64(rows * na)) * sizeof(float) + 512;
}

extern "C" int pdf_mil_explain(const pdf_mil_weights* w, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len, void* d_workspace,
                               float* d_logit, float* d_attn, float* d_contrib, float* d_dx, pdf_stream_t stream) {
  PDF_REQUIRE(w && n_bags > 0 && Lmax > 0 && d_bags && d_len && d_workspace && d_logit && d_attn && d_contrib, "pdf_mil_explain: bad arguments");
  PDF_REQUIRE((long long)n_bags * Lmax <= INT_MAX, "pdf_mil_explain: n_bags * Lmax must fit in an int");
  PDF_REQUIRE(w->D > 0 && w->H > 0 && w->H <= 2048 && w->A > 0, "pdf_mil_explain: bad dims");
  PDF_REQUIRE(w->w_inst && w->b_inst && w->w_v && w->b_v && w->w_w && w->b_w && w->w_cls && w->b_cls && (!w->gated || (w->w_u && w->b_u)),
              "pdf_mil_explain: null weight pointer");
  const size_t smem = (size_t)2 * Lmax * sizeof(float);
  PDF_REQUIRE(smem <= 200 * 1024, "pdf_mil_explain: bag too large for shared memory");
  cudaStream_t s = as_stream(stream);
  const int rows = n_bags * Lmax;
  const int H = w->H, A = w->A, D = w->D, NA = w->gated ? 2 * A : A;
  float* hbuf = reinterpret_cast<float*>(d_workspace);
  float* vu = hbuf + align64((size_t)rows * H);
  float* dh = vu + align64((size_t)rows * NA);
  float* dvu = dh + align64((size_t)rows * H);
  // the FP32 sweep path's GEMMs (pdf_mil_sweep with PDF_PREC_F32): the same h and attention pre-activations
  if (int rc = gemm_nt(d_bags, D, w->w_inst, D, hbuf, H, w->b_inst, rows, H, D, 1, s)) return rc;
  if (int rc = gemm_nt(hbuf, H, w->w_v, H, vu, NA, nullptr, rows, A, H, 0, s)) return rc;
  if (w->gated)
    if (int rc = gemm_nt(hbuf, H, w->w_u, H, vu + A, NA, nullptr, rows, A, H, 0, s)) return rc;
  if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(mil_explain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mil_explain_kernel<<<n_bags, 256, smem, s>>>(hbuf, vu, d_len, Lmax, *w, d_logit, d_attn, d_contrib, d_dx ? dh : nullptr,
                                               d_dx ? dvu : nullptr);
  PDF_CHECK_LAUNCH();
  if (!d_dx) return PDF_OK;
  // dh += dvu W_vu (attention layers), ReLU backward on h, dX = dh W_i
  if (int rc = pdf_gemm_f32(rows, H, A, dvu, NA, 1, w->w_v, H, 1, dh, H, nullptr, 0, 1, stream)) return rc;
  if (w->gated)
    if (int rc = pdf_gemm_f32(rows, H, A, dvu + A, NA, 1, w->w_u, H, 1, dh, H, nullptr, 0, 1, stream)) return rc;
  if (int rc = pdf_relu_mask_backward(dh, hbuf, nullptr, (size_t)rows * H, stream)) return rc;
  return pdf_gemm_f32(rows, D, H, dh, H, 1, w->w_inst, D, 1, d_dx, D, nullptr, 0, 0, stream);
}

extern "C" int pdf_gradcam(int n, int hw, int c, const float* d_fmap, const float* d_g, int out_h, int out_w, float* d_cam_small,
                           float* d_cam, pdf_stream_t stream) {
  PDF_REQUIRE(n > 0 && hw > 0 && c > 0 && out_h > 0 && out_w > 0 && d_fmap && d_g && d_cam, "pdf_gradcam: bad arguments");
  PDF_REQUIRE(c % 4 == 0 && (reinterpret_cast<uintptr_t>(d_fmap) & 15) == 0, "pdf_gradcam: c %% 4 == 0 and a 16-byte aligned feature map needed");
  PDF_REQUIRE(hw <= 64 && out_h <= 16384 && out_w <= 16384 && (long long)out_h * out_w <= INT_MAX, "pdf_gradcam: sizes out of range");
  const size_t smem = ((size_t)c + (size_t)hw * hw) * sizeof(float);
  PDF_REQUIRE(smem <= 200 * 1024, "pdf_gradcam: c too large for shared memory");
  cudaStream_t s = as_stream(stream);
  if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(gradcam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gradcam_kernel<<<n, 256, smem, s>>>(d_fmap, d_g, hw, c, out_h, out_w, d_cam_small, d_cam);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

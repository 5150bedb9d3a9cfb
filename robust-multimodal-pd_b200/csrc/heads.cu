// K3 / K4: MIL attention head and the batched missingness sweeps (Fusion-ModDrop, MoE), FP32.
// These are tiny, HBM/launch-bound kernels; the point is ONE launch over all bags / all (scenario, subject)
// pairs instead of the reference's per-bag and per-scenario Python loops
// (models/mil_attention.py:169-177, evaluation/evaluate.py:18-97).
#include "common.cuh"
#include "ops.cuh"

namespace pdf {

// ------------------------------------------------------------------------------------------------------
// C[M,N] = A[M,K] * B[N,K]^T (+bias[N]) (ReLU) ; row strides lda/ldb/ldc; FP32 FFMA, 64x64x16 tiles.
__global__ void __launch_bounds__(256)
gemm_nt_f32_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
                   const float* __restrict__ bias, int M, int N, int K, int relu) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
  const int lr = tid >> 2, lk = (tid & 3) * 4;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = k0 + lk + e;
      As[lk + e][lr] = (m0 + lr < M && k < K) ? __ldg(A + (size_t)(m0 + lr) * lda + k) : 0.f;
      Bs[lk + e][lr] = (n0 + lr < N && k < K) ? __ldg(B + (size_t)(n0 + lr) * ldb + k) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
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
      if (relu) v = fmaxf(v, 0.f);
      C[(size_t)m * ldc + n] = v;
    }
  }
}

int gemm_nt(const float* A, int lda, const float* B, int ldb, float* C, int ldc, const float* bias, int M, int N, int K,
                   int relu, cudaStream_t s) {
  dim3 grid(ceil_div(M, 64), ceil_div(N, 64));
  gemm_nt_f32_kernel<<<grid, 256, 0, s>>>(A, lda, B, ldb, C, ldc, bias, M, N, K, relu);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// ------------------------------------------------------------------------------------------------------
// MIL pooling: one block per bag.  h = ReLU(instance(x)) [n_bags*Lmax, H] is in `hbuf`; the attention scores come either
// ready-made (`scores`, tensor path: computed by the attention GEMM's epilogue) or as the pre-activations of the attention
// layer(s) `vu` [n_bags*Lmax, NA] (FP32 path; NA = 2A gated: v | u, else A).  Masked softmax over the bag, weighted pool,
// classifier, and the result is written for EVERY scenario: prob[s, bag] = live[s, bag] ? p : missing_prob -- the bag's
// probability does not depend on the scenario, only its presence does (evaluation/evaluate.py:32-37).
__global__ void __launch_bounds__(256)
mil_pool_kernel(const float* __restrict__ hbuf, const float* __restrict__ vu, const float* __restrict__ scores,
                const int32_t* __restrict__ lens, int Lmax, pdf_mil_weights w, int n_bags, int S, const uint8_t* __restrict__ live,
                float* __restrict__ prob) {
  extern __shared__ float sm[];
  float* s_score = sm;                 // [Lmax]
  __shared__ float s_red[8];
  const int bag = blockIdx.x;
  const int len = min(lens[bag], Lmax);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = w.H, A = w.A;
  bool any_live = len > 0;
  if (any_live && live) {
    any_live = false;
    for (int s = 0; s < S; ++s) any_live |= live[(size_t)s * n_bags + bag] != 0;
  }
  if (!any_live) {
    for (int s = tid; s < S; s += 256) prob[(size_t)s * n_bags + bag] = w.missing_prob;
    return;
  }
  const float* hb = hbuf + (size_t)bag * Lmax * H;
  if (scores) {
    for (int l = tid; l < len; l += 256) s_score[l] = scores[(size_t)bag * Lmax + l];
  } else {
    const int NA = w.gated ? 2 * A : A;
    for (int l = warp; l < len; l += 8) {
      const float* r = vu + ((size_t)bag * Lmax + l) * NA;
      float sc = 0.f;
      for (int a = lane; a < A; a += 32) {
        float t = tanhf(r[a] + __ldg(w.b_v + a));
        if (w.gated) t *= sigmoidf_(r[A + a] + __ldg(w.b_u + a));
        sc = fmaf(__ldg(w.w_w + a), t, sc);
      }
      sc = warp_sum(sc);
      if (lane == 0) s_score[l] = sc + __ldg(w.b_w);
    }
  }
  __syncthreads();
  // softmax over the valid instances (masked_fill(-1e9) on padding == exclusion)
  float mx = -INFINITY;
  for (int l = tid; l < len; l += 256) mx = fmaxf(mx, s_score[l]);
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = s_red[0];
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, s_red[i]);
  __syncthreads();
  float se = 0.f;
  for (int l = tid; l < len; l += 256) { const float e = expf(s_score[l] - mx); s_score[l] = e; se += e; }
  se = warp_sum(se);
  if (lane == 0) s_red[warp] = se;
  __syncthreads();
  se = 0.f;
  for (int i = 0; i < 8; ++i) se += s_red[i];
  for (int l = tid; l < len; l += 256) s_score[l] = s_score[l] / se;      // attention weights a_l (each element owned by one thread)
  __syncthreads();
  // pooled = sum_l a_l h_l ; z = w_cls . pooled + b.  Four independent accumulators: the bag's rows stream with four loads in
  // flight per thread instead of one dependent FMA chain per load (the kernel was latency-bound at 1.3 TB/s)
  float z = 0.f;
  for (int i = tid; i < H; i += 256) {
    float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
    int l = 0;
    for (; l + 4 <= len; l += 4) {
      p0 = fmaf(s_score[l], hb[(size_t)l * H + i], p0);
      p1 = fmaf(s_score[l + 1], hb[(size_t)(l + 1) * H + i], p1);
      p2 = fmaf(s_score[l + 2], hb[(size_t)(l + 2) * H + i], p2);
      p3 = fmaf(s_score[l + 3], hb[(size_t)(l + 3) * H + i], p3);
    }
    for (; l < len; ++l) p0 = fmaf(s_score[l], hb[(size_t)l * H + i], p0);
    z = fmaf(__ldg(w.w_cls + i), (p0 + p1) + (p2 + p3), z);
  }
  z = warp_sum(z);
  if (lane == 0) s_red[warp] = z;
  __syncthreads();
  float t = 0.f;
  for (int i = 0; i < 8; ++i) t += s_red[i];
  const float pr = sigmoidf_(t + __ldg(w.b_cls));
  for (int s = tid; s < S; s += 256) prob[(size_t)s * n_bags + bag] = (!live || live[(size_t)s * n_bags + bag]) ? pr : w.missing_prob;
}

// ------------------------------------------------------------------------------------------------------
// one dense layer evaluated by a warp: out[o] = act(sum_i W[o,i] in[i] + b[o]); in/out in shared memory
__device__ __forceinline__ void warp_dense(const float* __restrict__ W, const float* __restrict__ b, int n_in, int n_out,
                                           const float* in, float* out, int relu, int lane) {
  int o = 0;
  for (; o + 4 <= n_out; o += 4) {          // four independent dot products in flight (same summation order per output)
    const float* wr = W + (size_t)o * n_in;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int i = lane; i < n_in; i += 32) {
      const float x = in[i];
      a0 = fmaf(__ldg(wr + i), x, a0);
      a1 = fmaf(__ldg(wr + n_in + i), x, a1);
      a2 = fmaf(__ldg(wr + 2 * n_in + i), x, a2);
      a3 = fmaf(__ldg(wr + 3 * n_in + i), x, a3);
    }
#pragma unroll
    for (int s = 16; s; s >>= 1) {
      a0 += __shfl_xor_sync(0xffffffffu, a0, s);
      a1 += __shfl_xor_sync(0xffffffffu, a1, s);
      a2 += __shfl_xor_sync(0xffffffffu, a2, s);
      a3 += __shfl_xor_sync(0xffffffffu, a3, s);
    }
    if (lane < 4) {
      const float v = (lane == 0 ? a0 : lane == 1 ? a1 : lane == 2 ? a2 : a3) + __ldg(b + o + lane);
      out[o + lane] = relu ? fmaxf(v, 0.f) : v;
    }
  }
  for (; o < n_out; ++o) {
    const float* wr = W + (size_t)o * n_in;
    float acc = 0.f;
    for (int i = lane; i < n_in; i += 32) acc = fmaf(__ldg(wr + i), in[i], acc);
    acc = warp_sum(acc);
    if (lane == 0) { const float v = acc + __ldg(b + o); out[o] = relu ? fmaxf(v, 0.f) : v; }
  }
  __syncwarp();
}

constexpr int kMaxWidth = 1024;

// partials: [n_mods][N][h1] (layer-1 pre-activations per modality, no bias)
// kCoalitions: "scenario" s is the coalition bit set (mask_m = (s >> m) & 1, S = 2^M) and `masks` is not read; kLogit: the output is
// the last layer's value (the logit) instead of its sigmoid.  The explanations (fusion_explain.cu) evaluate every coalition this way.
template <bool kCoalitions, bool kLogit>
__global__ void __launch_bounds__(256)
moddrop_sweep_kernel(pdf_mlp net, const float* __restrict__ partials, const uint8_t* __restrict__ masks, int N, int S,
                     float* __restrict__ prob) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h1 = net.dims[1];
  int maxw = h1;
  for (int l = 2; l <= net.n_layers; ++l) maxw = max(maxw, net.dims[l]);
  float* bufA = sm + (size_t)warp * 2 * maxw;
  float* bufB = bufA + maxw;
  const int M = net.n_mods;
  // one warp per (scenario, subject) pair: a 32-subject batch under 7 scenarios still fills 28 blocks
  for (long long pair = (long long)blockIdx.x * 8 + warp; pair < (long long)N * S; pair += (long long)gridDim.x * 8) {
    {
      const int s = (int)(pair / N), n = (int)(pair - (long long)s * N);
      const uint8_t* mk = kCoalitions ? nullptr : masks + ((size_t)s * N + n) * M;
      const bool last0 = net.n_layers == 1;
      for (int i = lane; i < h1; i += 32) {
        float v = 0.f;
        for (int m = 0; m < M; ++m)
          if ((kCoalitions ? ((s >> m) & 1) != 0 : mk[m]) && net.mod_off[m + 1] > net.mod_off[m]) v += partials[((size_t)m * N + n) * h1 + i];
        v += __ldg(net.b[0] + i);
        bufA[i] = last0 ? v : fmaxf(v, 0.f);
      }
      __syncwarp();
      float* in = bufA;
      float* out = bufB;
      for (int l = 1; l < net.n_layers; ++l) {
        warp_dense(net.w[l], net.b[l], net.dims[l], net.dims[l + 1], in, out, l < net.n_layers - 1, lane);
        float* t = in; in = out; out = t;
      }
      if (lane == 0) prob[(size_t)s * N + n] = kLogit ? in[0] : sigmoidf_(in[0]);
      __syncwarp();
    }
  }
}

// Large S*N: a block takes a tile of TP (scenario, subject) pairs and runs layers 2.. as shared-memory-tiled FFMA GEMMs, so every
// weight element is fetched once per TILE instead of once per pair (the warp-per-pair kernel above re-reads 164 KB of weights per pair
// at the C2 widths: 1.1 TB of L2 traffic at N = 1e6, S = 7).  Same arithmetic, summation over k in ascending order per output.
template <int TP, bool kCoalitions, bool kLogit>
__global__ void __launch_bounds__(256)
moddrop_tile_kernel(pdf_mlp net, const float* __restrict__ partials, const uint8_t* __restrict__ masks, int N, int S, int maxw,
                    float* __restrict__ prob) {
  extern __shared__ float sm[];
  const int stride = maxw + 1;
  float* bufA = sm;                                  // [TP][stride]
  float* bufB = bufA + TP * stride;
  float* Ws = bufB + TP * stride;                    // [16][64 + 4]
  const int tid = threadIdx.x;
  const int M = net.n_mods, h1 = net.dims[1];
  const long long total = (long long)N * S;
  constexpr int RT = TP / 16;                        // rows per thread (thread grid 16 x 16)
  const int ty = tid >> 4, tx = tid & 15;
  for (long long p0 = (long long)blockIdx.x * TP; p0 < total; p0 += (long long)gridDim.x * TP) {
    // layer 1 from the per-modality partials
    for (int idx = tid; idx < TP * h1; idx += 256) {
      const int r = idx / h1, i = idx - r * h1;
      const long long pair = p0 + r;
      float v = 0.f;
      if (pair < total) {
        const int s = (int)(pair / N), n = (int)(pair - (long long)s * N);
        const uint8_t* mk = kCoalitions ? nullptr : masks + ((size_t)s * N + n) * M;
        for (int m = 0; m < M; ++m)
          if ((kCoalitions ? ((s >> m) & 1) != 0 : mk[m]) && net.mod_off[m + 1] > net.mod_off[m]) v += partials[((size_t)m * N + n) * h1 + i];
        v += __ldg(net.b[0] + i);
        if (net.n_layers > 1) v = fmaxf(v, 0.f);
      }
      bufA[r * stride + i] = v;
    }
    __syncthreads();
    float* in = bufA;
    float* out = bufB;
    for (int l = 1; l < net.n_layers; ++l) {
      const int n_in = net.dims[l], n_out = net.dims[l + 1];
      const float* W = net.w[l];
      const int relu = l < net.n_layers - 1;
      for (int c0 = 0; c0 < n_out; c0 += 64) {
        float acc[RT][4];
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        for (int k0 = 0; k0 < n_in; k0 += 16) {
          {   // W chunk: 64 output columns x 16 k  (thread -> column tid>>2, 4 consecutive k)
            const int col = c0 + (tid >> 2), kk = (tid & 3) * 4;
#pragma unroll
            for (int e = 0; e < 4; ++e)
              Ws[(kk + e) * 68 + (tid >> 2)] = (col < n_out && k0 + kk + e < n_in) ? __ldg(W + (size_t)col * n_in + k0 + kk + e) : 0.f;
          }
          __syncthreads();
          const int kmax = min(16, n_in - k0);
          for (int kk = 0; kk < kmax; ++kk) {
            float a[RT], b[4];
#pragma unroll
            for (int i = 0; i < RT; ++i) a[i] = in[(ty * RT + i) * stride + k0 + kk];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Ws[kk * 68 + tx * 4 + j];
#pragma unroll
            for (int i = 0; i < RT; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
          }
          __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int col = c0 + tx * 4 + j;
            if (col < n_out) {
              const float v = acc[i][j] + __ldg(net.b[l] + col);
              out[(ty * RT + i) * stride + col] = relu ? fmaxf(v, 0.f) : v;
            }
          }
      }
      __syncthreads();
      float* t = in; in = out; out = t;
    }
    for (int r = tid; r < TP; r += 256)
      if (p0 + r < total) prob[p0 + r] = kLogit ? in[r * stride] : sigmoidf_(in[r * stride]);       // prob is [S, N] = pair order
    __syncthreads();
  }
}

struct MoeArgs {
  pdf_moe net;
  const float* x[PDF_MAX_MODS];
};

// kCoalitions: as moddrop_sweep_kernel (S = 2^E, `masks` not read); the warps of subject 0 also write the router weights of every
// coalition to router_w [2^E, E].  The output is the gated sum itself either way: MoE has no single logit.
template <bool kCoalitions>
__global__ void __launch_bounds__(256)
moe_sweep_kernel(MoeArgs a, const uint8_t* __restrict__ masks, int N, int S, int maxw, float* __restrict__ prob,
                 float* __restrict__ router_w) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* bufA = sm + (size_t)warp * 2 * maxw;
  float* bufB = bufA + maxw;
  const int E = a.net.n_experts, R = a.net.router_hidden;
  // every warp first evaluates the experts on the all-zero input (a few thousand MACs, once per warp instead of once per subject)
  float e_zero[PDF_MAX_MODS];
  for (int e = 0; e < E; ++e) {
    const pdf_mlp& ex = a.net.expert[e];
    for (int i = lane; i < ex.dims[0]; i += 32) bufA[i] = 0.f;
    __syncwarp();
    float* in = bufA;
    float* out = bufB;
    for (int l = 0; l < ex.n_layers; ++l) {
      warp_dense(ex.w[l], ex.b[l], ex.dims[l], ex.dims[l + 1], in, out, l < ex.n_layers - 1, lane);
      float* t = in; in = out; out = t;
    }
    e_zero[e] = sigmoidf_(in[0]);
    __syncwarp();
  }
  for (int n = blockIdx.x * 8 + warp; n < N; n += gridDim.x * 8) {
    float e_x[PDF_MAX_MODS], e_0[PDF_MAX_MODS];
    for (int e = 0; e < E; ++e) {
      const pdf_mlp& ex = a.net.expert[e];
      e_0[e] = e_zero[e];                      // expert(0): the masked (all-zero) input gives the same output for every subject
      for (int i = lane; i < ex.dims[0]; i += 32) bufA[i] = a.x[e][(size_t)n * ex.dims[0] + i];
      __syncwarp();
      float* in = bufA;
      float* out = bufB;
      for (int l = 0; l < ex.n_layers; ++l) {
        warp_dense(ex.w[l], ex.b[l], ex.dims[l], ex.dims[l + 1], in, out, l < ex.n_layers - 1, lane);
        float* t = in; in = out; out = t;
      }
      e_x[e] = sigmoidf_(in[0]);
      __syncwarp();
    }
    for (int s = 0; s < S; ++s) {
      const uint8_t* mk = kCoalitions ? nullptr : masks + ((size_t)s * N + n) * E;
      // router: softmax(W1 relu(W0 mask + b0) + b1)
      for (int h = lane; h < R; h += 32) {
        float v = __ldg(a.net.b_r0 + h);
        for (int m = 0; m < E; ++m) v = fmaf(__ldg(a.net.w_r0 + h * E + m), (kCoalitions ? ((s >> m) & 1) != 0 : mk[m]) ? 1.f : 0.f, v);
        bufA[h] = fmaxf(v, 0.f);
      }
      __syncwarp();
      float logit[PDF_MAX_MODS];
      float mx = -INFINITY;
      for (int m = 0; m < E; ++m) {
        float v = 0.f;
        for (int h = lane; h < R; h += 32) v = fmaf(__ldg(a.net.w_r1 + m * R + h), bufA[h], v);
        v = warp_sum(v) + __ldg(a.net.b_r1 + m);
        logit[m] = v;
        mx = fmaxf(mx, v);
      }
      float se = 0.f;
      for (int m = 0; m < E; ++m) { logit[m] = expf(logit[m] - mx); se += logit[m]; }
      float o = 0.f;
      for (int m = 0; m < E; ++m) o += ((kCoalitions ? ((s >> m) & 1) != 0 : mk[m]) ? e_x[m] : e_0[m]) * (logit[m] / se);
      if (lane == 0) prob[(size_t)s * N + n] = o;
      if (kCoalitions && n == 0 && lane == 0)
        for (int m = 0; m < E; ++m) router_w[(size_t)s * E + m] = logit[m] / se;
      __syncwarp();
    }
  }
}

static bool g_moddrop_tiled = true;   // pdf_debug_set_moddrop_tiled

int check_mlp(const pdf_mlp& m, const char* what) {
  PDF_REQUIRE(m.n_layers >= 1 && m.n_layers <= PDF_MAX_LAYERS, "%s: n_layers out of range", what);
  PDF_REQUIRE(m.dims[m.n_layers] == 1, "%s: last layer must have one output", what);
  for (int l = 0; l < m.n_layers; ++l) {
    PDF_REQUIRE(m.w[l] && m.b[l] && m.dims[l] >= 0, "%s: null weights in layer %d", what, l);
    if (l > 0) PDF_REQUIRE(m.dims[l] >= 1 && m.dims[l] <= kMaxWidth, "%s: hidden width must be 1..%d", what, kMaxWidth);
  }
  return PDF_OK;
}

int check_moddrop(const pdf_mlp& net, const char* what) {
  if (int rc = check_mlp(net, what)) return rc;
  PDF_REQUIRE(net.n_mods >= 1 && net.n_mods <= PDF_MAX_MODS && net.mod_off[0] == 0 && net.mod_off[net.n_mods] == net.dims[0],
              "%s: modality offsets must tile [0, F)", what);
  PDF_REQUIRE(net.dims[1] <= kMaxWidth, "%s: first hidden width must be <= %d", what, kMaxWidth);
  return PDF_OK;
}

int check_moe(const pdf_moe& net, const float* const* d_x, const char* what) {
  PDF_REQUIRE(net.n_experts >= 1 && net.n_experts <= PDF_MAX_MODS && net.router_hidden >= 1 && net.router_hidden <= kMaxWidth &&
              net.w_r0 && net.b_r0 && net.w_r1 && net.b_r1, "%s: bad router", what);
  int maxw = net.router_hidden;
  for (int e = 0; e < net.n_experts; ++e) {
    if (int rc = check_mlp(net.expert[e], what)) return rc;
    PDF_REQUIRE(d_x[e] && net.expert[e].dims[0] >= 1 && net.expert[e].dims[0] <= 8192, "%s: expert input width 1..8192", what);
    for (int l = 0; l <= net.expert[e].n_layers; ++l) maxw = max(maxw, net.expert[e].dims[l]);
  }
  PDF_REQUIRE((size_t)8 * 2 * maxw * sizeof(float) <= 200 * 1024, "%s: layers too wide for shared memory", what);
  return PDF_OK;
}

int moddrop_partials(const pdf_mlp& net, int N, const float* d_x, float* partials, cudaStream_t s) {
  const int F = net.dims[0], h1 = net.dims[1];
  // linearity of layer 1: (x (.) mask) W1^T = sum_m mask_m * (x_m W1_m^T)  -> per-modality partials once, reused by every scenario
  for (int m = 0; m < net.n_mods; ++m) {
    const int d = net.mod_off[m + 1] - net.mod_off[m];
    if (d <= 0) continue;
    if (int rc = gemm_nt(d_x + net.mod_off[m], F, net.w[0] + net.mod_off[m], F, partials + (size_t)m * N * h1, h1, nullptr, N, h1, d, 0, s))
      return rc;
  }
  return PDF_OK;
}

template <bool kCoalitions, bool kLogit>
static int moddrop_launch(const pdf_mlp& net, int N, int S, const float* partials, const uint8_t* masks, long long sweep_pairs,
                          float* out, cudaStream_t s) {
  const int h1 = net.dims[1];
  int maxw = h1;
  for (int l = 2; l <= net.n_layers; ++l) maxw = max(maxw, net.dims[l]);
  const size_t smem = (size_t)8 * 2 * maxw * sizeof(float);
  if (smem > 48 * 1024)
    PDF_CHECK_CUDA(cudaFuncSetAttribute(moddrop_sweep_kernel<kCoalitions, kLogit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long pairs = (long long)N * S;
  if (g_moddrop_tiled && sweep_pairs >= 4096 && net.n_layers >= 2) {
    // batched path: tiles of 64 (32 for wide networks) pairs, layers 2.. as in-block GEMMs
    const int TP = maxw <= 384 ? 64 : 32;
    const size_t tsmem = ((size_t)2 * TP * (maxw + 1) + 16 * 68) * sizeof(float);
    if (tsmem <= 200 * 1024) {
      const int tblocks = (int)max(1LL, min((pairs + TP - 1) / TP, (long long)num_sms() * (tsmem > 100 * 1024 ? 1 : 2)));
      if (TP == 64) {
        PDF_CHECK_CUDA(cudaFuncSetAttribute(moddrop_tile_kernel<64, kCoalitions, kLogit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
        moddrop_tile_kernel<64, kCoalitions, kLogit><<<tblocks, 256, tsmem, s>>>(net, partials, masks, N, S, maxw, out);
      } else {
        PDF_CHECK_CUDA(cudaFuncSetAttribute(moddrop_tile_kernel<32, kCoalitions, kLogit>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
        moddrop_tile_kernel<32, kCoalitions, kLogit><<<tblocks, 256, tsmem, s>>>(net, partials, masks, N, S, maxw, out);
      }
      PDF_CHECK_LAUNCH();
      return PDF_OK;
    }
  }
  const int blocks = max(1, min(ceil_div(pairs, 8), num_sms() * 8));
  moddrop_sweep_kernel<kCoalitions, kLogit><<<blocks, 256, smem, s>>>(net, partials, masks, N, S, out);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

int moddrop_eval(const pdf_mlp& net, int N, int S, const float* partials, const uint8_t* masks, bool coalitions, long long sweep_pairs,
                 float* out, cudaStream_t s) {
  return coalitions ? moddrop_launch<true, true>(net, N, 1 << net.n_mods, partials, nullptr, sweep_pairs, out, s)
                    : moddrop_launch<false, false>(net, N, S, partials, masks, sweep_pairs, out, s);
}

int moe_eval(const pdf_moe& net, const float* const* d_x, int N, int S, const uint8_t* masks, float* router_w, float* out, cudaStream_t s) {
  MoeArgs a;
  a.net = net;
  int maxw = net.router_hidden;
  for (int e = 0; e < net.n_experts; ++e) {
    a.x[e] = d_x[e];
    for (int l = 0; l <= net.expert[e].n_layers; ++l) maxw = max(maxw, net.expert[e].dims[l]);
  }
  const size_t smem = (size_t)8 * 2 * maxw * sizeof(float);
  const int blocks = max(1, min(ceil_div(N, 8), num_sms() * 8));
  if (router_w) {
    if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(moe_sweep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    moe_sweep_kernel<true><<<blocks, 256, smem, s>>>(a, nullptr, N, 1 << net.n_experts, maxw, out, router_w);
  } else {
    if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(moe_sweep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    moe_sweep_kernel<false><<<blocks, 256, smem, s>>>(a, masks, N, S, maxw, out, nullptr);
  }
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

}  // namespace pdf

using namespace pdf;

extern "C" size_t pdf_mil_workspace_bytes(const pdf_mil_weights* w, int n_bags, int Lmax) {
  if (!w || n_bags <= 0 || Lmax <= 0) return 0;
  const size_t rows = (size_t)n_bags * Lmax;
  const size_t na = (size_t)(w->gated ? 2 * w->A : w->A);
  // h [rows, H] | attention pre-activations [rows, NA] (FP32 path) or scores [rows] (tensor path)
  return rows * w->H * sizeof(float) + rows * na * sizeof(float) + 512;
}

extern "C" int pdf_mil_sweep(const pdf_mil_weights* w, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len,
                             int n_scenarios, const uint8_t* d_live, int precision, void* d_workspace, float* d_prob,
                             pdf_stream_t stream) {
  PDF_REQUIRE(w && n_bags > 0 && Lmax > 0 && d_bags && d_len && d_workspace && d_prob && n_scenarios > 0, "pdf_mil_sweep: bad arguments");
  PDF_REQUIRE(w->D > 0 && w->H > 0 && w->H <= 2048 && w->A > 0, "pdf_mil_sweep: bad dims");
  PDF_REQUIRE(w->w_inst && w->b_inst && w->w_v && w->b_v && w->w_w && w->b_w && w->w_cls && w->b_cls && (!w->gated || (w->w_u && w->b_u)),
              "pdf_mil_sweep: null weight pointer");
  PDF_REQUIRE(precision == PDF_PREC_F32 || precision == PDF_PREC_TF32, "pdf_mil_sweep: precision must be PDF_PREC_F32 or PDF_PREC_TF32");
  cudaStream_t s = as_stream(stream);
  const int rows = n_bags * Lmax;
  const int NA = w->gated ? 2 * w->A : w->A;
  float* hbuf = reinterpret_cast<float*>(d_workspace);
  float* abuf = hbuf + (((size_t)rows * w->H + 63) & ~(size_t)63);
  const float* scores = nullptr;
  const float* vu = nullptr;
  if (precision == PDF_PREC_TF32) {
    // both linear layers on the tensor cores (kind::tf32 on the f32 operands); the attention GEMM reads [W_v; W_u] as ONE [2A, H]
    // matrix, so for the gated head w_u must directly follow w_v in memory (pd_fusion_b200/heads.py packs them)
    PDF_REQUIRE(gemm_tf32_supported(w->H, w->D) && gemm_tf32_supported(NA, w->H),
                "pdf_mil_sweep: the tensor path needs H and (2)A in {64,128,256}, D and H multiples of 32 (D=%d H=%d A=%d)", w->D, w->H, w->A);
    PDF_REQUIRE(!w->gated || (w->w_u == w->w_v + (size_t)w->A * w->H && w->b_u == w->b_v + w->A),
                "pdf_mil_sweep: the tensor path needs [w_v; w_u] and [b_v; b_u] contiguous");
    if (int rc = launch_gemm_tf32(d_bags, w->w_inst, rows, w->H, w->D, 0, 0, 0, w->b_inst, nullptr, nullptr, hbuf, s)) return rc;
    if (int rc = launch_gemm_tf32(hbuf, w->w_v, rows, NA, w->H, 1, w->gated, w->A, w->b_v, w->w_w, w->b_w, abuf, s)) return rc;
    scores = abuf;
  } else {
    // instance projection for every (padded) instance of every bag at once: M = n_bags * Lmax, then the attention layer(s)
    if (int rc = gemm_nt(d_bags, w->D, w->w_inst, w->D, hbuf, w->H, w->b_inst, rows, w->H, w->D, 1, s)) return rc;
    if (int rc = gemm_nt(hbuf, w->H, w->w_v, w->H, abuf, NA, nullptr, rows, w->A, w->H, 0, s)) return rc;
    if (w->gated)
      if (int rc = gemm_nt(hbuf, w->H, w->w_u, w->H, abuf + w->A, NA, nullptr, rows, w->A, w->H, 0, s)) return rc;
    vu = abuf;
  }
  const size_t smem = (size_t)Lmax * sizeof(float);
  PDF_REQUIRE(smem <= 200 * 1024, "pdf_mil_sweep: bag too large for shared memory");
  if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(mil_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mil_pool_kernel<<<n_bags, 256, smem, s>>>(hbuf, vu, scores, d_len, Lmax, *w, n_bags, n_scenarios, d_live, d_prob);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_mil_forward(const pdf_mil_weights* w, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len,
                               void* d_workspace, float* d_prob, pdf_stream_t stream) {
  return pdf_mil_sweep(w, n_bags, Lmax, d_bags, d_len, 1, nullptr, PDF_PREC_F32, d_workspace, d_prob, stream);
}

extern "C" size_t pdf_moddrop_workspace_bytes(const pdf_mlp* net, int n_subjects) {
  if (!net || n_subjects <= 0) return 0;
  return (size_t)net->n_mods * n_subjects * net->dims[1] * sizeof(float) + 256;
}

extern "C" int pdf_moddrop_sweep(const pdf_mlp* net, int n_subjects, int n_scenarios, const float* d_x, const uint8_t* d_masks,
                                 void* d_workspace, float* d_prob, pdf_stream_t stream) {
  PDF_REQUIRE(net && n_subjects > 0 && n_scenarios > 0 && d_x && d_masks && d_workspace && d_prob, "pdf_moddrop_sweep: bad arguments");
  if (int rc = check_moddrop(*net, "pdf_moddrop_sweep")) return rc;
  cudaStream_t s = as_stream(stream);
  float* partials = reinterpret_cast<float*>(d_workspace);
  if (int rc = moddrop_partials(*net, n_subjects, d_x, partials, s)) return rc;
  return moddrop_eval(*net, n_subjects, n_scenarios, partials, d_masks, false, (long long)n_subjects * n_scenarios, d_prob, s);
}

extern "C" int pdf_moe_sweep(const pdf_moe* net, int n_subjects, int n_scenarios, const float* const* d_x, const uint8_t* d_masks,
                             float* d_prob, pdf_stream_t stream) {
  PDF_REQUIRE(net && n_subjects > 0 && n_scenarios > 0 && d_x && d_masks && d_prob, "pdf_moe_sweep: bad arguments");
  if (int rc = check_moe(*net, d_x, "pdf_moe_sweep")) return rc;
  return moe_eval(*net, d_x, n_subjects, n_scenarios, d_masks, nullptr, d_prob, as_stream(stream));
}

/* A/B hook: 0 = the warp-per-pair ModDrop kernel for every size, 1 (default) = the tiled GEMM kernel from 4096 (scenario, subject) pairs up */
extern "C" int pdf_debug_set_moddrop_tiled(int enable) {
  pdf::g_moddrop_tiled = enable != 0;
  return PDF_OK;
}

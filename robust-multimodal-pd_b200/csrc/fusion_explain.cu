// Explanations of the fusion heads (Fusion-ModDrop, MoE): exact modality Shapley values and integrated gradients (IG).
//
// Both heads treat a missing modality as zeroed input, so the all-zero input is the baseline and the value of a coalition T of
// modalities is the head evaluated with every modality outside T set to 0.  The sweep kernels of heads.cu evaluate all 2^M coalitions
// once per subject (ModDrop: the logit; MoE: the gated probability, which has no single logit); shapley_combine_kernel then combines
// them per (scenario, subject) in float64.  M <= PDF_MAX_MODS = 8, so the Shapley values are exact, not sampled.
//
// IG from 0 along x(alpha) = alpha (x (.) m), midpoint rule alpha_k = (k + 1/2) / K.  Layer 1 is linear in its input, so
// z1(alpha) = alpha sum_m m_m P_m + b1 with the sweep's per-modality partials P_m = x_m W1_m^T: no step re-reads x or re-runs layer 1.
// mlp_ig_kernel runs layers 2.. forward and backward for a tile of (pair, k) rows and averages delta1 = d logit / d z1 over k; because
// W1^T is linear, the average gradient is ONE GEMM mean_k(delta1) W1, and ig = (x (.) m) (.) that gradient.  FP32, no atomics.
#include <algorithm>

#include "common.cuh"
#include "mlp_tile.cuh"
#include "ops.cuh"

namespace pdf {

constexpr int kMaxIgSteps = 256;

static size_t fx_align(size_t n) { return (n + 63) & ~(size_t)63; }     // floats -> 256-byte aligned workspace regions

__constant__ double c_fact[PDF_MAX_MODS + 1] = {1, 1, 2, 6, 24, 120, 720, 5040, 40320};

// ------------------------------------------------------------------------------------------------------
// One thread per (s, n, m).  v [2^M, N] = coalition values.  P = the modalities present under scenario s, minus the null players
// (zero-width modalities: no coalition value depends on them), and
//   phi_m = sum_{T subset P \ {m}} |T|! (|P| - |T| - 1)! / |P|! (v(T + m) - v(T))        (0 for m outside P)
// in float64.  Also value[s, n] = v(P) and base = v(empty), which does not depend on the subject.
__global__ void __launch_bounds__(256)
shapley_combine_kernel(const float* __restrict__ v, const uint8_t* __restrict__ masks, int N, int S, int M, unsigned null_players,
                       float* __restrict__ value, float* __restrict__ base, float* __restrict__ shap) {
  const long long total = (long long)S * N * M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pair = i / M;
    const int m = (int)(i - pair * M);
    const int n = (int)(pair % N);
    const uint8_t* mk = masks + pair * M;
    unsigned P = 0;
    for (int j = 0; j < M; ++j)
      if (mk[j]) P |= 1u << j;
    P &= ~null_players;
    if (m == 0) value[pair] = v[(size_t)P * N + n];
    if (i == 0) base[0] = v[0];
    double phi = 0.0;
    if ((P >> m) & 1u) {
      const int p = __popc(P);
      const unsigned R = P & ~(1u << m);
      for (unsigned T = R;; T = (T - 1) & R) {           // every subset of R, R first, the empty set last
        const int t = __popc(T);
        const double w = c_fact[t] * c_fact[p - t - 1] / c_fact[p];
        phi += w * ((double)v[(size_t)(T | (1u << m)) * N + n] - (double)v[(size_t)T * N + n]);
        if (T == 0) break;
      }
    }
    shap[i] = (float)phi;
  }
}

// Average gradient of the logit with respect to z1 along the IG path: dbar[pair, i] = (1/K) sum_k delta1(alpha_k)[i], k ascending.
// pair = s * N + n.  Layer 1 from the partials: masks [S, N, M] select and add the modalities' partials [M, N, h1] (the sweep's layer 1);
// masks == NULL reads partials [N, h1] as they are (an MoE expert, S = 1).  The tile holds TP rows = G pairs x Kc steps, pair-major:
// K <= TP gives G = TP / K pairs of all K steps; K > TP gives one pair in ceil(K / TP) chunks, summed into dbar in step order.
// Shared memory: the weight chunk, a per-row seed, then every hidden layer's activations [TP][width + 1] (the logit's, for a one-layer
// net), which the backward overwrites with that layer's delta.  Seed at the logit: 1 (ModDrop), or sigma'(z) (kSigmoidSeed: an MoE
// expert, whose output is sigmoid(z)).
template <int TP, bool kSigmoidSeed>
__global__ void __launch_bounds__(256)
mlp_ig_kernel(pdf_mlp net, const float* __restrict__ partials, const uint8_t* __restrict__ masks, int M, int N, int S, int K,
              float* __restrict__ dbar) {
  extern __shared__ float sm[];
  constexpr int RT = TP / 16;
  float* Ws = sm;                              // [16][68]
  float* seed = Ws + 16 * 68;                  // [TP]
  float* a1 = seed + TP;                       // layer 1, then layers 2 .. L-1 one after the other
  const int tid = threadIdx.x;
  const int L = net.n_layers, h1 = net.dims[1];
  const long long pairs = (long long)N * S;
  const int G = K <= TP ? TP / K : 1, Kc = K <= TP ? K : TP, chunks = (K + Kc - 1) / Kc;
  for (long long u = blockIdx.x; u * G < pairs; u += gridDim.x) {
    const long long pair0 = u * G;
    for (int ch = 0; ch < chunks; ++ch) {
      const int k0 = ch * Kc;
      // layer 1: z1 = alpha_k * sum_m m_m P_m + b1
      for (int idx = tid; idx < TP * h1; idx += 256) {
        const int r = idx / h1, i = idx - r * h1;
        const int g = r / Kc, k = k0 + r - g * Kc;
        const long long pair = pair0 + g;
        float z = 0.f;
        if (g < G && pair < pairs && k < K) {
          const int s = (int)(pair / N), n = (int)(pair - (long long)s * N);
          float p = 0.f;
          if (masks) {
            const uint8_t* mk = masks + pair * M;
            for (int m = 0; m < M; ++m)
              if (mk[m] && net.mod_off[m + 1] > net.mod_off[m]) p += partials[((size_t)m * N + n) * h1 + i];
          } else {
            p = partials[(size_t)n * h1 + i];
          }
          z = fmaf(((float)k + 0.5f) / (float)K, p, __ldg(net.b[0] + i));
          if (L > 1) z = fmaxf(z, 0.f);
        }
        a1[r * (h1 + 1) + i] = z;
      }
      __syncthreads();
      if (L == 1) {                            // a1 holds the logit: delta1 is the seed itself
        for (int r = tid; r < TP; r += 256) {
          const float p = 1.0f / (1.0f + expf(-a1[r * 2]));
          a1[r * 2] = kSigmoidSeed ? p * (1.f - p) : 1.f;
        }
      } else {
        // layers 2 .. L-1 forward, every activation kept
        float* in = a1;
        for (int l = 1; l < L - 1; ++l) {
          float* out = in + TP * (net.dims[l] + 1);
          const int os = net.dims[l + 1] + 1;
          const float* b = net.b[l];
          tile_layer<RT, false>(in, net.dims[l] + 1, net.w[l], net.dims[l], net.dims[l + 1], Ws,
                                [&](int r, int c, float acc) { out[r * os + c] = fmaxf(acc + __ldg(b + c), 0.f); });
          __syncthreads();
          in = out;
        }
        // the last hidden layer's delta: seed * w_L (.) [a > 0]
        const int H = net.dims[L - 1], hs = H + 1;
        const float* wL = net.w[L - 1];
        if (kSigmoidSeed) {
          for (int r = tid; r < TP; r += 256) {
            float z = 0.f;
            for (int i = 0; i < H; ++i) z = fmaf(__ldg(wL + i), in[r * hs + i], z);
            const float p = 1.0f / (1.0f + expf(-(z + __ldg(net.b[L - 1]))));
            seed[r] = p * (1.f - p);
          }
          __syncthreads();
        }
        for (int idx = tid; idx < TP * H; idx += 256) {
          const int r = idx / H, i = idx - r * H;
          float& a = in[r * hs + i];
          a = a > 0.f ? (kSigmoidSeed ? seed[r] : 1.f) * __ldg(wL + i) : 0.f;
        }
        __syncthreads();
        // backward through layers L-2 .. 1: delta_l = (delta_{l+1} W_{l+1}) (.) [a_l > 0], written over a_l
        for (int l = L - 2; l >= 1; --l) {
          float* dn = in;
          in -= TP * (net.dims[l] + 1);
          float* dl = in;
          const int ds = net.dims[l] + 1;
          tile_layer<RT, true>(dn, net.dims[l + 1] + 1, net.w[l], net.dims[l + 1], net.dims[l], Ws, [&](int r, int c, float acc) {
            float& a = dl[r * ds + c];
            a = a > 0.f ? acc : 0.f;
          });
          __syncthreads();
        }
      }
      __syncthreads();
      // sum over this chunk's steps in ascending k onto the previous chunks' sum; the last chunk divides by K
      const int kn = min(Kc, K - k0);
      for (int idx = tid; idx < G * h1; idx += 256) {
        const int g = idx / h1, i = idx - g * h1;
        const long long pair = pair0 + g;
        if (pair >= pairs) continue;
        float acc = ch == 0 ? 0.f : dbar[pair * h1 + i];
        for (int kk = 0; kk < kn; ++kk) acc += a1[(g * Kc + kk) * (h1 + 1) + i];
        dbar[pair * h1 + i] = ch == chunks - 1 ? acc / (float)K : acc;
      }
      __syncthreads();
    }
  }
}

// ModDrop: ig[pair, f] = (x (.) m_s)[n, f] * g[pair * g_rs + f], pair = s * N + n.  g is the GEMM's [S*N, F] output (g_rs = F, overwritten
// in place) or, for a one-layer net, w1 itself (g_rs = 0).  Features of an absent modality get exactly 0.
__global__ void __launch_bounds__(256)
moddrop_ig_finish_kernel(pdf_mlp net, const float* __restrict__ x, const uint8_t* __restrict__ masks, int N, int S, const float* g,
                         long long g_rs, float* ig) {
  const int F = net.dims[0], M = net.n_mods;
  const long long total = (long long)S * N * F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pair = i / F;
    const int f = (int)(i - pair * F), n = (int)(pair % N);
    int m = 0;
    while (m + 1 < M && f >= net.mod_off[m + 1]) ++m;
    const float gv = g[pair * g_rs + f];
    ig[i] = masks[pair * M + m] ? x[(size_t)n * F + f] * gv : 0.f;
  }
}

// MoE expert e of width d: ig[pair, f] = x[n, f] * w_e(c) * gbar[n, f], c = the coalition of (s, n), w_e(c) = router_w[c, e]; 0 where e
// is absent.  gbar [N, d] = mean_k(delta1) W1 of the expert, which does not depend on the scenario.
__global__ void __launch_bounds__(256)
moe_ig_finish_kernel(const float* __restrict__ x, int d, const uint8_t* __restrict__ masks, int E, int e, const float* __restrict__ router_w,
                     int N, int S, const float* __restrict__ gbar, float* __restrict__ ig) {
  const long long total = (long long)S * N * d;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pair = i / d;
    const int f = (int)(i - pair * d), n = (int)(pair % N);
    const uint8_t* mk = masks + pair * E;
    unsigned c = 0;
    for (int j = 0; j < E; ++j)
      if (mk[j]) c |= 1u << j;
    ig[i] = mk[e] ? x[(size_t)n * d + f] * (router_w[(size_t)c * E + e] * gbar[(size_t)n * d + f]) : 0.f;
  }
}

static int ew_grid(long long n) { return (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, (long long)num_sms() * 16)); }

template <int TP, bool kSigmoidSeed>
static int ig_launch_tp(const pdf_mlp& net, const float* partials, const uint8_t* masks, int M, int N, int S, int K, size_t smem,
                        float* dbar, cudaStream_t s) {
  const long long G = K <= TP ? TP / K : 1;
  const long long units = ((long long)N * S + G - 1) / G;
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (228 * 1024) / (smem + 1024)));
  const int blocks = (int)std::max<long long>(1, std::min<long long>(units, (long long)num_sms() * per_sm));
  if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(mlp_ig_kernel<TP, kSigmoidSeed>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mlp_ig_kernel<TP, kSigmoidSeed><<<blocks, 256, smem, s>>>(net, partials, masks, M, N, S, K, dbar);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

template <bool kSigmoidSeed>
static int ig_launch(const pdf_mlp& net, const float* partials, const uint8_t* masks, int M, int N, int S, int K, float* dbar, cudaStream_t s) {
  int tp = 0;
  size_t smem = 0;
  if (int rc = mlp_tile(net, &tp, &smem, "mlp_ig_kernel")) return rc;
  if (tp == 64) return ig_launch_tp<64, kSigmoidSeed>(net, partials, masks, M, N, S, K, smem, dbar, s);
  if (tp == 32) return ig_launch_tp<32, kSigmoidSeed>(net, partials, masks, M, N, S, K, smem, dbar, s);
  return ig_launch_tp<16, kSigmoidSeed>(net, partials, masks, M, N, S, K, smem, dbar, s);
}

static int check_steps(int steps, const void* d_ig, const char* what) {
  PDF_REQUIRE(steps >= 0 && steps <= kMaxIgSteps, "%s: steps must be 0..%d", what, kMaxIgSteps);
  PDF_REQUIRE(steps > 0 || !d_ig, "%s: integrated gradients (d_ig != NULL) need steps >= 1", what);
  return PDF_OK;
}

}  // namespace pdf

using namespace pdf;

extern "C" size_t pdf_moddrop_explain_workspace_bytes(const pdf_mlp* net, int n_subjects, int n_scenarios, int steps) {
  if (!net || n_subjects <= 0 || n_scenarios <= 0 || steps < 0 || net->n_mods < 1 || net->n_mods > PDF_MAX_MODS || net->n_layers < 1 ||
      net->n_layers > PDF_MAX_LAYERS || net->dims[1] <= 0)
    return 0;
  const size_t N = (size_t)n_subjects, h1 = (size_t)net->dims[1];
  // per-modality partials [M, N, h1] | coalition values [2^M, N] | with IG on a multi-layer net: mean delta1 [S*N, h1]
  size_t f = fx_align((size_t)net->n_mods * N * h1) + fx_align(((size_t)1 << net->n_mods) * N);
  if (steps > 0 && net->n_layers > 1) f += fx_align((size_t)n_scenarios * N * h1);
  return f * sizeof(float) + 256;
}

extern "C" int pdf_moddrop_explain(const pdf_mlp* net, int n_subjects, int n_scenarios, const float* d_x, const uint8_t* d_masks, int steps,
                                   void* d_workspace, float* d_value, float* d_base, float* d_shap, float* d_ig, pdf_stream_t stream) {
  const char* what = "pdf_moddrop_explain";
  PDF_REQUIRE(net && n_subjects > 0 && n_scenarios > 0 && d_x && d_masks && d_workspace && d_value && d_base && d_shap,
              "pdf_moddrop_explain: bad arguments");
  if (int rc = check_steps(steps, d_ig, what)) return rc;
  PDF_REQUIRE(net->n_mods >= 1 && net->n_mods <= PDF_MAX_MODS, "pdf_moddrop_explain: 1..%d modalities (got %d)", PDF_MAX_MODS, net->n_mods);
  if (int rc = check_moddrop(*net, what)) return rc;
  for (int m = 0; m < net->n_mods; ++m)
    PDF_REQUIRE(net->mod_off[m + 1] >= net->mod_off[m], "pdf_moddrop_explain: modality offsets must tile [0, F)");
  const int M = net->n_mods, F = net->dims[0], h1 = net->dims[1], L = net->n_layers;
  if (d_ig && L > 1) {
    int tp;
    size_t smem;
    if (int rc = mlp_tile(*net, &tp, &smem, what)) return rc;
  }
  cudaStream_t s = as_stream(stream);
  const size_t N = (size_t)n_subjects, S = (size_t)n_scenarios;
  float* partials = reinterpret_cast<float*>(d_workspace);
  float* v = partials + fx_align((size_t)M * N * h1);
  float* dbar = v + fx_align(((size_t)1 << M) * N);
  unsigned null_players = 0;
  for (int m = 0; m < M; ++m)
    if (net->mod_off[m + 1] == net->mod_off[m]) null_players |= 1u << m;
  if (int rc = moddrop_partials(*net, n_subjects, d_x, partials, s)) return rc;
  // every coalition once per subject, through the kernel the sweep of these S scenarios runs: v(P) is the sweep's logit bit for bit
  if (int rc = moddrop_eval(*net, n_subjects, 0, partials, nullptr, true, (long long)N * S, v, s)) return rc;
  shapley_combine_kernel<<<ew_grid((long long)(S * N * M)), 256, 0, s>>>(v, d_masks, n_subjects, n_scenarios, M, null_players, d_value,
                                                                         d_base, d_shap);
  PDF_CHECK_LAUNCH();
  if (!d_ig || F == 0) return PDF_OK;
  if (L > 1) {
    if (int rc = ig_launch<false>(*net, partials, d_masks, M, n_subjects, n_scenarios, steps, dbar, s)) return rc;
    if (int rc = pdf_gemm_f32((int)(S * N), F, h1, dbar, h1, 1, net->w[0], F, 1, d_ig, F, nullptr, 0, 0, stream)) return rc;
    moddrop_ig_finish_kernel<<<ew_grid((long long)(S * N * F)), 256, 0, s>>>(*net, d_x, d_masks, n_subjects, n_scenarios, d_ig, F, d_ig);
  } else {
    moddrop_ig_finish_kernel<<<ew_grid((long long)(S * N * F)), 256, 0, s>>>(*net, d_x, d_masks, n_subjects, n_scenarios, net->w[0], 0,
                                                                             d_ig);
  }
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" size_t pdf_moe_explain_workspace_bytes(const pdf_moe* net, int n_subjects, int n_scenarios, int steps) {
  if (!net || n_subjects <= 0 || n_scenarios <= 0 || steps < 0 || net->n_experts < 1 || net->n_experts > PDF_MAX_MODS) return 0;
  const size_t N = (size_t)n_subjects, E = (size_t)net->n_experts;
  // coalition values [2^E, N] | router weights [2^E, E] | with IG, reused expert by expert: partials and mean delta1 [N, max h1],
  // average input gradient [N, max d]
  size_t f = fx_align(((size_t)1 << E) * N) + fx_align(((size_t)1 << E) * E);
  if (steps > 0) {
    size_t h = 0, d = 0;
    for (size_t e = 0; e < E; ++e) {
      if (net->expert[e].n_layers < 1 || net->expert[e].dims[0] <= 0 || net->expert[e].dims[1] <= 0) return 0;
      h = std::max(h, (size_t)net->expert[e].dims[1]);
      d = std::max(d, (size_t)net->expert[e].dims[0]);
    }
    f += 2 * fx_align(N * h) + fx_align(N * d);
  }
  return f * sizeof(float) + 256;
}

extern "C" int pdf_moe_explain(const pdf_moe* net, int n_subjects, int n_scenarios, const float* const* d_x, const uint8_t* d_masks, int steps,
                               void* d_workspace, float* d_value, float* d_base, float* d_shap, float* const* d_ig, pdf_stream_t stream) {
  const char* what = "pdf_moe_explain";
  PDF_REQUIRE(net && n_subjects > 0 && n_scenarios > 0 && d_x && d_masks && d_workspace && d_value && d_base && d_shap,
              "pdf_moe_explain: bad arguments");
  if (int rc = check_steps(steps, d_ig, what)) return rc;
  PDF_REQUIRE(net->n_experts >= 1 && net->n_experts <= PDF_MAX_MODS, "pdf_moe_explain: 1..%d experts (got %d)", PDF_MAX_MODS, net->n_experts);
  if (int rc = check_moe(*net, d_x, what)) return rc;
  const int E = net->n_experts;
  if (d_ig) {
    for (int e = 0; e < E; ++e) {
      PDF_REQUIRE(d_ig[e], "pdf_moe_explain: null d_ig[%d]", e);
      int tp;
      size_t smem;
      if (int rc = mlp_tile(net->expert[e], &tp, &smem, what)) return rc;
    }
  }
  cudaStream_t s = as_stream(stream);
  const size_t N = (size_t)n_subjects, S = (size_t)n_scenarios;
  float* v = reinterpret_cast<float*>(d_workspace);
  float* rw = v + fx_align(((size_t)1 << E) * N);
  // every coalition once per subject, through the sweep's kernel: v(P) is the sweep's probability bit for bit
  if (int rc = moe_eval(*net, d_x, n_subjects, 0, nullptr, rw, v, s)) return rc;
  shapley_combine_kernel<<<ew_grid((long long)(S * N * E)), 256, 0, s>>>(v, d_masks, n_subjects, n_scenarios, E, 0u, d_value, d_base, d_shap);
  PDF_CHECK_LAUNCH();
  if (!d_ig) return PDF_OK;
  size_t h = 0;
  for (int e = 0; e < E; ++e) h = std::max(h, (size_t)net->expert[e].dims[1]);
  float* P = rw + fx_align(((size_t)1 << E) * E);
  float* dbar = P + fx_align(N * h);
  float* gbar = dbar + fx_align(N * h);
  // the expert's integral does not depend on the scenario: once per (n, e), scaled by the router weight of each scenario
  for (int e = 0; e < E; ++e) {
    const pdf_mlp& ex = net->expert[e];
    const int d = ex.dims[0], h1 = ex.dims[1];
    if (int rc = gemm_nt(d_x[e], d, ex.w[0], d, P, h1, nullptr, n_subjects, h1, d, 0, s)) return rc;
    if (int rc = ig_launch<true>(ex, P, nullptr, 1, n_subjects, 1, steps, dbar, s)) return rc;
    if (int rc = pdf_gemm_f32(n_subjects, d, h1, dbar, h1, 1, ex.w[0], d, 1, gbar, d, nullptr, 0, 0, stream)) return rc;
    moe_ig_finish_kernel<<<ew_grid((long long)(S * N * d)), 256, 0, s>>>(d_x[e], d, d_masks, E, e, rw, n_subjects, n_scenarios, gbar, d_ig[e]);
    PDF_CHECK_LAUNCH();
  }
  return PDF_OK;
}

// Monte-Carlo (MC) dropout of the ModDrop and MIL heads: T stochastic forward passes per (scenario, subject) with the heads' own
// nn.Dropout layers active, reduced to the mean probability, its spread and the entropy split into aleatoric and epistemic parts.
//
// Keep masks are stateless: unit j of row n, sample t, dropout layer l, instance i is dropped iff
//   philox4x32_10(key = seed, counter = (n, t, (l << 16) | i, 0x80000000 | (j >> 2))).word[j & 3] < thr,   thr = floor(p 2^32),
// and a kept unit is multiplied by (float)(1 / (1 - p)).  Sample t of row n therefore draws the same masks under every scenario
// (paired differences), results do not depend on S, N, T or the launch shape, and no mask is stored.  The top bit of counter word 3
// keeps these streams apart from the bootstrap's counters (u, b, 0, 0) under the same seed.  One Philox call gives the words of four
// consecutive units.
//
// ModDrop: layer 1 is the sweep's per-modality partials (x (.) m) W1^T = sum_m m_m P_m, computed once per subject; moddrop_mc_kernel
// adds them per (pair, sample) row, applies ReLU and the mask of hidden layer 0, and runs layers 2.. on the explanations' shared-memory
// FFMA tiles with the mask in each hidden layer's epilogue.  MIL: h = ReLU(x W_inst^T + b) does not depend on the sample and is
// computed once by the FP32 sweep's GEMM; mil_mc_kernel masks it per (bag, sample) and runs the attention layer(s), the masked softmax,
// the pooling and the classifier in pdf_mil_sweep's FP32 order.  Both write the sample probabilities; mc_stats reduces each
// (scenario, subject)'s T of them in float64, ascending t.  No atomics: calls are bit-identical.
#include <climits>
#include <cmath>

#include "common.cuh"
#include "mlp_tile.cuh"
#include "ops.cuh"

namespace pdf {

constexpr int kMaxMcSamples = 4096;
constexpr int kMaxMcInstances = 1 << 16;     // the instance index is the low half of counter word 2
constexpr int kMcStats = 5;

static size_t mc_align(size_t n) { return (n + 63) & ~(size_t)63; }     // floats -> 256-byte aligned workspace regions
static bool mc_aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

// the keep-mask words of units 4q .. 4q+3 of (row n, sample t, counter word 2 = (l << 16) | i); all kept when thr == 0
__device__ __forceinline__ void mc_words(uint2 key, uint32_t thr, uint32_t n, uint32_t t, uint32_t li, uint32_t q, uint32_t (&w)[4]) {
  if (thr == 0u) {
    w[0] = w[1] = w[2] = w[3] = 0xffffffffu;
    return;
  }
  const uint4 r = philox4x32_10(make_uint4(n, t, li, 0x80000000u | q), key);
  w[0] = r.x;
  w[1] = r.y;
  w[2] = r.z;
  w[3] = r.w;
}

__device__ __forceinline__ float mc_drop(float v, uint32_t word, uint32_t thr, float scale) { return word < thr ? 0.f : v * scale; }

__device__ __forceinline__ float mc_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float mc_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// binary entropy in nats, 0 ln 0 = 0
__device__ __forceinline__ double mc_entropy(double q) {
  return -(q > 0.0 ? q * log(q) : 0.0) - (q < 1.0 ? (1.0 - q) * log(1.0 - q) : 0.0);
}

// o[5] = mean, std (population), entropy of the mean, mean entropy, mutual information of T sample probabilities p[t * stride], float64,
// ascending t (the samples of MC dropout, stride 1, or the members of a deep ensemble).  The sums run over differences to the first sample, so T equal samples give exactly mean = p, std = 0 and mutual_info = 0.
__device__ void mc_stats(const float* __restrict__ p, int T, long long stride, double* __restrict__ o) {
  const double p0 = p[0], h0 = mc_entropy(p0);
  double sd = 0.0, sh = 0.0;
  for (int t = 0; t < T; ++t) {
    const double q = p[t * stride];
    sd += q - p0;
    sh += mc_entropy(q) - h0;
  }
  const double mean = p0 + sd / T;
  double v = 0.0;
  for (int t = 0; t < T; ++t) {
    const double d = (double)p[t * stride] - mean;
    v += d * d;
  }
  const double ent = mc_entropy(mean), eent = h0 + sh / T;
  o[0] = mean;
  o[1] = sqrt(v / T);
  o[2] = ent;
  o[3] = eent;
  o[4] = fmax(0.0, ent - eent);
}

// ------------------------------------------------------------------------------------------------------
// ModDrop: samples [S*N, T] = the probability of every (pair, sample), pair = s * N + n.  The tile holds TP rows = G pairs x Tc
// samples, pair-major (mlp_ig_kernel's layout): T <= TP gives G = TP / T pairs of all T samples; T > TP one pair in chunks of TP.
// Shared memory as mlp_tile sizes it: the weight chunk, a row slot (unused here), then every hidden layer's activations
// [TP][width + 1] one after the other (the logit's [TP][2] for a one-layer net, which has no dropout).
template <int TP>
__global__ void __launch_bounds__(256)
moddrop_mc_kernel(pdf_mlp net, const float* __restrict__ partials, const uint8_t* __restrict__ masks, int N, int S, int T, uint2 key,
                  uint32_t thr, float scale, float* __restrict__ samples) {
  extern __shared__ float sm[];
  constexpr int RT = TP / 16;
  float* Ws = sm;                              // [16][68]
  float* a1 = Ws + 16 * 68 + TP;               // layer 1, then layers 2 .. L-1 one after the other
  const int tid = threadIdx.x;
  const int L = net.n_layers, h1 = net.dims[1], M = net.n_mods;
  const long long pairs = (long long)N * S;
  const int G = T <= TP ? TP / T : 1, Tc = T <= TP ? T : TP, chunks = (T + Tc - 1) / Tc;
  for (long long u = blockIdx.x; u * G < pairs; u += gridDim.x) {
    const long long pair0 = u * G;
    for (int ch = 0; ch < chunks; ++ch) {
      const int t0 = ch * Tc;
      // layer 1 = sum_m m_m P_m + b1 (the sweep's order), ReLU, the mask of hidden layer 0: four units per thread and Philox call
      const int q1 = (h1 + 3) >> 2;
      for (int idx = tid; idx < TP * q1; idx += 256) {
        const int r = idx / q1, q = idx - r * q1;
        const int g = r / Tc, t = t0 + r - g * Tc;
        const long long pair = pair0 + g;
        const bool valid = g < G && pair < pairs && t < T;
        const int n = valid ? (int)(pair % N) : 0;
        uint32_t wd[4];
        mc_words(key, valid && L > 1 ? thr : 0u, (uint32_t)n, (uint32_t)t, 0u, (uint32_t)q, wd);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = 4 * q + e;
          if (i >= h1) break;
          float z = 0.f;
          if (valid) {
            const uint8_t* mk = masks + pair * M;
            for (int m = 0; m < M; ++m)
              if (mk[m] && net.mod_off[m + 1] > net.mod_off[m]) z += partials[((size_t)m * N + n) * h1 + i];
            z += __ldg(net.b[0] + i);
            if (L > 1) z = mc_drop(fmaxf(z, 0.f), wd[e], thr, scale);
          }
          a1[r * (h1 + 1) + i] = z;
        }
      }
      __syncthreads();
      // hidden layers 2 .. L-1: bias, ReLU, the mask of hidden layer l in the epilogue
      float* in = a1;
      for (int l = 1; l < L - 1; ++l) {
        float* out = in + TP * (net.dims[l] + 1);
        const int n_out = net.dims[l + 1], os = n_out + 1;
        const float* b = net.b[l];
        tile_layer<RT, false, true>(in, net.dims[l] + 1, net.w[l], net.dims[l], n_out, Ws, [&](int r, int c, const float* acc) {
          const int g = r / Tc, t = t0 + r - g * Tc;
          uint32_t wd[4];
          mc_words(key, thr, (uint32_t)((pair0 + g) % N), (uint32_t)t, (uint32_t)l << 16, (uint32_t)(c >> 2), wd);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c + j < n_out) out[r * os + c + j] = mc_drop(fmaxf(acc[j] + __ldg(b + c + j), 0.f), wd[j], thr, scale);
        });
        __syncthreads();
        in = out;
      }
      // the logit (the sweep tile's k-ascending dot product, then the bias), its sigmoid
      const int H = L > 1 ? net.dims[L - 1] : 1, hs = H + 1;
      const float* wL = net.w[L - 1];
      for (int r = tid; r < TP; r += 256) {
        const int g = r / Tc, t = t0 + r - g * Tc;
        const long long pair = pair0 + g;
        if (g >= G || pair >= pairs || t >= T) continue;
        float z;
        if (L > 1) {
          z = 0.f;
          for (int i = 0; i < H; ++i) z = fmaf(in[r * hs + i], __ldg(wL + i), z);
          z += __ldg(net.b[L - 1]);
        } else {
          z = in[r * hs];
        }
        samples[pair * T + t] = mc_sigmoid(z);
      }
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(256)
mc_stats_kernel(const float* __restrict__ samples, long long pairs, int T, double* __restrict__ stats) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (long long)gridDim.x * blockDim.x)
    mc_stats(samples + i * T, T, 1, stats + i * kMcStats);
}

// deep ensembles: probs [E, pairs] -> stats [pairs, 5], mc_stats over the members in ascending order
__global__ void __launch_bounds__(256)
ensemble_stats_kernel(const float* __restrict__ probs, int E, long long pairs, double* __restrict__ stats) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (long long)gridDim.x * blockDim.x)
    mc_stats(probs + i, E, pairs, stats + i * kMcStats);
}

// ------------------------------------------------------------------------------------------------------
// MIL: bagprob [n_bags, T] = the probability of sample t of every bag that is live under some scenario.  One bag per block at a time,
// its T samples one after the other.  Per sample, the bag's instances go through the tile TP rows at a time: masked h, the attention
// pre-activations (tile_layer, k ascending from 0 as gemm_nt_f32_kernel), the scores (mil_pool_kernel's FP32 branch) into
// scores [n_bags, Lmax] (global memory: L2-resident, so any Lmax fits); then mil_pool_kernel's softmax and four-accumulator pooling
// over the masked h.  A bag of one chunk keeps its masked h in the tile for the pooling; longer bags regenerate it chunk by chunk.
// Shared memory: the weight chunk, tile [TP][H + 1], vu [TP][NA + 1].
template <int TP>
__global__ void __launch_bounds__(256)
mil_mc_kernel(const float* __restrict__ hbuf, const int32_t* __restrict__ lens, int Lmax, pdf_mil_weights w, int n_bags, int S,
              const uint8_t* __restrict__ live, int T, uint2 key, uint32_t thr, float scale, float* scores, float* __restrict__ bagprob) {
  extern __shared__ float sm[];
  __shared__ float s_red[8];
  constexpr int RT = TP / 16;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = w.H, A = w.A, NA = w.gated ? 2 * A : A, hs = H + 1, vs = NA + 1, q4 = (H + 3) >> 2;
  float* Ws = sm;                              // [16][68]
  float* tile = Ws + 16 * 68;                  // [TP][H + 1]
  float* vu = tile + TP * hs;                  // [TP][NA + 1]
  for (int bag = blockIdx.x; bag < n_bags; bag += gridDim.x) {
    const int len = min(lens[bag], Lmax);
    bool any_live = len > 0;
    if (any_live && live) {
      any_live = false;
      for (int s = 0; s < S; ++s) any_live |= live[(size_t)s * n_bags + bag] != 0;
    }
    if (!any_live) continue;
    const float* hb = hbuf + (size_t)bag * Lmax * H;
    float* sc = scores + (size_t)bag * Lmax;
    const int chunks = (len + TP - 1) / TP;
    for (int t = 0; t < T; ++t) {
      // masked h of instances c0 .. c0 + TP - 1 (0 past the bag's end)
      auto load = [&](int c0) {
        for (int idx = tid; idx < TP * q4; idx += 256) {
          const int r = idx / q4, q = idx - r * q4, l = c0 + r;
          uint32_t wd[4];
          mc_words(key, l < len ? thr : 0u, (uint32_t)bag, (uint32_t)t, (uint32_t)l, (uint32_t)q, wd);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i = 4 * q + e;
            if (i < H) tile[r * hs + i] = l < len ? mc_drop(hb[(size_t)l * H + i], wd[e], thr, scale) : 0.f;
          }
        }
      };
      for (int ch = 0; ch < chunks; ++ch) {
        const int c0 = ch * TP;
        load(c0);
        __syncthreads();
        tile_layer<RT, false>(tile, hs, w.w_v, H, A, Ws, [&](int r, int c, float acc) { vu[r * vs + c] = acc; });
        if (w.gated) tile_layer<RT, false>(tile, hs, w.w_u, H, A, Ws, [&](int r, int c, float acc) { vu[r * vs + A + c] = acc; });
        __syncthreads();
        for (int r = warp; r < min(TP, len - c0); r += 8) {
          const float* rv = vu + r * vs;
          float s = 0.f;
          for (int a = lane; a < A; a += 32) {
            float th = tanhf(rv[a] + __ldg(w.b_v + a));
            if (w.gated) th *= mc_sigmoid(rv[A + a] + __ldg(w.b_u + a));
            s = fmaf(__ldg(w.w_w + a), th, s);
          }
          s = mc_warp_sum(s);
          if (lane == 0) sc[c0 + r] = s + __ldg(w.b_w);
        }
        __syncthreads();
      }
      // softmax over the bag's instances, as mil_pool_kernel
      float mx = -INFINITY;
      for (int l = tid; l < len; l += 256) mx = fmaxf(mx, sc[l]);
      for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0) s_red[warp] = mx;
      __syncthreads();
      mx = s_red[0];
      for (int i = 1; i < 8; ++i) mx = fmaxf(mx, s_red[i]);
      __syncthreads();
      float se = 0.f;
      for (int l = tid; l < len; l += 256) { const float e = expf(sc[l] - mx); sc[l] = e; se += e; }
      se = mc_warp_sum(se);
      if (lane == 0) s_red[warp] = se;
      __syncthreads();
      se = 0.f;
      for (int i = 0; i < 8; ++i) se += s_red[i];
      for (int l = tid; l < len; l += 256) sc[l] = sc[l] / se;
      __syncthreads();
      // pooling: mil_pool_kernel's four accumulators per column over groups of four instances, the rest into the first; chunks are
      // multiples of four instances, so the groups are the same
      float acc[8][4];
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f;
      for (int ch = 0; ch < chunks; ++ch) {
        const int c0 = ch * TP, lend = min(len, c0 + TP);
        if (chunks > 1) {
          load(c0);
          __syncthreads();
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int i = tid + k * 256;
          if (i >= H) continue;
          int l = c0;
          for (; l + 4 <= lend; l += 4) {
            const float* h4 = tile + (l - c0) * hs + i;
            acc[k][0] = fmaf(sc[l], h4[0], acc[k][0]);
            acc[k][1] = fmaf(sc[l + 1], h4[hs], acc[k][1]);
            acc[k][2] = fmaf(sc[l + 2], h4[2 * hs], acc[k][2]);
            acc[k][3] = fmaf(sc[l + 3], h4[3 * hs], acc[k][3]);
          }
          for (; l < lend; ++l) acc[k][0] = fmaf(sc[l], tile[(l - c0) * hs + i], acc[k][0]);
        }
        if (chunks > 1) __syncthreads();
      }
      float z = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = tid + k * 256;
        if (i < H) z = fmaf(__ldg(w.w_cls + i), (acc[k][0] + acc[k][1]) + (acc[k][2] + acc[k][3]), z);
      }
      z = mc_warp_sum(z);
      if (lane == 0) s_red[warp] = z;
      __syncthreads();
      float zt = 0.f;
      for (int i = 0; i < 8; ++i) zt += s_red[i];
      if (tid == 0) bagprob[(size_t)bag * T + t] = mc_sigmoid(zt + __ldg(w.b_cls));
      __syncthreads();                         // s_red, sc and the tile are reused by the next sample
    }
  }
}

// stats [S, n_bags, 5] and samples [S, n_bags, T] (when not NULL): live[s, b] && len[b] > 0 selects the bag's samples, anything else
// is missing_prob for every sample (mean = missing_prob, std = mutual_info = 0, as mc_stats gives for equal samples)
__global__ void __launch_bounds__(256)
mil_mc_stats_kernel(const float* __restrict__ bagprob, const int32_t* __restrict__ lens, int Lmax, const uint8_t* __restrict__ live,
                    int n_bags, int S, int T, float missing_prob, double* __restrict__ stats, float* __restrict__ samples) {
  const long long total = (long long)S * n_bags;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i % n_bags);
    const bool on = min(lens[b], Lmax) > 0 && (!live || live[i]);
    double* o = stats + i * kMcStats;
    if (on) {
      mc_stats(bagprob + (size_t)b * T, T, 1, o);
    } else {
      const double h = mc_entropy((double)missing_prob);
      o[0] = missing_prob;
      o[1] = 0.0;
      o[2] = h;
      o[3] = h;
      o[4] = 0.0;
    }
    if (samples)
      for (int t = 0; t < T; ++t) samples[i * T + t] = on ? bagprob[(size_t)b * T + t] : missing_prob;
  }
}

static int mc_grid(long long n) { return (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, (long long)num_sms() * 16)); }

static int check_mc(float p_drop, int n_samples, const char* what) {
  PDF_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "%s: p_drop must lie in [0, 1) (got %g)", what, (double)p_drop);
  PDF_REQUIRE(n_samples >= 1 && n_samples <= kMaxMcSamples, "%s: n_samples must be 1..%d (got %d)", what, kMaxMcSamples, n_samples);
  return PDF_OK;
}

// the drop threshold floor(p 2^32) and the kept units' factor (float)(1 / (1 - p)), in float64
static void mc_params(float p_drop, uint32_t* thr, float* scale) {
  *thr = (uint32_t)std::floor((double)p_drop * 4294967296.0);
  *scale = (float)(1.0 / (1.0 - (double)p_drop));
}

template <int TP>
static int moddrop_mc_launch(const pdf_mlp& net, const float* partials, const uint8_t* masks, int N, int S, int T, uint2 key, uint32_t thr,
                             float scale, size_t smem, float* samples, cudaStream_t s) {
  const long long G = T <= TP ? TP / T : 1;
  const long long units = ((long long)N * S + G - 1) / G;
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (228 * 1024) / (smem + 1024)));
  const int blocks = (int)std::max<long long>(1, std::min<long long>(units, (long long)num_sms() * per_sm));
  if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(moddrop_mc_kernel<TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  moddrop_mc_kernel<TP><<<blocks, 256, smem, s>>>(net, partials, masks, N, S, T, key, thr, scale, samples);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

// MIL tile rows: the bag length rounded up to 16, at most 64, fewer while the tile does not fit 227 KB (0: not even 16 rows fit)
static int mil_mc_tile(const pdf_mil_weights& w, int Lmax, size_t* smem) {
  const size_t NA = (size_t)(w.gated ? 2 * w.A : w.A);
  for (int tp = std::min(64, (Lmax + 15) / 16 * 16); tp >= 16; tp -= 16) {
    *smem = (16 * 68 + (size_t)tp * (w.H + 1) + (size_t)tp * (NA + 1)) * sizeof(float);
    if (*smem <= kMlpTileSmemMax) return tp;
  }
  return 0;
}

template <int TP>
static int mil_mc_launch(const float* hbuf, const int32_t* lens, int Lmax, const pdf_mil_weights& w, int n_bags, int S, const uint8_t* live,
                         int T, uint2 key, uint32_t thr, float scale, size_t smem, float* scores, float* bagprob, cudaStream_t s) {
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (228 * 1024) / (smem + 1024)));
  const int blocks = std::max(1, std::min(n_bags, num_sms() * per_sm));
  if (smem > 48 * 1024) PDF_CHECK_CUDA(cudaFuncSetAttribute(mil_mc_kernel<TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mil_mc_kernel<TP><<<blocks, 256, smem, s>>>(hbuf, lens, Lmax, w, n_bags, S, live, T, key, thr, scale, scores, bagprob);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

}  // namespace pdf

using namespace pdf;

extern "C" size_t pdf_moddrop_mc_workspace_bytes(const pdf_mlp* net, int n_subjects, int n_scenarios, int n_samples) {
  if (!net || n_subjects <= 0 || n_scenarios <= 0 || n_samples < 1 || n_samples > kMaxMcSamples || net->n_mods < 1 ||
      net->n_mods > PDF_MAX_MODS || net->n_layers < 1 || net->n_layers > PDF_MAX_LAYERS || net->dims[1] <= 0)
    return 0;
  const size_t N = (size_t)n_subjects, S = (size_t)n_scenarios, T = (size_t)n_samples;
  // per-modality partials [M, N, h1] | sample probabilities [S, N, T] (used when d_samples is NULL)
  return (mc_align((size_t)net->n_mods * N * (size_t)net->dims[1]) + mc_align(S * N * T)) * sizeof(float) + 256;
}

extern "C" int pdf_moddrop_mc(const pdf_mlp* net, float p_drop, int n_subjects, int n_scenarios, const float* d_x, const uint8_t* d_masks,
                              int n_samples, uint64_t seed, void* d_workspace, double* d_stats, float* d_samples, pdf_stream_t stream) {
  const char* what = "pdf_moddrop_mc";
  PDF_REQUIRE(net && n_subjects > 0 && n_scenarios > 0 && d_x && d_masks && d_workspace && d_stats, "pdf_moddrop_mc: bad arguments");
  if (int rc = check_mc(p_drop, n_samples, what)) return rc;
  PDF_REQUIRE(mc_aligned(d_x, 4) && mc_aligned(d_stats, 8) && mc_aligned(d_workspace, 256) && (!d_samples || mc_aligned(d_samples, 4)),
              "pdf_moddrop_mc: misaligned pointer (d_x, d_samples: 4 bytes; d_stats: 8; d_workspace: 256)");
  if (int rc = check_moddrop(*net, what)) return rc;
  for (int m = 0; m < net->n_mods; ++m)
    PDF_REQUIRE(net->mod_off[m + 1] >= net->mod_off[m], "pdf_moddrop_mc: modality offsets must tile [0, F)");
  int tp = 0;
  size_t smem = 0;
  if (int rc = mlp_tile(*net, &tp, &smem, what)) return rc;
  cudaStream_t s = as_stream(stream);
  const size_t N = (size_t)n_subjects, S = (size_t)n_scenarios, T = (size_t)n_samples;
  float* partials = reinterpret_cast<float*>(d_workspace);
  float* samples = d_samples ? d_samples : partials + mc_align((size_t)net->n_mods * N * (size_t)net->dims[1]);
  uint32_t thr;
  float scale;
  mc_params(p_drop, &thr, &scale);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  if (int rc = moddrop_partials(*net, n_subjects, d_x, partials, s)) return rc;
  int rc;
  if (tp == 64)
    rc = moddrop_mc_launch<64>(*net, partials, d_masks, n_subjects, n_scenarios, n_samples, key, thr, scale, smem, samples, s);
  else if (tp == 32)
    rc = moddrop_mc_launch<32>(*net, partials, d_masks, n_subjects, n_scenarios, n_samples, key, thr, scale, smem, samples, s);
  else
    rc = moddrop_mc_launch<16>(*net, partials, d_masks, n_subjects, n_scenarios, n_samples, key, thr, scale, smem, samples, s);
  if (rc) return rc;
  mc_stats_kernel<<<mc_grid((long long)(S * N)), 256, 0, s>>>(samples, (long long)(S * N), (int)T, d_stats);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" size_t pdf_mil_mc_workspace_bytes(const pdf_mil_weights* w, int n_bags, int Lmax, int n_samples) {
  if (!w || n_bags <= 0 || Lmax <= 0 || w->H <= 0 || w->A <= 0 || n_samples < 1 || n_samples > kMaxMcSamples) return 0;
  const size_t rows = (size_t)n_bags * Lmax;
  // h [rows, H] | scores [rows] | bag sample probabilities [n_bags, T]
  return (mc_align(rows * w->H) + mc_align(rows) + mc_align((size_t)n_bags * n_samples)) * sizeof(float) + 256;
}

extern "C" int pdf_mil_mc(const pdf_mil_weights* w, float p_drop, int n_bags, int Lmax, const float* d_bags, const int32_t* d_len,
                          int n_scenarios, const uint8_t* d_live, int n_samples, uint64_t seed, void* d_workspace, double* d_stats,
                          float* d_samples, pdf_stream_t stream) {
  const char* what = "pdf_mil_mc";
  PDF_REQUIRE(w && n_bags > 0 && Lmax > 0 && n_scenarios > 0 && d_bags && d_len && d_workspace && d_stats, "pdf_mil_mc: bad arguments");
  if (int rc = check_mc(p_drop, n_samples, what)) return rc;
  PDF_REQUIRE(mc_aligned(d_bags, 4) && mc_aligned(d_len, 4) && mc_aligned(d_stats, 8) && mc_aligned(d_workspace, 256) &&
              (!d_samples || mc_aligned(d_samples, 4)),
              "pdf_mil_mc: misaligned pointer (d_bags, d_len, d_samples: 4 bytes; d_stats: 8; d_workspace: 256)");
  PDF_REQUIRE(Lmax <= kMaxMcInstances && (long long)n_bags * Lmax <= INT_MAX, "pdf_mil_mc: Lmax must be <= %d and n_bags * Lmax fit an int",
              kMaxMcInstances);
  PDF_REQUIRE(w->D > 0 && w->H > 0 && w->H <= 2048 && w->A > 0, "pdf_mil_mc: bad dims");
  PDF_REQUIRE(w->w_inst && w->b_inst && w->w_v && w->b_v && w->w_w && w->b_w && w->w_cls && w->b_cls && (!w->gated || (w->w_u && w->b_u)),
              "pdf_mil_mc: null weight pointer");
  size_t smem = 0;
  const int tp = mil_mc_tile(*w, Lmax, &smem);
  PDF_REQUIRE(tp > 0, "pdf_mil_mc: H and the attention width too wide for the shared-memory tile (16 rows need more than 227 KB)");
  cudaStream_t s = as_stream(stream);
  const int rows = n_bags * Lmax, T = n_samples;
  float* hbuf = reinterpret_cast<float*>(d_workspace);
  float* scores = hbuf + mc_align((size_t)rows * w->H);
  float* bagprob = scores + mc_align((size_t)rows);
  uint32_t thr;
  float scale;
  mc_params(p_drop, &thr, &scale);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  // the FP32 sweep's instance projection: the same h as pdf_mil_sweep with PDF_PREC_F32
  if (int rc = gemm_nt(d_bags, w->D, w->w_inst, w->D, hbuf, w->H, w->b_inst, rows, w->H, w->D, 1, s)) return rc;
  int rc;
  switch (tp) {
    case 64: rc = mil_mc_launch<64>(hbuf, d_len, Lmax, *w, n_bags, n_scenarios, d_live, T, key, thr, scale, smem, scores, bagprob, s); break;
    case 48: rc = mil_mc_launch<48>(hbuf, d_len, Lmax, *w, n_bags, n_scenarios, d_live, T, key, thr, scale, smem, scores, bagprob, s); break;
    case 32: rc = mil_mc_launch<32>(hbuf, d_len, Lmax, *w, n_bags, n_scenarios, d_live, T, key, thr, scale, smem, scores, bagprob, s); break;
    default: rc = mil_mc_launch<16>(hbuf, d_len, Lmax, *w, n_bags, n_scenarios, d_live, T, key, thr, scale, smem, scores, bagprob, s); break;
  }
  if (rc) return rc;
  mil_mc_stats_kernel<<<mc_grid((long long)n_scenarios * n_bags), 256, 0, s>>>(bagprob, d_len, Lmax, d_live, n_bags, n_scenarios, T,
                                                                                 w->missing_prob, d_stats, d_samples);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

extern "C" int pdf_ensemble_stats(int n_members, long long pairs, const float* d_probs, double* d_stats, pdf_stream_t stream) {
  PDF_REQUIRE(n_members >= 1 && n_members <= 1024 && pairs > 0, "pdf_ensemble_stats: bad sizes (1 <= members <= 1024)");
  PDF_REQUIRE(d_probs && mc_aligned(d_probs, 4) && d_stats && mc_aligned(d_stats, 8), "pdf_ensemble_stats: null or misaligned pointer");
  ensemble_stats_kernel<<<mc_grid(pairs), 256, 0, as_stream(stream)>>>(d_probs, n_members, pairs, d_stats);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

// K2 (bf16 path): implicit-GEMM convolution on the 5th-gen tensor cores.
//
//   D[M = N*Ho*Wo, Cout] = im2col(X)[M, R*S*Cin] * W[Cout, R*S*Cin]^T      bf16 x bf16 -> f32 (TMEM)
//
//   warp 0 (one lane)  TMA producer: A tile [128 pixels x 64 ch] via im2col-mode TMA on the NHWC activation
//                      (padding / stride / image wrap handled by the TMA unit, zero fill), B tile [BLOCK_N x 64]
//                      of the K-major weight matrix; SWIZZLE_128B, STAGES-deep mbarrier ring
//   warp 1 (one lane)  tcgen05.mma cta_group::1 kind::f16, M=128, N=BLOCK_N, K=16 x4 per stage, accumulator in TMEM
//   warps 2..5         epilogue: tcgen05.ld 32x32b -> +bias (+residual) (ReLU) -> bf16 (or f32) NHWC store
//
// Relatives: conv3x3_tc.cu (64-channel 3x3, halo resident), conv3x3_hs.cu (3x3 stride 1, horizontal taps share a tile),
// conv_tc2.cu (CTA pairs, cta_group::2), the DUAL instantiation below (3x3 + the block's 1x1 downsample in one launch).
//
// Replaces the cuDNN/oneDNN convolutions torchvision's ResNet issues from `model(batch)`
// (data/openneuro_features.py:260, scripts/build_resnet2d_mil_embeddings.py:152).
#include "tc_common.cuh"
#include "ops.cuh"

namespace pdf {

static int g_conv_probe = 0;   // pdf_debug_set_conv_probe

struct TcParams {
  int M_total, Cout, Ho, Wo, stride, pad, S, cchunks, num_kb, relu, im2col, out_f32;
  int num_kb2;          // DUAL: k-blocks (= Cin/64) of the fused 1x1 convolution that shares the centre-tap A tiles
  const float* bias2;   // DUAL: its bias, and its bf16 output [M, Cout] (no ReLU, no residual)
  void* out2;
  int probe;            // timing probe (pdf_debug_set_conv_probe): bit 0 = epilogue only hands the accumulator back, bit 1 = no MMAs,
                        // bit 2 = epilogue without its global stores
  const float* bias;
  const __nv_bfloat16* residual;
  void* out;
};

constexpr int kBiasMax = 2048;

template <int BLOCK_N, int STAGES, int MT, bool DUAL = false>
struct SmemLayout {
  static constexpr int kBBytes = BLOCK_N * kBlockK * 2;
  static constexpr int kStage = MT * kABytes + kBBytes;
  static constexpr int kBarOff = STAGES * kStage;
  static constexpr int kNumBars = 2 * STAGES + 4;               // full/empty ring + acc_full[2] + acc_empty[2]
  static constexpr int kBiasOff = kBarOff + kNumBars * 8 + 16;   // f32 bias of every output channel (Cout <= kBiasMax), staged once
  static constexpr int kTotal = kBiasOff + (DUAL ? 2 : 1) * kBiasMax * 4;
  static constexpr int kDynamic = kTotal + 1024;                // slack for manual 1024-byte alignment
  static constexpr int kAccCols = (DUAL ? 2 : 1) * MT * BLOCK_N;   // TMEM columns of one accumulator set (DUAL: main | fused 1x1)
  static_assert(!DUAL || MT == 1, "the dual kernel uses one 128-row sub-tile per tile");
  static_assert(2 * kAccCols <= 512, "two accumulator sets must fit the 512 TMEM columns");
};

// Persistent, warp-specialised implicit-GEMM convolution.
//   MT   128-row M sub-tiles per tile (each with its own accumulator) sharing one B tile per k-block
//   two TMEM accumulator sets: the epilogue of tile t overlaps the TMA/MMA mainloop of tile t+1; the smem ring keeps
//   running across tiles.  Tiles are assigned round-robin (tile = blockIdx.x + i*gridDim.x), m fastest inside an n-tile
//   so that neighbouring CTAs share the weight tile in L2.
//   DUAL a ResNet BasicBlock's 1x1 stride-s downsample convolution reads exactly the centre-tap A tiles of the block's 3x3 stride-s
//        conv1: both are computed in one launch -- after the 9*Cin/64 k-blocks of the 3x3 the centre-tap tiles are loaded once
//        more against the 1x1 weights (tmap_b2) into a second accumulator, and the epilogue writes both outputs.  The separate
//        downsample launches were pure epilogue (profiles/r01_conv_probe.txt); here their stores hide under the next tile.
template <int BLOCK_N, int STAGES, int MT, bool DUAL = false>
__global__ void __launch_bounds__(192)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_b2, const TcParams p) {
  using L = SmemLayout<BLOCK_N, STAGES, MT, DUAL>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;          // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* smem = smem_raw + (base - raw_addr);
  const uint32_t bar_full = base + L::kBarOff;
  const uint32_t bar_empty = bar_full + STAGES * 8;
  const uint32_t bar_accfull = bar_empty + STAGES * 8;
  const uint32_t bar_accempty = bar_accfull + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kBarOff + L::kNumBars * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (p.M_total + kBlockM * MT - 1) / (kBlockM * MT);
  const int total_tiles = m_tiles * (p.Cout / BLOCK_N);
  // The bias vector lives in shared memory: a global load per 32-column chunk put one L2 latency on the epilogue's critical path,
  // which is the whole run time of the short-K (1x1 downsample) launches.  (Weights: not produced by the predecessor kernel.)
  float* s_bias = reinterpret_cast<float*>(smem + L::kBiasOff);
  const bool bias_staged = p.bias != nullptr && p.Cout <= kBiasMax;
  if (bias_staged)
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) s_bias[i] = __ldg(p.bias + i);
  if (DUAL)
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) s_bias[kBiasMax + i] = p.bias2 ? __ldg(p.bias2 + i) : 0.f;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_b);
    if (DUAL) prefetch_tmap(&tmap_b2);
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + s * 8, 1); mbar_init(bar_empty + s * 8, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar_accfull + a * 8, 1); mbar_init(bar_accempty + a * 8, 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 2 * L::kAccCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();   // the next kernel's prologue may overlap this kernel's tail ...
  pdl_wait();                // ... and this one touches activations only after its predecessor has completed

  if (warp == 0) {
    if (elect_one()) {
      uint32_t g = 0;   // k-block counter across tiles (ring position)
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int nt = tile / m_tiles, mtile = tile - nt * m_tiles;
        const int m0 = mtile * (kBlockM * MT), n0 = nt * BLOCK_N;
        const int n_sub = min(MT, (p.M_total - m0 + kBlockM - 1) / kBlockM);
        int n_img[MT], w0[MT], h0[MT];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          n_img[mt] = w0[mt] = h0[mt] = 0;
          if (p.im2col) {
            const int ms = m0 + mt * kBlockM;
            const int hw = p.Ho * p.Wo;
            n_img[mt] = ms / hw;
            const int rem = ms - n_img[mt] * hw;
            const int pp = rem / p.Wo, qq = rem - pp * p.Wo;
            w0[mt] = qq * p.stride - p.pad;
            h0[mt] = pp * p.stride - p.pad;
          }
        }
        const uint32_t tx_bytes = (uint32_t)(n_sub * kABytes + L::kBBytes);
        int tap = 0, cc = 0, r = 0, s = 0;
        for (int kb = 0; kb < p.num_kb; ++kb, ++g) {
          const uint32_t stage = g % STAGES, phase = (g / STAGES) & 1u;
          mbar_wait(bar_empty + stage * 8, phase ^ 1u);
          mbar_expect_tx(bar_full + stage * 8, tx_bytes);
          const uint32_t sa = base + stage * L::kStage, sb = sa + MT * kABytes;
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            if (mt < n_sub) {
              if (p.im2col)
                tma_load_im2col_4d(sa + mt * kABytes, &tmap_a, bar_full + stage * 8, cc * kBlockK, w0[mt], h0[mt], n_img[mt],
                                   (uint16_t)s, (uint16_t)r);
              else
                tma_load_2d(sa + mt * kABytes, &tmap_a, bar_full + stage * 8, kb * kBlockK, m0 + mt * kBlockM);
            }
          }
          tma_load_2d(sb, &tmap_b, bar_full + stage * 8, kb * kBlockK, n0);
          if (++cc == p.cchunks) { cc = 0; ++tap; if (++s == p.S) { s = 0; ++r; } }
        }
        if (DUAL) {   // centre tap (offset = pad in both directions) once more, against the 1x1 weights
          for (int kb = 0; kb < p.num_kb2; ++kb, ++g) {
            const uint32_t stage = g % STAGES, phase = (g / STAGES) & 1u;
            mbar_wait(bar_empty + stage * 8, phase ^ 1u);
            mbar_expect_tx(bar_full + stage * 8, tx_bytes);
            const uint32_t sa = base + stage * L::kStage, sb = sa + MT * kABytes;
            tma_load_im2col_4d(sa, &tmap_a, bar_full + stage * 8, kb * kBlockK, w0[0], h0[0], n_img[0], (uint16_t)p.pad, (uint16_t)p.pad);
            tma_load_2d(sb, &tmap_b2, bar_full + stage * 8, kb * kBlockK, n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(BLOCK_N);
      uint32_t g = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int mtile = tile % m_tiles;
        const int m0 = mtile * (kBlockM * MT);
        const int n_sub = min(MT, (p.M_total - m0 + kBlockM - 1) / kBlockM);
        const int acc = it & 1;
        mbar_wait(bar_accempty + acc * 8, ((uint32_t)(it >> 1) & 1u) ^ 1u);   // epilogue drained this accumulator set
        tc_fence_after();
        const uint32_t d0 = tmem_base + (uint32_t)(acc * L::kAccCols);
        for (int kb = 0; kb < p.num_kb; ++kb, ++g) {
          const uint32_t stage = g % STAGES, phase = (g / STAGES) & 1u;
          mbar_wait(bar_full + stage * 8, phase);
          tc_fence_after();
          const uint32_t a_lo = smem_desc_lo(base + stage * L::kStage), b_lo = a_lo + (uint32_t)(MT * kABytes / 16);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            if (mt < n_sub) {
              if (p.probe & 2) continue;
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k)   // advance 16 bf16 = 32 bytes (2 x 16-byte units) inside the swizzle row
                umma_f16_lo(d0 + mt * BLOCK_N, a_lo + (uint32_t)(mt * kABytes / 16 + k * 2), b_lo + (uint32_t)(k * 2), idesc,
                            (kb | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(bar_empty + stage * 8);   // frees the smem slot once these MMAs have read it
        }
        if (DUAL) {
          for (int kb = 0; kb < p.num_kb2; ++kb, ++g) {
            const uint32_t stage = g % STAGES, phase = (g / STAGES) & 1u;
            mbar_wait(bar_full + stage * 8, phase);
            tc_fence_after();
            const uint32_t a_lo = smem_desc_lo(base + stage * L::kStage), b_lo = a_lo + (uint32_t)(MT * kABytes / 16);
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k)
              umma_f16_lo(d0 + MT * BLOCK_N, a_lo + (uint32_t)(k * 2), b_lo + (uint32_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit(bar_empty + stage * 8);
          }
        }
        umma_commit(bar_accfull + acc * 8);     // accumulators of this tile complete
      }
    }
  } else {
    const int quad = warp & 3;                  // TMEM lanes [32*quad, 32*quad+32) belong to this warp
    const int row = quad * 32 + lane;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int nt = tile / m_tiles, mtile = tile - nt * m_tiles;
      const int m0 = mtile * (kBlockM * MT), n0 = nt * BLOCK_N;
      const int n_sub = min(MT, (p.M_total - m0 + kBlockM - 1) / kBlockM);
      const int acc = it & 1;
      // The whole tile's residual goes into registers BEFORE the wait for the accumulator: the epilogue warps idle through
      // the mainloop anyway, and a load issued per 32-column chunk would expose one DRAM latency per chunk (measured: the
      // residual convolutions ran 15-30 % longer than their twins without residual).
      constexpr int kCPT = BLOCK_N / 32;            // 32-column chunks per 128-row sub-tile
      uint32_t res[MT * kCPT][2][8];
      if (p.residual) {
#pragma unroll
        for (int ch = 0; ch < MT * kCPT; ++ch) {
          const int mt = ch / kCPT, c0 = (ch - mt * kCPT) * 32;
          const int m = m0 + mt * kBlockM + row;
          if (mt < n_sub && m < p.M_total) {
            const __nv_bfloat16* rp = p.residual + (size_t)m * p.Cout + n0 + c0;
            ldg256_nc(rp, res[ch][0]);
            ldg256_nc(rp + 16, res[ch][1]);
          }
        }
      }
      mbar_wait(bar_accfull + acc * 8, (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      if (!p.residual && !p.out_f32 && !(p.probe & 5)) {
        // no residual registers to index statically: a ROLLED loop over the chunks (1/8 of the code; the unrolled body below
        // misses the instruction cache on every tile, 9 % of the epilogue's stall samples in the short-K launches)
#pragma unroll 1
        for (int ch = 0; ch < n_sub * kCPT; ++ch) {
          const int mt = ch / kCPT, c0 = (ch - mt * kCPT) * 32;
          const int m = m0 + mt * kBlockM + row;
          const int col = n0 + c0;
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * L::kAccCols + mt * BLOCK_N + c0), v);
          if (m < p.M_total) {
            float f[32];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
              if (p.bias) b = bias_staged ? *reinterpret_cast<const float4*>(s_bias + col + i) : __ldg(reinterpret_cast<const float4*>(p.bias + col + i));
              f[i] = __uint_as_float(v[i]) + b.x; f[i + 1] = __uint_as_float(v[i + 1]) + b.y;
              f[i + 2] = __uint_as_float(v[i + 2]) + b.z; f[i + 3] = __uint_as_float(v[i + 3]) + b.w;
            }
            if (p.relu) {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
            }
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)m * p.Cout + col;
#pragma unroll
            for (int i = 0; i < 2; ++i)
              stg256(op + i * 16, pack_bf16x2(f[i * 16 + 0], f[i * 16 + 1]), pack_bf16x2(f[i * 16 + 2], f[i * 16 + 3]),
                     pack_bf16x2(f[i * 16 + 4], f[i * 16 + 5]), pack_bf16x2(f[i * 16 + 6], f[i * 16 + 7]),
                     pack_bf16x2(f[i * 16 + 8], f[i * 16 + 9]), pack_bf16x2(f[i * 16 + 10], f[i * 16 + 11]),
                     pack_bf16x2(f[i * 16 + 12], f[i * 16 + 13]), pack_bf16x2(f[i * 16 + 14], f[i * 16 + 15]));
          }
        }
      } else
#pragma unroll
      for (int ch = 0; ch < MT * kCPT; ++ch) {
        const int mt = ch / kCPT, c0 = (ch - mt * kCPT) * 32;
        if (mt >= n_sub || (p.probe & 1)) continue;
        const int m = m0 + mt * kBlockM + row;
        const bool mvalid = m < p.M_total;
        {
          const int col = n0 + c0;
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * L::kAccCols + mt * BLOCK_N + c0), v);
          if (mvalid) {
            float f[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
            if (p.bias) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                const float4 b = bias_staged ? *reinterpret_cast<const float4*>(s_bias + col + i)
                                             : __ldg(reinterpret_cast<const float4*>(p.bias + col + i));
                f[i] += b.x; f[i + 1] += b.y; f[i + 2] += b.z; f[i + 3] += b.w;
              }
            }
            if (p.residual) {
#pragma unroll
              for (int i = 0; i < 2; ++i) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  f[i * 16 + j * 2] += bf16_lo(res[ch][i][j]);
                  f[i * 16 + j * 2 + 1] += bf16_hi(res[ch][i][j]);
                }
              }
            }
            if (p.relu) {
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
            }
            if (p.probe & 4) {                       // timing probe: everything but the global stores
              if (f[0] == 1234.5678f) reinterpret_cast<float*>(p.out)[0] = f[1];
            } else if (p.out_f32) {
              float* op = reinterpret_cast<float*>(p.out) + (size_t)m * p.Cout + col;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                stg256(op + i * 8, __float_as_uint(f[8 * i]), __float_as_uint(f[8 * i + 1]), __float_as_uint(f[8 * i + 2]),
                       __float_as_uint(f[8 * i + 3]), __float_as_uint(f[8 * i + 4]), __float_as_uint(f[8 * i + 5]),
                       __float_as_uint(f[8 * i + 6]), __float_as_uint(f[8 * i + 7]));
            } else {
              __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)m * p.Cout + col;
#pragma unroll
              for (int i = 0; i < 2; ++i)
                stg256(op + i * 16, pack_bf16x2(f[i * 16 + 0], f[i * 16 + 1]), pack_bf16x2(f[i * 16 + 2], f[i * 16 + 3]),
                       pack_bf16x2(f[i * 16 + 4], f[i * 16 + 5]), pack_bf16x2(f[i * 16 + 6], f[i * 16 + 7]),
                       pack_bf16x2(f[i * 16 + 8], f[i * 16 + 9]), pack_bf16x2(f[i * 16 + 10], f[i * 16 + 11]),
                       pack_bf16x2(f[i * 16 + 12], f[i * 16 + 13]), pack_bf16x2(f[i * 16 + 14], f[i * 16 + 15]));
            }
          }
        }
      }
      if (DUAL && !(p.probe & 1)) {                 // second accumulator: the fused 1x1 convolution (+bias, no ReLU) -> out2
        const int m = m0 + row;
#pragma unroll
        for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
          const int col = n0 + c0;
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * L::kAccCols + MT * BLOCK_N + c0), v);   // (whole warp)
          if (m < p.M_total) {
            float f[32];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b = *reinterpret_cast<const float4*>(s_bias + kBiasMax + col + i);
              f[i] = __uint_as_float(v[i]) + b.x; f[i + 1] = __uint_as_float(v[i + 1]) + b.y;
              f[i + 2] = __uint_as_float(v[i + 2]) + b.z; f[i + 3] = __uint_as_float(v[i + 3]) + b.w;
            }
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out2) + (size_t)m * p.Cout + col;
#pragma unroll
            for (int i = 0; i < 2; ++i)
              stg256(op + i * 16, pack_bf16x2(f[i * 16 + 0], f[i * 16 + 1]), pack_bf16x2(f[i * 16 + 2], f[i * 16 + 3]),
                     pack_bf16x2(f[i * 16 + 4], f[i * 16 + 5]), pack_bf16x2(f[i * 16 + 6], f[i * 16 + 7]),
                     pack_bf16x2(f[i * 16 + 8], f[i * 16 + 9]), pack_bf16x2(f[i * 16 + 10], f[i * 16 + 11]),
                     pack_bf16x2(f[i * 16 + 12], f[i * 16 + 13]), pack_bf16x2(f[i * 16 + 14], f[i * 16 + 15]));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_accempty + acc * 8) : "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * L::kAccCols);
}

// Probe kernel: A (256 x 64) resident in smem, MMA reads rows [shift, shift+128) through a shifted descriptor.
template <int BLOCK_N>
__global__ void __launch_bounds__(128)
umma_shift_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int shift, int mode,
                  float* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  const uint32_t sa = base, sb = base + 2 * kABytes, bar = sb + BLOCK_N * 128, bar2 = bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 2 * kABytes + BLOCK_N * 128 + 16);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_init(bar2, 1); fence_barrier_init(); }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), BLOCK_N);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, 2 * kABytes + BLOCK_N * 128);
    tma_load_2d(sa, &tmap_a, bar, 0, 0);
    tma_load_2d(sa + kABytes, &tmap_a, bar, 0, 128);
    tma_load_2d(sb, &tmap_b, bar, 0, 0);
    mbar_wait(bar, 0);
    tc_fence_after();
    const uint32_t start = sa + (uint32_t)shift * 128u;
    for (int k = 0; k < 4; ++k) {
      uint64_t da = make_smem_desc(start + k * 32);
      if (mode == 1) da |= (uint64_t)((start >> 7) & 7u) << 49;
      umma_f16(tmem_base, da, make_smem_desc(sb + k * 32), make_idesc(BLOCK_N), k != 0 ? 1u : 0u);
    }
    umma_commit(bar2);
  }
  mbar_wait(bar2, 0);
  tc_fence_after();
  for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
    uint32_t v[32];
    tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
    for (int i = 0; i < 32; ++i) out[(size_t)(warp * 32 + lane) * BLOCK_N + c0 + i] = __uint_as_float(v[i]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BLOCK_N);
}

// Probe kernel: tensor-pipe rate of back-to-back SS MMAs (M=128, N, K=16) on resident operands.  mode bit 0: the A
// descriptor walks 9 row-shifted windows (the halo conv's access pattern) instead of one tile; out[cta] = cycles.
template <int BLOCK_N>
__global__ void __launch_bounds__(128)
umma_rate_kernel(int iters, int mode, unsigned long long* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  const uint32_t sa = base, sb = base + 3 * kABytes, bar = sb + BLOCK_N * 128;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 3 * kABytes + BLOCK_N * 128 + 16);
  const int warp = threadIdx.x >> 5;
  for (uint32_t i = threadIdx.x; i < (3 * kABytes + BLOCK_N * 128) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;
  if (threadIdx.x == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), BLOCK_N < 32 ? 32 : BLOCK_N);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0 && elect_one()) {
    constexpr uint32_t idesc = make_idesc(BLOCK_N);
    const uint32_t a_lo = smem_desc_lo(sa), b_lo = smem_desc_lo(sb);
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const uint32_t shift = (mode & 1) ? (uint32_t)((t / 3) * 58 + (t % 3)) * 8u : 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_lo(tmem_base, a_lo + shift + k * 2, b_lo + k * 2, idesc, 1u);
      }
    }
    umma_commit(bar);
    mbar_wait(bar, 0);
    out[blockIdx.x] = (unsigned long long)(clock64() - t0);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BLOCK_N < 32 ? 32 : BLOCK_N);
}

// ---------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn g_encode_tiled = nullptr;
static EncodeIm2colFn g_encode_im2col = nullptr;

int load_driver_entry_points() {
  if (g_encode_tiled && g_encode_im2col) return PDF_OK;
  PDF_CHECK_CUDA(cudaFree(0));  // make sure a context exists
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  PDF_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  PDF_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available from the driver");
  g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  fn = nullptr;
  PDF_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &qres));
  PDF_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeIm2col not available from the driver");
  g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
  return PDF_OK;
}

// [rows, cols] row-major bf16 matrix, box = [box_rows x 64 cols], 128-byte swizzle
int encode_2d(TensorMapBlob* out, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  static_assert(sizeof(CUtensorMap) == sizeof(TensorMapBlob), "CUtensorMap is 128 bytes");
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {cols * 2};
  const cuuint32_t box[2] = {(cuuint32_t)kBlockK, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr),
                              dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PDF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu box_rows=%u", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, box_rows);
  return PDF_OK;
}

// extra_w: widen the base-pixel bounding box by that many columns on the right (conv3x3_hs.cu traverses W + 2 positions per row);
// pixels: positions per load
int encode_im2col(TensorMapBlob* out, const pdf_op& op, int extra_w, int pixels) {
  const cuuint64_t dims[4] = {(cuuint64_t)op.c, (cuuint64_t)op.w, (cuuint64_t)op.h, (cuuint64_t)op.n};
  const cuuint64_t strides[3] = {(cuuint64_t)op.c * 2, (cuuint64_t)op.w * op.c * 2, (cuuint64_t)op.h * op.w * op.c * 2};
  // bounding box of the filter's base pixel: lower = -pad, upper = pad - (filter-1)   [W, H] order as CUTLASS passes them
  const int lower[2] = {-op.pad, -op.pad};
  const int upper[2] = {op.pad - (op.s - 1) + extra_w, op.pad - (op.r - 1)};
  const cuuint32_t estr[4] = {1, (cuuint32_t)op.stride, (cuuint32_t)op.stride, 1};
  CUresult r = g_encode_im2col(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(op.d_in),
                               dims, strides, lower, upper, (cuuint32_t)kBlockK, (cuuint32_t)pixels, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PDF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeIm2col failed (%d) nhwc=%d,%d,%d,%d rs=%d,%d stride=%d pad=%d", (int)r, op.n,
              op.h, op.w, op.c, op.r, op.s, op.stride, op.pad);
  // CUTLASS applies the same fix-up for drivers <= 13.1 on tensors smaller than 128 KiB
  int drv = 0;
  cudaDriverGetVersion(&drv);
  if (drv <= 13010 && (size_t)op.n * op.h * op.w * op.c * 2 < 131072) reinterpret_cast<uint64_t*>(out)[1] &= ~(1ull << 21);
  return PDF_OK;
}

// NHWC activation as a 4-D tiled map whose box is NR full padded rows (W+2 columns) of one image, 64 channels
static int encode_halo(TensorMapBlob* out, const pdf_op& op, int Wp, int NR) {
  const cuuint64_t dims[4] = {(cuuint64_t)op.c, (cuuint64_t)op.w, (cuuint64_t)op.h, (cuuint64_t)op.n};
  const cuuint64_t strides[3] = {(cuuint64_t)op.c * 2, (cuuint64_t)op.w * op.c * 2, (cuuint64_t)op.h * op.w * op.c * 2};
  const cuuint32_t box[4] = {(cuuint32_t)kBlockK, (cuuint32_t)Wp, (cuuint32_t)NR, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode_tiled(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(op.d_in), dims,
                              strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PDF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(4d halo) failed (%d) nhwc=%d,%d,%d,%d box=%d,%d", (int)r, op.n, op.h, op.w, op.c, Wp, NR);
  return PDF_OK;
}

static bool g_disable_halo = false;

int prepare_conv_tc(const pdf_op& op, TcConv* tc) {
  if (int rc = load_driver_entry_points()) return rc;
  PDF_REQUIRE(op.c % kBlockK == 0, "bf16 conv: Cin (%d) must be a multiple of 64", op.c);
  PDF_REQUIRE(op.k % 64 == 0, "bf16 conv: Cout (%d) must be a multiple of 64", op.k);
  PDF_REQUIRE(op.stride >= 1 && op.stride <= 8 && op.r == op.s, "bf16 conv: unsupported stride/filter");
  PDF_REQUIRE(op.ho == (op.h + 2 * op.pad - op.r) / op.stride + 1 && op.wo == (op.w + 2 * op.pad - op.s) / op.stride + 1,
              "bf16 conv: inconsistent output size");
  PDF_REQUIRE((reinterpret_cast<uintptr_t>(op.d_in) & 15) == 0 && (reinterpret_cast<uintptr_t>(op.d_weight) & 15) == 0 &&
              (reinterpret_cast<uintptr_t>(op.d_out) & 15) == 0, "bf16 conv: pointers must be 16-byte aligned");
  tc->pw = 0;
  if (pw_eligible(op)) return prepare_conv_pw(op, tc);   // 1x1 convs whose epilogue goes through shared memory (conv_pw.cu)
  PDF_REQUIRE(!op.d_weight3, "bf16 conv: a chained 1x1 convolution needs a 1x1 host convolution with bf16 output (conv_pw.cu)");
  PDF_REQUIRE(!op.sc_c, "bf16 conv: a shortcut segment needs a 1x1 host convolution with bf16 output (conv_pw.cu)");
  tc->block_n = (op.k % 256 == 0) ? 256 : (op.k % 128 == 0 ? 128 : 64);
  tc->im2col = !(op.r == 1 && op.s == 1 && op.stride == 1 && op.pad == 0);
  tc->M_total = op.n * op.ho * op.wo;
  tc->Cout = op.k; tc->Ho = op.ho; tc->Wo = op.wo; tc->stride = op.stride; tc->pad = op.pad; tc->R = op.r; tc->S = op.s;
  tc->cchunks = op.c / kBlockK;
  tc->relu = op.relu; tc->bias = op.d_bias; tc->residual = op.d_residual; tc->out = op.d_out; tc->out_f32 = op.out_f32;
  tc->n_images = op.n;
  tc->dual = 0;
  if (op.d_weight2) {   // fused 1x1 downsample (ResNet BasicBlock): see conv_tc_kernel<..., DUAL>
    PDF_REQUIRE(op.r == 3 && op.s == 3 && op.pad == 1 && op.k % 128 == 0 && op.k <= kBiasMax && op.d_out2 && !op.out_f32 && !op.d_residual,
                "bf16 conv: a fused 1x1 convolution needs a 3x3 pad-1 host conv with Cout %% 128 == 0, bf16 output, no residual");
    PDF_REQUIRE((reinterpret_cast<uintptr_t>(op.d_weight2) & 15) == 0 && (reinterpret_cast<uintptr_t>(op.d_out2) & 31) == 0,
                "bf16 conv: fused 1x1 pointers must be aligned");
    tc->dual = 1;
    tc->block_n = 128;
    tc->bias2 = op.d_bias2;
    tc->out2 = op.d_out2;
    if (int rc = encode_im2col(&tc->tmap_a, op)) return rc;
    if (int rc = encode_2d(&tc->tmap_ds, op.d_weight2, (uint64_t)op.k, (uint64_t)op.c, 128)) return rc;
    return encode_2d(&tc->tmap_b, op.d_weight, (uint64_t)op.k, (uint64_t)op.r * op.s * op.c, 128);
  }
  tc->hs = 0;
  if (hs_eligible(op)) {   // 3x3 stride-1: one activation tile per filter row serves its three taps (conv3x3_hs.cu)
    tc->hs = 1;
    if (int rc = encode_im2col(&tc->tmap_a, op, 2, kBlockM + 2)) return rc;
    return encode_2d(&tc->tmap_b, op.d_weight, (uint64_t)op.k, (uint64_t)op.r * op.s * op.c, 128);
  }
  tc->halo = (!g_disable_halo && !op.out_f32 && op.d_bias && halo_eligible(op)) ? 1 : 0;
  if (tc->halo) {
    tc->halo_wp = op.w + 2;
    tc->halo_nr = (tc->halo_wp - 1 + 255) / tc->halo_wp + 3;
    if (int rc = encode_halo(&tc->tmap_a, op, tc->halo_wp, tc->halo_nr)) return rc;
    return encode_2d(&tc->tmap_b, op.d_weight, (uint64_t)op.k, (uint64_t)op.r * op.s * op.c, 64);
  }
  if (tc->im2col) {
    if (int rc = encode_im2col(&tc->tmap_a, op)) return rc;
  } else {
    if (int rc = encode_2d(&tc->tmap_a, op.d_in, (uint64_t)tc->M_total, (uint64_t)op.c, kBlockM)) return rc;
  }
  if (tc->block_n >= 128) {   // one CTA's half of the weight tile, for the cta_group::2 pair kernel
    if (int rc = encode_2d(&tc->tmap_b2, op.d_weight, (uint64_t)op.k, (uint64_t)op.r * op.s * op.c, (uint32_t)tc->block_n / 2)) return rc;
  }
  return encode_2d(&tc->tmap_b, op.d_weight, (uint64_t)op.k, (uint64_t)op.r * op.s * op.c, (uint32_t)tc->block_n);
}

int prepare_stem_tc(const pdf_op& op, TcConv* tc) {
  if (int rc = load_driver_entry_points()) return rc;
  PDF_REQUIRE((reinterpret_cast<uintptr_t>(op.d_weight) & 15) == 0, "fused stem: weight pointer must be 16-byte aligned");
  if (int rc = encode_2d(&tc->tmap_b, op.d_weight, 128, 128, 128)) return rc;   // [2 variants x 64 channels, K = 96 padded to 128]
  // zero-padded one-channel images [n, rows, pitch]: box = one 39 x 40 patch, no swizzle (stem_tc.cu)
  int pitch = 0, rows = 0;
  if (int rc = pdf_stem_padded_dims(op.h, &pitch, &rows)) return rc;
  PDF_REQUIRE((reinterpret_cast<uintptr_t>(op.d_in) & 15) == 0, "fused stem: input pointer must be 16-byte aligned");
  const cuuint64_t dims[3] = {(cuuint64_t)pitch, (cuuint64_t)rows, (cuuint64_t)op.n};
  const cuuint64_t strides[2] = {(cuuint64_t)pitch * 2, (cuuint64_t)pitch * rows * 2};
  const cuuint32_t box[3] = {40, 39, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode_tiled(reinterpret_cast<CUtensorMap*>(&tc->tmap_a), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(op.d_in),
                              dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PDF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(stem patch) failed (%d) n=%d rows=%d pitch=%d", (int)r, op.n, rows, pitch);
  return PDF_OK;
}

template <int BLOCK_N, int STAGES, int MT, bool DUAL = false>
static int launch_tc(const TcConv& tc, cudaStream_t s) {
  using L = SmemLayout<BLOCK_N, STAGES, MT, DUAL>;
  static bool configured = false;
  if (!configured) {
    PDF_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BLOCK_N, STAGES, MT, DUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kDynamic));
    configured = true;
  }
  TcParams p;
  p.M_total = tc.M_total; p.Cout = tc.Cout; p.Ho = tc.Ho; p.Wo = tc.Wo; p.stride = tc.stride; p.pad = tc.pad; p.S = tc.S;
  p.cchunks = tc.cchunks; p.num_kb = tc.R * tc.S * tc.cchunks; p.relu = tc.relu; p.im2col = tc.im2col; p.out_f32 = tc.out_f32;
  p.bias = tc.bias; p.residual = reinterpret_cast<const __nv_bfloat16*>(tc.residual); p.out = tc.out;
  p.num_kb2 = DUAL ? tc.cchunks : 0; p.bias2 = DUAL ? tc.bias2 : nullptr; p.out2 = DUAL ? tc.out2 : nullptr;
  p.probe = g_conv_probe;
  const int total_tiles = ceil_div(tc.M_total, kBlockM * MT) * (tc.Cout / BLOCK_N);
  const int ctas_per_sm = max(1, min(2, (int)((225 * 1024) / L::kDynamic)));
  const int grid = max(1, min(total_tiles, num_sms() * ctas_per_sm));
  const CUtensorMap& ta = *reinterpret_cast<const CUtensorMap*>(&tc.tmap_a);
  const CUtensorMap& tb = *reinterpret_cast<const CUtensorMap*>(&tc.tmap_b);
  const CUtensorMap& tb2 = DUAL ? *reinterpret_cast<const CUtensorMap*>(&tc.tmap_ds) : tb;
  PDF_CHECK_CUDA(launch_pdl(conv_tc_kernel<BLOCK_N, STAGES, MT, DUAL>, dim3(grid), dim3(192), (size_t)L::kDynamic, s, ta, tb, tb2, p));
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

int launch_conv_tc(const TcConv& tc, cudaStream_t s) {
  if (tc.pw) return launch_conv_pw(tc, s);
  if (tc.dual) return launch_tc<128, 6, 1, true>(tc, s);     // 3x3 conv + the block's 1x1 downsample in one launch
  if (tc.hs) return launch_conv3x3_hs(tc, s);                // 3x3 stride-1: horizontal taps share one activation tile
  if (tc.halo) return launch_conv3x3_halo(tc, s);
  if (pair_eligible(tc)) return launch_conv_tc2(tc, s);      // cta_group::2: two SMs per 256-row tile (conv_tc2.cu)
  // two 128-row sub-tiles per CTA when the mainloop is long enough to amortise the single-tile prologue/epilogue and
  // there are still >= 1.5 waves of CTAs
  // N=128 tiles pair two 128-row sub-tiles per B tile when there is enough work for every SM
  const long tiles2 = (long)ceil_div(tc.M_total, 2 * kBlockM) * (tc.Cout / tc.block_n);
  const bool pair = tiles2 >= 2L * num_sms();
  switch (tc.block_n) {
    case 256: return launch_tc<256, 4, 1>(tc, s);                                        // 2 x 256 TMEM columns
    case 128: return pair ? launch_tc<128, 4, 2>(tc, s) : launch_tc<128, 3, 1>(tc, s);
    case 64: return pair ? launch_tc<64, 4, 2>(tc, s) : launch_tc<64, 4, 1>(tc, s);
  }
  set_error("launch_conv_tc: bad block_n %d", tc.block_n);
  return PDF_ERR_ARG;
}

}  // namespace pdf

// C[M,N] f32 = A[M,K] bf16 * B[N,K]^T bf16 : exercises TMA(2D) -> tcgen05.mma -> tcgen05.ld end to end
extern "C" int pdf_selftest_umma(int M, int N, int K, const void* d_a_bf16, const void* d_b_bf16, float* d_c, pdf_stream_t stream) {
  using namespace pdf;
  PDF_REQUIRE(M > 0 && N % 64 == 0 && K % 64 == 0 && d_a_bf16 && d_b_bf16 && d_c, "pdf_selftest_umma: need N,K multiples of 64");
  pdf_op op;
  memset(&op, 0, sizeof(op));
  op.kind = PDF_OP_CONV; op.precision = PDF_PREC_BF16;
  op.n = 1; op.h = 1; op.w = M; op.c = K; op.k = N; op.r = 1; op.s = 1; op.stride = 1; op.pad = 0; op.ho = 1; op.wo = M;
  op.relu = 0; op.out_f32 = 1; op.d_in = d_a_bf16; op.d_weight = d_b_bf16; op.d_out = d_c;
  TcConv tc;
  memset(&tc, 0, sizeof(tc));
  if (int rc = prepare_conv_tc(op, &tc)) return rc;
  return launch_conv_tc(tc, as_stream(stream));
}

extern "C" int pdf_selftest_umma_shift(int N, int shift, int mode, const void* d_a_bf16, const void* d_b_bf16, float* d_c,
                                       pdf_stream_t stream) {
  using namespace pdf;
  PDF_REQUIRE(N == 64 && shift >= 0 && shift <= 128 && d_a_bf16 && d_b_bf16 && d_c, "pdf_selftest_umma_shift: N must be 64, shift 0..128");
  if (int rc = load_driver_entry_points()) return rc;
  TensorMapBlob ta, tb;
  if (int rc = encode_2d(&ta, d_a_bf16, 256, 64, 128)) return rc;
  if (int rc = encode_2d(&tb, d_b_bf16, 64, 64, 64)) return rc;
  const int smem = 2 * kABytes + 64 * 128 + 64 + 1024;
  PDF_CHECK_CUDA(cudaFuncSetAttribute(umma_shift_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  umma_shift_kernel<64><<<1, 128, smem, as_stream(stream)>>>(*reinterpret_cast<const CUtensorMap*>(&ta),
                                                             *reinterpret_cast<const CUtensorMap*>(&tb), shift, mode, d_c);
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

/* test hook: 1 = route 3x3 s1 64->64 convs through the generic im2col kernel (A/B comparison of the halo kernel) */
extern "C" int pdf_debug_disable_halo(int disable) {
  pdf::g_disable_halo = disable != 0;
  return PDF_OK;
}

/* timing probe for conv_tc_kernel (results are garbage while set): bit 0 = the epilogue only hands the accumulator back,
 * bit 1 = the MMA issuer skips the MMAs (TMA ring and commits still run); 0 = normal */
extern "C" int pdf_debug_set_conv_probe(int mode) {
  pdf::g_conv_probe = mode;
  return PDF_OK;
}

/* probe: cycles for `iters` x 36 back-to-back MMAs (M=128, N, K=16) per CTA, one CTA per SM; d_cycles[grid] */
extern "C" int pdf_selftest_umma_rate(int N, int iters, int mode, int grid, unsigned long long* d_cycles, pdf_stream_t stream) {
  using namespace pdf;
  PDF_REQUIRE((N == 64 || N == 128 || N == 256) && iters > 0 && grid > 0 && d_cycles, "pdf_selftest_umma_rate: bad arguments");
  if (mode & 2) return launch_umma2_rate(N, iters, mode & 1, max(1, grid / 2), d_cycles, as_stream(stream));   // CTA pairs (cta_group::2)
  const int smem = 3 * kABytes + N * 128 + 64 + 1024;
  cudaStream_t s = as_stream(stream);
  if (N == 64) {
    PDF_CHECK_CUDA(cudaFuncSetAttribute(umma_rate_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    umma_rate_kernel<64><<<grid, 128, smem, s>>>(iters, mode, d_cycles);
  } else if (N == 128) {
    PDF_CHECK_CUDA(cudaFuncSetAttribute(umma_rate_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    umma_rate_kernel<128><<<grid, 128, smem, s>>>(iters, mode, d_cycles);
  } else {
    PDF_CHECK_CUDA(cudaFuncSetAttribute(umma_rate_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    umma_rate_kernel<256><<<grid, 128, smem, s>>>(iters, mode, d_cycles);
  }
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

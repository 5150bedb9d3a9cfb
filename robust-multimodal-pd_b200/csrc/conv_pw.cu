// K2 (bf16 path): pointwise (1x1) convolutions of the ResNet50 bottleneck, epilogue through shared memory.
//
//   Y[M, Cout] = relu?( X[M, Cin] * W[Cout, Cin]^T + bias (+ R[M, Cout]) )                 bf16 x bf16 -> f32 (TMEM) -> bf16
//   optional shortcut segment:  Y = relu( [X | Xs] * [W | Ws]^T + bias )                      (instead of a residual R)
//   optional chain:  T[M, N2] = relu( Y[M, Cout] * W3[N2, Cout]^T + bias3 )               (the NEXT block's 1x1 reduce conv)
//
// Why a second kernel next to conv_tc.cu: the bottleneck's expansion convs and downsamples have K = 64..512 and N = 256..2048,
// i.e. a few hundred tensor-pipe cycles per 128 x 128 output tile against 64 KB of residual + output traffic -- they are bound
// by how the EPILOGUE moves bytes.  conv_tc_kernel's row-per-lane global accesses (every lane of a warp in a different
// 128-byte line) ran them at 2x their HBM floor (profiles/r01_op_times_resnet50.txt, r01_conv_probe_resnet50.txt).  Here
//
//   * the residual tile is fetched by TMA into a 128B-swizzled staging buffer, one unit ahead of the epilogue;
//   * the epilogue warps read TMEM, add bias + residual (conflict-free 16-byte shared-memory accesses), apply ReLU and write
//     the bf16 result IN PLACE into the staging buffer;
//   * one thread hands the buffer to the TMA unit (cp.async.bulk.tensor store): full-line writes, no LSU involvement;
//   * the same buffer -- it has exactly the K-major SWIZZLE_128B layout of an MMA A operand -- feeds the chained GEMM:
//     the next block's 1x1 reduce convolution accumulates over the N-chunks of the tile in a third TMEM accumulator, so that
//     conv never re-reads the (4x wider) block output from HBM: its launch disappears;
//   * a Bottleneck's projection shortcut (downsample 1x1 conv + BN of the block input x, added before the ReLU) is the same GEMM
//     as conv3 over K: the last k-blocks of the mainloop come from a second map over x (2-D at stride 1, im2col-mode at stride 2)
//     and multiply the shortcut's columns of the host-concatenated weights [W3 | Wds].  The downsample's 4x-wide output is then
//     never written nor read back as a residual, and its launch disappears.
//
// Work unit = (128-row M tile, NC-column N chunk), N fastest: one CTA owns all chunks of its M tiles (persistent, round-robin).
//   warp 0 (one lane)  TMA producer: residual tile of unit u | A/B k-blocks of unit u | chained-weight k-blocks of unit u-1
//   warp 1 (one lane)  tcgen05.mma issuer: main GEMM of unit u, then the chained GEMM of unit u-1 (its Y tile is ready by then)
//   warps 2..9         epilogue (two warps per TMEM lane quarter, alternating 32-column chunks)
//
// Replaces the cuDNN 1x1 convolutions + BatchNorm + add + ReLU torchvision's Bottleneck.forward issues from `model(batch)`
// (scripts/build_resnet2d_mil_embeddings.py:148-156, data/openneuro_features.py:257-262).
#include "tc_common.cuh"
#include "ops.cuh"

namespace pdf {

static int g_pw_mode = 1;   // pdf_debug_set_pw: 0 = never, 1 = default policy, 2 = every eligible 1x1 convolution
static int g_pw_prefetch = 0;   // pdf_debug_set_pw_prefetch: L2 prefetch of the next row tile's A operand
static int g_pw_mc = 0;     // pdf_debug_set_pw_multicast: 0 (default) = single CTAs, 1 = weight-multicast CTA pairs where K >= 128

constexpr int kPwMaxStages = 6;     // ring depth and staging-buffer count are launch parameters (pdf_debug_set_pw_config)
constexpr int kPwMaxRy = 4;         // staging buffers (residual in / output out / chained A operand)
static int g_pw_stages = 0, g_pw_ry = 0;   // 0 = per-launch default (launch_pw)
constexpr int kPwEpiWarps = 8;
constexpr int kPwThreads = 64 + 32 * kPwEpiWarps;
constexpr int kPwBiasMax = 2048;

struct PwParams {
  int M_total, Cout, K, n_chunks, m_tiles, relu, im2col, has_res;
  int Ho, Wo, stride;           // im2col (strided 1x1) geometry
  int kb_main;                  // k-blocks read through tmap_a; k-blocks kb_main .. K/64-1 are the shortcut segment (tmap_sc)
  int sc_im2col, sc_stride;     // shortcut segment: 1 = im2col-mode map at sc_stride (2), 0 = 2-D map over [M, sc_c]
  int N2;                       // chained output channels
  int stages, nry;              // ring depth, staging buffers
  int bias_staged;              // 1: bias vector copied to shared memory at kernel start, 0: read from global memory (L1-resident)
  int l2_prefetch;              // 1: prefetch the next row tile's A k-blocks into L2
  const float* bias;
  const float* bias3;
  __nv_bfloat16* out3;
};

template <int NC>
struct PwSmem {
  static constexpr int kStageBytes = (NC == 128) ? 32768 : (kABytes + NC * 128);   // NC=128: A | B contiguous = one [256 x 64] chained-weight tile
  static constexpr int kRyBytes = NC * 256;                                         // 128 rows x NC channels bf16 = NC/64 sub-tiles of 16 KB
  // layout: ring [stages] | staging [nry] | barriers | TMEM slot | bias
  static constexpr int kNumBars = 2 * kPwMaxStages + 4 + 3 * kPwMaxRy + 2;
  // tail: barriers | TMEM slot | chained bias [256] | bias [bias_floats] (0 = the epilogue reads the bias from global memory)
  static int dynamic_bytes(int stages, int nry, int bias_floats) {
    return stages * kStageBytes + nry * kRyBytes + kNumBars * 8 + 16 + 16 + (256 + bias_floats) * 4 + 1024;
  }
};

__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kPwEpiWarps) : "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- weight multicast (MC): two CTAs of a cluster own DIFFERENT 128-row tiles but walk the SAME sequence of weight tiles (main B
// k-blocks and chained W3 blocks).  Each CTA fetches HALF of every weight tile and multicasts it into both CTAs' rings, so a unit
// costs each SM 160 instead of 224 KB of L2 requests in stage 3 (A 64 + B 32 + W3 32 + residual 32).  MEASURED: no gain (9.34 vs
// 9.23 ms on the ResNet50 stack, per-launch times unchanged) -- a stage still needs its full 32 KB to land before the MMAs start and
// the ring holds the same three stages, so halving the REQUESTS does not raise the bytes in flight per unit of work; only a real
// cta_group::2 tile (half of B RESIDENT per CTA: 24 KB stages, a deeper ring) would.  Kept as a tested opt-in
// (pdf_debug_set_pw_multicast / PDFUSION_B200_PW_MC=1); bit-identical to the single-CTA launches.  The MMAs stay cta_group::1 (each CTA
// its own accumulators); only the ring is shared: a stage is free once BOTH CTAs' MMAs have read it (multicast tcgen05.commit, "empty"
// barriers count two arrivals), and its "full" barrier collects the CTA's own A load plus both weight halves.
__device__ __forceinline__ uint32_t pw_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void pw_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, uint16_t mask) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}

// Packed float32 pairs (Blackwell FADD2) and the fused ReLU + bf16x2 pack (F2FP.RELU): the epilogue of a 128 x 128 unit was ~36 ALU
// instructions per 8 channels (8 bias adds, 8 bf16 unpacks, 8 residual adds, 8 max, 4 packs) on 8 warps -- in stages 2-4, where the
// unit's MMAs take 0.5 us, the epilogue WAS the unit time.  With pairs: 4 + 8 + 4 + 4.
__device__ __forceinline__ uint64_t f2_pack(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint32_t f2_to_bf16x2(uint64_t v, bool relu) {     // low half = first element
  uint32_t lo, hi, r;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
  if (relu) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  return r;
}
__device__ __forceinline__ uint64_t bf16x2_to_f2(uint32_t w) { return f2_pack(w << 16, w & 0xffff0000u); }

template <int NC, bool CHAIN, bool MC>
__global__ void __launch_bounds__(kPwThreads, 1)
conv_pw_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_res,
               const __grid_constant__ CUtensorMap tmap_w3, const __grid_constant__ CUtensorMap tmap_sc, const PwParams p) {
  using L = PwSmem<NC>;
  constexpr int kSub = NC / 64;                   // 64-channel sub-tiles of a staging buffer
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  const int kPwStages = p.stages, kPwRy = p.nry;
  const uint32_t s_ring = base, s_ry = base + (uint32_t)(kPwStages * L::kStageBytes);
  const uint32_t bar_off = (uint32_t)(kPwStages * L::kStageBytes + kPwRy * L::kRyBytes);
  const uint32_t bar_full = base + bar_off;
  const uint32_t bar_empty = bar_full + 8 * kPwMaxStages;
  const uint32_t bar_accfull = bar_empty + 8 * kPwMaxStages;
  const uint32_t bar_accempty = bar_accfull + 16;
  const uint32_t bar_resfull = bar_accempty + 16;
  const uint32_t bar_ryfree = bar_resfull + 8 * kPwMaxRy;
  const uint32_t bar_yready = bar_ryfree + 8 * kPwMaxRy;
  const uint32_t bar_acc2full = bar_yready + 8 * kPwMaxRy;
  const uint32_t bar_acc2empty = bar_acc2full + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + bar_off + L::kNumBars * 8);
  float* s_bias3 = reinterpret_cast<float*>(smem + bar_off + L::kNumBars * 8 + 16);
  float* s_bias = s_bias3 + 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (p.bias_staged)
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) s_bias[i] = p.bias ? __ldg(p.bias + i) : 0.f;
  if (CHAIN)
    for (int i = threadIdx.x; i < p.N2; i += blockDim.x) s_bias3[i] = p.bias3 ? __ldg(p.bias3 + i) : 0.f;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmap_a); prefetch_tmap(&tmap_b); prefetch_tmap(&tmap_out);
    if (p.has_res) prefetch_tmap(&tmap_res);
    if (CHAIN) prefetch_tmap(&tmap_w3);
    if (p.kb_main < p.K / kBlockK) prefetch_tmap(&tmap_sc);
    for (int s = 0; s < kPwStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, MC ? 2 : 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar_accfull + 8 * a, 1); mbar_init(bar_accempty + 8 * a, kPwEpiWarps); }
    for (int b = 0; b < kPwRy; ++b) {
      mbar_init(bar_resfull + 8 * b, 1);
      mbar_init(bar_ryfree + 8 * b, CHAIN ? 2 : 1);     // TMA store has read the buffer (+ the chained MMAs have)
      mbar_init(bar_yready + 8 * b, 1);
    }
    mbar_init(bar_acc2full, 1);
    mbar_init(bar_acc2empty, kPwEpiWarps);
    fence_barrier_init();
  }
  constexpr uint32_t kTmemCols = CHAIN ? 512 : 2 * NC;
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_acc2 = tmem_base + 2 * NC;
  if (MC) pw_cluster_sync();                     // both CTAs' barriers exist before any multicast load / commit reaches them
  pdl_launch_dependents();
  pdl_wait();

  // M tiles of this CTA: tile(ti).  MC: cluster c of gridDim/2 walks tile PAIRS c, c + gridDim/2, ...; both CTAs run the same
  // number of units (a pair's second tile may lie past the end: its loads are zero-filled, its stores clipped)
  const uint32_t rank = MC ? pw_cluster_rank() : 0u;
  const int n_walkers = MC ? (int)gridDim.x / 2 : (int)gridDim.x;
  const int walker = MC ? (int)blockIdx.x / 2 : (int)blockIdx.x;
  const int n_items = MC ? (p.m_tiles + 1) / 2 : p.m_tiles;
  const int my_tiles = (n_items - walker + n_walkers - 1) / n_walkers;
  auto tile_of = [&](int ti) { return MC ? (walker + ti * n_walkers) * 2 + (int)rank : walker + ti * n_walkers; };
  const int n_units = my_tiles * p.n_chunks;
  const int num_kb = p.K / kBlockK;

  if (warp == 0) {
    if (elect_one()) {
      uint32_t g = 0;
      auto ring_wait = [&](uint32_t& stage) {
        stage = g % kPwStages;
        mbar_wait(bar_empty + 8 * stage, ((g / kPwStages) & 1u) ^ 1u);
        ++g;
      };
      auto load_chain = [&](int v) {                // chained-weight k-blocks of unit v: W3[:, nc*NC + j*64 .. +64]
        const int nc = v % p.n_chunks;
        for (int j = 0; j < kSub; ++j) {
          uint32_t stage;
          ring_wait(stage);
          mbar_expect_tx(bar_full + 8 * stage, (uint32_t)p.N2 * 128u);
          const uint32_t dst = s_ring + stage * L::kStageBytes + (p.N2 > 128 ? 0 : kABytes);
          if (MC)      // this CTA's half of the [N2 x 64] block (tmap_w3's box is N2/2 rows), into both rings
            tma_load_2d_mc(dst + rank * (uint32_t)(p.N2 * 64), &tmap_w3, bar_full + 8 * stage, nc * NC + j * 64, (int)rank * (p.N2 / 2), (uint16_t)3);
          else tma_load_2d(dst, &tmap_w3, bar_full + 8 * stage, nc * NC + j * 64, 0);
        }
      };
      for (int u = 0; u < n_units; ++u) {
        const int ti = u / p.n_chunks, nc = u - ti * p.n_chunks;
        const int m0 = tile_of(ti) * kBlockM, n0 = nc * NC;
        if (p.l2_prefetch && nc == 0 && !p.im2col && ti + 1 < my_tiles) {
          // the NEXT row tile's A k-blocks into L2 while this tile's n_chunks units run: its first ring fills then hit L2 instead of
          // paying the HBM latency inside the ring (pdf_debug_set_pw_prefetch)
          const int m1 = tile_of(ti + 1) * kBlockM;
          for (int kb = 0; kb < p.kb_main; ++kb)
            asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
                         ::"l"(reinterpret_cast<uint64_t>(&tmap_a)), "r"(kb * kBlockK), "r"(m1) : "memory");
        }
        if (p.has_res) {
          const int b = u % kPwRy;
          mbar_wait(bar_ryfree + 8 * b, (((uint32_t)(u / kPwRy)) & 1u) ^ 1u);
          mbar_expect_tx(bar_resfull + 8 * b, (uint32_t)L::kRyBytes);
          for (int s = 0; s < kSub; ++s) tma_load_2d(s_ry + b * L::kRyBytes + s * kABytes, &tmap_res, bar_resfull + 8 * b, n0 + s * 64, m0);
        }
        int n_img = 0, pp = 0, qq = 0;             // first output pixel of the tile (im2col-mode loads)
        if (p.im2col || p.sc_im2col) {
          const int hw = p.Ho * p.Wo;
          n_img = m0 / hw;
          const int rem = m0 - n_img * hw;
          pp = rem / p.Wo; qq = rem - pp * p.Wo;
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          uint32_t stage;
          ring_wait(stage);
          mbar_expect_tx(bar_full + 8 * stage, (uint32_t)(kABytes + NC * 128));
          const uint32_t sa = s_ring + stage * L::kStageBytes;
          const int kc = (kb - p.kb_main) * kBlockK;    // channel of the shortcut segment (kb >= kb_main)
          if (kb < p.kb_main) {
            if (p.im2col) tma_load_im2col_4d(sa, &tmap_a, bar_full + 8 * stage, kb * kBlockK, qq * p.stride, pp * p.stride, n_img, 0, 0);
            else tma_load_2d(sa, &tmap_a, bar_full + 8 * stage, kb * kBlockK, m0);
          } else if (p.sc_im2col) {
            tma_load_im2col_4d(sa, &tmap_sc, bar_full + 8 * stage, kc, qq * p.sc_stride, pp * p.sc_stride, n_img, 0, 0);
          } else {
            tma_load_2d(sa, &tmap_sc, bar_full + 8 * stage, kc, m0);
          }
          if (MC)      // this CTA's half of the [NC x 64] weight tile (tmap_b's box is NC/2 rows), into both rings
            tma_load_2d_mc(sa + kABytes + rank * (uint32_t)(NC * 64), &tmap_b, bar_full + 8 * stage, kb * kBlockK, n0 + (int)rank * (NC / 2), (uint16_t)3);
          else tma_load_2d(sa + kABytes, &tmap_b, bar_full + 8 * stage, kb * kBlockK, n0);
        }
        if (CHAIN && u > 0) load_chain(u - 1);
      }
      if (CHAIN && n_units > 0) load_chain(n_units - 1);
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(NC);
      const uint32_t idesc2 = make_idesc(CHAIN ? p.N2 : NC);
      uint32_t g = 0;
      auto do_chain = [&](int v) {                  // acc2 (+)= Y tile of unit v (staging buffer) x chained weights
        const int ti = v / p.n_chunks, nc = v - ti * p.n_chunks;
        const int b = v % kPwRy;
        if (nc == 0) { mbar_wait(bar_acc2empty, ((uint32_t)ti & 1u) ^ 1u); }
        mbar_wait(bar_yready + 8 * b, ((uint32_t)(v / kPwRy)) & 1u);
        tc_fence_after();
        for (int j = 0; j < kSub; ++j, ++g) {
          const uint32_t stage = g % kPwStages;
          mbar_wait(bar_full + 8 * stage, (g / kPwStages) & 1u);
          tc_fence_after();
          const uint32_t a_lo = smem_desc_lo(s_ry + b * L::kRyBytes + j * kABytes);
          const uint32_t b_lo = smem_desc_lo(s_ring + stage * L::kStageBytes + (p.N2 > 128 ? 0 : kABytes));
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k)
            umma_f16_lo(tmem_acc2, a_lo + (uint32_t)(k * 2), b_lo + (uint32_t)(k * 2), idesc2, (nc | j | k) != 0 ? 1u : 0u);
          if (MC) umma_commit_mc(bar_empty + 8 * stage, (uint16_t)3); else umma_commit(bar_empty + 8 * stage);
        }
        umma_commit(bar_ryfree + 8 * b);
        if (nc == p.n_chunks - 1) umma_commit(bar_acc2full);
      };
      for (int u = 0; u < n_units; ++u) {
        const int acc = u & 1;
        mbar_wait(bar_accempty + 8 * acc, (((uint32_t)(u >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d0 = tmem_base + (uint32_t)(acc * NC);
        for (int kb = 0; kb < num_kb; ++kb, ++g) {
          const uint32_t stage = g % kPwStages;
          mbar_wait(bar_full + 8 * stage, (g / kPwStages) & 1u);
          tc_fence_after();
          const uint32_t a_lo = smem_desc_lo(s_ring + stage * L::kStageBytes), b_lo = a_lo + (uint32_t)(kABytes / 16);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k)
            umma_f16_lo(d0, a_lo + (uint32_t)(k * 2), b_lo + (uint32_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
          if (MC) umma_commit_mc(bar_empty + 8 * stage, (uint16_t)3); else umma_commit(bar_empty + 8 * stage);
        }
        umma_commit(bar_accfull + 8 * acc);
        if (CHAIN && u > 0) do_chain(u - 1);
      }
      if (CHAIN && n_units > 0) do_chain(n_units - 1);
    }
  } else {
    const int ew = warp - 2;                        // 0..7
    const int quad = warp & 3;                      // TMEM lane quarter this warp may read
    const int half = ew >> 2;                       // which 32-column chunks (alternating) this warp handles
    const int row = quad * 32 + lane;
    const uint32_t row_off = (uint32_t)row * 128u;
    const uint32_t sw = (uint32_t)(row & 7);
    const bool leader = (ew == 0 && lane == 0);
    constexpr int kChunks = NC / 32;

    auto acc2_epilogue = [&](int ti) {              // chained conv output of M tile ti: relu(acc2 + bias3) -> out3 (bf16)
      mbar_wait(bar_acc2full, (uint32_t)ti & 1u);
      tc_fence_after();
      const int m = tile_of(ti) * kBlockM + row;
      const int chunks2 = p.N2 / 32;
      for (int ch = half; ch < chunks2; ch += 2) {
        uint32_t v[32];
        tmem_ld32(tmem_acc2 + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ch * 32), v);
        if (m < p.M_total) {
          uint32_t h[16];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(s_bias3 + ch * 32 + i);
            h[i / 2] = f2_to_bf16x2(f2_add(f2_pack(v[i], v[i + 1]), b.x), true);
            h[i / 2 + 1] = f2_to_bf16x2(f2_add(f2_pack(v[i + 2], v[i + 3]), b.y), true);
          }
          __nv_bfloat16* op = p.out3 + (size_t)m * p.N2 + ch * 32;
#pragma unroll
          for (int i = 0; i < 2; ++i)
            stg256(op + i * 16, h[i * 8 + 0], h[i * 8 + 1], h[i * 8 + 2], h[i * 8 + 3], h[i * 8 + 4], h[i * 8 + 5], h[i * 8 + 6], h[i * 8 + 7]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc2empty);
    };

    for (int u = 0; u < n_units; ++u) {
      const int ti = u / p.n_chunks, nc = u - ti * p.n_chunks;
      const int m0 = tile_of(ti) * kBlockM, n0 = nc * NC;
      const int b = u % kPwRy, acc = u & 1;
      const uint32_t ry = s_ry + b * L::kRyBytes;
      if (p.has_res) mbar_wait(bar_resfull + 8 * b, ((uint32_t)(u / kPwRy)) & 1u);
      else mbar_wait(bar_ryfree + 8 * b, (((uint32_t)(u / kPwRy)) & 1u) ^ 1u);
      mbar_wait(bar_accfull + 8 * acc, ((uint32_t)(u >> 1)) & 1u);
      tc_fence_after();
#pragma unroll
      for (int ci = 0; ci < kChunks / 2; ++ci) {
        const int ch = ci * 2 + half;
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * NC + ch * 32), v);
        const uint32_t sub = ry + (uint32_t)(ch >> 1) * kABytes + row_off;      // 64-channel sub-tile, this thread's 128-byte row
        const float* bp = (p.bias_staged ? s_bias : p.bias) + n0 + ch * 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {                                          // 8 channels = one 16-byte unit
          const uint32_t addr = sub + ((((uint32_t)((ch & 1) * 4 + q)) ^ sw) << 4);
          const ulonglong2 b0 = *reinterpret_cast<const ulonglong2*>(bp + q * 8), b1 = *reinterpret_cast<const ulonglong2*>(bp + q * 8 + 4);
          uint64_t p0 = f2_add(f2_pack(v[q * 8 + 0], v[q * 8 + 1]), b0.x), p1 = f2_add(f2_pack(v[q * 8 + 2], v[q * 8 + 3]), b0.y);
          uint64_t p2 = f2_add(f2_pack(v[q * 8 + 4], v[q * 8 + 5]), b1.x), p3 = f2_add(f2_pack(v[q * 8 + 6], v[q * 8 + 7]), b1.y);
          if (p.has_res) {
            const uint4 r = lds128(addr);
            p0 = f2_add(p0, bf16x2_to_f2(r.x)); p1 = f2_add(p1, bf16x2_to_f2(r.y));
            p2 = f2_add(p2, bf16x2_to_f2(r.z)); p3 = f2_add(p3, bf16x2_to_f2(r.w));
          }
          uint4 o;
          const bool relu = p.relu != 0;
          o.x = f2_to_bf16x2(p0, relu); o.y = f2_to_bf16x2(p1, relu); o.z = f2_to_bf16x2(p2, relu); o.w = f2_to_bf16x2(p3, relu);
          sts128(addr, o);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_accempty + 8 * acc);        // the MMA issuer may overwrite this accumulator
      if (leader && u > 0) {                                     // the PREVIOUS unit's store was issued a whole tile of arithmetic ago: it
        bulk_wait_read<0>();                                     // has read its staging buffer -- hand the buffer back now (not after this
        mbar_arrive(bar_ryfree + 8 * ((u - 1) % kPwRy));         // unit's store), the next residual tile streams in under the rest
      }
      fence_proxy_async();                                       // staging-buffer writes -> visible to the TMA unit / tensor core
      epi_bar_sync();
      if (leader) {
#pragma unroll
        for (int s = 0; s < kSub; ++s) tma_store_2d(&tmap_out, ry + s * kABytes, n0 + s * 64, m0);
        bulk_commit();
        if (CHAIN) mbar_arrive(bar_yready + 8 * b);
      }
      // the chained accumulator of the previous M tile is complete once the chained MMAs of its last chunk (issued after the
      // main MMAs of THIS unit) have run
      if (CHAIN && nc == 0 && ti > 0) acc2_epilogue(ti - 1);
    }
    if (CHAIN && my_tiles > 0) acc2_epilogue(my_tiles - 1);
    if (leader) bulk_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (MC) pw_cluster_sync();                     // the peer's multicast loads / commits must not target a CTA that has exited
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------- host side
bool pw_eligible(const pdf_op& op) {
  if (g_pw_mode == 0) return false;
  if (!(op.kind == PDF_OP_CONV && op.precision == PDF_PREC_BF16 && op.r == 1 && op.s == 1 && op.pad == 0 && !op.out_f32 && !op.d_weight2))
    return false;
  if (op.c % 64 != 0 || op.k % 64 != 0 || op.k > kPwBiasMax || op.sc_c % 64 != 0) return false;
  if (op.d_weight3 || op.sc_c) return true;
  if (g_pw_mode == 2) return true;
  // default policy (profiles/r02_op_times_resnet50_pw*.txt): every N chunk of a tile re-streams the A tile, so long-K reduce
  // convs and downsamples stay on conv_tc_kernel's 256-wide tiles; the epilogue-bound short-K launches come here
  if (op.c <= 256) return true;
  return op.d_residual != nullptr && op.c <= 512;
}

int prepare_conv_pw(const pdf_op& op, TcConv* tc) {
  if (int rc = load_driver_entry_points()) return rc;
  const int NC = (op.k % 128 == 0) ? 128 : 64;
  PDF_REQUIRE((reinterpret_cast<uintptr_t>(op.d_in) & 15) == 0 && (reinterpret_cast<uintptr_t>(op.d_weight) & 15) == 0 &&
              (reinterpret_cast<uintptr_t>(op.d_out) & 15) == 0 && (reinterpret_cast<uintptr_t>(op.d_residual) & 15) == 0,
              "pointwise conv: pointers must be 16-byte aligned");
  tc->pw = NC;
  tc->Cin = op.c;
  tc->M_total = op.n * op.ho * op.wo;
  tc->Cout = op.k; tc->Ho = op.ho; tc->Wo = op.wo; tc->stride = op.stride; tc->pad = 0; tc->R = 1; tc->S = 1;
  tc->cchunks = op.c / kBlockK;
  tc->relu = op.relu; tc->bias = op.d_bias; tc->residual = op.sc_c ? nullptr : op.d_residual; tc->out = op.d_out; tc->out_f32 = 0;
  tc->n_images = op.n;
  tc->im2col = op.stride != 1;
  tc->k3 = 0; tc->bias3 = nullptr; tc->out3 = nullptr;
  tc->sc_kb = op.sc_c / kBlockK; tc->sc_im2col = 0;
  if (tc->im2col) {
    if (int rc = encode_im2col(&tc->tmap_a, op)) return rc;
  } else {
    if (int rc = encode_2d(&tc->tmap_a, op.d_in, (uint64_t)tc->M_total, (uint64_t)op.c, kBlockM)) return rc;
  }
  if (op.sc_c) {        // shortcut segment: d_residual is the block input x [N, sc_h, sc_w, sc_c], read at stride 1 or 2
    const int sc_h = op.sc_hw >> 16, sc_w = op.sc_hw & 0xffff;
    PDF_REQUIRE(op.stride == 1 && op.d_residual && (reinterpret_cast<uintptr_t>(op.d_residual) & 15) == 0,
                "pointwise conv: a shortcut segment needs a stride-1 host convolution and d_residual = x, 16-byte aligned");
    pdf_op xs = op;
    xs.d_in = op.d_residual; xs.h = sc_h; xs.w = sc_w; xs.c = op.sc_c;
    if (sc_h == op.ho && sc_w == op.wo) {
      if (int rc = encode_2d(&tc->tmap_sc, op.d_residual, (uint64_t)tc->M_total, (uint64_t)op.sc_c, kBlockM)) return rc;
    } else {
      xs.stride = 2; xs.ho = op.ho; xs.wo = op.wo;
      tc->sc_im2col = 1;
      if (int rc = encode_im2col(&tc->tmap_sc, xs)) return rc;
    }
  }
  // weight-multicast CTA pairs (see the kernel): where the weight tiles are a large share of a unit's ring traffic
  tc->pw_mc = (g_pw_mc && NC == 128 && op.c >= 128 && (!op.d_weight3 || op.k3 % 2 == 0)) ? 1 : 0;
  const uint64_t k_total = (uint64_t)op.c + (uint64_t)op.sc_c;     // weights [K][c + sc_c]: conv3's columns, then the shortcut's
  if (int rc = encode_2d(&tc->tmap_b, op.d_weight, (uint64_t)op.k, k_total, (uint32_t)(tc->pw_mc ? NC / 2 : NC))) return rc;
  if (int rc = encode_2d(&tc->tmap_out, op.d_out, (uint64_t)tc->M_total, (uint64_t)op.k, kBlockM)) return rc;
  if (tc->residual)
    if (int rc = encode_2d(&tc->tmap_res, op.d_residual, (uint64_t)tc->M_total, (uint64_t)op.k, kBlockM)) return rc;
  if (op.d_weight3) {
    PDF_REQUIRE(NC == 128 && (op.k3 == 64 || op.k3 == 128 || op.k3 == 256) && op.d_out3 &&
                (reinterpret_cast<uintptr_t>(op.d_weight3) & 15) == 0 && (reinterpret_cast<uintptr_t>(op.d_out3) & 31) == 0,
                "pointwise conv: a chained 1x1 convolution needs Cout %% 128 == 0, k3 in {64,128,256} and aligned pointers");
    tc->k3 = op.k3; tc->bias3 = op.d_bias3; tc->out3 = op.d_out3;
    if (int rc = encode_2d(&tc->tmap_w3, op.d_weight3, (uint64_t)op.k3, (uint64_t)op.k, (uint32_t)(tc->pw_mc ? op.k3 / 2 : op.k3))) return rc;
  }
  return PDF_OK;
}

template <int NC, bool CHAIN, bool MC>
static int launch_pw(const TcConv& tc, cudaStream_t s) {
  using L = PwSmem<NC>;
  // measured (profiles/r02_pw_cfg.txt): launches that fetch a residual tile want the third staging buffer (the residual of unit
  // u+1 streams in while unit u is still in its buffer), the others the fourth ring stage.  Launches with a shortcut segment fetch
  // no residual and run a 2-4x longer k-loop: they want the fourth ring stage also when chained (profiles/r03_pw_cfg_shortcut.txt)
  const bool wants_staging = tc.residual != nullptr || (CHAIN && !tc.sc_kb);
  int stages = g_pw_stages ? g_pw_stages : (wants_staging ? 3 : 4), nry = g_pw_ry ? g_pw_ry : (wants_staging ? 3 : 2);
  // the bias vector is staged in shared memory when it fits next to the requested ring; a deeper ring wins over bias staging
  // (the epilogue then reads the bias through L1), and the ring shrinks only when even that does not fit
  int bias_floats = tc.Cout;
  if (L::dynamic_bytes(stages, nry, bias_floats) > 227 * 1024 && tc.bias != nullptr) bias_floats = 0;
  while (L::dynamic_bytes(stages, nry, bias_floats) > 227 * 1024 && stages > 2) --stages;
  const int smem = L::dynamic_bytes(stages, nry, bias_floats);
  static int configured = 0;
  if (smem > configured) {
    PDF_CHECK_CUDA(cudaFuncSetAttribute(conv_pw_kernel<NC, CHAIN, MC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  PwParams p;
  p.stages = stages; p.nry = nry; p.bias_staged = bias_floats > 0 || tc.bias == nullptr;
  p.l2_prefetch = g_pw_prefetch;
  p.M_total = tc.M_total; p.Cout = tc.Cout; p.K = tc.Cin + tc.sc_kb * kBlockK; p.n_chunks = tc.Cout / NC; p.m_tiles = ceil_div(tc.M_total, kBlockM);
  p.relu = tc.relu; p.im2col = tc.im2col; p.has_res = tc.residual != nullptr;
  p.Ho = tc.Ho; p.Wo = tc.Wo; p.stride = tc.stride;
  p.kb_main = tc.Cin / kBlockK; p.sc_im2col = tc.sc_im2col; p.sc_stride = tc.sc_im2col ? 2 : 1;
  p.N2 = tc.k3; p.bias = tc.bias; p.bias3 = tc.bias3; p.out3 = reinterpret_cast<__nv_bfloat16*>(tc.out3);
  int grid = max(1, min(p.m_tiles, num_sms()));
  if (MC) grid = max(2, min((p.m_tiles + 1) / 2 * 2, num_sms() / 2 * 2));      // whole clusters of two CTAs
  const CUtensorMap& ta = *reinterpret_cast<const CUtensorMap*>(&tc.tmap_a);
  const CUtensorMap& tb = *reinterpret_cast<const CUtensorMap*>(&tc.tmap_b);
  const CUtensorMap& to = *reinterpret_cast<const CUtensorMap*>(&tc.tmap_out);
  const CUtensorMap& tr = p.has_res ? *reinterpret_cast<const CUtensorMap*>(&tc.tmap_res) : to;
  const CUtensorMap& tw = CHAIN ? *reinterpret_cast<const CUtensorMap*>(&tc.tmap_w3) : tb;
  const CUtensorMap& tsc = tc.sc_kb ? *reinterpret_cast<const CUtensorMap*>(&tc.tmap_sc) : ta;
  if (MC) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kPwThreads); cfg.dynamicSmemBytes = (size_t)smem; cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2; attr[1].val.clusterDim.y = 1; attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 2;
    PDF_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_pw_kernel<NC, CHAIN, MC>, ta, tb, to, tr, tw, tsc, p));
  } else {
    PDF_CHECK_CUDA(launch_pdl(conv_pw_kernel<NC, CHAIN, MC>, dim3(grid), dim3(kPwThreads), (size_t)smem, s, ta, tb, to, tr, tw, tsc, p));
  }
  PDF_CHECK_LAUNCH();
  return PDF_OK;
}

int launch_conv_pw(const TcConv& tc, cudaStream_t s) {
  if (tc.pw == 128 && tc.pw_mc) return tc.k3 ? launch_pw<128, true, true>(tc, s) : launch_pw<128, false, true>(tc, s);
  if (tc.pw == 128) return tc.k3 ? launch_pw<128, true, false>(tc, s) : launch_pw<128, false, false>(tc, s);
  if (tc.pw == 64) return launch_pw<64, false, false>(tc, s);
  set_error("launch_conv_pw: bad chunk width %d", tc.pw);
  return PDF_ERR_ARG;
}

}  // namespace pdf

/* tuning / A-B hook: 0 = 1x1 convolutions stay on conv_tc_kernel, 1 = default policy, 2 = every eligible 1x1 convolution uses
 * conv_pw_kernel.  Takes effect for plans created afterwards. */
extern "C" int pdf_debug_set_pw_config(int stages, int staging_buffers) {
  if (stages == 0 && staging_buffers == 0) { pdf::g_pw_stages = pdf::g_pw_ry = 0; return PDF_OK; }   // back to the defaults
  if (stages < 2 || stages > pdf::kPwMaxStages || staging_buffers < 2 || staging_buffers > pdf::kPwMaxRy) {
    pdf::set_error("pdf_debug_set_pw_config: stages in [2,%d], staging buffers in [2,%d]", pdf::kPwMaxStages, pdf::kPwMaxRy);
    return PDF_ERR_ARG;
  }
  pdf::g_pw_stages = stages; pdf::g_pw_ry = staging_buffers;
  return PDF_OK;
}
/* 0 (default) = single CTAs everywhere, 1 = weight-multicast CTA pairs for the pointwise launches with Cin >= 128 (measured neutral).
 * Takes effect for plans created afterwards. */
extern "C" int pdf_debug_set_pw_multicast(int enable) {
  pdf::g_pw_mc = enable != 0;
  return PDF_OK;
}
extern "C" int pdf_debug_set_pw_prefetch(int enable) {
  pdf::g_pw_prefetch = enable != 0;
  return PDF_OK;
}
extern "C" int pdf_debug_set_pw(int mode) {
  pdf::g_pw_mode = mode;
  return PDF_OK;
}

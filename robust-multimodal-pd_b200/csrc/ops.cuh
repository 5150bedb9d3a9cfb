// Internal launch entry points shared by plan.cu.
#pragma once
#include "common.cuh"

namespace pdf {

int launch_conv_f32(const pdf_op& op, cudaStream_t s);
int launch_maxpool(const pdf_op& op, cudaStream_t s);
int launch_avgpool(const pdf_op& op, cudaStream_t s);
int launch_stem_im2col(const pdf_op& op, cudaStream_t s);


// tcgen05 path: one prepared launch per bf16 conv op (tensor maps are 128-byte opaque blobs)
struct alignas(64) TensorMapBlob { unsigned char bytes[128]; };

struct TcConv {
  TensorMapBlob tmap_a, tmap_b;
  TensorMapBlob tmap_b2;   // weight map with a [BLOCK_N/2 x 64] box (one CTA's half of B in the CTA-pair kernel)
  TensorMapBlob tmap_ds;   // dual kernel: weights [Cout, Cin] of the fused 1x1 convolution
  int dual;                // 1: the launch also computes that 1x1 convolution of the same input (centre-tap tiles) into out2
  const float* bias2;
  void* out2;
  int block_n;      // 64 | 128 | 256
  int im2col;       // 1: A through im2col-mode TMA, 0: plain 2D tile of the [M, C] matrix (1x1 stride-1)
  int M_total, Cout, Ho, Wo, stride, pad, R, S, cchunks, relu;
  const float* bias;
  const void* residual;   // bf16 [M, Cout]
  void* out;              // bf16 [M, Cout] or f32 when out_f32
  int out_f32;
  int hs;                 // 1: horizontally-shared 3x3 stride-1 kernel (conv3x3_hs.cu); tmap_a traverses W+2 positions per row
  int halo;               // 1: halo-resident 3x3 kernel (conv3x3_tc.cu); tmap_a is then a 4-D tiled map
  int halo_wp, halo_nr, n_images;
  // pointwise kernel (conv_pw.cu): 1x1 convolution whose epilogue goes through shared memory (TMA residual load, TMA store),
  // optionally chained with the NEXT 1x1 convolution (out3 = relu(out * W3^T + bias3)) while the output tile is still on chip
  int pw;                  // 0 | NC (64 or 128): the launch goes to conv_pw_kernel<NC, ...>
  int pw_mc;               // 1: weight-multicast CTA pairs (tmap_b / tmap_w3 boxes hold half the rows)
  int Cin;
  TensorMapBlob tmap_out, tmap_res, tmap_w3;
  int k3;                  // chained output channels (0 = no chain)
  const float* bias3;
  void* out3;
  // shortcut segment (Bottleneck projection shortcut computed as the last k-blocks of conv3's GEMM): Cin counts conv3's own channels
  TensorMapBlob tmap_sc;   // block input x: 2-D [M, sc_c] map at stride 1, im2col-mode map at stride 2
  int sc_kb;               // k-blocks of the shortcut segment (0 = none)
  int sc_im2col;
};

int load_driver_entry_points();
// [rows, cols] row-major bf16 matrix, box = [box_rows x 64 cols], 128-byte swizzle
int encode_2d(TensorMapBlob* out, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
int encode_im2col(TensorMapBlob* out, const pdf_op& op, int extra_w = 0, int pixels = 128);
int prepare_conv_tc(const pdf_op& op, TcConv* out);
int prepare_stem_tc(const pdf_op& op, TcConv* out);   // weight map -> out->tmap_b, padded-image patch map -> out->tmap_a
int launch_stem_fused(const pdf_op& op, const TensorMapBlob& tmap_w, const TensorMapBlob& tmap_in, cudaStream_t s);
int launch_conv_tc(const TcConv& tc, cudaStream_t s);
bool pair_eligible(const TcConv& tc);
int launch_conv_tc2(const TcConv& tc, cudaStream_t s);   // cta_group::2 pair kernel (conv_tc2.cu)
int launch_umma2_rate(int N, int iters, int mode, int pairs, unsigned long long* d_cycles, cudaStream_t s);   // probe
bool halo_eligible(const pdf_op& op);
bool hs_eligible(const pdf_op& op);
int launch_conv3x3_hs(const TcConv& tc, cudaStream_t s);
int launch_conv3x3_halo(const TcConv& tc, cudaStream_t s);
// tcgen05 kind::tf32 GEMM on f32 operands (mil_tc.cu): mode 0 out[M,N] = relu(A B^T + bias); mode 1 out[M] = attention score
bool gemm_tf32_supported(int N, int K);
int launch_gemm_tf32(const float* A, const float* B, int M, int N, int K, int mode, int gated, int A_dim, const float* bias,
                     const float* w_w, const float* b_w, float* out, cudaStream_t s);
// FP32 FFMA GEMM C[M,N] = A[M,K] B[N,K]^T (+bias) (ReLU) of the MIL head (heads.cu: gemm_nt_f32_kernel); also used by explain.cu so
// that explanations see the same h and attention pre-activations as pdf_mil_sweep's FP32 path
int gemm_nt(const float* A, int lda, const float* B, int ldb, float* C, int ldc, const float* bias, int M, int N, int K, int relu,
            cudaStream_t s);
// Fusion heads (heads.cu), shared with their explanations (fusion_explain.cu).  check_*: the sweeps' argument checks.
// moddrop_partials: partials[m] = x_m W1_m^T [N, h1] per modality of nonzero width (layer 1 without bias).
// moddrop_eval: layers 2.. under S scenario masks -> prob [S, N]; coalitions = true: under all 2^M coalitions (mask_m = (c >> m) & 1,
// masks not read) -> logit [2^M, N].  The kernel (tiled or warp per pair) is the one pdf_moddrop_sweep picks for sweep_pairs pairs.
// moe_eval: router, experts and gated sum under S scenario masks -> [S, N]; router_w != NULL: under all 2^E coalitions instead, and
// router_w [2^E, E] receives the router weights of every coalition.
int check_mlp(const pdf_mlp& m, const char* what);
int check_moddrop(const pdf_mlp& net, const char* what);
int check_moe(const pdf_moe& net, const float* const* d_x, const char* what);
int moddrop_partials(const pdf_mlp& net, int N, const float* d_x, float* partials, cudaStream_t s);
int moddrop_eval(const pdf_mlp& net, int N, int S, const float* partials, const uint8_t* masks, bool coalitions, long long sweep_pairs,
                 float* out, cudaStream_t s);
int moe_eval(const pdf_moe& net, const float* const* d_x, int N, int S, const uint8_t* masks, float* router_w, float* out, cudaStream_t s);
bool pw_eligible(const pdf_op& op);
int prepare_conv_pw(const pdf_op& op, TcConv* tc);
int launch_conv_pw(const TcConv& tc, cudaStream_t s);

}  // namespace pdf

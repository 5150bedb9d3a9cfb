// Shared-memory FFMA tiles of MLP rows, shared by the explanations (fusion_explain.cu) and the Monte-Carlo dropout kernels
// (uncertainty.cu).
#pragma once
#include <algorithm>

#include "common.cuh"

namespace pdf {

constexpr size_t kMlpTileSmemMax = 227 * 1024;

// ------------------------------------------------------------------------------------------------------
// One linear layer on the rows of a tile: out(r, c) = sum_k in[r][k] W(k, c), k ascending, 64-column x 16-k weight chunks in shared
// memory, a 16 x 16 thread grid with RT rows x 4 columns each (moddrop_tile_kernel's loop).  kBackward = false: W(k, c) = W[c * n_in + k]
// (the forward x W^T, W [n_out, n_in]); true: W(k, c) = W[k * n_out + c] (delta W, W [n_in, n_out]).  epi(r, c, acc) takes every
// valid output; it may overwrite any buffer but `in`.  kQuad: epi(r, c, acc4) instead takes a thread's four consecutive columns
// c .. c+3 (c a multiple of 4; those >= n_out hold 0 and must be ignored) at once.
template <int RT, bool kBackward, bool kQuad = false, typename Epi>
__device__ __forceinline__ void tile_layer(const float* in, int in_stride, const float* __restrict__ W, int n_in, int n_out, float* Ws,
                                           Epi epi) {
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  for (int c0 = 0; c0 < n_out; c0 += 64) {
    float acc[RT][4];
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < n_in; k0 += 16) {
      if (!kBackward) {
        const int col = c0 + (tid >> 2), kk = (tid & 3) * 4;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          Ws[(kk + e) * 68 + (tid >> 2)] = (col < n_out && k0 + kk + e < n_in) ? __ldg(W + (size_t)col * n_in + k0 + kk + e) : 0.f;
      } else {
        const int kk = tid >> 4, cc = (tid & 15) * 4;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          Ws[kk * 68 + cc + e] = (c0 + cc + e < n_out && k0 + kk < n_in) ? __ldg(W + (size_t)(k0 + kk) * n_out + c0 + cc + e) : 0.f;
      }
      __syncthreads();
      const int kmax = min(16, n_in - k0);
      for (int kk = 0; kk < kmax; ++kk) {
        float a[RT], b[4];
#pragma unroll
        for (int i = 0; i < RT; ++i) a[i] = in[(ty * RT + i) * in_stride + k0 + kk];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = Ws[kk * 68 + tx * 4 + j];
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
    if constexpr (kQuad) {
#pragma unroll
      for (int i = 0; i < RT; ++i)
        if (c0 + tx * 4 < n_out) epi(ty * RT + i, c0 + tx * 4, acc[i]);
    } else {
#pragma unroll
      for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (c0 + tx * 4 + j < n_out) epi(ty * RT + i, c0 + tx * 4 + j, acc[i][j]);
    }
  }
}

// The widest tile (64, 32 or 16 rows) of an MLP's (row, layer) activations that fits 227 KB: the 16 x 68 weight chunk, one float per
// row, and every hidden layer's activations [rows][width + 1] one after the other (the logit's [rows][2], for a one-layer net).
inline int mlp_tile(const pdf_mlp& net, int* tp, size_t* smem, const char* what) {
  size_t widths = 0;
  for (int l = 1; l <= std::max(net.n_layers - 1, 1); ++l) widths += (size_t)net.dims[l] + 1;
  for (int t = 64; t >= 16; t /= 2) {
    const size_t b = (16 * 68 + (size_t)t + (size_t)t * widths) * sizeof(float);
    if (b <= kMlpTileSmemMax) {
      *tp = t;
      *smem = b;
      return PDF_OK;
    }
  }
  set_error("%s: hidden layers too wide for the shared-memory tile (%zu activations per row; 16 rows need more than 227 KB)", what,
            widths);
  return PDF_ERR_ARG;
}

}  // namespace pdf

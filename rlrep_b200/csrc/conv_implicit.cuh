// Implicit "full correlation" of a 32-channel NHWC map with a 3x3 kernel on the tcgen05 GEMM (see conv_implicit.cu):
// the shared core of the encoder's data gradient (conv.cu) and the decoder's stride-1 transposed convolutions
// (deconv.cu).
#pragma once
#include "agent.cuh"

namespace rlrep {

// Scratch for one full correlation at a time: the zero-padded input grid, the output grid and the repacked weights.
// K groups of the implicit weight-gradient GEMM (GemmArgs::k_groups), measured at B = 256: 1 and 2 groups 131 us, 4 groups
// 117 us
constexpr int kWgradGroups = 4;
constexpr int kScatterMaxBlocks = kNumSMs * 16;  // grid cap of the scatter pass (its per-CTA column partials)
struct FullCorrScratch {
  float *padded = nullptr, *out_grid = nullptr, *w_flip = nullptr, *wfold = nullptr, *colsum_partial = nullptr;
  void want(DeviceArena& a, int batch, int max_hi) {
    const size_t rows = (size_t)batch * (max_hi + 4) * (max_hi + 4);
    a.want(&padded, rows * 32);
    a.want(&out_grid, rows * 32);
    a.want(&w_flip, 32 * 288);
    a.want(&wfold, kWgradGroups * 128 * 768);
    a.want(&colsum_partial, (size_t)kScatterMaxBlocks * 32);
  }
};

enum FullCorrWeights : int {
  FC_CONV_DGRAD = 0,   // W is a conv weight [32 (co), (ky, kx, ci)]: out channel n = ci, contraction over co
  FC_DECONV_FWD = 1,   // W is a transposed-conv weight [(ky, kx, co), ci]: out channel n = co, contraction over ci
};

// out[b, oy, ox, n] = act(bias[n] + sum_{ky, kx, c} in[b, oy - ky, ox - kx, c] * Wt[n, (ky, kx), c]) * (mask > 0),
// in [B, Hi, Hi, 32] (zero outside), out / mask [B, Hi + 2, Hi + 2, 32]; bias and mask may be null.
void full_correlation_3x3(GemmRunner& g, cudaStream_t s, int B, int Hi, const float* in, const float* W, int weights,
                          const float* bias, int act, const float* mask, float* out, FullCorrScratch& scratch);

// Weight gradient of a 3x3 valid convolution / stride-1 transposed convolution without a column matrix:
//   G[n, (ky, kx), c] = sum_{b, y, x} small[b, y, x, n] * map[b, y + ky, x + kx, c]
// small [B, Hg - 2, Hg - 2, 32] (the convolution's output gradient, or the transposed convolution's input), map
// [B, Hg, Hg, 32] (the convolution's input, or the transposed convolution's output gradient) FOLLOWED BY 2 Hg + 5 readable
// rows of finite values.  `small` is copied onto the map's grid (zero outside) and folded four rows to one; the GEMM's TMA
// producer reads `map` through the shifted view of GemmArgs::conv_wgrad_hi.  Tensor-core path only; B % 4 == 0.
// transposed = false writes dW[n * ld + (ky * 3 + kx) * 32 + c], true writes dW[((ky * 3 + kx) * 32 + c) * ld + n].
// small_colsum != nullptr: also small_colsum[n] = sum over pixels of small[., n] -- the convolution's bias gradient, a
// by-product of the pass that copies `small` onto the grid (saves a separate read of the gradient map).
void conv3x3_wgrad_implicit(GemmRunner& g, cudaStream_t s, int B, int Hg, const float* small, const float* map, float* dW,
                            int ld_dw, bool transposed, FullCorrScratch& scratch, float* small_colsum = nullptr);

// Forward pass of a STRIDE-2 3x3 transposed convolution (+ bias + ReLU) without the [rows, 288] column matrix:
//   out[b, oy, ox, co] = relu(bias[co] + sum over (ky, kx) with oy - ky = 2 iy, ox - kx = 2 ix of in[b, iy, ix, :] . W[(ky, kx, co), :])
// in [B, Hi, Hi, 32], out [B, Ho, Ho, 32] (Ho = 2 Hi + 1 or 2 Hi + 2), W [288, 32] = [(ky, kx, co), ci].  The four output
// parity classes (oy % 2, ox % 2) are four stride-1 problems with 4 / 2 / 2 / 1 taps on the zero-padded input grid: four
// launches of the halo kernel with a tap list and a stride-2 compacting store.  Returns false (nothing launched) when the
// halo kernel does not take this shape / precision: the caller falls back to GEMM + col2im.
bool deconv3x3_s2_forward(GemmRunner& g, cudaStream_t s, int B, int Hi, int Ho, const float* in, const float* W,
                          const float* bias, float* out, FullCorrScratch& scratch);

// Valid 3x3 convolution of dY-like maps with MN-major weights, for the data gradient of a stride-1 transposed convolution:
// out[b, y, x, n] = (mask > 0) * sum_{ky, kx, c} in[b, y + ky, x + kx, c] * W[(ky * 3 + kx) * 32 + c, n], W [288, 32].
void valid_conv_3x3_wt(GemmRunner& g, cudaStream_t s, int B, int Hi, const float* in, const float* W, const float* mask,
                       float* out, FullCorrScratch& scratch);

// Valid 3x3 convolution of a dense NHWC map without a column matrix: out[b, oy, ox, n] = act(bias[n] + sum_{ky, kx, c}
// in[b, oy + ky, ox + kx, c] * W[n, (ky, kx), c]), in [B, Hi, Hi, 32], out [B, Hi - 2, Hi - 2, 32].  The GEMM runs on the
// input's own grid (rows whose window crosses the border are computed and dropped by the compaction).
void valid_conv_3x3(GemmRunner& g, cudaStream_t s, int B, int Hi, const float* in, const float* W, int ldw,
                    const float* bias, int act, float* out, FullCorrScratch& scratch);

}  // namespace rlrep

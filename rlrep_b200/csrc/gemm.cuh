// GEMM entry points of the library.
//
//   C[M,N] = epilogue( sum_k A(m,k) * B(n,k) )
//
// Operand addressing ("major" = which index is contiguous in memory):
//   K-major  A:  A(m,k) = A[m*lda + k]      (activations X[B,in], weights W[out,in] as used by y = x W^T)
//   MN-major A:  A(m,k) = A[k*lda + m]      (transposed views: dY^T in wgrad, W in dgrad)
// and the same for B with (n,k).  All three linear-layer passes map onto this one contraction:
//   forward  Y  = X  W^T : A = X  (K-major),  B = W  (K-major)
//   dgrad    dX = dY W   : A = dY (K-major),  B = W  (MN-major, k = out index)
//   wgrad    dW = dY^T X : A = dY (MN-major), B = X  (MN-major, k = batch index)
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "epilogue.cuh"

namespace rlrep {

struct GemmArgs {
  int M = 0, N = 0, K = 0;
  const float* A = nullptr;
  int lda = 0;
  bool a_mn = false;
  // Optional second K-segment of A (CUDA-core path, K-major A only): columns [K1, K) come from A2.
  // Lets first layers read cat(s, a) / cat(s', a') straight from two buffers without a concat pass.
  const float* A2 = nullptr;
  int lda2 = 0;
  int K1 = 0;
  // Implicit 3x3 convolution over an NHWC matrix (K-major A only): conv_w > 0 makes A a [M, 32] matrix of pixels on a
  // grid conv_w wide and k-block t (K = 9 * 32) reads rows m + (t / 3) * conv_w + (t % 3), i.e.
  //   C[m, n] = sum_{ky, kx, c} A[m + ky * conv_w + kx, c] * B(n, (ky * 3 + kx) * 32 + c)
  // with rows past M read as zero.  No column matrix is materialised: the TMA producer shifts its row coordinate.
  int conv_w = 0;
  // Implicit weight gradient of that convolution (tensor-core path, both operands MN-major): conv_wgrad_hi = Hi > 0 makes B
  // the convolution's INPUT, a dense [rows, 32] NHWC map on a grid Hi wide, read through the view
  //   B(k, n = ky * 256 + q * 32 + c) = X[4 k + q + ky * Hi, c],   q = 0..7 (6, 7: padding), ky = 0..2   (N = 768),
  // i.e. with A = the output gradient on the same grid folded four rows to one ([rows / 4, 128], zero where the window
  // leaves the image) the product C[(f, n), (ky, q, c)] holds dW[n, (ky, kx), c] = sum_f C[(f, n), (ky, kx + f, c)].
  // No column matrix exists; K = rows / 4, and 2 Hi + 7 rows of finite values must be readable behind the map (they meet
  // zeros of A, or land in the padding columns nobody reads).
  int conv_wgrad_hi = 0;
  // Compacting store of an implicit convolution (halo kernel only, GemmRunner::run_compact): the GEMM's rows live on a grid
  // compact_wp wide; only rows with x < compact_ho and y < compact_ho are stored, at row (b * ho + y) * ho + x of C -- and
  // of epi.aux / epi.pre_out, which are indexed by the compact row too.
  int compact_wp = 0, compact_ho = 0;
  // Generalisations used by the stride-2 transposed convolution (one launch per output parity class): the valid extent in x
  // (0: compact_ho), an output stride / offset -- grid (b, y, x) goes to output row (b * out_w + s*y + oy) * out_w + s*x + ox
  // (out_w = 0: compact_ho) -- and a subset / reordering of the nine taps: tap i reads rows shifted by conv_tap_shift[i]
  // and multiplies by weight k-block conv_tap_kb[i] (conv_ntaps = 0: the nine taps (ky, kx) -> shift ky * conv_w + kx).
  int compact_hx = 0, compact_stride = 1, compact_oy = 0, compact_ox = 0, compact_out_w = 0;
  int conv_ntaps = 0;
  int conv_tap_shift[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int conv_tap_kb[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  // K groups (tensor-core path, one tile per CTA): the K range is cut into k_groups parts, each reduced by its own split-K
  // cluster into its own output matrix -- k_groups matrices of ceil(M / 128) * 128 rows (pitch ldc) behind each other at C,
  // which the caller sums.  For GEMMs with K ~ 1e5 and a handful of tiles, where a cluster's 8 CTAs are not enough.
  int k_groups = 1;
  const float* B = nullptr;
  int ldb = 0;
  bool b_mn = false;
  float* C = nullptr;
  int ldc = 0;
  Epilogue epi;
};

// ---- tcgen05 path (TF32 inputs, FP32 accumulate in TMEM, TMA-fed) ----
struct TcGemmPlan {
  CUtensorMap tmA, tmB;
  GemmArgs args;
  int bn = 0;
  int split_k = 1;
  int kb_per_split = 0;
  int stages = 0;       // TMA ring depth (shallow for short K-slices so two CTAs share an SM)
  bool push = false;    // split-K partials pushed into the owner CTA's shared memory (see gemm_tc_kernel.cuh)
  bool persistent = false;  // one CTA per SM walks the tiles with a double-buffered TMEM accumulator (no split-K)
  int k_groups = 1;         // GemmArgs::k_groups as planned (1 when the K range is too short to cut)
  int halo_rows = 0;        // > 0: implicit convolution with the tile's halo in shared memory (gemm_conv_halo_kernel)
  float* ws = nullptr;  // unused (split-K reduces over DSMEM); kept for ABI stability of rlrep_gemm
};

// True when the operands satisfy TMA's constraints (16-byte aligned base, ld % 4 == 0, no A2 segment).
bool tc_eligible(const GemmArgs& a);
// bn / split_k = 0 picks them automatically from a cost model whose wave count comes from the occupancy API.
// sm_share in (0, 1]: fraction of the GPU this GEMM may count on (0.5 when two kernel chains run on two streams).
TcGemmPlan make_tc_plan(const GemmArgs& a, int bn, int split_k, float* ws, size_t ws_floats, double sm_share = 1.0);
void launch_tc(const TcGemmPlan& p, cudaStream_t stream);
// Debug builds (-DRLREP_GEMM_TRACE): %globaltimer stamps of CTA (0,0,0) of the last tcgen05 GEMM.
void read_gemm_trace(unsigned long long* out16);
// Debug aid: device buffer of 80 uint64 the persistent kernel's CTA 0 stamps its first 16 tiles into (nullptr = off).
void set_gemm_debug_buffer(unsigned long long* dev80);

// TMA descriptor of one GEMM operand over fp32 memory, typed TFLOAT32 (the TMA unit rounds on the way into shared
// memory): K-major = matrix [mn, K] with row pitch ld, box box_mn x 32, SWIZZLE_128B; MN-major = matrix [K, mn] viewed as
// (mn % 32, k, mn / 32), box {32, 32, box_mn / 32}, SWIZZLE_128B_ATOM_32B (see gemm_tc_kernel.cuh).
CUtensorMap make_operand_map(const float* base, bool mn_major, int mn, int K, int ld, int box_mn);

// ---- CUDA-core path (exact FP32 FFMA; small-K / small-N layers and the strict-fp32 mode) ----
void launch_simt(const GemmArgs& a, cudaStream_t stream);

}  // namespace rlrep

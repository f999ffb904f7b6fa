// Full correlation  out[oy, ox] = sum_taps in[oy - ky, ox - kx] W[ky, kx]  (the data gradient of a 3x3 convolution, and
// the forward pass of a stride-1 ConvTranspose2d) WITHOUT a column matrix.
//
// Version 1 ran it as  col = X W^T  ([B*Hi*Hi, 32] x [288, 32]^T, a K = 32 GEMM with 30k one-k-block tiles) followed by
// a gather-form col2im: ~500 us per layer at B = 256, 6x the HBM time of its traffic, because every 128 x 32 tile pays
// the whole TMA -> MMA -> epilogue latency for a single k-block.  Here the input is copied once onto a zero-padded
// grid (Hi + 4 wide, so that every tap of every valid output is an in-grid read), and the GEMM's TMA producer walks the
// nine taps by SHIFTING ITS ROW COORDINATE on that grid (GemmArgs::conv_w): one K = 288 GEMM, A re-read from L2 only,
// output on the same grid, then one compaction pass that also applies the ReLU mask.  Taps are visited in flipped
// order (t -> 8 - t) so all shifts are non-negative; the weights are repacked to match ([32, 9 * 32], 37 KB).
#include "conv_implicit.cuh"
#include "kernels.cuh"

#include <algorithm>

namespace rlrep {

namespace {

int grid_for(long long work, int threads) {
  const long long want = (work + threads - 1) / threads;
  return (int)std::max<long long>(1, std::min<long long>(want, (long long)kNumSMs * 16));
}

// padded[b, y, x] = in[b, y - 2, x - 2] inside, zero on the two-pixel frame; Wp = Hi + 4
__global__ void pad_grid_kernel(const float4* __restrict__ in, int B, int Hi, float4* __restrict__ padded) {
  const int Wp = Hi + 4;
  const long long total = (long long)B * Wp * Wp * 8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i & 7);
    const long long pix = i >> 3;
    const int x = (int)(pix % Wp) - 2, y = (int)((pix / Wp) % Wp) - 2, b = (int)(pix / ((long long)Wp * Wp));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (x >= 0 && x < Hi && y >= 0 && y < Hi) v = in[(((long long)b * Hi + y) * Hi + x) * 8 + c4];
    padded[i] = v;
  }
}

// w_flip[n, t * 32 + c] = Wt[n, 8 - t, c] for the two weight layouts (conv_implicit.cuh)
__global__ void repack_flip_kernel(const float* __restrict__ W, int weights, float* __restrict__ w_flip) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 32 * 288) return;
  const int n = i / 288, r = i - n * 288, t = r >> 5, c = r & 31;
  const int tap = 8 - t;
  w_flip[i] = weights == FC_CONV_DGRAD ? W[c * 288 + tap * 32 + n] : W[(tap * 32 + n) * 32 + c];
}

// w_rep[co, t * 32 + ci] = W[(t * 32 + co) * 32 + ci]: the transposed-conv weight [(ky, kx, co), ci] as nine K-major k-blocks
__global__ void repack_deconv_kernel(const float* __restrict__ W, float* __restrict__ w_rep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 32 * 288) return;
  const int co = i / 288, r = i - co * 288, t = r >> 5, ci = r & 31;
  w_rep[i] = W[(t * 32 + co) * 32 + ci];
}

// out[b, y, x] = grid[b, y, x] (y, x < Ho) * (mask > 0)
__global__ void compact_grid_kernel(const float4* __restrict__ grid, int B, int Wp, int Ho, const float4* __restrict__ mask,
                                    float4* __restrict__ out) {
  const long long total = (long long)B * Ho * Ho * 8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i & 7);
    const long long pix = i >> 3;
    const int x = (int)(pix % Ho), y = (int)((pix / Ho) % Ho), b = (int)(pix / ((long long)Ho * Ho));
    float4 v = grid[(((long long)b * Wp + y) * Wp + x) * 8 + c4];
    if (mask != nullptr) {
      const float4 m = mask[i];
      v = make_float4(m.x > 0.f ? v.x : 0.f, m.y > 0.f ? v.y : 0.f, m.z > 0.f ? v.z : 0.f, m.w > 0.f ? v.w : 0.f);
    }
    out[i] = v;
  }
}

// in [B, Hs, Hs, 32] onto a grid Hg wide (zero outside); colsum_partial != nullptr: per-CTA column sums of `in` as well
// ([gridDim.x][32], fixed order inside the CTA) -- every element of `in` is read exactly once by this pass
__global__ void __launch_bounds__(256) scatter_to_grid_kernel(const float4* __restrict__ in, int B, int Hs, int Hg,
                                                              float4* __restrict__ grid, float* __restrict__ colsum_partial) {
  __shared__ float4 part[32][8];
  const long long total = (long long)B * Hg * Hg * 8;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i & 7);
    const int pix = (int)(i >> 3);
    const int b = pix / (Hg * Hg), rem = pix - b * Hg * Hg, y = rem / Hg, x = rem - y * Hg;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (x < Hs && y < Hs) v = in[(((long long)b * Hs + y) * Hs + x) * 8 + c4];
    grid[i] = v;
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  if (colsum_partial == nullptr) return;
  part[threadIdx.x >> 3][threadIdx.x & 7] = acc;  // the grid-stride step is a multiple of 8: a thread keeps its columns
  __syncthreads();
  if (threadIdx.x < 8) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q = 0; q < 32; ++q) {
      const float4 a = part[q][threadIdx.x];
      t.x += a.x; t.y += a.y; t.z += a.z; t.w += a.w;
    }
    reinterpret_cast<float4*>(colsum_partial + (size_t)blockIdx.x * 32)[threadIdx.x] = t;
  }
}
// G[n, (ky, kx), c] = sum_f C[(f, n), (ky, kx + f, c)] over the four folded rows, C [128, 768] (fixed order)
__global__ void diag_tap_sum_kernel(const float* __restrict__ C, int groups, float* __restrict__ dW, int ld_dw,
                                    int transposed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 32 * 288) return;
  const int n = i / 288, r = i - n * 288, t = r >> 5, c = r & 31, ky = t / 3, kx = t - 3 * ky;
  float acc = 0.f;
  for (int g = 0; g < groups; ++g)  // the GEMM's K groups, then the four folded rows: fixed order
    for (int f = 0; f < 4; ++f)
      acc += C[(size_t)g * 128 * 768 + (size_t)(f * 32 + n) * 768 + ky * 256 + (kx + f) * 32 + c];
  if (transposed) dW[(size_t)r * ld_dw + n] = acc;
  else dW[(size_t)n * ld_dw + r] = acc;
}

}  // namespace

void conv3x3_wgrad_implicit(GemmRunner& g, cudaStream_t s, int B, int Hg, const float* small, const float* map, float* dW,
                            int ld_dw, bool transposed, FullCorrScratch& sc, float* small_colsum) {
  const long long rows = (long long)B * Hg * Hg;
  RLREP_CHECK(rows % 4 == 0 && rows * 8 < (1LL << 31), "implicit weight gradient: batch must be a multiple of 4 (and < 2^28 pixels)");
  // with column partials: 4 CTAs per SM -- the second stage is one CTA walking [blocks][32] partials (8 us for 2,368)
  const int blocks = small_colsum != nullptr ? std::min(grid_for(rows * 8, 256), kNumSMs * 4) : grid_for(rows * 8, 256);
  RLREP_CHECK(blocks <= kScatterMaxBlocks, "scatter grid larger than its partial buffer");
  scatter_to_grid_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<const float4*>(small), B, Hg - 2, Hg,
                                              reinterpret_cast<float4*>(sc.padded),
                                              small_colsum != nullptr ? sc.colsum_partial : nullptr);
  RLREP_LAUNCHED_W("scatter_to_grid", s, 4.0 * 32 * ((double)B * (Hg - 2) * (Hg - 2) + rows), 0.0);
  if (small_colsum != nullptr) launch_colsum_finish(sc.colsum_partial, blocks, 32, small_colsum, s);
  GemmArgs a;
  a.M = 128; a.N = 768; a.K = (int)(rows / 4);
  a.A = sc.padded; a.lda = 128; a.a_mn = true;
  a.B = map; a.ldb = 128; a.b_mn = true;
  a.conv_wgrad_hi = Hg;
  a.C = sc.wfold; a.ldc = 768;
  // nine or eighteen tiles x a split-K cluster of 8 leave half the GPU idle and every CTA with ~10 MB to stream: cut K
  // into groups with their own output matrices (summed by diag_tap_sum)
  a.k_groups = kWgradGroups;
  const int groups = (a.k_groups > 1 && ceil_div(a.K, 32) >= 64 * a.k_groups) ? a.k_groups : 1;  // make_tc_plan's rule
  g.run(a, s);
  diag_tap_sum_kernel<<<ceil_div(32 * 288, 256), 256, 0, s>>>(sc.wfold, groups, dW, ld_dw, transposed ? 1 : 0);
  RLREP_LAUNCHED("diag_tap_sum", s);
}

bool deconv3x3_s2_forward(GemmRunner& g, cudaStream_t s, int B, int Hi, int Ho, const float* in, const float* W,
                          const float* bias, float* out, FullCorrScratch& sc) {
  const int Wp = Hi + 4;
  const long long rows = (long long)B * Wp * Wp;
  GemmArgs a;
  a.M = (int)rows; a.N = 32; a.K = 288;
  a.A = sc.padded; a.lda = 32; a.conv_w = Wp;
  a.B = sc.w_flip; a.ldb = 288;
  a.C = out; a.ldc = 32;
  a.epi.bias = bias;
  a.epi.act = ACT_RELU;
  a.compact_stride = 2;
  a.compact_out_w = Ho;
  for (int par = 0; par < 4; ++par) {
    const int py = par >> 1, px = par & 1;
    GemmArgs c = a;
    c.compact_oy = py; c.compact_ox = px;
    const int hy = (Ho - py + 1) / 2, hx = (Ho - px + 1) / 2;  // outputs oy = 2 y + py < Ho
    c.compact_hx = hx;
    // taps: ky = py + 2 dy (dy = 0, 1 while ky <= 2) reads in[y - dy] = padded[y + 2 - dy]
    int n = 0;
    for (int dy = 0; py + 2 * dy <= 2; ++dy)
      for (int dx = 0; px + 2 * dx <= 2; ++dx) {
        c.conv_tap_shift[n] = (2 - dy) * Wp + (2 - dx);
        c.conv_tap_kb[n] = (py + 2 * dy) * 3 + (px + 2 * dx);
        ++n;
      }
    c.conv_ntaps = n;
    if (par == 0) {
      // probe first: nothing is launched (not even the padding pass) unless the halo kernel takes this GEMM
      if (!g.compact_supported(c, Wp, hy)) return false;
      pad_grid_kernel<<<grid_for(rows * 8, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(in), B, Hi,
                                                             reinterpret_cast<float4*>(sc.padded));
      RLREP_LAUNCHED_W("pad_grid", s, 4.0 * 32 * ((double)B * Hi * Hi + rows), 0.0);
      repack_deconv_kernel<<<ceil_div(32 * 288, 256), 256, 0, s>>>(W, sc.w_flip);
      RLREP_LAUNCHED("repack_deconv", s);
    }
    RLREP_CHECK(g.run_compact(c, Wp, hy, s), "stride-2 transposed convolution: the halo kernel refused a parity class");
  }
  return true;
}

void valid_conv_3x3_wt(GemmRunner& g, cudaStream_t s, int B, int Hi, const float* in, const float* W, const float* mask,
                       float* out, FullCorrScratch& sc) {
  const int Ho = Hi - 2;
  GemmArgs a;
  a.M = B * Hi * Hi; a.N = 32; a.K = 288;
  a.A = in; a.lda = 32; a.conv_w = Hi;
  a.B = W; a.ldb = 32; a.b_mn = true;
  a.ldc = 32;
  {  // the halo kernel stores the valid rows at their compact positions (x mask) itself
    GemmArgs c = a;
    c.C = out;
    if (mask != nullptr) { c.epi.dact = DACT_RELU_OUT; c.epi.aux = mask; c.epi.ld_aux = 32; }
    if (g.run_compact(c, Hi, Ho, s)) return;
  }
  a.C = sc.out_grid;
  g.run(a, s);
  compact_grid_kernel<<<grid_for((long long)B * Ho * Ho * 8, 256), 256, 0, s>>>(
      reinterpret_cast<const float4*>(sc.out_grid), B, Hi, Ho, reinterpret_cast<const float4*>(mask),
      reinterpret_cast<float4*>(out));
  RLREP_LAUNCHED_W("compact_grid", s, 4.0 * 32 * ((double)B * Ho * Ho * (mask ? 3 : 2)), 0.0);
}

void full_correlation_3x3(GemmRunner& g, cudaStream_t s, int B, int Hi, const float* in, const float* W, int weights,
                          const float* bias, int act, const float* mask, float* out, FullCorrScratch& sc) {
  const int Wp = Hi + 4, Ho = Hi + 2;
  const long long rows = (long long)B * Wp * Wp;
  pad_grid_kernel<<<grid_for(rows * 8, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(in), B, Hi,
                                                         reinterpret_cast<float4*>(sc.padded));
  RLREP_LAUNCHED_W("pad_grid", s, 4.0 * 32 * ((double)B * Hi * Hi + rows), 0.0);
  repack_flip_kernel<<<ceil_div(32 * 288, 256), 256, 0, s>>>(W, weights, sc.w_flip);
  RLREP_LAUNCHED("repack_flip", s);
  GemmArgs a;
  a.M = (int)rows; a.N = 32; a.K = 288;
  a.A = sc.padded; a.lda = 32; a.conv_w = Wp;
  a.B = sc.w_flip; a.ldb = 288;
  a.ldc = 32;
  a.epi.bias = bias;
  a.epi.act = act;
  {
    GemmArgs c = a;
    c.C = out;
    if (mask != nullptr) { c.epi.dact = DACT_RELU_OUT; c.epi.aux = mask; c.epi.ld_aux = 32; }
    if (g.run_compact(c, Wp, Ho, s)) return;
  }
  a.C = sc.out_grid;
  g.run(a, s);
  compact_grid_kernel<<<grid_for((long long)B * Ho * Ho * 8, 256), 256, 0, s>>>(
      reinterpret_cast<const float4*>(sc.out_grid), B, Wp, Ho, reinterpret_cast<const float4*>(mask),
      reinterpret_cast<float4*>(out));
  RLREP_LAUNCHED_W("compact_grid", s, 4.0 * 32 * ((double)B * Ho * Ho * (mask ? 3 : 2)), 0.0);
}

void valid_conv_3x3(GemmRunner& g, cudaStream_t s, int B, int Hi, const float* in, const float* W, int ldw,
                    const float* bias, int act, float* out, FullCorrScratch& sc) {
  const int Ho = Hi - 2;
  GemmArgs a;
  a.M = B * Hi * Hi; a.N = 32; a.K = 288;
  a.A = in; a.lda = 32; a.conv_w = Hi;
  a.B = W; a.ldb = ldw;
  a.ldc = 32;
  a.epi.bias = bias;
  a.epi.act = act;
  {
    GemmArgs c = a;
    c.C = out;
    if (g.run_compact(c, Hi, Ho, s)) return;
  }
  a.C = sc.out_grid;
  g.run(a, s);
  compact_grid_kernel<<<grid_for((long long)B * Ho * Ho * 8, 256), 256, 0, s>>>(
      reinterpret_cast<const float4*>(sc.out_grid), B, Hi, Ho, nullptr, reinterpret_cast<float4*>(out));
  RLREP_LAUNCHED_W("compact_grid", s, 4.0 * 32 * ((double)B * Ho * Ho * 2), 0.0);
}

}  // namespace rlrep

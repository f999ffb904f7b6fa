// DrQ-v2 pixel encoder (reference: agent/diffsrdrq/network_arch/drqv2.py:21-57,138-167; the same 4-conv stack is
// agent/mulvdrq/drqv2.py:52-96): RandomShiftsAug (replicate-pad 4 + integer shift) -> x / 255 - 0.5 ->
// Conv 3x3 s2 (C -> 32) + ReLU -> 3 x [Conv 3x3 s1 (32 -> 32) + ReLU] -> flatten, forward and backward.
//
// First building block of the pixel agents (SURVEY.md 8a rows a16 / a17, kernel K15).  Activations are kept NHWC
// ([B, H, W, 32] == a row-major [B*H*W, 32] matrix, so a GEMM output IS the next layer's activation).
//   * layer 1 (stride 2, C input channels): explicit im2col -- augmentation, uint8 -> float and the normalisation fused into
//     it, so the frames are read once as bytes -- then a GEMM with the bias + ReLU epilogue; backward: dW = dY^T col.
//   * layers 2-4 (3x3, stride 1, 32 -> 32), TF32 path: NO column matrices.  Forward = implicit convolution on the input's
//     own grid (the halo kernel, gemm_tc_kernel.cuh: one TMA box per tile, nine taps as shifted UMMA descriptors, valid
//     rows stored compactly); data gradient = implicit full correlation on a zero-padded grid (conv_implicit.cu); weight
//     gradient = a GEMM whose B operand reads the input map through a shifted 4-D TMA view (GemmArgs::conv_wgrad_hi).
//   * strict-fp32 mode and batches that are not a multiple of 4: layers 2-4 run forward as explicit im2col + GEMM and their
//     weight gradient as a folded GEMM over the column matrix; the data gradient is the implicit full correlation.
#include "conv.cuh"
#include "layout.cuh"

#include <algorithm>

namespace rlrep {

namespace {

constexpr int kPad = 4;  // RandomShiftsAug(pad=4)
constexpr int kMaxK1 = 512;  // padded first-layer column count the im2col kernel's tap table holds (C <= 56 channels)

__global__ void im2col_u8_aug_kernel(const unsigned char* __restrict__ obs, const int* __restrict__ shifts, int B, int C,
                                     int H, int Ho, float4* __restrict__ col, int ldk) {
  // one thread per (output pixel, four consecutive k), k = c * 9 + ky * 3 + kx -- the reference's weight layout
  // [32, C, 3, 3] flattened; 16-byte stores, consecutive threads on consecutive pieces of a row; byte loads served by L1.
  // obs / 255.0 - 0.5 (op by op like torch) comes from a 256-entry table built with exactly those two operations, and all
  // index arithmetic is 32-bit (checked by the constructor): the IEEE divisions and 64-bit div / mod by run-time values
  // were most of this kernel's instructions (100 us for a 165 MB write).
  __shared__ float lut[256];
  __shared__ __align__(16) int tap_off[kMaxK1];  // per column k: (c * H * H) << 4 | ky << 2 | kx, or -1 for the padding columns
  for (int p = threadIdx.x; p < 256; p += blockDim.x) lut[p] = __fsub_rn(__fdiv_rn((float)p, 255.0f), 0.5f);
  for (int k = threadIdx.x; k < ldk; k += blockDim.x) {
    const int c = k / 9, r9 = k - 9 * c, ky = r9 / 3, kx = r9 - 3 * ky;
    tap_off[k] = k < C * 9 ? ((c * H * H) << 4) | (ky << 2) | kx : -1;
  }
  __syncthreads();
  const int q4 = ldk >> 2, HoHo = Ho * Ho;
  const int total = B * HoHo * q4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int row = i / q4, q = i - row * q4;
    const int b = row / HoHo, rem = row - b * HoHo, oy = rem / Ho, ox = rem - oy * Ho;
    int sx = 0, sy = 0;
    if (shifts != nullptr) {  // padded[i + sy, j + sx] with replicate padding == clamp(i + sy - pad)
      sx = shifts[2 * b] - kPad;
      sy = shifts[2 * b + 1] - kPad;
    }
    const unsigned char* img = obs + (size_t)b * C * H * H;
    float v[4];
#pragma unroll
    const int4 t4 = *reinterpret_cast<const int4*>(tap_off + 4 * q);  // the column decomposition comes from the table
    const int tt[4] = {t4.x, t4.y, t4.z, t4.w};
    const int by = 2 * oy + sy, bx = 2 * ox + sx;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      v[e] = 0.f;
      if (tt[e] >= 0) {
        const int iy = min(max(by + ((tt[e] >> 2) & 3), 0), H - 1), ix = min(max(bx + (tt[e] & 3), 0), H - 1);
        v[e] = lut[img[(tt[e] >> 4) + iy * H + ix]];
      }
    }
    col[i] = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// act [B, H, H, 32] -> col [B*Ho*Ho, 288], k = (ky*3 + kx) * 32 + c; one float4 per thread (8 per tap)
__global__ void im2col_nhwc32_kernel(const float4* __restrict__ act, int B, int H, int Ho, float4* __restrict__ col) {
  const long long total = (long long)B * Ho * Ho * 72;  // 288 / 4 float4 per row
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(i % 72);
    const long long row = i / 72;
    const int tap = q >> 3, c4 = q & 7;
    const int ky = tap / 3, kx = tap % 3;
    const int ox = (int)(row % Ho), oy = (int)((row / Ho) % Ho), b = (int)(row / ((long long)Ho * Ho));
    col[i] = act[(((long long)b * H + oy + ky) * H + ox + kx) * 8 + c4];
  }
}

// dW[o, k] = sum_p C[p*32 + o, p*ldk + k]: the diagonal blocks of the folded weight-gradient GEMM (see backward())
__global__ void diag_block_sum_kernel(const float* __restrict__ C, int ldc, int P, int ldk, float* __restrict__ dW,
                                      int ld_dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 32 * ldk) return;
  const int o = i / ldk, k = i - o * ldk;
  float acc = 0.f;
  for (int p = 0; p < P; ++p) acc += C[(size_t)(p * 32 + o) * ldc + p * ldk + k];  // fixed order
  dW[(size_t)o * ld_dw + k] = acc;
}

int grid_for(long long work, int threads) {
  const long long want = (work + threads - 1) / threads;
  return (int)std::min<long long>(want, (long long)kNumSMs * 16);
}

}  // namespace

ConvEncoder::ConvEncoder(int batch, int in_channels, int height, Precision prec, cudaStream_t s, bool with_target)
    : B_(batch), C_(in_channels), H_(height), stream_(s) {
  RLREP_CHECK(B_ > 0 && C_ > 0 && H_ >= 16, "bad encoder dimensions");
  RLREP_CHECK((long long)B_ * H_ * H_ * (C_ * 9 + 32) / 4 < (1LL << 31), "encoder batch too large for 32-bit column indexing");
  RLREP_CHECK(round_up32(C_ * 9) <= kMaxK1 && (long long)C_ * H_ * H_ < (1 << 27), "too many input channels for the im2col tap table");
  hw_[0] = (H_ - 3) / 2 + 1;  // 84 -> 41
  for (int l = 1; l < 4; ++l) hw_[l] = hw_[l - 1] - 2;  // 39, 37, 35
  K1_ = C_ * 9;
  ldk1_ = round_up32(K1_);
  g_.name = "encoder";
  // layer 1 keeps the reference's [32, C*3*3] layout; layers 2-4 are stored [32, (ky, kx, c)] (permuted at the API)
  conv_[0] = add_linear(g_, "convnet.0", 32, K1_);  // exported as "encoder.convnet.N" by the DrQ handle
  for (int l = 1; l < 4; ++l) conv_[l] = add_linear(g_, "convnet." + std::to_string(2 * l), 32, 288);
  if (with_target) g_.n_target = g_.n;
  g_.want(arena_);
  implicit_wgrad_ = prec == PREC_TF32 && B_ % 4 == 0;
  arena_.want(&col_[0], rows(0) * ldk1_);
  if (!implicit_wgrad_)  // 1.2 GB at B = 256 that the implicit path never allocates
    for (int l = 1; l < 4; ++l) arena_.want(&col_[l], rows(l) * 288);
  for (int l = 0; l < 4; ++l) {
    // + slack rows (zero from the arena, never written): the implicit weight gradient reads up to 2 Hi + 5 rows past a map
    arena_.want(&act_[l], (rows(l) + 2 * hw_[l] + 8) * 32);
    arena_.want(&dact_[l], rows(l) * 32);
  }
  corr_.want(arena_, B_, hw_[1]);
  arena_.want(&bias_partial_, kBiasChunks * 32);
  arena_.want(&wfold_, (size_t)32 * kFold * 288 * kFold);
  arena_.commit();
  gemm_.init(prec, 0);
}

void ConvEncoder::forward(const unsigned char* obs_dev, const int* shifts_dev, float* feat_dev, int ld_feat, bool target,
                          bool no_grad) {
  cudaStream_t s = stream_;
  RLREP_CHECK(!target || g_.n_target == g_.n, "this encoder has no target copy");
  backward_ready_ = !target && !no_grad;
  im2col_u8_aug_kernel<<<grid_for((long long)rows(0) * (ldk1_ / 4), 256), 256, 0, s>>>(
      obs_dev, shifts_dev, B_, C_, H_, hw_[0], reinterpret_cast<float4*>(col_[0]), ldk1_);
  RLREP_LAUNCHED_W("im2col_u8_aug", s, (double)B_ * C_ * H_ * H_ + 4.0 * rows(0) * ldk1_, 0.0);
  linear_fwd(gemm_, s, (int)rows(0), Mat{col_[0], ldk1_}, conv_[0].view(g_, target), ACT_RELU, act_[0], 32);
  for (int l = 1; l < 4; ++l) {
    if (target || no_grad || implicit_wgrad_) {
      // no backward pass follows (target / no-grad evaluation), so no column matrix is needed: implicit convolution
      const Linear w = conv_[l].view(g_, target);
      valid_conv_3x3(gemm_, s, B_, hw_[l - 1], act_[l - 1], w.W, w.ld, w.b, ACT_RELU, act_[l], corr_);
      continue;
    }
    im2col_nhwc32_kernel<<<grid_for((long long)rows(l) * 72, 256), 256, 0, s>>>(
        reinterpret_cast<const float4*>(act_[l - 1]), B_, hw_[l - 1], hw_[l], reinterpret_cast<float4*>(col_[l]));
    RLREP_LAUNCHED_W("im2col_nhwc32", s, 4.0 * (rows(l - 1) * 32 + rows(l) * 288), 0.0);
    linear_fwd(gemm_, s, (int)rows(l), Mat{col_[l], 288}, conv_[l].view(g_, target), ACT_RELU, act_[l], 32);
  }
  const int P = hw_[3] * hw_[3];
  launch_nhwc_to_cp(act_[3], B_, P, feat_dev, ld_feat > 0 ? ld_feat : (long long)P * 32, s);
  RLREP_LAUNCHED_W("nhwc_to_nchw", s, 8.0 * B_ * P * 32, 0.0);
}

void ConvEncoder::backward(const float* dfeat_dev, int ld_dfeat) {
  RLREP_CHECK(backward_ready_, "encoder backward() needs the last forward to have run with gradients: after a target "
                               "or no_grad forward (or none) the maps it differentiates belong to no such input");
  cudaStream_t s = stream_;
  const int P = hw_[3] * hw_[3];
  launch_cp_to_nhwc(dfeat_dev, ld_dfeat > 0 ? ld_dfeat : (long long)P * 32, B_, P, /*mask=*/act_[3], dact_[3], s);
  RLREP_LAUNCHED_W("nchw_to_nhwc_relu_bwd", s, 12.0 * B_ * P * 32, 0.0);
  for (int l = 3; l >= 0; --l) {
    const Linear w = conv_[l].view(g_);
    const Mat dy{dact_[l], 32};
    const Mat col = l == 0 ? Mat{col_[0], ldk1_} : Mat{col_[l], 288};
    // dW = dY^T col is a [32, 9 C_in] output over K = B*Ho*Wo ~ 4e5 rows: 32 of the tile's 128 rows and at most 8
    // split-K CTAs per N-tile would leave the GPU idle.  Fold kFold consecutive rows into one: dY as [rows / F, 32 F],
    // col as [rows / F, ldk F]; their product is an [32 F, ldk F] matrix whose F diagonal blocks sum to dW.  Same
    // tensor-core work as before (the tile is now full), K shrinks F-fold and the N-tiles multiply F-fold.
    if (l > 0 && implicit_wgrad_) {
      // no column matrix: dY goes onto the input's grid (55 MB at B = 256 instead of the 450 MB col), and the GEMM's TMA
      // producer reads the input map through the shifted (ky, q, c) view (gemm.cuh conv_wgrad_hi)
      conv3x3_wgrad_implicit(gemm_, s, B_, hw_[l - 1], dact_[l], act_[l - 1], w.dW, w.ld, /*transposed=*/false, corr_,
                             /*small_colsum=*/w.db);  // the bias gradient rides in the scatter pass
    } else if (rows(l) % kFold == 0) {
      GemmArgs a;
      a.M = 32 * kFold; a.N = col.ld * kFold; a.K = (int)(rows(l) / kFold);
      a.A = dy.p; a.lda = 32 * kFold; a.a_mn = true;
      a.B = col.p; a.ldb = col.ld * kFold; a.b_mn = true;
      a.C = wfold_; a.ldc = a.N;
      gemm_.run(a, s);
      diag_block_sum_kernel<<<ceil_div(32 * col.ld, 256), 256, 0, s>>>(wfold_, a.N, kFold, col.ld, w.dW, w.ld);
      RLREP_LAUNCHED("diag_block_sum", s);
    } else {
      linear_wgrad(gemm_, s, (int)rows(l), dy, col, w, Mat(), 0, /*bias_grad=*/false);
    }
    if (!(l > 0 && implicit_wgrad_)) launch_colsum_tall(dy.p, 32, rows(l), 32, bias_partial_, kBiasChunks, w.db, s);
    if (l == 0) break;
    // dX = full correlation of dY with W (x ReLU mask), the taps walked by the GEMM's TMA producer (conv_implicit.cu)
    full_correlation_3x3(gemm_, s, B_, hw_[l], dact_[l], w.W, FC_CONV_DGRAD, nullptr, ACT_NONE, act_[l - 1], dact_[l - 1],
                         corr_);
  }
}

}  // namespace rlrep

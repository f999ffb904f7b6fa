// muLV-Rep pixel decoder (reference: agent/mulvdrq/drqv2.py:98-117): x.view(B, 32, 35, 35) ->
// 3 x [ConvTranspose2d(32, 32, 3, stride 1) + ReLU] -> ConvTranspose2d(32, 32, 3, stride 2) + ReLU ->
// Conv2d(32, 3, kernel 2, padding 1): 35 -> 37 -> 39 -> 41 -> 83 -> 84, forward, L1 loss and backward.
//
// A transposed convolution is the data-gradient of a convolution, so it runs on the encoder's machinery with the roles
// swapped (conv.cu): activations NHWC.  Forward: the stride-1 layers are implicit full correlations (conv_implicit.cu); the
// stride-2 layer runs as four parity classes on the halo kernel, or where that kernel does not apply as
// colT [B*Hi*Hi, 9*32] = X [B*Hi*Hi, 32] x Wd^T  (tcgen05 GEMM, K = 32) followed by the gather-form col2im (+ bias + ReLU).
// Backward  dcolT = im2col(dY) (stride 1 or 2),  dX = dcolT Wd (x ReLU mask),  dWd = dcolT^T X.  Wd[(ky*3 + kx)*32 + co, ci] = W_ref[ci, co, ky, kx] (permuted at the
// API).  The 3-channel output layer is a direct CUDA-core kernel (384 FMAs per pixel) fused with nothing; its weight
// gradient is a two-pass deterministic reduction.
#include "deconv.cuh"
#include "layout.cuh"

#include <algorithm>

#include "reduce.cuh"

namespace rlrep {

namespace {

int grid_for(long long work, int threads) {
  const long long want = (work + threads - 1) / threads;
  return (int)std::max<long long>(1, std::min<long long>(want, (long long)kNumSMs * 16));
}

// Y[b, y, x, co] = relu(bias[co] + sum over taps with (y - ky) = S*iy, (x - kx) = S*ix of colT[(b, iy, ix), tap, co])
template <int S>
__global__ void col2im_bias_relu_kernel(const float4* __restrict__ colT, const float4* __restrict__ bias, int B, int Hi,
                                        int Ho, float4* __restrict__ y) {
  const long long total = (long long)B * Ho * Ho * 8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i & 7);
    const long long pix = i >> 3;
    const int ox = (int)(pix % Ho), oy = (int)((pix / Ho) % Ho), b = (int)(pix / ((long long)Ho * Ho));
    float4 acc = __ldg(bias + c4);
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int ty = oy - ky;
      if (ty < 0 || (S == 2 && (ty & 1))) continue;
      const int iy = ty / S;
      if (iy >= Hi) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int tx = ox - kx;
        if (tx < 0 || (S == 2 && (tx & 1))) continue;
        const int ix = tx / S;
        if (ix >= Hi) continue;
        const float4 g = colT[(((long long)b * Hi + iy) * Hi + ix) * 72 + (ky * 3 + kx) * 8 + c4];
        acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
      }
    }
    y[i] = make_float4(fmaxf(acc.x, 0.f), fmaxf(acc.y, 0.f), fmaxf(acc.z, 0.f), fmaxf(acc.w, 0.f));
  }
}

// dcolT[(b, iy, ix), tap, c] = dY[b, S*iy + ky, S*ix + kx, c]
template <int S>
__global__ void im2col_strided_kernel(const float4* __restrict__ dy, int B, int Hi, int Ho, float4* __restrict__ col) {
  const long long total = (long long)B * Hi * Hi * 72;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(i % 72);
    const long long row = i / 72;
    const int tap = q >> 3, c4 = q & 7;
    const int ky = tap / 3, kx = tap % 3;
    const int ix = (int)(row % Hi), iy = (int)((row / Hi) % Hi), b = (int)(row / ((long long)Hi * Hi));
    col[i] = dy[(((long long)b * Ho + S * iy + ky) * Ho + S * ix + kx) * 8 + c4];
  }
}

// Output layer Conv2d(32 -> 3, kernel 2, padding 1) on X [B, 83, 83, 32]: eight lanes per output pixel (one float4 of
// channels each, so a tap is one coalesced 128-byte row), shuffle-reduced; pred [B*84*84, 4] (channel 3 unused).
// w_s[(tap*32 + c)*3 + o] = W[o, c, ky, kx] staged in shared memory.
template <int KS>
__global__ void __launch_bounds__(256) out_conv_fwd_kernel(const float4* __restrict__ x, const float* __restrict__ W,
                                                           const float* __restrict__ bias, int B, int Hi, int Ho,
                                                           float4* __restrict__ pred) {
  constexpr int T = KS * KS, Q = 4, COLS = Q + KS - 1;  // Q consecutive output pixels per thread, their input columns
  // w_s[(tap * 32 + c) * 3 + o] = W[o, c, tap]: a thread's 12 weights of a tap are three aligned float4.  The kernel is
  // bound by these shared-memory reads (ncu: 218 M wavefronts per launch at 1024 frames), so every weight fetched is used
  // for FOUR pixels: a thread keeps the (KS + 3) x KS window of its channel group in registers.
  __shared__ __align__(16) float w_s[T * 32 * 3];
  for (int i = threadIdx.x; i < T * 96; i += 256) {
    const int o = i % 3, c = (i / 3) % 32, tap = i / 96;
    w_s[i] = W[(o * 32 + c) * T + tap];
  }
  __syncthreads();
  const int c4 = threadIdx.x & 7;
  const float b0 = bias[0], b1 = bias[1], b2 = bias[2];
  // 32-bit index arithmetic (the constructor checks that every index fits); eight lanes (channel groups) per pixel quad
  const int quads_x = (Ho + Q - 1) / Q, total = B * Ho * quads_x;
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; i < ((total + 3) & ~3); i += (gridDim.x * blockDim.x) >> 3) {
    float acc[Q][3];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[q][0] = acc[q][1] = acc[q][2] = 0.f;
    int b = 0, oy = 0, ox0 = 0;
    if (i < total) {
      const int row = i / quads_x;
      ox0 = (i - row * quads_x) * Q;
      b = row / Ho;
      oy = row - b * Ho;
      float4 v[KS][COLS];
#pragma unroll
      for (int ky = 0; ky < KS; ++ky) {
        const int iy = oy + ky - 1;
#pragma unroll
        for (int cx = 0; cx < COLS; ++cx) {
          const int ix = ox0 + cx - 1;
          const bool ok = iy >= 0 && iy < Hi && ix >= 0 && ix < Hi;
          v[ky][cx] = ok ? x[((b * Hi + iy) * Hi + ix) * 8 + c4] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int ky = 0; ky < KS; ++ky)
#pragma unroll
        for (int kx = 0; kx < KS; ++kx) {
          const float4* wq = reinterpret_cast<const float4*>(w_s + (ky * KS + kx) * 96 + c4 * 12);
          const float4 q0 = wq[0], q1 = wq[1], q2 = wq[2];
          const float wc[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
#pragma unroll
          for (int q = 0; q < Q; ++q) {
            const float4 t = v[ky][q + kx];
#pragma unroll
            for (int o = 0; o < 3; ++o)
              acc[q][o] = fmaf(t.x, wc[o], fmaf(t.y, wc[3 + o], fmaf(t.z, wc[6 + o], fmaf(t.w, wc[9 + o], acc[q][o]))));
          }
        }
    }
#pragma unroll
    for (int sh = 4; sh > 0; sh >>= 1)  // fixed-order reduction over the eight channel groups
#pragma unroll
      for (int q = 0; q < Q; ++q)
#pragma unroll
        for (int o = 0; o < 3; ++o) acc[q][o] += __shfl_xor_sync(0xffffffffu, acc[q][o], sh);
    if (i < total && c4 < Q && ox0 + c4 < Ho) {  // lane q of the group stores pixel q
      float r0 = 0.f, r1 = 0.f, r2 = 0.f;
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (q == c4) { r0 = acc[q][0]; r1 = acc[q][1]; r2 = acc[q][2]; }
      pred[(b * Ho + oy) * Ho + ox0 + c4] = make_float4(r0 + b0, r1 + b1, r2 + b2, 0.f);
    }
  }
}

// dpred = scale * sign(pred - (t / 255 - 0.5)); partial[block] = sum |diff|.  target uint8 [B, 3, Ho, Ho].
__global__ void __launch_bounds__(256) l1_loss_kernel(const float4* __restrict__ pred, const unsigned char* __restrict__ tgt,
                                                      int B, int Ho, float scale, float4* __restrict__ dpred,
                                                      float* __restrict__ partial) {
  __shared__ float scratch[33];
  const long long P = (long long)Ho * Ho, total = (long long)B * P;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / P, p = i - b * P;
    const float4 v = pred[i];
    const unsigned char* t = tgt + b * 3 * P + p;
    const float d0 = v.x - __fsub_rn(__fdiv_rn((float)t[0], 255.0f), 0.5f);
    const float d1 = v.y - __fsub_rn(__fdiv_rn((float)t[P], 255.0f), 0.5f);
    const float d2 = v.z - __fsub_rn(__fdiv_rn((float)t[2 * P], 255.0f), 0.5f);
    acc += fabsf(d0) + fabsf(d1) + fabsf(d2);
    dpred[i] = make_float4(d0 > 0.f ? scale : (d0 < 0.f ? -scale : 0.f), d1 > 0.f ? scale : (d1 < 0.f ? -scale : 0.f),
                           d2 > 0.f ? scale : (d2 < 0.f ? -scale : 0.f), 0.f);
  }
  acc = block_sum<256>(acc, scratch);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}
// Latent Diff-SR reconstruction loss (latent_diff_sr.py:242): sum((pred - target)^2) / n_frames with
// target = frame / 255 - 0.5 and frame = the shift-augmented uint8 frame (replicate padding == clamped lookup; a null
// shift table means no augmentation).  dpred = scale * 2 * diff; partial[block] = sum diff^2.
__global__ void __launch_bounds__(256) mse_sum_loss_kernel(const float4* __restrict__ pred, const unsigned char* __restrict__ tgt,
                                                           const int* __restrict__ shifts, int B, int Ho, float scale,
                                                           float4* __restrict__ dpred, float* __restrict__ partial) {
  __shared__ float scratch[33];
  const long long P = (long long)Ho * Ho, total = (long long)B * P;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / P, p = i - b * P;
    int y = (int)(p / Ho), x = (int)(p - (long long)y * Ho);
    if (shifts != nullptr) {
      x = min(max(x + shifts[2 * b] - 4, 0), Ho - 1);
      y = min(max(y + shifts[2 * b + 1] - 4, 0), Ho - 1);
    }
    const float4 v = pred[i];
    const unsigned char* t = tgt + b * 3 * P + (long long)y * Ho + x;
    const float d0 = v.x - __fsub_rn(__fdiv_rn((float)t[0], 255.0f), 0.5f);
    const float d1 = v.y - __fsub_rn(__fdiv_rn((float)t[P], 255.0f), 0.5f);
    const float d2 = v.z - __fsub_rn(__fdiv_rn((float)t[2 * P], 255.0f), 0.5f);
    acc = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, acc)));
    dpred[i] = make_float4(2.f * scale * d0, 2.f * scale * d1, 2.f * scale * d2, 0.f);
  }
  acc = block_sum<256>(acc, scratch);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}
__global__ void mse_sum_finalize_kernel(const float* __restrict__ partial, int n, float inv_frames, float* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float s = 0.f;
  for (int i = 0; i < n; ++i) s += partial[i];
  out[0] = s * inv_frames;
}

// out[0] = 10 * sum(partial) / count  (fixed order)
__global__ void l1_finalize_kernel(const float* __restrict__ partial, int n, float inv_count, float* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float s = 0.f;
  for (int i = 0; i < n; ++i) s += partial[i];
  out[0] = 10.f * s * inv_count;
}

// dX[b, iy, ix, c] = relu'(X) * sum_{tap, o} dpred[b, iy - ky + 1, ix - kx + 1, o] * W[o, c, ky, kx]
template <int KS>
__global__ void __launch_bounds__(256) out_conv_dgrad_kernel(const float4* __restrict__ dpred, const float* __restrict__ W,
                                                             const float4* __restrict__ x, int B, int Hi, int Ho,
                                                             float4* __restrict__ dx) {
  constexpr int T = KS * KS, Q = 4, COLS = Q + KS - 1;
  // like the forward kernel: weights from shared memory once per FOUR input pixels of a thread's channel group; the
  // (KS + 3) x KS window of output gradients (one float4 = three channels each) lives in registers
  __shared__ __align__(16) float w_s[T * 32 * 3];  // [(tap * 32 + c) * 3 + o]
  for (int i = threadIdx.x; i < T * 96; i += 256) {
    const int o = i % 3, c = (i / 3) % 32, tap = i / 96;
    w_s[i] = W[(o * 32 + c) * T + tap];
  }
  __syncthreads();
  const int c4 = threadIdx.x & 7;
  const int quads_x = (Hi + Q - 1) / Q, total = B * Hi * quads_x * 8;  // 32-bit index arithmetic (checked by the constructor)
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int quad = i >> 3;  // (i & 7) == c4: the grid-stride step is a multiple of 8
    const int row = quad / quads_x, ix0 = (quad - row * quads_x) * Q;
    const int b = row / Hi, iy = row - b * Hi;
    // dX[iy, ix] = sum_{ky, kx} dpred[iy - ky + 1, ix - kx + 1] . W[:, c, ky, kx]: window columns ox = ix0 - (KS - 2) + cx
    float4 g[KS][COLS];
#pragma unroll
    for (int ky = 0; ky < KS; ++ky) {
      const int oy = iy - ky + 1;
#pragma unroll
      for (int cx = 0; cx < COLS; ++cx) {
        const int ox = ix0 - (KS - 2) + cx;
        const bool ok = oy >= 0 && oy < Ho && ox >= 0 && ox < Ho;
        g[ky][cx] = ok ? dpred[(b * Ho + oy) * Ho + ox] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float acc[Q][4];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f;
#pragma unroll
    for (int ky = 0; ky < KS; ++ky)
#pragma unroll
      for (int kx = 0; kx < KS; ++kx) {
        const float4* wq = reinterpret_cast<const float4*>(w_s + (ky * KS + kx) * 96 + c4 * 12);
        const float4 q0 = wq[0], q1 = wq[1], q2 = wq[2];
        const float w[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          // input pixel ix0 + q, tap kx reads output column ox = ix0 + q - kx + 1 = window index q - kx + 1 + (KS - 2)
          const float4 t = g[ky][q - kx + KS - 1];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            acc[q][j] = fmaf(t.x, w[3 * j], fmaf(t.y, w[3 * j + 1], fmaf(t.z, w[3 * j + 2], acc[q][j])));
        }
      }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int ix = ix0 + q;
      if (ix < Hi) {
        const int o = ((b * Hi + iy) * Hi + ix) * 8 + c4;
        const float4 xv = x[o];
        dx[o] = make_float4(xv.x > 0.f ? acc[q][0] : 0.f, xv.y > 0.f ? acc[q][1] : 0.f, xv.z > 0.f ? acc[q][2] : 0.f,
                            xv.w > 0.f ? acc[q][3] : 0.f);
      }
    }
  }
}

// Pass 1 of dW[o, c, tap] = sum_pixels dpred[pix, o] * X[pix + tap - 1, c] and db[o] = sum dpred[pix, o]:
// lane = input channel; each warp walks whole output ROWS with a sliding KS x KS window of the input in registers, so a
// pixel costs KS new loads (the window's next column) instead of KS * KS, and the next four columns are in flight while
// the current four pixels are accumulated; partial[block] = [3 T * 32 weight sums | 3 bias sums | pad].
template <int KS>
__global__ void __launch_bounds__(256, 3) out_conv_wgrad_kernel(const float4* __restrict__ dpred, const float* __restrict__ x,
                                                             int B, int Hi, int Ho, float* __restrict__ partial) {
  constexpr int T = KS * KS, NA = 3 * T, PS = NA * 32 + 4;  // accumulators per lane, partial stride
  constexpr int U = 4;
  __shared__ float red[8][PS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_rows = B * Ho;  // (b, oy) pairs; 32-bit index arithmetic (checked by the launcher)
  const int nw = gridDim.x * 8, gw = blockIdx.x * 8 + warp;
  const int per = (n_rows + nw - 1) / nw;
  const int r0 = min(gw * per, n_rows), r1 = min(r0 + per, n_rows);
  float acc[NA];
#pragma unroll
  for (int j = 0; j < NA; ++j) acc[j] = 0.f;
  float bsum = 0.f;
  for (int r = r0; r < r1; ++r) {
    const int b = r / Ho, oy = r - b * Ho;
    const float* xrow[KS];  // input row of tap row ky (nullptr outside the image)
#pragma unroll
    for (int ky = 0; ky < KS; ++ky) {
      const int iy = oy + ky - 1;
      xrow[ky] = (iy >= 0 && iy < Hi) ? x + (size_t)((b * Hi + iy) * Hi) * 32 + lane : nullptr;
    }
    auto ld = [&](int ky, int ix) { return (xrow[ky] != nullptr && ix >= 0 && ix < Hi) ? xrow[ky][ix * 32] : 0.f; };
    float win[KS][KS];  // win[ky][kx] = X[iy, ox + kx - 1] for the current output pixel
#pragma unroll
    for (int ky = 0; ky < KS; ++ky) {
      win[ky][0] = 0.f;
#pragma unroll
      for (int kx = 1; kx < KS; ++kx) win[ky][kx] = ld(ky, kx - 1);
    }
    const float4* grow = dpred + (size_t)r * Ho;
    for (int ox = 0; ox < Ho; ox += U) {
      float4 g[U];
      float nxt[U][KS];  // the window's next column for pixel ox + u + 1: ix = ox + u + KS - 1
#pragma unroll
      for (int u = 0; u < U; ++u) {
        g[u] = ox + u < Ho ? grow[ox + u] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int ky = 0; ky < KS; ++ky) nxt[u][ky] = ld(ky, ox + u + KS - 1);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (lane < 3) bsum += lane == 0 ? g[u].x : (lane == 1 ? g[u].y : g[u].z);
#pragma unroll
        for (int ky = 0; ky < KS; ++ky)
#pragma unroll
          for (int kx = 0; kx < KS; ++kx) {
            const int tap = ky * KS + kx;
            acc[tap * 3 + 0] = fmaf(g[u].x, win[ky][kx], acc[tap * 3 + 0]);
            acc[tap * 3 + 1] = fmaf(g[u].y, win[ky][kx], acc[tap * 3 + 1]);
            acc[tap * 3 + 2] = fmaf(g[u].z, win[ky][kx], acc[tap * 3 + 2]);
          }
#pragma unroll
        for (int ky = 0; ky < KS; ++ky) {
#pragma unroll
          for (int kx = 0; kx + 1 < KS; ++kx) win[ky][kx] = win[ky][kx + 1];
          win[ky][KS - 1] = nxt[u][ky];
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NA; ++j) red[warp][j * 32 + lane] = acc[j];
  if (lane < 3) red[warp][NA * 32 + lane] = bsum;
  __syncthreads();
  for (int k = threadIdx.x; k < NA * 32 + 3; k += 256) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][k];
    partial[(size_t)blockIdx.x * PS + k] = s;
  }
}
// Pass 2: dW[o, c, tap] (reference layout [3, 32, 2, 2]) and db[o] from the per-block partials, fixed order.
template <int KS>
__global__ void out_conv_wgrad_finish_kernel(const float* __restrict__ partial, int n_blocks, float* __restrict__ dW,
                                             float* __restrict__ db) {
  constexpr int T = KS * KS, NA = 3 * T, PS = NA * 32 + 4;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= NA * 32 + 3) return;
  float s = 0.f;
  for (int i = 0; i < n_blocks; ++i) s += partial[(size_t)i * PS + k];
  if (k < NA * 32) {
    const int j = k / 32, c = k % 32, tap = j / 3, o = j % 3;
    dW[(o * 32 + c) * T + tap] = s;
  } else {
    db[k - NA * 32] = s;
  }
}

// dW[n, c] = sum_p C[(p*288 + n)*ldc + p*32 + c]: the diagonal blocks of the folded weight-gradient GEMM (backward())
__global__ void diag_block_sum_288x32_kernel(const float* __restrict__ C, int ldc, int P, float* __restrict__ dW) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 288 * 32) return;
  const int n = i >> 5, c = i & 31;
  float acc = 0.f;
  for (int p = 0; p < P; ++p) acc += C[(size_t)(p * 288 + n) * ldc + p * 32 + c];  // fixed order
  dW[i] = acc;
}

// [B*P, 4] -> [B, 3, P]
__global__ void pred_to_nchw_kernel(const float4* __restrict__ pred, int B, long long P, float* __restrict__ out) {
  const long long total = (long long)B * P;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / P, p = i - b * P;
    const float4 v = pred[i];
    out[b * 3 * P + p] = v.x;
    out[b * 3 * P + P + p] = v.y;
    out[b * 3 * P + 2 * P + p] = v.z;
  }
}

}  // namespace

ConvDecoder::ConvDecoder(int batch, Precision prec, cudaStream_t s, int out_kernel, bool with_target)
    : B_(batch), ks_(out_kernel), stream_(s) {
  RLREP_CHECK(B_ > 0 && (ks_ == 2 || ks_ == 3), "bad decoder batch / output kernel size");
  RLREP_CHECK((long long)B_ * 84 * 84 * 32 < (1LL << 31), "decoder batch too large for the output layer's 32-bit indexing");
  // out_kernel 2: muLV-Rep (stride-2 layer 41 -> 83, Conv2d k2 p1 -> 84); out_kernel 3: the latent Diff-SR VAE
  // (stride-2 layer with output_padding 1: 41 -> 84, Conv2d k3 p1 -> 84)
  if (ks_ == 3) hw_[4] = 84;
  g_.name = "decoder";
  for (int l = 0; l < 4; ++l) {  // stored [(ky, kx, co), ci]; exported as the reference's [ci, co, ky, kx]
    w_off_[l] = g_.add("deconvnet." + std::to_string(2 * l) + ".weight", 288, 32);
    b_off_[l] = g_.add("deconvnet." + std::to_string(2 * l) + ".bias", 32, 1);
  }
  w_off_[4] = g_.add("deconvnet.8.weight", 3, 32 * ks_ * ks_);  // the reference's [3, 32, k, k] flattened
  b_off_[4] = g_.add("deconvnet.8.bias", 3, 1);
  if (with_target) g_.n_target = g_.n;
  g_.want(arena_);
  for (int i = 0; i < 5; ++i) {
    arena_.want(&act_[i], rows(i) * 32);
    // + slack rows (zero from the arena, never written): the implicit weight gradient reads up to 2 H + 5 rows past the map
    arena_.want(&dact_[i], (rows(i) + 2 * hw_[i] + 8) * 32);
  }
  arena_.want(&col_, rows(3) * 288);  // the largest GEMM side: 41 x 41 pixels per image
  arena_.want(&pred_, rows(5) * 4);
  arena_.want(&dpred_, rows(5) * 4);
  arena_.want(&loss_partial_, kLossBlocks);
  arena_.want(&wg_partial_, (size_t)kWgBlocks * (96 * ks_ * ks_ + 4));
  arena_.want(&bias_partial_, kBiasChunks * 32);
  arena_.want(&wfold_, (size_t)288 * kFold * 32 * kFold);
  corr_.want(arena_, B_, hw_[3]);  // grids up to (hw_[3] + 4)^2: the stride-2 layer's padded input
  // the stride-1 layers' backward pass without column matrices (TF32 path); otherwise im2col + folded GEMM
  implicit_bwd_ = prec == PREC_TF32 && B_ % 4 == 0;
  arena_.commit();
  gemm_.init(prec, 0);
}

Linear ConvDecoder::layer(int l) const {
  Linear w;
  w.W = g_.p + w_off_[l];
  w.dW = g_.g + w_off_[l];
  w.b = nullptr;  // the bias is added after col2im, not per tap
  w.db = nullptr;
  w.out = 288; w.in = 32; w.ld = 32; w.out_alloc = 288;
  return w;
}

void ConvDecoder::forward(const float* x_dev, int ld_x) {
  cudaStream_t s = stream_;
  const int P0 = hw_[0] * hw_[0];
  launch_cp_to_nhwc(x_dev, ld_x > 0 ? ld_x : (long long)P0 * 32, B_, P0, nullptr, act_[0], s);
  RLREP_LAUNCHED_W("nchw_to_nhwc", s, 8.0 * B_ * P0 * 32, 0.0);
  for (int l = 0; l < 4; ++l) {
    const int Hi = hw_[l], Ho = hw_[l + 1];
    if (l < 3) {  // stride 1: a full correlation, the taps walked by the GEMM's TMA producer
      full_correlation_3x3(gemm_, s, B_, Hi, act_[l], g_.p + w_off_[l], FC_DECONV_FWD, g_.p + b_off_[l], ACT_RELU, nullptr,
                           act_[l + 1], corr_);
      continue;
    }
    if (deconv3x3_s2_forward(gemm_, s, B_, Hi, Ho, act_[l], g_.p + w_off_[l], g_.p + b_off_[l], act_[l + 1], corr_))
      continue;  // stride 2: four parity classes on the halo kernel, no [rows, 288] matrix
    linear_fwd(gemm_, s, (int)rows(l), Mat{act_[l], 32}, layer(l), ACT_NONE, col_, 288);
    const float4* colT = reinterpret_cast<const float4*>(col_);
    const float4* bias = reinterpret_cast<const float4*>(g_.p + b_off_[l]);
    float4* y = reinterpret_cast<float4*>(act_[l + 1]);
    col2im_bias_relu_kernel<2><<<grid_for(rows(l + 1) * 8, 256), 256, 0, s>>>(colT, bias, B_, Hi, Ho, y);
    RLREP_LAUNCHED_W("col2im_bias_relu", s, 4.0 * (rows(l) * 288 + rows(l + 1) * 32), 0.0);
  }
  if (ks_ == 2)
    out_conv_fwd_kernel<2><<<grid_for(rows(5) * 2, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(act_[4]),
                                                                    g_.p + w_off_[4], g_.p + b_off_[4], B_, hw_[4], hw_[5],
                                                                    reinterpret_cast<float4*>(pred_));
  else
    out_conv_fwd_kernel<3><<<grid_for(rows(5) * 2, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(act_[4]),
                                                                    g_.p + w_off_[4], g_.p + b_off_[4], B_, hw_[4], hw_[5],
                                                                    reinterpret_cast<float4*>(pred_));
  RLREP_LAUNCHED_W("out_conv_fwd", s, 4.0 * (rows(4) * 32 + rows(5) * 4), 2.0 * rows(5) * 384);
}

void ConvDecoder::l1_loss(const unsigned char* target_dev, float grad_scale, float* loss_out_dev) {
  cudaStream_t s = stream_;
  const float count = (float)rows(5) * 3.f;
  l1_loss_kernel<<<kLossBlocks, 256, 0, s>>>(reinterpret_cast<const float4*>(pred_), target_dev, B_, hw_[5],
                                            grad_scale * 10.f / count, reinterpret_cast<float4*>(dpred_), loss_partial_);
  RLREP_LAUNCHED_W("l1_loss", s, rows(5) * 35.0, 0.0);
  l1_finalize_kernel<<<1, 32, 0, s>>>(loss_partial_, kLossBlocks, 1.f / count, loss_out_dev);
  RLREP_LAUNCHED("l1_finalize", s);
}

void ConvDecoder::mse_sum_loss(const unsigned char* target_dev, const int* shifts_dev, float grad_scale, float* loss_out_dev) {
  cudaStream_t s = stream_;
  mse_sum_loss_kernel<<<kLossBlocks, 256, 0, s>>>(reinterpret_cast<const float4*>(pred_), target_dev, shifts_dev, B_, hw_[5],
                                                 grad_scale / (float)B_, reinterpret_cast<float4*>(dpred_), loss_partial_);
  RLREP_LAUNCHED_W("mse_sum_loss", s, rows(5) * 35.0, 0.0);
  mse_sum_finalize_kernel<<<1, 32, 0, s>>>(loss_partial_, kLossBlocks, 1.f / (float)B_, loss_out_dev);
  RLREP_LAUNCHED("mse_sum_finalize", s);
}

void ConvDecoder::backward(float* dx_dev, int ld_dx) {
  cudaStream_t s = stream_;
  // ---- output layer
  if (ks_ == 2)
    out_conv_wgrad_kernel<2><<<kWgBlocks2, 256, 0, s>>>(reinterpret_cast<const float4*>(dpred_), act_[4], B_, hw_[4], hw_[5],
                                                      wg_partial_);
  else
    out_conv_wgrad_kernel<3><<<kWgBlocks, 256, 0, s>>>(reinterpret_cast<const float4*>(dpred_), act_[4], B_, hw_[4], hw_[5],
                                                      wg_partial_);
  RLREP_LAUNCHED_W("out_conv_wgrad", s, 4.0 * (rows(4) * 32 + rows(5) * 4), 2.0 * rows(5) * 384);
  if (ks_ == 2) out_conv_wgrad_finish_kernel<2><<<2, 256, 0, s>>>(wg_partial_, kWgBlocks2, g_.g + w_off_[4], g_.g + b_off_[4]);
  else out_conv_wgrad_finish_kernel<3><<<4, 256, 0, s>>>(wg_partial_, kWgBlocks, g_.g + w_off_[4], g_.g + b_off_[4]);
  RLREP_LAUNCHED("out_conv_wgrad_finish", s);
  if (ks_ == 2)
    out_conv_dgrad_kernel<2><<<grid_for(rows(4) * 2 + 2048, 256), 256, 0, s>>>(
        reinterpret_cast<const float4*>(dpred_), g_.p + w_off_[4], reinterpret_cast<const float4*>(act_[4]), B_, hw_[4],
        hw_[5], reinterpret_cast<float4*>(dact_[4]));
  else
    out_conv_dgrad_kernel<3><<<grid_for(rows(4) * 2 + 2048, 256), 256, 0, s>>>(
        reinterpret_cast<const float4*>(dpred_), g_.p + w_off_[4], reinterpret_cast<const float4*>(act_[4]), B_, hw_[4],
        hw_[5], reinterpret_cast<float4*>(dact_[4]));
  RLREP_LAUNCHED_W("out_conv_dgrad", s, 4.0 * (rows(5) * 4 + 2.0 * rows(4) * 32), 2.0 * rows(4) * 384);
  // ---- transposed convolutions, last to first; dact_[l + 1] already carries the ReLU mask of its layer
  for (int l = 3; l >= 0; --l) {
    const int Hi = hw_[l], Ho = hw_[l + 1];
    const Linear w = layer(l);
    launch_colsum_tall(dact_[l + 1], 32, rows(l + 1), 32, bias_partial_, kBiasChunks, g_.g + b_off_[l], s);
    if (implicit_bwd_ && l < 3) {
      // stride 1: dWd[(tap, co), ci] = sum X[b, y, x, ci] dY[b, y + ky, x + kx, co] and dX = valid convolution of dY with
      // Wd (x ReLU mask; the decoder input, l == 0, is a plain linear output) -- neither builds the [rows, 288] matrix
      conv3x3_wgrad_implicit(gemm_, s, B_, Ho, act_[l], dact_[l + 1], w.dW, 32, /*transposed=*/true, corr_);
      valid_conv_3x3_wt(gemm_, s, B_, Ho, dact_[l + 1], w.W, l > 0 ? act_[l] : nullptr, dact_[l], corr_);
      continue;
    }
    const float4* dy = reinterpret_cast<const float4*>(dact_[l + 1]);
    float4* col = reinterpret_cast<float4*>(col_);
    if (l < 3) im2col_strided_kernel<1><<<grid_for(rows(l) * 72, 256), 256, 0, s>>>(dy, B_, Hi, Ho, col);
    else im2col_strided_kernel<2><<<grid_for(rows(l) * 72, 256), 256, 0, s>>>(dy, B_, Hi, Ho, col);
    RLREP_LAUNCHED_W("im2col_strided", s, 4.0 * (rows(l + 1) * 32 + rows(l) * 288), 0.0);
    // dWd = dcolT^T X is a [288, 32] output over K = B*Hi*Hi rows: three M-tiles x at most 8 split-K CTAs would leave
    // the GPU idle.  Fold kFold consecutive rows into one (conv.cu does the same): [rows/F, 288 F]^T [rows/F, 32 F] is a
    // [288 F, 32 F] matrix whose F diagonal blocks sum to dWd -- F x the tensor-core work, F x F the parallelism.
    if (rows(l) % kFold == 0) {
      GemmArgs a;
      a.M = 288 * kFold; a.N = 32 * kFold; a.K = (int)(rows(l) / kFold);
      a.A = col_; a.lda = 288 * kFold; a.a_mn = true;
      a.B = act_[l]; a.ldb = 32 * kFold; a.b_mn = true;
      a.C = wfold_; a.ldc = a.N;
      gemm_.run(a, s);
      diag_block_sum_288x32_kernel<<<ceil_div(288 * 32, 256), 256, 0, s>>>(wfold_, a.N, kFold, w.dW);
      RLREP_LAUNCHED("diag_block_sum", s);
    } else {
      linear_wgrad(gemm_, s, (int)rows(l), Mat{col_, 288}, Mat{act_[l], 32}, w, Mat(), 0, /*bias_grad=*/false);
    }
    // the decoder input (l == 0) is a plain linear output: no ReLU mask
    linear_dgrad(gemm_, s, (int)rows(l), Mat{col_, 288}, w, l > 0 ? DACT_RELU_OUT : DACT_NONE,
                 l > 0 ? Mat{act_[l], 32} : Mat(), dact_[l], 32);
  }
  const int P0 = hw_[0] * hw_[0];
  launch_nhwc_to_cp(dact_[0], B_, P0, dx_dev, ld_dx > 0 ? ld_dx : (long long)P0 * 32, s);
  RLREP_LAUNCHED_W("nhwc_to_nchw", s, 8.0 * B_ * P0 * 32, 0.0);
}

void ConvDecoder::copy_pred(float* pred_nchw_dev, bool grad) {
  const long long P = (long long)hw_[5] * hw_[5];
  pred_to_nchw_kernel<<<grid_for((long long)B_ * P, 256), 256, 0, stream_>>>(
      reinterpret_cast<const float4*>(grad ? dpred_ : pred_), B_, P, pred_nchw_dev);
  RLREP_LAUNCHED("pred_to_nchw", stream_);
}

}  // namespace rlrep

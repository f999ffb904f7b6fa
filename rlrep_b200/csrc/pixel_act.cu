// Small-batch policy of the pixel agents: DrQ-v2's select_action (agent/diffsrdrq/drqv2.py:74-82) and muLV-Rep's act
// (agent/mulvdrq/drqv2.py:270-282) share it.  x / 255 - 0.5 -> Conv 3x3 s2 (C -> 32) + ReLU -> 3 x [Conv 3x3 s1 (32 -> 32)
// + ReLU] -> flatten -> actor.trunk (Linear F -> bn, LayerNorm, tanh) -> actor.policy (Linear bn -> H, ReLU, H -> H, ReLU,
// H -> A) -> tanh -> TruncatedNormal.sample(clip=None).
//
// Up to kPixelActRows observations per pass, IEEE fp32 FMA on CUDA cores throughout: at these sizes acting is bound by
// latency, not by tensor throughput.  The convolutions run straight from the frames and the NHWC activations (no column
// matrices), one CTA per (observation, band of output rows), weights and the input band in shared memory.  The trunk's
// 39,200-wide weight, the only part of an act that moves real bytes, is streamed once per pass by a split-K kernel over
// all SMs.  The policy MLP runs on the exact-fp32 SIMT GEMMs (gemm_simt.cu) and the sample on the update's kernel.
//
// Every output element is summed over the same terms in the same order however the rows are chunked or the work is
// tiled: the band height changes only the grid, the trunk's split count is a constant, and the SIMT GEMMs sum each
// output the same way at every M.  linear_fwd does widen the A-wide head to N = 32 from 64 rows on (pad_n), and
// launch_simt's rowthread branches depend on M, but those need an MN-major A, which linear_fwd never passes; the kernels
// it reaches (skinny_rowwarp: lane-strided K and a fixed shuffle tree per output; gemm_tiled: k ascending per output)
// compute every output independently of M and N.  So an observation's action does not depend on the batch it is acted
// on with.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "pixel_act.cuh"
#include "reduce.cuh"
#include "staging.cuh"

namespace rlrep {

namespace {

constexpr int kWPitch = 36;    // conv weights transposed to wT[k][co]: 16-byte rows for float4 reads of 4 channels
constexpr int kXPitch = 33;    // NHWC input band, one pixel per 33 floats: the 4 pixels a warp reads hit 4 banks
constexpr int kMaxThreads = 512;  // conv CTAs: 8 threads per output column (4 channels each), columns looped past 64
constexpr int kTrunkSplits = kNumSMs;  // FIXED: the trunk's K split must not follow the batch
constexpr int kTrunkThreads = 256;
constexpr int kFinishThreads = 128;
constexpr size_t kMaxSmem = 227 * 1024;

// Layer 1 on uint8 frames [N, C, H, H]: out NHWC [N, Ho, Ho, 32].  k = c * 9 + ky * 3 + kx (the reference's [32, C, 3, 3]).
template <int R>
__global__ void __launch_bounds__(kMaxThreads) act_conv_s2_kernel(const unsigned char* __restrict__ obs, int C, int H,
                                                                  const float* __restrict__ W, int ldw,
                                                                  const float* __restrict__ bias, float* __restrict__ out) {
  extern __shared__ __align__(16) float sm[];
  const int Ho = (H - 3) / 2 + 1, K = C * 9, rows_in = 2 * R + 1;
  float* wT = sm;                 // [K][kWPitch]
  float* lut = wT + K * kWPitch;  // [256]
  float* xs = lut + 256;          // [C][2R + 1][H]
  const int n = blockIdx.y, oy0 = blockIdx.x * R;
  // obs / 255.0 - 0.5 op by op like torch (the same table as im2col_u8_aug_kernel, conv.cu)
  for (int p = threadIdx.x; p < 256; p += blockDim.x) lut[p] = __fsub_rn(__fdiv_rn((float)p, 255.0f), 0.5f);
  for (int i = threadIdx.x; i < 32 * K; i += blockDim.x) {
    const int co = i / K, k = i - co * K;
    wT[k * kWPitch + co] = __ldg(W + (size_t)co * ldw + k);
  }
  __syncthreads();
  const unsigned char* img = obs + (size_t)n * C * H * H;
  for (int i = threadIdx.x; i < C * rows_in * H; i += blockDim.x) {
    const int cr = i / H, x = i - cr * H, c = cr / rows_in, iy = 2 * oy0 + cr - c * rows_in;
    xs[i] = iy < H ? lut[img[((size_t)c * H + iy) * H + x]] : 0.f;
  }
  __syncthreads();
  const int cg = threadIdx.x & 7;
  const float4 b = *reinterpret_cast<const float4*>(bias + cg * 4);
  for (int x = threadIdx.x >> 3; x < Ho; x += blockDim.x >> 3) {
    float acc[R][4];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[r][i] = 0.f;
    for (int c = 0; c < C; ++c) {
      const float* xc = xs + c * rows_in * H + 2 * x;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int ky = t / 3, kx = t % 3;
        const float4 w = *reinterpret_cast<const float4*>(wT + (c * 9 + t) * kWPitch + cg * 4);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float v = xc[(2 * r + ky) * H + kx];
          acc[r][0] = fmaf(v, w.x, acc[r][0]);
          acc[r][1] = fmaf(v, w.y, acc[r][1]);
          acc[r][2] = fmaf(v, w.z, acc[r][2]);
          acc[r][3] = fmaf(v, w.w, acc[r][3]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int oy = oy0 + r;
      if (oy >= Ho) break;
      const float4 o = make_float4(fmaxf(__fadd_rn(acc[r][0], b.x), 0.f), fmaxf(__fadd_rn(acc[r][1], b.y), 0.f),
                                   fmaxf(__fadd_rn(acc[r][2], b.z), 0.f), fmaxf(__fadd_rn(acc[r][3], b.w), 0.f));
      *reinterpret_cast<float4*>(out + (((size_t)n * Ho + oy) * Ho + x) * 32 + cg * 4) = o;
    }
  }
}

// Layers 2-4, 3x3 stride 1, 32 -> 32 on NHWC [N, Hi, Hi, 32].  k = (ky * 3 + kx) * 32 + c (the stored layout).
// feat = 0: out NHWC [N, Ho, Ho, 32];  feat = 1: out [N, 32 * Ho * Ho] in the reference's (channel, row, column) flatten
// order, the column order of actor.trunk.0.weight.
template <int R>
__global__ void __launch_bounds__(kMaxThreads) act_conv_s1_kernel(const float* __restrict__ in, int Hi,
                                                                  const float* __restrict__ W, int ldw,
                                                                  const float* __restrict__ bias, float* __restrict__ out,
                                                                  int feat) {
  extern __shared__ __align__(16) float sm[];
  const int Ho = Hi - 2;
  float* wT = sm;                  // [288][kWPitch]
  float* xs = wT + 288 * kWPitch;  // [R + 2][Hi][kXPitch]
  const int n = blockIdx.y, oy0 = blockIdx.x * R;
  for (int i = threadIdx.x; i < 32 * 288; i += blockDim.x) {
    const int co = i / 288, k = i - co * 288;
    wT[k * kWPitch + co] = __ldg(W + (size_t)co * ldw + k);
  }
  const float* src = in + ((size_t)n * Hi + oy0) * Hi * 32;
  const int valid = min(R + 2, Hi - oy0) * Hi * 32;
  for (int i = threadIdx.x; i < (R + 2) * Hi * 32; i += blockDim.x)
    xs[(i >> 5) * kXPitch + (i & 31)] = i < valid ? __ldg(src + i) : 0.f;
  __syncthreads();
  const int cg = threadIdx.x & 7;
  const float4 b = *reinterpret_cast<const float4*>(bias + cg * 4);
  const float bb[4] = {b.x, b.y, b.z, b.w};
  for (int x = threadIdx.x >> 3; x < Ho; x += blockDim.x >> 3) {
    float acc[R][4];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[r][i] = 0.f;
#pragma unroll 1
    for (int t = 0; t < 9; ++t) {
      const int ky = t / 3, kx = t % 3;
      const float* xp = xs + (ky * Hi + x + kx) * kXPitch;
      const float* wp = wT + t * 32 * kWPitch + cg * 4;
#pragma unroll 8
      for (int c = 0; c < 32; ++c) {
        const float4 w = *reinterpret_cast<const float4*>(wp + c * kWPitch);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float v = xp[r * Hi * kXPitch + c];
          acc[r][0] = fmaf(v, w.x, acc[r][0]);
          acc[r][1] = fmaf(v, w.y, acc[r][1]);
          acc[r][2] = fmaf(v, w.z, acc[r][2]);
          acc[r][3] = fmaf(v, w.w, acc[r][3]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int oy = oy0 + r;
      if (oy >= Ho) break;
      float o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = fmaxf(__fadd_rn(acc[r][i], bb[i]), 0.f);
      if (feat) {
        float* f = out + (size_t)n * 32 * Ho * Ho + (size_t)(cg * 4) * Ho * Ho + oy * Ho + x;
#pragma unroll
        for (int i = 0; i < 4; ++i) f[(size_t)i * Ho * Ho] = o[i];
      } else {
        *reinterpret_cast<float4*>(out + (((size_t)n * Ho + oy) * Ho + x) * 32 + cg * 4) = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
  }
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}

// Float4 columns [c0, c1) of the K range of split s.
__host__ __device__ __forceinline__ int split_begin(int s, int F4) { return (int)((long long)s * F4 / kTrunkSplits); }

// partial[s, n, j] = sum over split s's slice of k of x[n, k] * W[j, k], k ascending.  The CTA copies the feature slice
// of every row ([4 NT rows, <= P4 float4]) into shared memory, then the weight slice in groups of jg rows (all of it at
// once for the shipped widths), each with all its loads in flight at once.  Each thread computes 4 x 4 tiles (rows
// n = nt + NT * a, outputs j = j0 + jt + JT * b: consecutive lanes read consecutive weight rows, which the pitch
// P4 = 1 mod 8 float4 puts on distinct banks).  Neither the grouping nor the tiling changes any output's sum.
__global__ void __launch_bounds__(kTrunkThreads) act_trunk_splitk_kernel(const float* __restrict__ x, int N, int F,
                                                                         const float* __restrict__ W, int ldw, int bn,
                                                                         int P4, int jg, float* __restrict__ partial) {
  extern __shared__ __align__(16) float4 sm4[];
  const int F4 = F / 4, s = blockIdx.x;
  const int c0 = split_begin(s, F4), w4 = split_begin(s + 1, F4) - c0;
  const int NT = (N + 3) / 4, bn4 = (bn + 3) & ~3;
  float4* xs = sm4;                // [4 NT][P4]
  float4* ws = sm4 + 4 * NT * P4;  // [jg][P4]
  const float4* W4 = reinterpret_cast<const float4*>(W);
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (int i = threadIdx.x; i < 4 * NT * w4; i += kTrunkThreads) {
    const int r = i / w4, c = i - r * w4;
    if (r < N) cp_async16(xs + r * P4 + c, x4 + (size_t)r * F4 + c0 + c);
    else xs[r * P4 + c] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int j0 = 0; j0 < bn4; j0 += jg) {
    const int JT = min(jg, bn4 - j0) / 4;
    if (j0 > 0) __syncthreads();  // the previous group's tiles are done with ws
    for (int i = threadIdx.x; i < 4 * JT * w4; i += kTrunkThreads) {
      const int j = i / w4, c = i - j * w4;  // rows [bn, bn4) are the weight's zero padding rows
      cp_async16(ws + j * P4 + c, W4 + (size_t)(j0 + j) * (ldw / 4) + c0 + c);
    }
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::);
    __syncthreads();
    for (int t = threadIdx.x; t < NT * JT; t += kTrunkThreads) {
      const int jt = t % JT, nt = t / JT;
      float acc[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
#pragma unroll 2
      for (int c = 0; c < w4; ++c) {
        float4 xv[4], wv[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) xv[a] = xs[(nt + NT * a) * P4 + c];
#pragma unroll
        for (int b = 0; b < 4; ++b) wv[b] = ws[(jt + JT * b) * P4 + c];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            float v = acc[a][b];
            v = fmaf(xv[a].x, wv[b].x, v);
            v = fmaf(xv[a].y, wv[b].y, v);
            v = fmaf(xv[a].z, wv[b].z, v);
            acc[a][b] = fmaf(xv[a].w, wv[b].w, v);
          }
      }
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int n = nt + NT * a;
        if (n >= N) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int j = j0 + jt + JT * b;
          if (j < bn) partial[((size_t)s * N + n) * bn + j] = acc[a][b];
        }
      }
    }
  }
}

// One CTA per observation: sum the partials in split order, + bias, LayerNorm (eps 1e-5), tanh -> out [N, ld_out]
// (columns [bn, ld_out) zero).  Any bn: the pre-activations are kept in shared memory (bn floats).
__global__ void __launch_bounds__(kFinishThreads) act_trunk_finish_kernel(const float* __restrict__ partial, int N, int bn,
                                                                          const float* __restrict__ bias,
                                                                          const float* __restrict__ gamma,
                                                                          const float* __restrict__ beta,
                                                                          float* __restrict__ out, int ld_out) {
  extern __shared__ float pre[];  // [bn]
  __shared__ float scratch[33];
  const int n = blockIdx.x;
  float sum = 0.f;
  for (int j = threadIdx.x; j < bn; j += kFinishThreads) {
    const float* p = partial + (size_t)n * bn + j;
    float v = 0.f;
#pragma unroll 8
    for (int s = 0; s < kTrunkSplits; ++s) v = __fadd_rn(v, p[(size_t)s * N * bn]);
    v = __fadd_rn(v, bias[j]);
    pre[j] = v;
    sum += v;
  }
  const float mean = block_sum<kFinishThreads>(sum, scratch) / (float)bn;
  float sq = 0.f;
  for (int j = threadIdx.x; j < bn; j += kFinishThreads) {
    const float d = pre[j] - mean;
    sq = fmaf(d, d, sq);
  }
  const float rs = 1.0f / sqrtf(block_sum<kFinishThreads>(sq, scratch) / (float)bn + 1e-5f);
  for (int j = threadIdx.x; j < ld_out; j += kFinishThreads)
    out[(size_t)n * ld_out + j] = j < bn ? tanhf(fmaf((pre[j] - mean) * rs, gamma[j], beta[j])) : 0.f;
}

size_t conv_s2_smem(int C, int H, int R) { return sizeof(float) * ((size_t)C * 9 * kWPitch + 256 + (size_t)C * (2 * R + 1) * H); }
size_t conv_s1_smem(int Hi, int R) { return sizeof(float) * (288 * kWPitch + (size_t)(R + 2) * Hi * kXPitch); }
int trunk_pitch4(int F) {  // float4 pitch of the trunk kernel's slices: >= the widest slice, = 1 (mod 8)
  const int w4 = (F / 4 + kTrunkSplits - 1) / kTrunkSplits;
  return w4 + ((1 - w4) % 8 + 8) % 8;
}
size_t trunk_smem(int rows, int jg, int F) { return sizeof(float4) * (size_t)(4 * ((rows + 3) / 4) + jg) * trunk_pitch4(F); }
int conv_threads(int Ho) { return 8 * std::min(Ho, kMaxThreads / 8); }

}  // namespace

PixelPolicy::PixelPolicy(int channels, int height, int action_dim, const PixelPolicyWeights& w, cudaStream_t s)
    : C_(channels), H_(height), A_(action_dim), LA_(round_up32(action_dim)), bn_(w.trunk.out), LB_(round_up32(w.trunk.out)),
      hid_(w.policy[0].out), frame_bytes_((size_t)channels * height * height), w_(w), stream_(s) {
  hw_[0] = (H_ - 3) / 2 + 1;
  for (int l = 1; l < 4; ++l) hw_[l] = hw_[l - 1] - 2;
  const int F = 32 * hw_[3] * hw_[3];
  RLREP_CHECK(hw_[3] > 0, "pixel act: frame height out of range");
  RLREP_CHECK(bn_ > 0 && w.trunk.in == F && w.trunk.ld % 4 == 0 && w.trunk.out_alloc >= 4 * ((bn_ + 3) / 4),
              "pixel act: trunk shape");
  RLREP_CHECK(w.policy[0].in == bn_ && w.policy[1].in == hid_ && w.policy[2].in == hid_ && w.policy[2].out == A_,
              "pixel act: policy shapes");
  // Rows per pass: kPixelActRows unless the trunk's feature slices of that many rows (plus 4 weight rows) would not fit
  // in shared memory; then weight rows per trunk pass: all of them when they fit (the shipped widths), else groups.
  const size_t row_bytes = sizeof(float4) * trunk_pitch4(F);
  chunk_ = kPixelActRows;
  while (chunk_ > 4 && (size_t)(chunk_ + 4) * row_bytes > kMaxSmem) chunk_ -= 4;
  RLREP_CHECK((size_t)(chunk_ + 4) * row_bytes <= kMaxSmem, "pixel act: frames too large for the trunk kernel");
  jg_ = std::min(4 * ((bn_ + 3) / 4), (int)((kMaxSmem / row_bytes - chunk_) & ~size_t(3)));
  const size_t s2 = conv_s2_smem(C_, H_, 2), s1 = conv_s1_smem(hw_[0], 2), tr = trunk_smem(chunk_, jg_, F);
  RLREP_CHECK(std::max({s2, s1, tr}) <= kMaxSmem, "pixel act: frames too large for the convolution kernels");
  RLREP_CUDA(cudaFuncSetAttribute(act_conv_s2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2));
  RLREP_CUDA(cudaFuncSetAttribute(act_conv_s2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2));
  RLREP_CUDA(cudaFuncSetAttribute(act_conv_s1_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1));
  RLREP_CUDA(cudaFuncSetAttribute(act_conv_s1_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1));
  RLREP_CUDA(cudaFuncSetAttribute(act_trunk_splitk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tr));
  gemm_.init(PREC_FP32, 0);
}

PixelPolicy::~PixelPolicy() {
  if (stage_host_) cudaFreeHost(stage_host_);
  if (out_host_) cudaFreeHost(out_host_);
}

// Nothing is allocated before the first act; the arena then grows to the largest chunk seen (at most chunk_ rows).
void PixelPolicy::reserve(int rows) {
  if (rows <= cap_) return;
  RLREP_CUDA(cudaStreamSynchronize(stream_));
  arena_.release();
  if (stage_host_) RLREP_CUDA(cudaFreeHost(stage_host_));
  if (out_host_) RLREP_CUDA(cudaFreeHost(out_host_));
  stage_host_ = nullptr;
  out_host_ = nullptr;
  cap_ = rows;
  const size_t r = (size_t)rows;
  arena_.want(&frames_, r * frame_bytes_);
  arena_.want(&act_a_, r * hw_[0] * hw_[0] * 32);  // layers 1 and 3
  arena_.want(&act_b_, r * hw_[1] * hw_[1] * 32);  // layer 2
  arena_.want(&feat_, r * 32 * hw_[3] * hw_[3]);
  arena_.want(&partial_, (size_t)kTrunkSplits * r * bn_);
  arena_.want(&th_, r * LB_);
  arena_.want(&h1_, r * hid_);
  arena_.want(&h2_, r * hid_);
  arena_.want(&raw_, r * LA_);
  arena_.want(&mu_, r * A_);
  arena_.want(&eps_, r * A_);
  arena_.want(&action_, r * A_);
  arena_.commit();
  RLREP_CUDA(cudaMallocHost(&stage_host_, r * frame_bytes_ + 16 + r * A_ * sizeof(float)));
  RLREP_CUDA(cudaMallocHost(&out_host_, r * A_ * sizeof(float)));
}

void PixelPolicy::act(const unsigned char* obs, const float* eps_host, float stddev, int n, float* actions_host) {
  RLREP_CHECK(n > 0 && obs != nullptr && actions_host != nullptr, "bad act arguments");
  cudaStream_t s = stream_;
  const bool on_device = is_device_pointer(obs);
  reserve(std::min(n, chunk_));
  float* eps_stage = reinterpret_cast<float*>(stage_host_ + ((cap_ * frame_bytes_ + 15) & ~size_t(15)));
  for (int r0 = 0; r0 < n; r0 += chunk_) {
    const int rows = std::min(chunk_, n - r0);
    const size_t bytes = (size_t)rows * frame_bytes_, ebytes = (size_t)rows * A_ * sizeof(float);
    const unsigned char* src = obs + (size_t)r0 * frame_bytes_;
    if (on_device) {
      RLREP_CUDA(cudaMemcpyAsync(frames_, src, bytes, cudaMemcpyDeviceToDevice, s));
    } else {
      unsigned char* cursor = stage_host_;
      stage_h2d(cursor, frames_, src, bytes, s);
    }
    if (eps_host) {
      std::memcpy(eps_stage, eps_host + (size_t)r0 * A_, ebytes);
      RLREP_CUDA(cudaMemcpyAsync(eps_, eps_stage, ebytes, cudaMemcpyHostToDevice, s));
    } else {
      RLREP_CUDA(cudaMemsetAsync(eps_, 0, ebytes, s));  // the mean: x = mu + 0 * 0, clamped like a sample
    }
    forward(rows, eps_host ? stddev : 0.f);
    RLREP_CUDA(cudaMemcpyAsync(out_host_, action_, ebytes, cudaMemcpyDeviceToHost, s));
    RLREP_CUDA(cudaStreamSynchronize(s));  // also frees the pinned staging for the next chunk
    std::memcpy(actions_host + (size_t)r0 * A_, out_host_, ebytes);
  }
}

void PixelPolicy::forward(int rows, float stddev) {
  cudaStream_t s = stream_;
  const int F = 32 * hw_[3] * hw_[3];
  // Bands of two output rows once there are enough of them to fill the SMs, else one (N = 1: 35-41 CTAs per layer).
  const int R = rows * ((hw_[1] + 1) / 2) >= kNumSMs ? 2 : 1;
  {
    const Linear& l = w_.conv[0];
    const dim3 grid(ceil_div(hw_[0], R), rows);
    const size_t smem = conv_s2_smem(C_, H_, R);
    if (R == 2) act_conv_s2_kernel<2><<<grid, conv_threads(hw_[0]), smem, s>>>(frames_, C_, H_, l.W, l.ld, l.b, act_a_);
    else act_conv_s2_kernel<1><<<grid, conv_threads(hw_[0]), smem, s>>>(frames_, C_, H_, l.W, l.ld, l.b, act_a_);
    RLREP_LAUNCHED_W("act_conv_s2", s, (double)rows * frame_bytes_ + 4.0 * rows * hw_[0] * hw_[0] * 32,
                     2.0 * rows * hw_[0] * hw_[0] * 32 * C_ * 9);
  }
  const float* ins[3] = {act_a_, act_b_, act_a_};
  float* outs[3] = {act_b_, act_a_, feat_};
  for (int l = 1; l < 4; ++l) {
    const Linear& w = w_.conv[l];
    const int Hi = hw_[l - 1], Ho = hw_[l];
    const dim3 grid(ceil_div(Ho, R), rows);
    const size_t smem = conv_s1_smem(Hi, R);
    const int feat = l == 3 ? 1 : 0;
    if (R == 2) act_conv_s1_kernel<2><<<grid, conv_threads(Ho), smem, s>>>(ins[l - 1], Hi, w.W, w.ld, w.b, outs[l - 1], feat);
    else act_conv_s1_kernel<1><<<grid, conv_threads(Ho), smem, s>>>(ins[l - 1], Hi, w.W, w.ld, w.b, outs[l - 1], feat);
    RLREP_LAUNCHED_W("act_conv_s1", s, 4.0 * rows * (Hi * Hi + Ho * Ho) * 32, 2.0 * rows * Ho * Ho * 32 * 288);
  }
  act_trunk_splitk_kernel<<<kTrunkSplits, kTrunkThreads, trunk_smem(rows, jg_, F), s>>>(
      feat_, rows, F, w_.trunk.W, w_.trunk.ld, bn_, trunk_pitch4(F), jg_, partial_);
  RLREP_LAUNCHED_W("act_trunk_splitk", s, 4.0 * ((double)bn_ * F + (double)rows * F + (double)kTrunkSplits * rows * bn_),
                   2.0 * rows * bn_ * F);
  act_trunk_finish_kernel<<<rows, kFinishThreads, bn_ * sizeof(float), s>>>(partial_, rows, bn_, w_.trunk.b, w_.ln_w, w_.ln_b, th_, LB_);
  RLREP_LAUNCHED("act_trunk_finish", s);
  linear_fwd(gemm_, s, rows, Mat{th_, LB_}, w_.policy[0], ACT_RELU, h1_, hid_);
  linear_fwd(gemm_, s, rows, Mat{h1_, hid_}, w_.policy[1], ACT_RELU, h2_, hid_);
  linear_fwd(gemm_, s, rows, Mat{h2_, hid_}, w_.policy[2], ACT_NONE, raw_, LA_);
  launch_trunc_normal_sample(raw_, LA_, rows, A_, eps_, stddev, INFINITY, mu_, action_, A_, s);  // clip=None
}

}  // namespace rlrep

// Non-GEMM kernels of the update step.  See kernels.cuh for the contract of each launcher.
#include <cmath>

#include "common.cuh"
#include "epilogue.cuh"
#include "kernels.cuh"
#include "ptx.cuh"
#include "reduce.cuh"

namespace rlrep {

namespace {

// ------------------------------------------------------------------------------------------- tick
__device__ __forceinline__ AdamHyper adam_hyper(double lr, long long t) {
  // torch.optim.Adam (single-tensor path): step_size = lr / (1 - beta1^t); denom uses sqrt(1 - beta2^t).
  const double bc1 = 1.0 - pow(0.9, (double)t);
  const double bc2 = 1.0 - pow(0.999, (double)t);
  AdamHyper h;
  h.step_size = (float)(lr / bc1);
  h.bc2_sqrt = (float)sqrt(bc2);
  return h;
}

template <bool MEMBERS>
__global__ void tick_kernel(Control* c, const TickParams p, long long mstride) {
  // One warp: every lane reads the counters, then each of the (k_feat + 5) independent results -- two double-precision
  // pow() each -- is computed by its own lane instead of one after the other (7.5 us -> ~2 us at the head of every update).
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const int lane = threadIdx.x;
  if (blockIdx.x != 0 || lane >= 32) return;
  c = member_ptr(c, member_offset<MEMBERS>(mstride));
  const long long t_feat = c->t_feat, t_critic = c->t_critic, t_actor = c->t_actor, t_alpha = c->t_alpha;
  const int steps = c->steps + 1;
  const double log_alpha = c->log_alpha;
  __syncwarp();
  const int k = p.k_feat;
  if (lane < k) c->feat[lane] = adam_hyper(p.lr_feat, t_feat + lane + 1);
  if (lane == k && p.critic_steps) c->critic = adam_hyper(p.lr_critic, t_critic + 1);
  if (lane == k + 1) c->actor = adam_hyper(p.lr_actor, t_actor + 1);
  if (lane == k + 2) c->alpha_step_size = p.lr_alpha / (1.0 - pow(0.9, (double)(t_alpha + 1)));
  if (lane == k + 3) c->alpha_bc2_sqrt = sqrt(1.0 - pow(0.999, (double)(t_alpha + 1)));
  if (lane == k + 4) {
    c->alpha = (float)exp(log_alpha);
    c->steps = steps;
    c->polyak_critic = (steps % p.period == 0) ? 1 : 0;
    c->t_feat = t_feat + k;
    if (p.critic_steps) c->t_critic = t_critic + 1;
    c->t_actor = t_actor + 1;
    c->t_alpha = t_alpha + 1;
  }
}

// ------------------------------------------------------------------------------------------- ring
template <bool MEMBERS>
__global__ void gather_kernel(const float4* __restrict__ ring, int rec4, const long long* __restrict__ idx, int B,
                              float4* __restrict__ out, const float* const* ring_slot, long long mstride) {
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const long long off = member_offset<MEMBERS>(mstride);
  if constexpr (MEMBERS) ring = reinterpret_cast<const float4*>(*member_ptr(ring_slot, off));
  idx = member_ptr(idx, off);
  out = member_ptr(out, off);
  const int total = B * rec4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / rec4, c = i - b * rec4;
    out[i] = __ldg(ring + (size_t)idx[b] * rec4 + c);
  }
}
__global__ void ring_write_kernel(float4* __restrict__ ring, int rec4, long long capacity, long long start,
                                  const float4* __restrict__ rows, int n) {
  const int total = n * rec4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / rec4, c = i - b * rec4;
    ring[(size_t)((start + b) % capacity) * rec4 + c] = rows[i];
  }
}

// ------------------------------------------------------------------------------------------- contrastive CE
// One CTA per row: online max/sum pass, then rewrite the row as the CE gradient.
__global__ void __launch_bounds__(256) ce_rows_kernel(float* __restrict__ logits, int ld, int cols, int diag_off,
                                                      float inv_batch, float* __restrict__ loss_rows) {
  __shared__ float scratch[33];
  const int row = blockIdx.x;
  float* l = logits + (size_t)row * ld;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < cols; j += 256) mx = fmaxf(mx, l[j]);
  mx = block_max<256>(mx, scratch);
  float sum = 0.f;
  for (int j = threadIdx.x; j < cols; j += 256) sum += expf(l[j] - mx);
  sum = block_sum<256>(sum, scratch);
  const float lse = mx + logf(sum);
  const int dj = diag_off + row;  // column of this row's positive
  if (threadIdx.x == 0) loss_rows[row] = lse - l[dj];
  __syncthreads();
  for (int j = threadIdx.x; j < cols; j += 256) {
    const float pr = expf(l[j] - lse);
    l[j] = (pr - (j == dj ? 1.f : 0.f)) * inv_batch;
  }
}

// ------------------------------------------------------------------------------------------- N = 1 heads
// One 128-thread CTA per (row, job): 256 rows spread over 256+ CTAs, every thread has its few 128-bit loads in flight
// at once, then a fixed-order block reduction.  Two jobs (the twin Q heads) share one launch through blockIdx.y.
struct RowDotJobs {
  RowDotJob j[2];
};
template <bool MEMBERS>
__global__ void __launch_bounds__(128) rowdot_kernel(const RowDotJobs jobs, int rows, long long mstride) {
  __shared__ float scratch[33];
  const long long off = member_offset<MEMBERS>(mstride);
  const RowDotJob& jb = jobs.j[blockIdx.y];
  const float* X = member_ptr(jb.X, off);
  const int row = blockIdx.x;
  const float* x = X + (size_t)row * jb.ld;
  const float* w = member_ptr(jb.w, off);
  const int D = jb.D;
  float acc = 0.f;
  if (((jb.ld | D) & 3) == 0 && ((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(w)) & 15) == 0) {
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* w4 = reinterpret_cast<const float4*>(w);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
    for (int j = threadIdx.x; j < D / 4; j += 128) {
      const float4 xv = x4[j];
      const float4 wv = __ldg(w4 + j);
      a0 = fmaf(xv.x, wv.x, a0); a1 = fmaf(xv.y, wv.y, a1); a2 = fmaf(xv.z, wv.z, a2); a3 = fmaf(xv.w, wv.w, a3);
    }
    acc = (a0 + a1) + (a2 + a3);
  } else {
    for (int j = threadIdx.x; j < D; j += 128) acc = fmaf(x[j], __ldg(w + j), acc);
  }
  acc = block_sum<128>(acc, scratch);
  if (threadIdx.x == 0) member_ptr(jb.y, off)[row] = acc + (jb.b ? __ldg(member_ptr(jb.b, off)) : 0.f);
}

// 32 columns x 8 row-slices per CTA; fixed-order smem reduction across the slices.
template <bool MEMBERS>
__global__ void __launch_bounds__(256) colreduce_kernel(const float* __restrict__ X, int ld, int rows, int cols,
                                                        const float* __restrict__ u, float* __restrict__ out,
                                                        int accumulate, long long mstride) {
  __shared__ float part[8][33];
  const long long off = member_offset<MEMBERS>(mstride);
  X = member_ptr(X, off); u = member_ptr(u, off); out = member_ptr(out, off);
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  float acc = 0.f;
  if (j < cols) {
    for (int i = ty; i < rows; i += 8) {
      const float x = X[(size_t)i * ld + j];
      acc = u ? fmaf(__ldg(u + i), x, acc) : acc + x;
    }
  }
  part[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && j < cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += part[k][tx];
    out[j] = accumulate ? out[j] + t : t;
  }
}

// Column sums over very tall matrices (conv bias gradients: 4e5 rows x 32 columns): stage 1 reduces a row chunk per
// CTA into partial[chunk, cols], stage 2 sums the chunks in a fixed order.
__global__ void __launch_bounds__(256) colsum_tall_stage1_kernel(const float* __restrict__ X, int ld, long long rows,
                                                                 int cols, int rows_per_cta, float* __restrict__ partial) {
  __shared__ float part[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < rows ? r0 + rows_per_cta : rows;
  float acc = 0.f;
  if (j < cols)
    for (long long i = r0 + ty; i < r1; i += 8) acc += X[i * ld + j];
  part[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && j < cols) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) t += part[q][tx];
    partial[(long long)blockIdx.y * cols + j] = t;
  }
}
// The conv-shaped case (32 dense columns: the bias gradients of the pixel agents' layers, ~430k rows): float4 loads, 32 rows
// per trip and four trips in flight per thread -- the one-load-per-thread loop above leaves HBM waiting on latency (31 us for
// 55 MB).  Fixed summation order per thread, then over the 32 row groups.
__global__ void __launch_bounds__(256) colsum_tall32_stage1_kernel(const float4* __restrict__ X, long long rows,
                                                                   int rows_per_cta, float* __restrict__ partial) {
  __shared__ float4 part[32][9];
  const int c4 = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < rows ? r0 + rows_per_cta : rows;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  long long i = r0 + rg;
  for (; i + 96 < r1; i += 128) {
    const float4 a = X[i * 8 + c4], b = X[(i + 32) * 8 + c4], c = X[(i + 64) * 8 + c4], d = X[(i + 96) * 8 + c4];
    acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
    acc.x += c.x; acc.y += c.y; acc.z += c.z; acc.w += c.w;
    acc.x += d.x; acc.y += d.y; acc.z += d.z; acc.w += d.w;
  }
  for (; i < r1; i += 32) {
    const float4 a = X[i * 8 + c4];
    acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
  }
  part[rg][c4] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
    for (int q = 0; q < 32; ++q) {
      const float4 a = part[q][threadIdx.x];
      t.x += a.x; t.y += a.y; t.z += a.z; t.w += a.w;
    }
    reinterpret_cast<float4*>(partial + (long long)blockIdx.y * 32)[threadIdx.x] = t;
  }
}
// 32 columns x 32 chunk-slices per 1024-thread CTA: every slice adds its chunks with four independent accumulators (the loads
// of a slice are all in flight together; with 8 slices and one accumulator 2,368 partials took 10 us), then a fixed-order
// combination of the 32 slices.
__global__ void __launch_bounds__(1024) colsum_tall_stage2_kernel(const float* __restrict__ partial, int chunks, int cols,
                                                                  float* __restrict__ out) {
  __shared__ float part[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
  if (j < cols) {
    int c = ty;
    for (; c + 96 < chunks; c += 128) {
      t0 += partial[(long long)c * cols + j];
      t1 += partial[(long long)(c + 32) * cols + j];
      t2 += partial[(long long)(c + 64) * cols + j];
      t3 += partial[(long long)(c + 96) * cols + j];
    }
    for (; c < chunks; c += 32) t0 += partial[(long long)c * cols + j];
  }
  part[ty][tx] = (t0 + t1) + (t2 + t3);
  __syncthreads();
  if (ty == 0 && j < cols) {
    float v = 0.f;
#pragma unroll
    for (int q = 0; q < 32; ++q) v += part[q][tx];
    out[j] = v;
  }
}

struct ColJobs {
  ColJob j[kMaxColJobs];
};
// 32 columns x 32 row-slices per 1024-thread CTA: at B = 256 every thread issues its 8 loads back to back (one
// memory round trip for the whole reduction instead of 32 dependent-latency steps), then a fixed-order smem tree.
template <bool MEMBERS>
__global__ void __launch_bounds__(1024) colreduce_multi_kernel(const ColJobs jobs, long long mstride) {
  __shared__ float part[32][33];
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const long long off = member_offset<MEMBERS>(mstride);
  const ColJob& jb = jobs.j[blockIdx.y];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  if (blockIdx.x * 32 >= jb.cols) return;
  float acc = 0.f;
  if (j < jb.cols) {
    const float* x = member_ptr(jb.X, off) + j;
    int i = ty;
    for (; i + 7 * 32 < jb.rows; i += 8 * 32) {
      float v[8], w[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = x[(size_t)(i + q * 32) * jb.ld];
      if (jb.u) {
#pragma unroll
        for (int q = 0; q < 8; ++q) w[q] = __ldg(member_ptr(jb.u, off) + i + q * 32);
#pragma unroll
        for (int q = 0; q < 8; ++q) acc = fmaf(w[q], v[q], acc);
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) acc += v[q];
      }
    }
    for (; i < jb.rows; i += 32) {
      const float v = x[(size_t)i * jb.ld];
      acc = jb.u ? fmaf(__ldg(member_ptr(jb.u, off) + i), v, acc) : acc + v;
    }
  }
  part[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && j < jb.cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) t += part[k][tx];
    member_ptr(jb.out, off)[j] = t;
  }
}

template <bool MEMBERS>
__global__ void outer_dact_kernel(const float* __restrict__ u, const float* __restrict__ w, int rows, int cols,
                                  const float* __restrict__ aux, int ld_aux, int dact, float* __restrict__ out,
                                  int ld_out, long long mstride) {
  const long long off = member_offset<MEMBERS>(mstride);
  u = member_ptr(u, off); w = member_ptr(w, off); aux = member_ptr(aux, off); out = member_ptr(out, off);
  const size_t total = (size_t)rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i - (size_t)r * cols);
    float v = __ldg(u + r) * __ldg(w + c);
    if (dact != DACT_NONE) v *= apply_dact(aux[(size_t)r * ld_aux + c], dact);
    out[(size_t)r * ld_out + c] = v;
  }
}

// ------------------------------------------------------------------------------------------- feature loss
__global__ void __launch_bounds__(256) feature_loss_finalize_kernel(const float* __restrict__ loss_rows, int rows,
                                                                    const float* __restrict__ pred,
                                                                    const float* __restrict__ reward, int ld_r,
                                                                    float inv_batch, float* __restrict__ dpred,
                                                                    float* __restrict__ metrics) {
  __shared__ float scratch[33];
  float ce = 0.f, se = 0.f;
  for (int i = threadIdx.x; i < rows; i += 256) {
    ce += loss_rows[i];
    const float d = pred[i] - reward[(size_t)i * ld_r];
    se = fmaf(d, d, se);
    dpred[i] = d * inv_batch;
  }
  ce = block_sum<256>(ce, scratch);
  se = block_sum<256>(se, scratch);
  if (threadIdx.x == 0) {
    const float model = ce * inv_batch;
    const float r = 0.5f * (se * inv_batch);
    metrics[0] = model + r;
    metrics[1] = model;
    metrics[2] = r;
  }
}

// ce_rows + rowdot(theta) + feature_loss_finalize in ONE launch (the chained CTRL feature step): CTA i does row i's
// log-sum-exp / gradient rewrite and its reward-head prediction; the last CTA to finish (an arrival counter) adds up the
// per-row terms in the fixed order of feature_loss_finalize_kernel and writes the three metrics.
__global__ void __launch_bounds__(256) contrastive_head_kernel(float* __restrict__ logits, int ld, int cols, int diag_off,
                                                               float inv_batch, const float* __restrict__ z, int ldz, int D,
                                                               const float* __restrict__ theta_w,
                                                               const float* __restrict__ theta_b,
                                                               const float* __restrict__ reward, int ld_r,
                                                               float* __restrict__ loss_rows, float* __restrict__ pred,
                                                               float* __restrict__ dpred, float* __restrict__ metrics,
                                                               unsigned* __restrict__ counter, int rows) {
  __shared__ float scratch[33];
  __shared__ bool last;
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const int row = blockIdx.x;
  float* l = logits + (size_t)row * ld;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < cols; j += 256) mx = fmaxf(mx, l[j]);
  mx = block_max<256>(mx, scratch);
  float sum = 0.f;
  for (int j = threadIdx.x; j < cols; j += 256) sum += expf(l[j] - mx);
  sum = block_sum<256>(sum, scratch);
  const float lse = mx + logf(sum);
  const int dj = diag_off + row;
  const float loss = lse - l[dj];
  __syncthreads();
  for (int j = threadIdx.x; j < cols; j += 256) {
    const float pr = expf(l[j] - lse);
    l[j] = (pr - (j == dj ? 1.f : 0.f)) * inv_batch;
  }
  // reward head: pred = <z_row, theta.w> + theta.b
  const float* x = z + (size_t)row * ldz;
  float acc = 0.f;
  if (((ldz | D) & 3) == 0 && ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(theta_w)) & 15) == 0) {
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* w4 = reinterpret_cast<const float4*>(theta_w);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int j = threadIdx.x; j < D / 4; j += 256) {
      const float4 xv = x4[j];
      const float4 wv = __ldg(w4 + j);
      a0 = fmaf(xv.x, wv.x, a0); a1 = fmaf(xv.y, wv.y, a1); a2 = fmaf(xv.z, wv.z, a2); a3 = fmaf(xv.w, wv.w, a3);
    }
    acc = (a0 + a1) + (a2 + a3);
  } else {
    for (int j = threadIdx.x; j < D; j += 256) acc = fmaf(x[j], __ldg(theta_w + j), acc);
  }
  acc = block_sum<256>(acc, scratch);
  if (threadIdx.x == 0) {
    const float p = acc + __ldg(theta_b);
    loss_rows[row] = loss;
    pred[row] = p;
    dpred[row] = (p - reward[(size_t)row * ld_r]) * inv_batch;
    __threadfence();
    last = atomicAdd(counter, 1u) == (unsigned)(rows - 1);
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  float ce = 0.f, se = 0.f;
  for (int i = threadIdx.x; i < rows; i += 256) {
    ce += __ldcg(loss_rows + i);
    const float d = __ldcg(pred + i) - reward[(size_t)i * ld_r];
    se = fmaf(d, d, se);
  }
  ce = block_sum<256>(ce, scratch);
  se = block_sum<256>(se, scratch);
  if (threadIdx.x == 0) {
    const float model = ce * inv_batch;
    const float r = 0.5f * (se * inv_batch);
    metrics[0] = model + r;
    metrics[1] = model;
    metrics[2] = r;
    *counter = 0;  // re-armed for the next launch
  }
}

// ------------------------------------------------------------------------------------------- actor
constexpr float kLogStdMin = -5.f, kLogStdMax = 2.f;  // sac_agent.py:64

// One warp per row: lane j handles action dimension j (+32, ...), the log-prob terms are warp-reduced, and -- when
// `obs` is given -- all lanes copy the S observation columns in front of the action so that `action - S` becomes the
// contiguous cat(obs, action) row the next network's first layer reads (row pitch lda).  blockIdx.y selects the job.
struct ActorSampleJobs {
  ActorSampleJob j[2];
};
template <bool MEMBERS>
__global__ void actor_sample_kernel(const ActorSampleJobs jobs, int ld_head, int B, int A, int lda, int S,
                                    long long mstride) {
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const ActorSampleJob& jb = jobs.j[blockIdx.y];
  const long long off = member_offset<MEMBERS>(mstride);
  const float* __restrict__ head = member_ptr(jb.head, off);
  const float* __restrict__ eps = member_ptr(jb.eps, off);
  float* __restrict__ action = member_ptr(jb.action, off);
  float* __restrict__ logp = member_ptr(jb.logp, off);
  const float* __restrict__ obs = member_ptr(jb.obs, off);
  const int ld_obs = jb.ld_obs;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* h = head + (size_t)b * ld_head;
  float lp = 0.f;
  for (int j = lane; j < A; j += 32) {
    const float mu = h[j];
    const float ls = kLogStdMin + 0.5f * (kLogStdMax - kLogStdMin) * (tanhf(h[A + j]) + 1.f);
    const float sd = expf(ls);
    const float u = mu + eps[(size_t)b * A + j] * sd;
    const float d = u - mu;
    // Normal.log_prob: -(u-mu)^2 / (2 var) - log(std) - log(sqrt(2 pi))
    const float base = -(d * d) / (2.f * sd * sd) - logf(sd) - 0.91893853320467267f;
    // TanhTransform.log_abs_det_jacobian: 2 (log 2 - u - softplus(-2u)), softplus with torch's threshold 20
    const float z = -2.f * u;
    const float sp = z > 20.f ? z : log1pf(expf(z));
    const float ladj = 2.f * (0.69314718055994531f - u - sp);
    lp += -ladj + base;
    action[(size_t)b * lda + j] = tanhf(u);
  }
  // torch sums the A terms left to right; a shuffle tree differs from that by rounding only (<= 1e-7 relative)
  lp = warp_sum(lp);
  if (lane == 0) logp[b] = lp;
  if (obs != nullptr) {
    float* dst = action + (size_t)b * lda - S;
    const float* src = obs + (size_t)b * ld_obs;
    for (int j = lane; j < S; j += 32) dst[j] = src[j];
  }
}

// select_action (sac_agent.py:89-96) as ONE launch: CTA r evaluates the whole tanh-Gaussian policy for row r of `in`
// ([state (S) | eps (A)] per row, row pitch S + A) -- trunk 0 / 2 / 4 with ELU in shared memory, one warp per output unit
// with the lanes striding over the inputs -- and writes tanh(mu) (explore = 0) or tanh(mu + std * eps).  `in` and `out` may
// be mapped pinned host memory: the kernel then reads the observation and writes the action over PCIe itself and the host
// only synchronises, no copy calls (the path main.py takes once per environment step).
template <bool MEMBERS>
__global__ void __launch_bounds__(256) actor_act_kernel(const float* __restrict__ in, int S, int A, int H,
                                                        const float* __restrict__ W0, int ld0, const float* __restrict__ b0,
                                                        const float* __restrict__ W1, int ld1, const float* __restrict__ b1,
                                                        const float* __restrict__ W2, int ld2, const float* __restrict__ b2,
                                                        int explore, float* __restrict__ out, long long mstride) {
  extern __shared__ float sm[];
  const long long off = member_offset<MEMBERS>(mstride);
  W0 = member_ptr(W0, off); b0 = member_ptr(b0, off); W1 = member_ptr(W1, off); b1 = member_ptr(b1, off);
  W2 = member_ptr(W2, off); b2 = member_ptr(b2, off);
  float* x = sm;                 // [S]
  float* h1 = x + ((S + 3) & ~3);  // [H]
  float* h2 = h1 + H;            // [H]
  float* hd = h2 + H;            // [2A]
  const int row = (MEMBERS ? blockIdx.z * gridDim.x : 0) + blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const float* r = in + (size_t)row * (S + A);
  for (int j = threadIdx.x; j < S; j += blockDim.x) x[j] = r[j];
  __syncthreads();
  auto layer = [&](const float* __restrict__ W, int ld, const float* __restrict__ b, const float* src, int n_in, float* dst,
                   int n_out, bool elu) {
    for (int o = warp; o < n_out; o += nw) {
      const float* w = W + (size_t)o * ld;
      float acc = 0.f;
      for (int j = lane; j < n_in; j += 32) acc = fmaf(__ldg(w + j), src[j], acc);
      acc = warp_sum(acc);
      if (lane == 0) {
        const float v = acc + __ldg(b + o);
        dst[o] = elu ? (v > 0.f ? v : expm1f(v)) : v;
      }
    }
    __syncthreads();
  };
  layer(W0, ld0, b0, x, S, h1, H, true);
  layer(W1, ld1, b1, h1, H, h2, H, true);
  layer(W2, ld2, b2, h2, H, hd, 2 * A, false);
  for (int j = threadIdx.x; j < A; j += blockDim.x) {
    float u = hd[j];
    if (explore) {
      const float ls = kLogStdMin + 0.5f * (kLogStdMax - kLogStdMin) * (tanhf(hd[A + j]) + 1.f);
      u += r[S + j] * expf(ls);
    }
    out[(size_t)row * A + j] = tanhf(u);
  }
}

template <bool MEMBERS>
__global__ void actor_sample_bwd_kernel(const float* __restrict__ head, int ld_head, int B, int A,
                                        const float* __restrict__ eps, const float* __restrict__ d_action, int ldd,
                                        const float* __restrict__ dlogp_scalar, float* __restrict__ dhead, int ld_dh,
                                        long long mstride) {
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const long long off = member_offset<MEMBERS>(mstride);
  head = member_ptr(head, off); eps = member_ptr(eps, off); d_action = member_ptr(d_action, off);
  dlogp_scalar = member_ptr(dlogp_scalar, off); dhead = member_ptr(dhead, off);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * A) return;
  const int b = i / A, j = i - b * A;
  const float* h = head + (size_t)b * ld_head;
  const float glp = *dlogp_scalar;
  const float mu = h[j];
  const float t = tanhf(h[A + j]);
  const float ls = kLogStdMin + 0.5f * (kLogStdMax - kLogStdMin) * (t + 1.f);
  const float sd = expf(ls);
  const float e = eps[i];
  const float a = tanhf(mu + e * sd);
  // dL/du: through a = tanh(u) and through log pi (d(-ladj)/du = 2 tanh(u); the Gaussian term cancels)
  const float du = d_action[(size_t)b * ldd + j] * (1.f - a * a) + glp * 2.f * a;
  const float dsd = du * e - glp / sd;
  dhead[(size_t)b * ld_dh + j] = du;
  dhead[(size_t)b * ld_dh + A + j] = dsd * sd * (0.5f * (kLogStdMax - kLogStdMin)) * (1.f - t * t);
}

// ------------------------------------------------------------------------------------------- critic loss
template <bool MEMBERS>
__global__ void __launch_bounds__(256) td_critic_loss_kernel(const float* __restrict__ reward,
                                                             const float* __restrict__ done, int ld_rd,
                                                             const float* __restrict__ nq1,
                                                             const float* __restrict__ nq2,
                                                             const float* __restrict__ logp2,
                                                             const float* __restrict__ q1, const float* __restrict__ q2,
                                                             int B, int norm_B, float gamma,
                                                             const Control* __restrict__ c, float* __restrict__ dq1,
                                                             float* __restrict__ dq2, float* __restrict__ metrics,
                                                             long long mstride) {
  __shared__ float scratch[33];
  const long long off = member_offset<MEMBERS>(mstride);
  reward = member_ptr(reward, off); done = member_ptr(done, off); nq1 = member_ptr(nq1, off); nq2 = member_ptr(nq2, off);
  logp2 = member_ptr(logp2, off); q1 = member_ptr(q1, off); q2 = member_ptr(q2, off); c = member_ptr(c, off);
  dq1 = member_ptr(dq1, off); dq2 = member_ptr(dq2, off); metrics = member_ptr(metrics, off);
  const float alpha = c->alpha;
  const float inv_b = 1.f / (float)norm_B;
  float l1 = 0.f, l2 = 0.f, s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < B; i += 256) {
    const float nq = fminf(nq1[i], nq2[i]) - alpha * logp2[i];
    const float y = reward[(size_t)i * ld_rd] + (1.f - done[(size_t)i * ld_rd]) * gamma * nq;
    const float e1 = q1[i] - y, e2 = q2[i] - y;
    l1 = fmaf(e1, e1, l1);
    l2 = fmaf(e2, e2, l2);
    s1 += q1[i];
    s2 += q2[i];
    dq1[i] = 2.f * e1 * inv_b;
    dq2[i] = 2.f * e2 * inv_b;
  }
  l1 = block_sum<256>(l1, scratch);
  l2 = block_sum<256>(l2, scratch);
  s1 = block_sum<256>(s1, scratch);
  s2 = block_sum<256>(s2, scratch);
  if (threadIdx.x == 0) {
    metrics[0] = l1 * inv_b;
    metrics[1] = l2 * inv_b;
    metrics[2] = s1 * inv_b;
    metrics[3] = s2 * inv_b;
  }
}

template <bool MEMBERS>
__global__ void __launch_bounds__(256) actor_alpha_loss_kernel(const float* __restrict__ q1,
                                                               const float* __restrict__ q2,
                                                               const float* __restrict__ logp, int B,
                                                               float target_entropy, int learn_alpha, Control* c,
                                                               float* __restrict__ dq1, float* __restrict__ dq2,
                                                               float* __restrict__ dlogp_scalar,
                                                               float* __restrict__ metrics, long long mstride) {
  __shared__ float scratch[33];
  const long long off = member_offset<MEMBERS>(mstride);
  q1 = member_ptr(q1, off); q2 = member_ptr(q2, off); logp = member_ptr(logp, off); c = member_ptr(c, off);
  dq1 = member_ptr(dq1, off); dq2 = member_ptr(dq2, off); dlogp_scalar = member_ptr(dlogp_scalar, off);
  metrics = member_ptr(metrics, off);
  const float alpha = c->alpha;
  const float inv_b = 1.f / (float)B;
  float la = 0.f, ent = 0.f, raw = 0.f;
  for (int i = threadIdx.x; i < B; i += 256) {
    const float a = q1[i], b = q2[i];
    la += alpha * logp[i] - fminf(a, b);
    ent += alpha * (-logp[i] - target_entropy);
    raw += -logp[i] - target_entropy;
    // torch.min backward: the smaller input gets the gradient, a tie splits it
    const float g = -inv_b;
    dq1[i] = a < b ? g : (a == b ? 0.5f * g : 0.f);
    dq2[i] = b < a ? g : (a == b ? 0.5f * g : 0.f);
  }
  la = block_sum<256>(la, scratch);
  ent = block_sum<256>(ent, scratch);
  raw = block_sum<256>(raw, scratch);
  if (threadIdx.x == 0) {
    *dlogp_scalar = alpha * inv_b;
    metrics[0] = la * inv_b;
    const float alpha_loss = ent * inv_b;
    metrics[1] = alpha_loss;
    if (learn_alpha) {
      // autograd: d/d alpha = fp32 mean(-logp - H); d/d log_alpha = that (cast to float64) * exp(log_alpha)
      const double g = (double)(raw * inv_b) * exp(c->log_alpha);
      c->la_m = c->la_m + (1.0 - 0.9) * (g - c->la_m);
      c->la_v = c->la_v * 0.999 + (1.0 - 0.999) * g * g;
      const double denom = sqrt(c->la_v) / c->alpha_bc2_sqrt + 1e-8;
      c->log_alpha = c->log_alpha - c->alpha_step_size * (c->la_m / denom);
    }
    metrics[2] = (float)exp(c->log_alpha);
  }
}

// ------------------------------------------------------------------------------------------- fused SAC heads (chained path)
// The N = 1 heads of the twin critic, the loss on them and the way back to the hidden layer are row-local except for the
// loss means: ONE launch with a CTA per batch row replaces rowdot x2 + td_critic_loss + outer_dact x2 (critic step) and
// rowdot + actor_alpha_loss + outer_dact x2 (actor step); the last CTA to finish (arrival counter) runs the reductions of
// td_critic_loss_kernel / actor_alpha_loss_kernel unchanged, so metrics and the temperature step are bit-identical.
__device__ __forceinline__ float head_dot(const float* __restrict__ x, const float* __restrict__ w, int D, int tid) {
  float acc = 0.f;
  if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w)) & 15) == 0) {
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* w4 = reinterpret_cast<const float4*>(w);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int j = tid; j < D / 4; j += 256) {
      const float4 xv = x4[j];
      const float4 wv = __ldg(w4 + j);
      a0 = fmaf(xv.x, wv.x, a0); a1 = fmaf(xv.y, wv.y, a1); a2 = fmaf(xv.z, wv.z, a2); a3 = fmaf(xv.w, wv.w, a3);
    }
    acc = (a0 + a1) + (a2 + a3);
  } else {
    for (int j = tid; j < D; j += 256) acc = fmaf(x[j], __ldg(w + j), acc);
  }
  return acc;
}
// dhid[row, 0:H] = dq1 * w2 * elu'(hid[row, 0:H]), dhid[row, H:2H] = dq2 * w5 * elu'(hid[row, H:2H])  (outer_dact, ELU_OUT)
__device__ __forceinline__ void head_backward_row(const float* __restrict__ hid, const float* __restrict__ w2,
                                                  const float* __restrict__ w5, float dq1, float dq2, int H,
                                                  float* __restrict__ dhid, int tid) {
  for (int j = tid; j < 2 * H; j += 256) {
    const bool second = j >= H;
    float v = (second ? dq2 : dq1) * __ldg((second ? w5 : w2) + (second ? j - H : j));
    v *= apply_dact(hid[j], DACT_ELU_OUT);
    dhid[j] = v;
  }
}

__global__ void __launch_bounds__(256) critic_td_head_kernel(const CriticHeadArgs a) {
  __shared__ float scratch[33];
  __shared__ float bc[2];
  __shared__ bool last;
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const int row = blockIdx.x, tid = threadIdx.x, H = a.H;
  const float* ht = a.hid_t + (size_t)row * a.ldh;
  const float* h = a.hid + (size_t)row * a.ldh;
  float nq1 = block_sum<256>(head_dot(ht, a.w2t, H, tid), scratch);
  float nq2 = block_sum<256>(head_dot(ht + H, a.w5t, H, tid), scratch);
  float q1 = block_sum<256>(head_dot(h, a.w2, H, tid), scratch);
  float q2 = block_sum<256>(head_dot(h + H, a.w5, H, tid), scratch);
  if (tid == 0) {
    nq1 += __ldg(a.b2t); nq2 += __ldg(a.b5t); q1 += __ldg(a.b2); q2 += __ldg(a.b5);
    const float alpha = a.c->alpha, inv_b = 1.f / (float)a.B;
    const float nq = fminf(nq1, nq2) - alpha * a.logp2[row];
    const float y = a.reward[(size_t)row * a.ld_rd] + (1.f - a.done[(size_t)row * a.ld_rd]) * a.gamma * nq;
    const float e1 = q1 - y, e2 = q2 - y;
    a.nq1[row] = nq1; a.nq2[row] = nq2; a.q1[row] = q1; a.q2[row] = q2;
    bc[0] = 2.f * e1 * inv_b;
    bc[1] = 2.f * e2 * inv_b;
    a.dq1[row] = bc[0];
    a.dq2[row] = bc[1];
  }
  __syncthreads();
  head_backward_row(h, a.w2, a.w5, bc[0], bc[1], H, a.dhid + (size_t)row * a.ld_dh, tid);
  if (tid == 0) {
    __threadfence();
    last = atomicAdd(a.counter, 1u) == (unsigned)(a.B - 1);
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // td_critic_loss_kernel's reductions, same order
  const float alpha = a.c->alpha, inv_b = 1.f / (float)a.B;
  float l1 = 0.f, l2 = 0.f, s1 = 0.f, s2 = 0.f;
  for (int i = tid; i < a.B; i += 256) {
    const float nq = fminf(__ldcg(a.nq1 + i), __ldcg(a.nq2 + i)) - alpha * a.logp2[i];
    const float y = a.reward[(size_t)i * a.ld_rd] + (1.f - a.done[(size_t)i * a.ld_rd]) * a.gamma * nq;
    const float v1 = __ldcg(a.q1 + i), v2 = __ldcg(a.q2 + i);
    const float e1 = v1 - y, e2 = v2 - y;
    l1 = fmaf(e1, e1, l1);
    l2 = fmaf(e2, e2, l2);
    s1 += v1;
    s2 += v2;
  }
  l1 = block_sum<256>(l1, scratch);
  l2 = block_sum<256>(l2, scratch);
  s1 = block_sum<256>(s1, scratch);
  s2 = block_sum<256>(s2, scratch);
  if (tid == 0) {
    a.metrics[0] = l1 * inv_b;
    a.metrics[1] = l2 * inv_b;
    a.metrics[2] = s1 * inv_b;
    a.metrics[3] = s2 * inv_b;
    *a.counter = 0;  // re-armed for the next launch
  }
}

__global__ void __launch_bounds__(256) actor_head_kernel(const ActorHeadArgs a) {
  __shared__ float scratch[33];
  __shared__ float bc[2];
  __shared__ bool last;
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const int row = blockIdx.x, tid = threadIdx.x, H = a.H;
  const float* h = a.hid + (size_t)row * a.ldh;
  float q1 = block_sum<256>(head_dot(h, a.w2, H, tid), scratch);
  float q2 = block_sum<256>(head_dot(h + H, a.w5, H, tid), scratch);
  if (tid == 0) {
    q1 += __ldg(a.b2); q2 += __ldg(a.b5);
    a.q1[row] = q1; a.q2[row] = q2;
    // torch.min backward: the smaller input gets the gradient, a tie splits it
    const float g = -1.f / (float)a.B;
    bc[0] = q1 < q2 ? g : (q1 == q2 ? 0.5f * g : 0.f);
    bc[1] = q2 < q1 ? g : (q1 == q2 ? 0.5f * g : 0.f);
    a.dq1[row] = bc[0];
    a.dq2[row] = bc[1];
  }
  __syncthreads();
  head_backward_row(h, a.w2, a.w5, bc[0], bc[1], H, a.dhid + (size_t)row * a.ld_dh, tid);
  if (tid == 0) {
    __threadfence();
    last = atomicAdd(a.counter, 1u) == (unsigned)(a.B - 1);
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // actor_alpha_loss_kernel's reductions and temperature step, same order
  Control* c = a.c;
  const float alpha = c->alpha, inv_b = 1.f / (float)a.B;
  float la = 0.f, ent = 0.f, raw = 0.f;
  for (int i = tid; i < a.B; i += 256) {
    const float v1 = __ldcg(a.q1 + i), v2 = __ldcg(a.q2 + i);
    la += alpha * a.logp[i] - fminf(v1, v2);
    ent += alpha * (-a.logp[i] - a.target_entropy);
    raw += -a.logp[i] - a.target_entropy;
  }
  la = block_sum<256>(la, scratch);
  ent = block_sum<256>(ent, scratch);
  raw = block_sum<256>(raw, scratch);
  if (tid == 0) {
    *a.dlogp_scalar = alpha * inv_b;
    a.metrics[0] = la * inv_b;
    a.metrics[1] = ent * inv_b;
    if (a.learn_alpha) {
      const double g = (double)(raw * inv_b) * exp(c->log_alpha);
      c->la_m = c->la_m + (1.0 - 0.9) * (g - c->la_m);
      c->la_v = c->la_v * 0.999 + (1.0 - 0.999) * g * g;
      const double denom = sqrt(c->la_v) / c->alpha_bc2_sqrt + 1e-8;
      c->log_alpha = c->log_alpha - c->alpha_step_size * (c->la_m / denom);
    }
    a.metrics[2] = (float)exp(c->log_alpha);
    *a.counter = 0;
  }
}

// Batch-sharded variant of the kernel above (agent_ctrlsac_dp.cu): the rank's rows contribute partial means over the
// GLOBAL batch; the temperature step runs after the partials have been all-reduced.
__global__ void __launch_bounds__(256) actor_loss_partial_kernel(const float* __restrict__ q1,
                                                                 const float* __restrict__ q2,
                                                                 const float* __restrict__ logp, int B, int norm_B,
                                                                 float target_entropy, const Control* __restrict__ c,
                                                                 float* __restrict__ dq1, float* __restrict__ dq2,
                                                                 float* __restrict__ dlogp_scalar,
                                                                 float* __restrict__ partial) {
  __shared__ float scratch[33];
  const float alpha = c->alpha;
  const float inv_b = 1.f / (float)norm_B;
  float la = 0.f, raw = 0.f;
  for (int i = threadIdx.x; i < B; i += 256) {
    const float a = q1[i], b = q2[i];
    la += alpha * logp[i] - fminf(a, b);
    raw += -logp[i] - target_entropy;
    const float g = -inv_b;
    dq1[i] = a < b ? g : (a == b ? 0.5f * g : 0.f);
    dq2[i] = b < a ? g : (a == b ? 0.5f * g : 0.f);
  }
  la = block_sum<256>(la, scratch);
  raw = block_sum<256>(raw, scratch);
  if (threadIdx.x == 0) {
    *dlogp_scalar = alpha * inv_b;
    partial[0] = la * inv_b;   // this rank's share of mean(alpha * logp - min(q1, q2))
    partial[1] = raw * inv_b;  // this rank's share of mean(-logp - target_entropy)
  }
}
__global__ void alpha_step_kernel(const float* __restrict__ reduced, int learn_alpha, Control* c,
                                  float* __restrict__ metrics) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  metrics[0] = reduced[0];
  metrics[1] = c->alpha * reduced[1];  // mean(alpha * (-logp - H).detach())
  if (learn_alpha) {
    const double g = (double)reduced[1] * exp(c->log_alpha);
    c->la_m = c->la_m + (1.0 - 0.9) * (g - c->la_m);
    c->la_v = c->la_v * 0.999 + (1.0 - 0.999) * g * g;
    const double denom = sqrt(c->la_v) / c->alpha_bc2_sqrt + 1e-8;
    c->log_alpha = c->log_alpha - c->alpha_step_size * (c->la_m / denom);
  }
  metrics[2] = (float)exp(c->log_alpha);
}
// x[i, j] *= dact(aux[i, j])  (the tanh derivative of mu after the reduce-scatter of its gradient)
__global__ void mul_dact_kernel(float* __restrict__ x, const float* __restrict__ aux, size_t n, int dact) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    x[i] *= apply_dact(aux[i], dact);
}

// ------------------------------------------------------------------------------------------- Adam + Polyak
__device__ __forceinline__ float adam_elem(float& p, float g, float& m, float& v, float ss, float bc2s) {
  // torch/optim/adam.py _single_tensor_adam: lerp, mul+addcmul, sqrt/bc2_sqrt + eps, addcdiv.
  constexpr float w1 = (float)(1.0 - 0.9), b2 = 0.999f, w2 = (float)(1.0 - 0.999), eps = 1e-8f;
  m = fmaf(w1, g - m, m);
  v = fmaf(w2 * g, g, v * b2);
  const float denom = sqrtf(v) / bc2s + eps;
  p = p - ss * (m / denom);
  return p;
}

template <bool MEMBERS>
__global__ void __launch_bounds__(256) adam_polyak_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                                          float4* __restrict__ m, float4* __restrict__ v, size_t n4,
                                                          const AdamHyper* __restrict__ hyper,
                                                          float4* __restrict__ target, size_t n4_polyak, float tau,
                                                          const int* __restrict__ polyak_flag, long long mstride) {
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const long long off = member_offset<MEMBERS>(mstride);
  p = member_ptr(p, off); g = member_ptr(g, off); m = member_ptr(m, off); v = member_ptr(v, off);
  hyper = member_ptr(hyper, off); target = member_ptr(target, off); polyak_flag = member_ptr(polyak_flag, off);
  const float ss = hyper->step_size, bc2s = hyper->bc2_sqrt;
  const bool do_polyak = target != nullptr && (polyak_flag == nullptr || *polyak_flag != 0);
  const float omt = 1.f - tau;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    // m, v, g and the Polyak target are touched once per optimiser step: stream them through L2 (evict-first) so the
    // weights p -- which every GEMM until the next step re-reads -- stay L2-resident instead of being flushed by the
    // optimiser's own 200 MB sweep.
    float4 pv = p[i], mv = __ldcs(m + i), vv = __ldcs(v + i);
    const float4 gv = __ldcs(g + i);
    adam_elem(pv.x, gv.x, mv.x, vv.x, ss, bc2s);
    adam_elem(pv.y, gv.y, mv.y, vv.y, ss, bc2s);
    adam_elem(pv.z, gv.z, mv.z, vv.z, ss, bc2s);
    adam_elem(pv.w, gv.w, mv.w, vv.w, ss, bc2s);
    p[i] = pv;
    __stcs(m + i, mv);
    __stcs(v + i, vv);
    if (do_polyak && i < n4_polyak) {
      float4 t = __ldcs(target + i);
      // tau * param + (1 - tau) * target, each op rounded separately (no FMA) like the reference's tensor ops
      t.x = __fadd_rn(__fmul_rn(tau, pv.x), __fmul_rn(omt, t.x));
      t.y = __fadd_rn(__fmul_rn(tau, pv.y), __fmul_rn(omt, t.y));
      t.z = __fadd_rn(__fmul_rn(tau, pv.z), __fmul_rn(omt, t.z));
      t.w = __fadd_rn(__fmul_rn(tau, pv.w), __fmul_rn(omt, t.w));
      __stcs(target + i, t);
    }
  }
}

__global__ void __launch_bounds__(256) polyak_kernel(const float4* __restrict__ p, float4* __restrict__ target,
                                                     size_t n4, float tau, const int* __restrict__ polyak_flag) {
  if (polyak_flag != nullptr && *polyak_flag == 0) return;
  const float omt = 1.f - tau;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 pv = p[i];
    float4 t = target[i];
    t.x = __fadd_rn(__fmul_rn(tau, pv.x), __fmul_rn(omt, t.x));
    t.y = __fadd_rn(__fmul_rn(tau, pv.y), __fmul_rn(omt, t.y));
    t.z = __fadd_rn(__fmul_rn(tau, pv.z), __fmul_rn(omt, t.z));
    t.w = __fadd_rn(__fmul_rn(tau, pv.w), __fmul_rn(omt, t.w));
    target[i] = t;
  }
}

// ------------------------------------------------------------------------------------------- LV-Rep / VL-SAC
constexpr float kLogSigMin = -20.f, kLogSigMax = 2.f;  // networks/vae.py:9-10
__device__ __forceinline__ float clamp_ls(float raw) { return fminf(fmaxf(raw, kLogSigMin), kLogSigMax); }
__device__ __forceinline__ float clamp_grad(float raw) { return (raw >= kLogSigMin && raw <= kLogSigMax) ? 1.f : 0.f; }

struct ColSegments {
  ColSegment s[3];
  int n;
};
__global__ void pack_columns_kernel(const float* __restrict__ in, int ld_in, float* __restrict__ out, int ld_out, int rows,
                                    const ColSegments segs, int width) {
  const size_t total = (size_t)rows * width;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / width);
    int c = (int)(i - (size_t)r * width);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (k < segs.n) {
        if (c < segs.s[k].len) {
          out[(size_t)r * ld_out + segs.s[k].dst + c] = in[(size_t)r * ld_in + segs.s[k].src + c];
          break;
        }
        c -= segs.s[k].len;
      }
    }
  }
}

__global__ void vae_sample_kernel(const float* __restrict__ head, int ld_head, int B, int D, const float* __restrict__ eps,
                                  float* __restrict__ z) {
  const int total = B * D;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / D, d = i - b * D;
    const float* h = head + (size_t)b * ld_head;
    z[i] = h[d] + eps[i] * expf(clamp_ls(h[D + d]));
  }
}

__global__ void __launch_bounds__(256) vae_recon_loss_kernel(const float* __restrict__ xr, int ld_xr,
                                                             const float* __restrict__ next_state,
                                                             const float* __restrict__ reward, int ld_rec, int B, int S,
                                                             float* __restrict__ dxr, float* __restrict__ partial) {
  __shared__ float scratch[33];
  const float gs = 1.f / ((float)B * (float)S), gr = 1.f / (float)B;
  float se_s = 0.f, se_r = 0.f;
  const int total = B * ld_xr;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
    const int b = i / ld_xr, c = i - b * ld_xr;
    float g = 0.f;
    if (c < S) {
      const float d = xr[i] - next_state[(size_t)b * ld_rec + c];
      se_s = fmaf(d, d, se_s);
      g = d * gs;
    } else if (c == S) {
      const float d = xr[i] - reward[(size_t)b * ld_rec];
      se_r = fmaf(d, d, se_r);
      g = d * gr;
    }
    dxr[i] = g;
  }
  se_s = block_sum<256>(se_s, scratch);
  se_r = block_sum<256>(se_r, scratch);
  if (threadIdx.x == 0) {
    partial[2 * blockIdx.x] = se_s;
    partial[2 * blockIdx.x + 1] = se_r;
  }
}

__global__ void __launch_bounds__(256) vae_kl_bwd_kernel(const float* __restrict__ enc_head,
                                                         const float* __restrict__ prior_head, int ld_head, int B, int D,
                                                         const float* __restrict__ eps, const float* __restrict__ dz,
                                                         float* __restrict__ d_enc, float* __restrict__ d_prior,
                                                         float* __restrict__ partial) {
  __shared__ float scratch[33];
  const int total = B * D;
  const float g = 1.f / (float)total;
  float kl_sum = 0.f;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
    const int b = i / D, d = i - b * D;
    const float* he = enc_head + (size_t)b * ld_head;
    const float* hp = prior_head + (size_t)b * ld_head;
    const float m1 = he[d], raw1 = he[D + d], m2 = hp[d], raw2 = hp[D + d];
    const float ls1 = clamp_ls(raw1), ls2 = clamp_ls(raw2);
    const float var1 = expf(2.f * ls1), var2 = expf(2.f * ls2);
    const float diff = m1 - m2;
    const float q = (var1 + diff * diff) / var2;
    kl_sum += ls2 - ls1 + 0.5f * q - 0.5f;
    const float dzi = dz[i];
    const float dm = g * diff / var2;
    d_enc[(size_t)b * ld_head + d] = dzi + dm;
    d_enc[(size_t)b * ld_head + D + d] = (dzi * eps[i] * expf(ls1) + g * (var1 / var2 - 1.f)) * clamp_grad(raw1);
    d_prior[(size_t)b * ld_head + d] = -dm;
    d_prior[(size_t)b * ld_head + D + d] = g * (1.f - q) * clamp_grad(raw2);
  }
  kl_sum = block_sum<256>(kl_sum, scratch);
  if (threadIdx.x == 0) partial[blockIdx.x] = kl_sum;
}

__global__ void vae_finalize_kernel(const float* __restrict__ recon_partial, int n_recon,
                                    const float* __restrict__ kl_partial, int n_kl, int B, int S, int D,
                                    float* __restrict__ metrics) {
  // one warp: lane l adds partials l, l + 32, ... in order, then a fixed shuffle tree (a single thread walking 3 x 296
  // partials was 5+ us at the tail of every feature step)
  if (blockIdx.x != 0 || threadIdx.x >= 32) return;
  float se_s = 0.f, se_r = 0.f, kl = 0.f;
  for (int i = threadIdx.x; i < n_recon; i += 32) { se_s += recon_partial[2 * i]; se_r += recon_partial[2 * i + 1]; }
  for (int i = threadIdx.x; i < n_kl; i += 32) kl += kl_partial[i];
  se_s = warp_sum(se_s);
  se_r = warp_sum(se_r);
  kl = warp_sum(kl);
  if (threadIdx.x != 0) return;
  const float s_loss = 0.5f * (se_s / ((float)B * (float)S));
  const float r_loss = 0.5f * (se_r / (float)B);
  const float ml = r_loss + s_loss;
  const float kl_mean = kl / ((float)B * (float)D);
  metrics[0] = ml + kl_mean;
  metrics[1] = ml;
  metrics[2] = kl_mean;
  metrics[3] = s_loss;
  metrics[4] = r_loss;
}

// x[(b, j), d] = mean[b, d] + exp(clamp(log_std[b, d])) * noise[j, d].  One thread per (b, four columns): the head is read and
// exponentiated once and the NN rows are written as float4 (per element with 64-bit div / mod and NN x the expf this
// took 21 us for a 21 MB write); the scalar kernel keeps unaligned shapes.
__global__ void noise_expand4_kernel(const float* __restrict__ head, int ld_head, int B, int D,
                                     const float* __restrict__ noise, int NN, float* __restrict__ x) {
  const int D4 = D >> 2, total = B * D4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / D4, d = (i - b * D4) << 2;
    const float* h = head + (size_t)b * ld_head;
    const float4 m = *reinterpret_cast<const float4*>(h + d);
    const float4 r = *reinterpret_cast<const float4*>(h + D + d);
    const float4 sd = make_float4(expf(clamp_ls(r.x)), expf(clamp_ls(r.y)), expf(clamp_ls(r.z)), expf(clamp_ls(r.w)));
    float4* out = reinterpret_cast<float4*>(x + ((size_t)b * NN) * D + d);
    for (int j = 0; j < NN; ++j) {
      const float4 n = __ldg(reinterpret_cast<const float4*>(noise + (size_t)j * D + d));
      out[(size_t)j * D4] = make_float4(m.x + sd.x * n.x, m.y + sd.y * n.y, m.z + sd.z * n.z, m.w + sd.w * n.w);
    }
  }
}
__global__ void noise_expand_kernel(const float* __restrict__ head, int ld_head, int B, int D,
                                    const float* __restrict__ noise, int NN, float* __restrict__ x) {
  const size_t total = (size_t)B * NN * D;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const size_t row = i / D;
    const int j = (int)(row % NN), b = (int)(row / NN);
    const float* h = head + (size_t)b * ld_head;
    x[i] = h[d] + expf(clamp_ls(h[D + d])) * __ldg(noise + (size_t)j * D + d);
  }
}

__global__ void noise_expand_bwd_kernel(const float* __restrict__ dx, const float* __restrict__ head, int ld_head, int B,
                                        int D, const float* __restrict__ noise, int NN, float* __restrict__ d_head) {
  const int total = B * D;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / D, d = i - b * D;
    float sm = 0.f, sn = 0.f;
    for (int j = 0; j < NN; ++j) {
      const float g = dx[((size_t)b * NN + j) * D + d];
      sm += g;
      sn = fmaf(g, __ldg(noise + (size_t)j * D + d), sn);
    }
    const float raw = head[(size_t)b * ld_head + D + d];
    d_head[(size_t)b * ld_head + d] = sm;
    d_head[(size_t)b * ld_head + D + d] = sn * expf(clamp_ls(raw)) * clamp_grad(raw);
  }
}

__global__ void group_mean_kernel(const float* __restrict__ hid, int ld, int B, int NN, int C, float* __restrict__ out) {
  const int total = B * C;
  const float inv = 1.f / (float)NN;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / C, c = i - b * C;
    float acc = 0.f;
    for (int j = 0; j < NN; ++j) acc += hid[((size_t)b * NN + j) * ld + c];
    out[i] = acc * inv;
  }
}

__global__ void group_mean_bwd_kernel(const float* __restrict__ dmean, const float* __restrict__ hid, int ld, int B, int NN,
                                      int C, float* __restrict__ dhid, float* __restrict__ colsum_partial) {
  const int total = B * C;
  const float inv = 1.f / (float)NN;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / C, c = i - b * C;
    const float g = dmean[i] * inv;
    float acc = 0.f;
    for (int j = 0; j < NN; ++j) {
      const size_t o = ((size_t)b * NN + j) * ld + c;
      const float v = g * apply_dact(hid[o], DACT_ELU_OUT);
      dhid[o] = v;
      acc += v;
    }
    colsum_partial[i] = acc;
  }
}

__global__ void kgroup_finish_kernel(const float* __restrict__ ws, int groups, int M, int N, int ldw, size_t group_stride,
                                     float* __restrict__ C, int ldc, const Epilogue epi) {
  const size_t total = (size_t)M * N;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int m = (int)(i / N), n = (int)(i - (size_t)m * N);
    float acc = 0.f;
    for (int g = 0; g < groups; ++g) acc += ws[(size_t)g * group_stride + (size_t)m * ldw + n];
    float* cp = C + (size_t)m * ldc + n;
    *cp = epilogue_apply<-1, -1>(epi, acc, m, n, cp);
  }
}

int grid_for(size_t work_items, int threads, int per_sm = 8) {
  size_t blocks = (work_items + threads - 1) / threads;
  const size_t cap = (size_t)kNumSMs * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace

void launch_tick(Control* c, const TickParams& p, cudaStream_t s, Members mb) {
  RLREP_CHECK(p.k_feat <= kMaxFeatureSteps, "too many feature steps per update");
  launch_pdl((mb.n > 1 ? tick_kernel<true> : tick_kernel<false>), dim3(1, 1, mb.n), 32, 0, s, c, p, mb.stride);
  RLREP_LAUNCHED("tick", s);
}

void launch_gather(const float* ring, int rec4, const long long* idx, int B, float* out, cudaStream_t s, Members mb,
                   const float* const* ring_slot) {
  launch_pdl((mb.n > 1 ? gather_kernel<true> : gather_kernel<false>), dim3(grid_for((size_t)B * rec4, 256), 1, mb.n), 256, 0, s, reinterpret_cast<const float4*>(ring),
             rec4, idx, B, reinterpret_cast<float4*>(out), ring_slot, mb.stride);
  RLREP_LAUNCHED_W("gather", s, 2.0 * 16.0 * (double)B * rec4 * mb.n, 0.0);
}

void launch_ring_write(float* ring, int rec4, long long capacity, long long start, const float* rows, int n,
                       cudaStream_t s) {
  if (n <= 0) return;
  ring_write_kernel<<<grid_for((size_t)n * rec4, 256), 256, 0, s>>>(reinterpret_cast<float4*>(ring), rec4, capacity,
                                                                   start, reinterpret_cast<const float4*>(rows), n);
  RLREP_LAUNCHED("ring_write", s);
}

void launch_ce_rows(float* logits, int ld, int rows, int cols, int diag_off, float inv_batch, float* loss_rows,
                    cudaStream_t s) {
  ce_rows_kernel<<<rows, 256, 0, s>>>(logits, ld, cols, diag_off, inv_batch, loss_rows);
  RLREP_LAUNCHED_W("ce_rows", s, 3.0 * 4.0 * (double)rows * cols, 0.0);
}

void launch_rowdot(const float* X, int ld, int rows, int D, const float* w, const float* b, float* y, cudaStream_t s,
                   Members mb) {
  RowDotJobs js;
  js.j[0] = RowDotJob{X, w, b, y, ld, D};
  js.j[1] = js.j[0];
  (mb.n > 1 ? rowdot_kernel<true> : rowdot_kernel<false>)<<<dim3(rows, 1, mb.n), 128, 0, s>>>(js, rows, mb.stride);
  RLREP_LAUNCHED("rowdot", s);
}
void launch_rowdot_pair(const RowDotJob& a, const RowDotJob& b, int rows, cudaStream_t s) {
  RowDotJobs js;
  js.j[0] = a;
  js.j[1] = b;
  rowdot_kernel<false><<<dim3(rows, 2), 128, 0, s>>>(js, rows, 0LL);
  RLREP_LAUNCHED("rowdot", s);
}

void launch_colreduce(const float* X, int ld, int rows, int cols, const float* u, float* out, int accumulate,
                      cudaStream_t s, Members mb) {
  (mb.n > 1 ? colreduce_kernel<true> : colreduce_kernel<false>)<<<dim3(ceil_div(cols, 32), 1, mb.n), 256, 0, s>>>(X, ld, rows, cols, u, out, accumulate, mb.stride);
  RLREP_LAUNCHED("colreduce", s);
}

void launch_colsum_tall(const float* X, int ld, long long rows, int cols, float* partial, int chunks, float* out,
                        cudaStream_t s) {
  const int rows_per = (int)((rows + chunks - 1) / chunks);
  if (cols == 32 && ld == 32 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(partial) & 15) == 0)
    colsum_tall32_stage1_kernel<<<dim3(1, chunks), 256, 0, s>>>(reinterpret_cast<const float4*>(X), rows, rows_per, partial);
  else
    colsum_tall_stage1_kernel<<<dim3(ceil_div(cols, 32), chunks), 256, 0, s>>>(X, ld, rows, cols, rows_per, partial);
  RLREP_LAUNCHED_W("colsum_tall", s, 4.0 * (double)rows * cols, 0.0);
  colsum_tall_stage2_kernel<<<ceil_div(cols, 32), 1024, 0, s>>>(partial, chunks, cols, out);
  RLREP_LAUNCHED("colsum_tall_final", s);
}

void launch_kgroup_finish(const float* ws, int groups, int M, int N, int ldw, size_t group_stride, float* C, int ldc,
                          const Epilogue& epi, cudaStream_t s) {
  const size_t total = (size_t)M * N;
  kgroup_finish_kernel<<<grid_for(total, 256, 16), 256, 0, s>>>(ws, groups, M, N, ldw, group_stride, C, ldc, epi);
  RLREP_LAUNCHED_W("kgroup_finish", s, 4.0 * (double)total * (groups + 1), 0.0);
}

void launch_colsum_finish(const float* partial, int chunks, int cols, float* out, cudaStream_t s) {
  colsum_tall_stage2_kernel<<<ceil_div(cols, 32), 1024, 0, s>>>(partial, chunks, cols, out);
  RLREP_LAUNCHED("colsum_tall_final", s);
}

void launch_colreduce_multi(const ColJob* jobs, int n_jobs, cudaStream_t s, Members mb) {
  RLREP_CHECK(n_jobs >= 1 && n_jobs <= kMaxColJobs, "too many column-reduction jobs for one launch");
  ColJobs js;
  int max_cols = 0;
  for (int i = 0; i < n_jobs; ++i) {
    js.j[i] = jobs[i];
    if (jobs[i].cols > max_cols) max_cols = jobs[i].cols;
  }
  launch_pdl((mb.n > 1 ? colreduce_multi_kernel<true> : colreduce_multi_kernel<false>), dim3(ceil_div(max_cols, 32), n_jobs, mb.n), 1024, 0, s, js, mb.stride);
  RLREP_LAUNCHED("colreduce_multi", s);
}

void launch_outer_dact(const float* u, const float* w, int rows, int cols, const float* aux, int ld_aux, int dact,
                       float* out, int ld_out, cudaStream_t s, Members mb) {
  (mb.n > 1 ? outer_dact_kernel<true> : outer_dact_kernel<false>)<<<dim3(grid_for((size_t)rows * cols, 256), 1, mb.n), 256, 0, s>>>(u, w, rows, cols, aux, ld_aux, dact,
                                                                                      out, ld_out, mb.stride);
  RLREP_LAUNCHED("outer_dact", s);
}

void launch_feature_loss_finalize(const float* loss_rows, int rows, const float* pred, const float* reward, int ld_r,
                                  float inv_batch, float* dpred, float* metrics, cudaStream_t s) {
  feature_loss_finalize_kernel<<<1, 256, 0, s>>>(loss_rows, rows, pred, reward, ld_r, inv_batch, dpred, metrics);
  RLREP_LAUNCHED("feature_loss_finalize", s);
}

void launch_contrastive_head(float* logits, int ld, int rows, int cols, int diag_off, float inv_batch, const float* z, int ldz,
                             int D, const float* theta_w, const float* theta_b, const float* reward, int ld_r,
                             float* loss_rows, float* pred, float* dpred, float* metrics, unsigned* counter,
                             cudaStream_t s) {
  launch_pdl(contrastive_head_kernel, rows, 256, 0, s, logits, ld, cols, diag_off, inv_batch, z, ldz, D, theta_w, theta_b,
             reward, ld_r, loss_rows, pred, dpred, metrics, counter, rows);
  RLREP_LAUNCHED_W("contrastive_head", s, 3.0 * 4.0 * (double)rows * cols + 4.0 * (double)rows * D, 0.0);
}

void launch_critic_td_head(const CriticHeadArgs& a, cudaStream_t s) {
  launch_pdl(critic_td_head_kernel, a.B, 256, 0, s, a);
  RLREP_LAUNCHED_W("critic_td_head", s, 4.0 * a.B * (4.0 * a.H + 2.0 * a.H), 0.0);
}
void launch_actor_head(const ActorHeadArgs& a, cudaStream_t s) {
  launch_pdl(actor_head_kernel, a.B, 256, 0, s, a);
  RLREP_LAUNCHED_W("actor_head", s, 4.0 * a.B * (4.0 * a.H), 0.0);
}

void launch_actor_sample(const float* head, int ld_head, int B, int A, const float* eps, float* action, int lda,
                         float* logp, cudaStream_t s, const float* obs, int ld_obs, int S, Members mb) {
  ActorSampleJobs js;
  js.j[0] = ActorSampleJob{head, eps, action, logp, obs, ld_obs};
  js.j[1] = js.j[0];
  launch_pdl((mb.n > 1 ? actor_sample_kernel<true> : actor_sample_kernel<false>), dim3(ceil_div(B * 32, 128), 1, mb.n), 128, 0, s, js, ld_head, B, A, lda, S, mb.stride);
  RLREP_LAUNCHED("actor_sample", s);
}
void launch_actor_sample_pair(const ActorSampleJob& j0, const ActorSampleJob& j1, int ld_head, int B, int A, int lda, int S,
                              cudaStream_t s) {
  ActorSampleJobs js;
  js.j[0] = j0;
  js.j[1] = j1;
  launch_pdl(actor_sample_kernel<false>, dim3(ceil_div(B * 32, 128), 2), 128, 0, s, js, ld_head, B, A, lda, S, 0LL);
  RLREP_LAUNCHED("actor_sample", s);
}

void launch_actor_act(const float* in, int rows, int S, int A, int H, const float* W0, int ld0, const float* b0,
                      const float* W1, int ld1, const float* b1, const float* W2, int ld2, const float* b2, int explore,
                      float* out, cudaStream_t s, Members mb) {
  const size_t smem = (size_t)(((S + 3) & ~3) + 2 * H + 2 * A) * sizeof(float);
  RLREP_CHECK(smem <= 48 * 1024, "actor too wide for the one-launch select_action kernel");
  (mb.n > 1 ? actor_act_kernel<true> : actor_act_kernel<false>)<<<dim3(rows, 1, mb.n), 256, smem, s>>>(in, S, A, H, W0, ld0, b0, W1, ld1, b1, W2, ld2, b2, explore, out,
                                                         mb.stride);
  RLREP_LAUNCHED("actor_act", s);
}

void launch_actor_sample_bwd(const float* head, int ld_head, int B, int A, const float* eps, const float* d_action,
                             int ldd, const float* dlogp_scalar, float* dhead, int ld_dhead, cudaStream_t s, Members mb) {
  launch_pdl((mb.n > 1 ? actor_sample_bwd_kernel<true> : actor_sample_bwd_kernel<false>), dim3(ceil_div(B * A, 128), 1, mb.n), 128, 0, s, head, ld_head, B, A, eps, d_action, ldd,
             dlogp_scalar, dhead, ld_dhead, mb.stride);
  RLREP_LAUNCHED("actor_sample_bwd", s);
}

void launch_td_critic_loss(const float* reward, const float* done, int ld_rd, const float* nq1, const float* nq2,
                           const float* logp2, const float* q1, const float* q2, int B, float gamma, const Control* c,
                           float* dq1, float* dq2, float* metrics, cudaStream_t s, int norm_B, Members mb) {
  (mb.n > 1 ? td_critic_loss_kernel<true> : td_critic_loss_kernel<false>)<<<dim3(1, 1, mb.n), 256, 0, s>>>(reward, done, ld_rd, nq1, nq2, logp2, q1, q2, B,
                                                         norm_B > 0 ? norm_B : B, gamma, c, dq1, dq2, metrics, mb.stride);
  RLREP_LAUNCHED("td_critic_loss", s);
}

void launch_actor_alpha_loss(const float* q1, const float* q2, const float* logp, int B, float target_entropy,
                             int learn_alpha, Control* c, float* dq1, float* dq2, float* dlogp_scalar, float* metrics,
                             cudaStream_t s, Members mb) {
  (mb.n > 1 ? actor_alpha_loss_kernel<true> : actor_alpha_loss_kernel<false>)<<<dim3(1, 1, mb.n), 256, 0, s>>>(q1, q2, logp, B, target_entropy, learn_alpha, c, dq1, dq2,
                                                           dlogp_scalar, metrics, mb.stride);
  RLREP_LAUNCHED("actor_alpha_loss", s);
}

void launch_actor_loss_partial(const float* q1, const float* q2, const float* logp, int B, int norm_B,
                               float target_entropy, const Control* c, float* dq1, float* dq2, float* dlogp_scalar,
                               float* partial, cudaStream_t s) {
  actor_loss_partial_kernel<<<1, 256, 0, s>>>(q1, q2, logp, B, norm_B, target_entropy, c, dq1, dq2, dlogp_scalar, partial);
  RLREP_LAUNCHED("actor_loss_partial", s);
}
void launch_alpha_step(const float* reduced, int learn_alpha, Control* c, float* metrics, cudaStream_t s) {
  alpha_step_kernel<<<1, 32, 0, s>>>(reduced, learn_alpha, c, metrics);
  RLREP_LAUNCHED("alpha_step", s);
}
void launch_mul_dact(float* x, const float* aux, size_t n, int dact, cudaStream_t s) {
  mul_dact_kernel<<<grid_for(n, 256), 256, 0, s>>>(x, aux, n, dact);
  RLREP_LAUNCHED_W("mul_dact", s, 12.0 * (double)n, 0.0);
}

void launch_pack_columns(const float* in, int ld_in, float* out, int ld_out, int rows, const ColSegment* segs, int n_segs,
                         cudaStream_t s) {
  RLREP_CHECK(n_segs >= 1 && n_segs <= 3, "pack_columns takes 1..3 segments");
  ColSegments cs;
  cs.n = n_segs;
  int width = 0;
  for (int i = 0; i < n_segs; ++i) {
    cs.s[i] = segs[i];
    width += segs[i].len;
  }
  pack_columns_kernel<<<grid_for((size_t)rows * width, 256), 256, 0, s>>>(in, ld_in, out, ld_out, rows, cs, width);
  RLREP_LAUNCHED("pack_columns", s);
}
void launch_vae_sample(const float* head, int ld_head, int B, int D, const float* eps, float* z, cudaStream_t s) {
  vae_sample_kernel<<<grid_for((size_t)B * D, 256), 256, 0, s>>>(head, ld_head, B, D, eps, z);
  RLREP_LAUNCHED("vae_sample", s);
}
void launch_vae_recon_loss(const float* xr, int ld_xr, const float* next_state, const float* reward, int ld_rec, int B,
                           int S, float* dxr, float* partial, int n_blocks, cudaStream_t s) {
  vae_recon_loss_kernel<<<n_blocks, 256, 0, s>>>(xr, ld_xr, next_state, reward, ld_rec, B, S, dxr, partial);
  RLREP_LAUNCHED("vae_recon_loss", s);
}
void launch_vae_kl_bwd(const float* enc_head, const float* prior_head, int ld_head, int B, int D, const float* eps,
                       const float* dz, float* d_enc, float* d_prior, float* partial, int n_blocks, cudaStream_t s) {
  vae_kl_bwd_kernel<<<n_blocks, 256, 0, s>>>(enc_head, prior_head, ld_head, B, D, eps, dz, d_enc, d_prior, partial);
  RLREP_LAUNCHED("vae_kl_bwd", s);
}
void launch_vae_finalize(const float* recon_partial, int n_recon, const float* kl_partial, int n_kl, int B, int S, int D,
                         float* metrics, cudaStream_t s) {
  vae_finalize_kernel<<<1, 32, 0, s>>>(recon_partial, n_recon, kl_partial, n_kl, B, S, D, metrics);
  RLREP_LAUNCHED("vae_finalize", s);
}
void launch_noise_expand(const float* head, int ld_head, int B, int D, const float* noise, int NN, float* x,
                         cudaStream_t s) {
  const bool vec = (D & 3) == 0 && (ld_head & 3) == 0 && (long long)B * NN * D < (1LL << 31) &&
                   ((reinterpret_cast<uintptr_t>(head) | reinterpret_cast<uintptr_t>(noise) | reinterpret_cast<uintptr_t>(x)) & 15) == 0;
  if (vec) noise_expand4_kernel<<<grid_for((size_t)B * (D / 4), 256, 16), 256, 0, s>>>(head, ld_head, B, D, noise, NN, x);
  else noise_expand_kernel<<<grid_for((size_t)B * NN * D, 256, 16), 256, 0, s>>>(head, ld_head, B, D, noise, NN, x);
  RLREP_LAUNCHED("noise_expand", s);
}
void launch_noise_expand_bwd(const float* dx, const float* head, int ld_head, int B, int D, const float* noise, int NN,
                             float* d_head, cudaStream_t s) {
  noise_expand_bwd_kernel<<<grid_for((size_t)B * D, 256), 256, 0, s>>>(dx, head, ld_head, B, D, noise, NN, d_head);
  RLREP_LAUNCHED("noise_expand_bwd", s);
}
void launch_group_mean(const float* hid, int ld, int B, int NN, int C, float* out, cudaStream_t s) {
  group_mean_kernel<<<grid_for((size_t)B * C, 256), 256, 0, s>>>(hid, ld, B, NN, C, out);
  RLREP_LAUNCHED("group_mean", s);
}
void launch_group_mean_bwd(const float* dmean, const float* hid, int ld, int B, int NN, int C, float* dhid,
                           float* colsum_partial, cudaStream_t s) {
  group_mean_bwd_kernel<<<grid_for((size_t)B * C, 256), 256, 0, s>>>(dmean, hid, ld, B, NN, C, dhid, colsum_partial);
  RLREP_LAUNCHED("group_mean_bwd", s);
}

void launch_adam_polyak(float* p, const float* g, float* m, float* v, size_t n, const AdamHyper* hyper, float* target,
                        size_t n_polyak, float tau, const int* polyak_flag, cudaStream_t s, Members mb) {
  RLREP_CHECK(n % 4 == 0 && n_polyak % 4 == 0, "optimizer arenas are padded to float4");
  const size_t n4 = n / 4;
  launch_pdl((mb.n > 1 ? adam_polyak_kernel<true> : adam_polyak_kernel<false>), dim3(grid_for(n4, 256, 16), 1, mb.n), 256, 0, s, reinterpret_cast<float4*>(p),
             reinterpret_cast<const float4*>(g), reinterpret_cast<float4*>(m), reinterpret_cast<float4*>(v), n4, hyper,
             reinterpret_cast<float4*>(target), n_polyak / 4, tau, polyak_flag, mb.stride);
  // 28 B/param (p, g, m, v read; p, m, v written) + 12 B/param of Polyak (p is already in registers: target read +
  // written = 8 B; counted as 12 like SURVEY.md 8d counts a stand-alone Polyak) -- a gated Polyak fires every 2nd step
  const double polyak = target ? 12.0 * (double)n_polyak * (polyak_flag ? 0.5 : 1.0) : 0.0;
  RLREP_LAUNCHED_W("adam_polyak", s, 28.0 * (double)n + polyak, 0.0);
}

void launch_polyak(const float* p, float* target, size_t n, float tau, const int* polyak_flag, cudaStream_t s) {
  RLREP_CHECK(n % 4 == 0, "optimizer arenas are padded to float4");
  polyak_kernel<<<grid_for(n / 4, 256, 16), 256, 0, s>>>(reinterpret_cast<const float4*>(p),
                                                        reinterpret_cast<float4*>(target), n / 4, tau, polyak_flag);
  RLREP_LAUNCHED_W("polyak", s, 12.0 * (double)n * (polyak_flag ? 0.5 : 1.0), 0.0);
}

}  // namespace rlrep

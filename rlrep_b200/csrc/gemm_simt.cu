// CUDA-core FP32 GEMMs (FFMA, exact fp32 products and accumulation) with the shared epilogue.
// Used for the layers tensor cores cannot help: K = 17/23-wide input layers (optionally reading the
// concatenated input from two buffers), the 6/12/17/23-wide heads and their gradients, and for the strict-fp32
// mode of the library (IEEE fp32 multiply-add, like torch with allow_tf32 = False).
//
// Three kernels, picked by shape:
//   gemm_tiled_kernel     64x64 output tile per 256-thread CTA, BK = 16, 4x4 register micro-tile, operands staged
//                         through shared memory with a register prefetch of the next k-tile (one global round trip
//                         per k-tile is hidden behind the FMAs of the previous one).
//   skinny_rowwarp_kernel N <= 32 outputs per row, A K-major: one warp per output row, lanes stride over K, warp
//                         shuffle reduction (d_action = dh1 W1[:, S:], actor head forward).
//   skinny_rowthread_kernel N <= 32 outputs per row, A MN-major: one thread per output row, K split over the 8
//                         warps of the CTA and reduced through shared memory in a fixed order (first-layer and
//                         head weight gradients; also the transposed problem when M <= 32).
#include "common.cuh"
#include "gemm.cuh"

namespace rlrep {

namespace {

constexpr int TBM = 64, TBN = 64, TBK = 16;

struct SimtParams {
  int M, N, K, K1;
  int conv_w;          // implicit 3x3 convolution over a K-major [M, 32] pixel matrix (gemm.cuh); 0 = plain GEMM
  const float* A;
  long long sam, sak;  // A(m,k) = A[m*sam + k*sak]
  const float* A2;
  long long sam2;      // second K segment (K-major only): A2[m*sam2 + (k-K1)]
  const float* B;
  long long sbn, sbk;  // B(n,k) = B[n*sbn + k*sbk]
  float* C;
  long long scm, scn;  // C(m,n) = C[m*scm + n*scn]
  long long mstride;   // population GEMM (members.cuh): bytes between consecutive members' operands
};
// The operands of member blockIdx.z (members.cuh).
template <bool MEMBERS>
__device__ __forceinline__ SimtParams member_params(SimtParams p, Epilogue& epi) {
  const long long off = member_offset<MEMBERS>(p.mstride);
  p.A = member_ptr(p.A, off);
  p.A2 = member_ptr(p.A2, off);
  p.B = member_ptr(p.B, off);
  p.C = member_ptr(p.C, off);
  epi = member_epilogue(epi, off);
  return p;
}

template <int ACT, int DACT>
__device__ __forceinline__ void store_micro_tile(const SimtParams& p, const Epilogue& epi, const float (&acc)[4][4], int m0,
                                                 int n0, int tx, int ty) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.N) continue;
      float* cp = p.C + (long long)m * p.scm + (long long)n * p.scn;
      *cp = epilogue_apply<ACT, DACT>(epi, acc[i][j], m, n, cp);
    }
  }
}
template <int ACT, int DACT>
__device__ __forceinline__ void store_one(const Epilogue& epi, float v, int m, int n, float* cp) {
  *cp = epilogue_apply<ACT, DACT>(epi, v, m, n, cp);
}

// ------------------------------------------------------------------------------------------------ tiled
template <bool MEMBERS>
__device__ __forceinline__ void gemm_tiled(const SimtParams& pm, const Epilogue& epi_in) {
  Epilogue epi = epi_in;
  const SimtParams p = member_params<MEMBERS>(pm, epi);
  __shared__ __align__(16) float As[TBK][TBM + 4];
  __shared__ __align__(16) float Bs[TBK][TBN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * TBM, n0 = blockIdx.x * TBN;
  const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, each 4x4 outputs
  float acc[4][4] = {};

  const bool a_kmajor = (p.sak == 1);
  const bool b_kmajor = (p.sbk == 1);
  constexpr int PER = (TBM * TBK) / 256;  // 4 elements of each operand tile per thread
  int a_mm[PER], a_kk[PER], b_nn[PER], b_kk[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int idx = tid + i * 256;
    if (a_kmajor) { a_kk[i] = idx % TBK; a_mm[i] = idx / TBK; } else { a_mm[i] = idx % TBM; a_kk[i] = idx / TBM; }
    if (b_kmajor) { b_kk[i] = idx % TBK; b_nn[i] = idx / TBK; } else { b_nn[i] = idx % TBN; b_kk[i] = idx / TBN; }
  }
  float ra[PER], rb[PER];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int m = m0 + a_mm[i], k = k0 + a_kk[i];
      bool ok = m < p.M && k < p.K;
      const bool seg2 = p.A2 != nullptr && k >= p.K1;
      const float* src = seg2 ? p.A2 + (long long)m * p.sam2 + (k - p.K1) : p.A + (long long)m * p.sam + (long long)k * p.sak;
      if (p.conv_w > 0) {
        const int t = k >> 5;
        const long long row = (long long)m + (t / 3) * p.conv_w + (t % 3);
        ok = ok && row < p.M;
        src = p.A + row * p.sam + (k & 31);
      }
      ra[i] = ok ? __ldg(ok ? src : p.A) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int n = n0 + b_nn[i], k = k0 + b_kk[i];
      const bool ok = n < p.N && k < p.K;
      rb[i] = ok ? __ldg(ok ? p.B + (long long)n * p.sbn + (long long)k * p.sbk : p.B) : 0.f;
    }
  };

  fetch(0);
  for (int k0 = 0; k0 < p.K; k0 += TBK) {
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      As[a_kk[i]][a_mm[i]] = ra[i];
      Bs[b_kk[i]][b_nn[i]] = rb[i];
    }
    __syncthreads();
    if (k0 + TBK < p.K) fetch(k0 + TBK);  // in flight while this tile is consumed
#pragma unroll
    for (int kk = 0; kk < TBK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#define RLREP_STORE(A, D) store_micro_tile<A, D>(p, epi, acc, m0, n0, tx, ty)
  RLREP_EPILOGUE_SWITCH(epi, RLREP_STORE);
#undef RLREP_STORE
}

// ------------------------------------------------------------------------------------------------ skinny: warp per row
// One output at a time: both operand streams advance by a constant stride, so the inner loop is two loads and an FMA.
template <bool MEMBERS>
__device__ __forceinline__ void skinny_rowwarp(const SimtParams& pm, const Epilogue& epi_in) {
  Epilogue epi = epi_in;
  const SimtParams p = member_params<MEMBERS>(pm, epi);
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (m >= p.M) return;
  const float* arow = p.A + (long long)m * p.sam;
  float mine = 0.f;
#pragma unroll 1
  for (int n = 0; n < p.N; ++n) {
    const float* bp = p.B + (long long)n * p.sbn + (long long)lane * p.sbk;
    const long long bstep = 32 * p.sbk;
    float acc = 0.f;
#pragma unroll 8
    for (int k = lane; k < p.K; k += 32) {
      acc = fmaf(__ldg(arow + k), __ldg(bp), acc);
      bp += bstep;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == n) mine = acc;
  }
  if (lane < p.N) {
    float* cp = p.C + (long long)m * p.scm + (long long)lane * p.scn;
#define RLREP_STORE(A, D) store_one<A, D>(epi, mine, m, lane, cp)
    RLREP_EPILOGUE_SWITCH(epi, RLREP_STORE);
#undef RLREP_STORE
  }
}

// ------------------------------------------------------------------------------------------------ skinny: thread per row
// B must be contiguous in n (sbn == 1): the N loads of a k-step then use immediate offsets from one base pointer.
template <int NT, bool MEMBERS>
__device__ __forceinline__ void skinny_rowthread(const SimtParams& pm, const Epilogue& epi_in, int swapped) {
  Epilogue epi = epi_in;
  const SimtParams p = member_params<MEMBERS>(pm, epi);
  __shared__ float red[8][32][NT + 1];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int m = blockIdx.x * 32 + lane;
  float acc[NT];
#pragma unroll
  for (int n = 0; n < NT; ++n) acc[n] = 0.f;
  if (m < p.M) {
    const float* ap = p.A + (long long)slice * p.sak + m;  // sam == 1: coalesced over rows
    const float* bk = p.B + (long long)slice * p.sbk;      // uniform across the warp: broadcast loads
    const long long astep = 8 * p.sak, bstep = 8 * p.sbk;
#pragma unroll 2
    for (int k = slice; k < p.K; k += 8) {
      const float a = __ldg(ap);
#pragma unroll
      for (int n = 0; n < NT; ++n)
        if (n < p.N) acc[n] = fmaf(a, __ldg(bk + n), acc[n]);
      ap += astep;
      bk += bstep;
    }
  }
#pragma unroll
  for (int n = 0; n < NT; ++n) red[slice][lane][n] = acc[n];
  __syncthreads();
  for (int o = threadIdx.x; o < 32 * p.N; o += 256) {
    const int r = o / p.N, n = o - r * p.N;
    const int mm = blockIdx.x * 32 + r;
    if (mm >= p.M) continue;
    float v = 0.f;
#pragma unroll
    for (int s = 0; s < 8; ++s) v += red[s][r][n];  // fixed order
    float* cp = p.C + (long long)mm * p.scm + (long long)n * p.scn;
    // in swapped mode rows/cols of this kernel are cols/rows of the caller's C: the epilogue sees the caller's indices
    const int em = swapped ? n : mm, en = swapped ? mm : n;
#define RLREP_STORE(A, D) store_one<A, D>(epi, v, em, en, cp)
    RLREP_EPILOGUE_SWITCH(epi, RLREP_STORE);
#undef RLREP_STORE
  }
}

// The kernels: the lone form, and the population form (SimtParams::mstride, member = blockIdx.z).
__global__ void __launch_bounds__(256) gemm_tiled_kernel(const SimtParams p, const Epilogue epi) {
  gemm_tiled<false>(p, epi);
}
__global__ void __launch_bounds__(256) gemm_tiled_members_kernel(const SimtParams p, const Epilogue epi) {
  gemm_tiled<true>(p, epi);
}
__global__ void __launch_bounds__(256) skinny_rowwarp_kernel(const SimtParams p, const Epilogue epi) {
  skinny_rowwarp<false>(p, epi);
}
__global__ void __launch_bounds__(256) skinny_rowwarp_members_kernel(const SimtParams p, const Epilogue epi) {
  skinny_rowwarp<true>(p, epi);
}
template <int NT>
__global__ void __launch_bounds__(256) skinny_rowthread_kernel(const SimtParams p, const Epilogue epi, int swapped) {
  skinny_rowthread<NT, false>(p, epi, swapped);
}
template <int NT>
__global__ void __launch_bounds__(256) skinny_rowthread_members_kernel(const SimtParams p, const Epilogue epi, int swapped) {
  skinny_rowthread<NT, true>(p, epi, swapped);
}

void launch_rowwarp(const SimtParams& p, const Epilogue& e, int members, cudaStream_t s) {
  (members > 1 ? skinny_rowwarp_members_kernel : skinny_rowwarp_kernel)<<<dim3(ceil_div(p.M * 32, 256), 1, members), 256, 0, s>>>(p, e);
  RLREP_LAUNCHED_W("skinny_rowwarp", s, 4.0 * ((double)p.M * p.K + (double)p.N * p.K + (double)p.M * p.N), 2.0 * p.M * p.N * p.K);
}
template <int NT>
void launch_rowthread(const SimtParams& p, const Epilogue& e, int swapped, int members, cudaStream_t s) {
  (members > 1 ? skinny_rowthread_members_kernel<NT> : skinny_rowthread_kernel<NT>)<<<dim3(ceil_div(p.M, 32), 1, members), 256, 0, s>>>(
      p, e, swapped);
  RLREP_LAUNCHED_W("skinny_rowthread", s, 4.0 * ((double)p.M * p.K + (double)p.N * p.K + (double)p.M * p.N), 2.0 * p.M * p.N * p.K);
}

}  // namespace

void launch_simt(const GemmArgs& a, cudaStream_t stream) {
  RLREP_CHECK(a.M > 0 && a.N > 0 && a.K > 0, "empty GEMM");
  RLREP_CHECK(a.A2 == nullptr || !a.a_mn, "two-segment A requires a K-major A");
  SimtParams p;
  RLREP_CHECK(a.conv_w == 0 || (!a.a_mn && a.A2 == nullptr && a.K == 9 * 32), "implicit convolution needs a K-major [M, 32] A");
  RLREP_CHECK(a.conv_wgrad_hi == 0, "the implicit conv weight gradient exists on the tensor-core path only");
  p.M = a.M; p.N = a.N; p.K = a.K; p.K1 = a.A2 ? a.K1 : a.K;
  p.conv_w = a.conv_w;
  p.A = a.A;
  p.sam = a.a_mn ? 1 : a.lda;
  p.sak = a.a_mn ? a.lda : 1;
  p.A2 = a.A2;
  p.sam2 = a.lda2;
  p.B = a.B;
  p.sbn = a.b_mn ? 1 : a.ldb;
  p.sbk = a.b_mn ? a.ldb : 1;
  p.C = a.C;
  p.scm = a.ldc;
  p.scn = 1;
  p.mstride = a.mb.stride;
  const int nm = a.mb.n;
  const bool plain_epi = a.epi.pre_out == nullptr;  // pre_out uses (m, n) addressing the skinny kernels do not remap
  if (a.A2 == nullptr && plain_epi && a.N <= 32 && !a.a_mn && a.K >= 64 && a.conv_w == 0) {
    launch_rowwarp(p, a.epi, nm, stream);
    return;
  }
  if (a.A2 == nullptr && plain_epi && a.N <= 32 && a.a_mn && a.b_mn && a.M >= 64) {
    if (a.N <= 8) launch_rowthread<8>(p, a.epi, 0, nm, stream);
    else if (a.N <= 16) launch_rowthread<16>(p, a.epi, 0, nm, stream);
    else launch_rowthread<32>(p, a.epi, 0, nm, stream);
    return;
  }
  if (a.A2 == nullptr && plain_epi && a.M <= 32 && a.a_mn && a.b_mn && a.N >= 64) {
    // transposed problem: rows' = n (B is contiguous in n), cols' = m
    SimtParams q = p;
    q.M = a.N; q.N = a.M;
    q.A = a.B; q.sam = 1; q.sak = a.ldb;
    q.B = a.A; q.sbn = 1; q.sbk = a.lda;
    q.scm = 1; q.scn = a.ldc;
    if (q.N <= 8) launch_rowthread<8>(q, a.epi, 1, nm, stream);
    else if (q.N <= 16) launch_rowthread<16>(q, a.epi, 1, nm, stream);
    else launch_rowthread<32>(q, a.epi, 1, nm, stream);
    return;
  }
  dim3 grid(ceil_div(a.N, TBN), ceil_div(a.M, TBM), nm);
  (nm > 1 ? gemm_tiled_members_kernel : gemm_tiled_kernel)<<<grid, 256, 0, stream>>>(p, a.epi);
  RLREP_LAUNCHED_W("gemm_simt", stream, 4.0 * ((double)p.M * p.K + (double)p.N * p.K + (double)p.M * p.N), 2.0 * p.M * p.N * p.K);
}

}  // namespace rlrep

// tcgen05 TF32 GEMM for sm_100a: TMA-fed shared-memory ring -> tcgen05.mma (kind::tf32) with the FP32
// accumulator in TMEM -> staged, coalesced epilogue with fused bias / activation / activation-derivative.
//
// One CTA computes one 128 x BN output tile over a K-slice.  Split-K runs as a THREAD-BLOCK CLUSTER along
// gridDim.z (1, 2, 4 or 8 CTAs): every CTA stages its partial accumulator in its own shared memory, the cluster
// synchronises, and CTA r reduces rows [r*128/s, (r+1)*128/s) of the tile by reading all peers' slices over
// distributed shared memory in a fixed order (deterministic), applies the epilogue and writes C with fully
// coalesced 16-byte stores.  No global workspace, no second kernel, no atomics.
//   warp 0     : TMA producer (one elected lane)
//   warp 1     : MMA issuer (one elected lane)
//   warps 2..5 : TMEM -> shared staging (warp w owns TMEM lanes 32*(w&3) ..); warp 2 owns TMEM alloc/dealloc
//   all 16 warps: reduce + epilogue + store (the store phase is issue-bound, so it gets every warp the CTA has)
//
// Operands stay FP32 in HBM; the tensor maps are typed TFLOAT32 so the TMA unit rounds to TF32 on the way
// into shared memory and the weights are never re-materialised in a second precision.
//
// Both K-major and MN-major operands are supported (see gemm.cuh), so forward, dgrad and wgrad all run
// here without transposed copies of weights or activations:
//   K-major  tile: rows x 32 fp32 (128 B) per k-block, one TMA box, SWIZZLE_128B, SBO = 1024 B;
//                  the 4 UMMA_K=8 slices of a k-block advance the descriptor start address by 32 B.
//   MN-major tile: 32 k-rows x 32 fp32 boxes (4 KB each), one per 32 rows of M/N.  tcgen05 accepts exactly one
//                  layout for MN-major tf32: SWIZZLE_128B_BASE32B (32-byte chunks XOR k-row % 4, 4-row atoms),
//                  which TMA writes with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.  LBO = 4096 B between boxes,
//                  SBO = 512 B between 4-k-row groups; the 4 UMMA_K=8 slices advance the start by 1024 B.
//
// This header holds the device code and the per-variant launcher; it is included by the gemm_tc_inst_*.cu units (one
// per (BN, A-major) pair so the 16 kernel variants compile in parallel) and by gemm_tc.cu for the tile constants.
#pragma once
#include <algorithm>
#include <cstdint>

#include "common.cuh"
#include "gemm.cuh"
#include "ptx.cuh"

namespace rlrep {
namespace tc {

constexpr int BM = 128;           // UMMA M (cta_group::1)
constexpr int BK = 32;            // fp32 elements per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 8;         // tf32
constexpr int kThreads = 512;     // 16 warps: 2 issue the pipeline, 4 drain TMEM, all 16 run the store phase
constexpr int kSmemBudget = 200 * 1024;

__host__ __device__ constexpr int stage_bytes(int bn) { return (BM + bn) * BK * 4; }
__host__ __device__ constexpr int min_stages_fwd(int bn) { return bn >= 256 ? 3 : 2; }
__host__ __device__ constexpr int num_stages(int bn) {
  return kSmemBudget / stage_bytes(bn) > 8 ? 8 : kSmemBudget / stage_bytes(bn);
}
// Split-K "push" mode: every CTA owns BM / splits rows of the tile; the TMEM-drain warps write each partial row straight
// into the OWNER's shared memory (st.shared::cluster), one cluster barrier later the owner sums its `splits` slots
// locally in a fixed order.  The slots live behind the operand ring (peers may push while this CTA is still in its main
// loop).  Compared with staging locally and pulling over DSMEM this removes the dependent remote-load latency, the
// second cluster barrier and the local staging pass from the tail of every split-K GEMM.
__host__ __device__ constexpr int slots_bytes(int bn) { return BM * (bn + 4) * 4; }
__host__ __device__ constexpr int smem_bytes(int bn, int stages, bool push = false) {
  return stages * stage_bytes(bn) + 1024 + 256 + (push ? slots_bytes(bn) : 0);
}
constexpr int kMaxSmem = 227 * 1024;
__host__ __device__ constexpr bool push_possible(int bn) { return smem_bytes(bn, min_stages_fwd(bn), true) <= kMaxSmem; }
__host__ __device__ constexpr int max_stages_push(int bn) {
  return (kMaxSmem - 1024 - 256 - slots_bytes(bn)) / stage_bytes(bn) > 8
             ? 8
             : (kMaxSmem - 1024 - 256 - slots_bytes(bn)) / stage_bytes(bn);
}
__host__ __device__ constexpr int smem_bytes(int bn) { return smem_bytes(bn, num_stages(bn)); }
// Fewest stages whose ring still holds the fp32 staging tile [BM, bn + 4] of the store phase.
__host__ __device__ constexpr int min_stages(int bn) { return (BM * (bn + 4) * 4 + stage_bytes(bn) - 1) / stage_bytes(bn); }

// One launcher per (BN, A-major) pair, each defined in its own translation unit (gemm_tc_inst_*.cu).
#define RLREP_TC_DECL(BN, AMN)                                           \
  void launch_tc_##BN##_##AMN(const TcGemmPlan& p, cudaStream_t stream); \
  int max_clusters_##BN##_##AMN(bool b_mn, int split_k, int stages, bool push);
RLREP_TC_DECL(32, 0) RLREP_TC_DECL(32, 1) RLREP_TC_DECL(64, 0) RLREP_TC_DECL(64, 1)
RLREP_TC_DECL(128, 0) RLREP_TC_DECL(128, 1) RLREP_TC_DECL(256, 0) RLREP_TC_DECL(256, 1)
#undef RLREP_TC_DECL

#ifdef RLREP_TC_DEVICE_CODE
// Optional in-kernel timeline (nanoseconds from %globaltimer) of CTA (0,0,0); one copy per translation unit, read back
// through the reader the last launch registered (rlrep_gemm_trace).
__device__ unsigned long long g_gemm_trace[16];
extern void (*g_trace_reader)(unsigned long long*);
// Debug aid for the persistent kernel: when set (rlrep_gemm_set_debug_buffer), CTA 0 stamps %globaltimer for its first 16
// tiles into dbg[role * 16 + tile], role = 0 TMA issued, 1 first operands landed, 2 accumulator committed, 3 epilogue
// sees the accumulator, 4 epilogue done.
extern unsigned long long* g_persist_dbg;
static void read_trace_here(unsigned long long* out16) {
  RLREP_CUDA(cudaMemcpyFromSymbol(out16, g_gemm_trace, sizeof(unsigned long long) * 16));
}

namespace {

__device__ __forceinline__ void trace(int slot) {
#ifdef RLREP_GEMM_TRACE
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
    g_gemm_trace[slot] = t;
  }
#endif
}

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct TileStore {  // what the store phase needs to know about the tile (run-time so the functions below are shared)
  uint32_t stage_addr;  // shared-memory address of this CTA's staged fp32 tile (pull) / of its reduction slots (push)
  uint32_t peer_stride; // push mode: bytes between the slots of consecutive source CTAs (0 = pull over DSMEM)
  int row_bias;         // row of the staged tile that local row 0 of this CTA's slice maps to (pull: row0, push: 0)
  int lds;              // staging row pitch in floats
  int c4_shift;         // log2(BN / 4)
  int splits;           // cluster size along K
  int row0, rows_per;   // rows of the tile this CTA reduces and stores
  int m0, n0, M, N;
  float* C;
  int ldc;
};

template <int S>
__device__ __forceinline__ float4 load_reduced_n(uint32_t off) {
  float4 v[S];
#pragma unroll
  for (int p = 0; p < S; ++p) v[p] = ptx::ld_dsmem_f4(off, p);  // all peers in flight at once
  float4 acc = v[0];
#pragma unroll
  for (int p = 1; p < S; ++p) {  // fixed order over the cluster => deterministic
    acc.x += v[p].x; acc.y += v[p].y; acc.z += v[p].z; acc.w += v[p].w;
  }
  return acc;
}
template <int S>
__device__ __forceinline__ float4 load_reduced_local(uint32_t off, uint32_t stride) {
  float4 v[S];
#pragma unroll
  for (int p = 0; p < S; ++p) v[p] = ptx::ld_shared_f4(off + p * stride);
  float4 acc = v[0];
#pragma unroll
  for (int p = 1; p < S; ++p) {  // same fixed order as the DSMEM pull: bit-identical results in both modes
    acc.x += v[p].x; acc.y += v[p].y; acc.z += v[p].z; acc.w += v[p].w;
  }
  return acc;
}
__device__ __forceinline__ float4 load_reduced(const TileStore& t, uint32_t off) {
  if (t.peer_stride != 0) {
    switch (t.splits) {
      case 2: return load_reduced_local<2>(off, t.peer_stride);
      case 4: return load_reduced_local<4>(off, t.peer_stride);
      default: return load_reduced_local<8>(off, t.peer_stride);
    }
  }
  switch (t.splits) {
    case 1: return ptx::ld_shared_f4(off);
    case 2: return load_reduced_n<2>(off);
    case 4: return load_reduced_n<4>(off);
    default: return load_reduced_n<8>(off);
  }
}

// Store phase, fast path: interior tile, every pointer 16-byte aligned, N % 4 == 0.  ACT / DACT / BIAS / EXTRAS are
// compile-time so the loop carries only the instructions the layer needs (the step is issue-bound here: few warps
// per SM, so every instruction counts).  Four float4 per thread are loaded before any is consumed.
template <int ACT, int DACT, bool BIAS, bool EXTRAS>
__device__ __noinline__ bool store_tile_fast(const TileStore t, const Epilogue* __restrict__ ep) {
  const Epilogue& epi = *ep;
  constexpr int U = 4;
  const int nthr = blockDim.x;
  const int total = t.rows_per << t.c4_shift;
  const int c4_mask = (1 << t.c4_shift) - 1;
  auto one = [&](int idx, float4 acc) {
    const int rr = t.row0 + (idx >> t.c4_shift), c4 = idx & c4_mask;
    const int gm = t.m0 + rr, gn = t.n0 + c4 * 4;
    float v[4] = {acc.x, acc.y, acc.z, acc.w};
    if constexpr (EXTRAS) {
      const float sc = epi.scale;
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] *= sc;
      if (epi.r1_u) {
        const float u = __ldg(epi.r1_u + gm);
        const float4 w = __ldg(reinterpret_cast<const float4*>(epi.r1_v + gn));
        v[0] = fmaf(u, w.x, v[0]); v[1] = fmaf(u, w.y, v[1]); v[2] = fmaf(u, w.z, v[2]); v[3] = fmaf(u, w.w, v[3]);
      }
    }
    if constexpr (BIAS) {
      if (!EXTRAS || epi.bias != nullptr) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(epi.bias + gn));
        v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
      }
    }
    if constexpr (EXTRAS) {
      if (epi.pre_out)
        *reinterpret_cast<float4*>(epi.pre_out + (size_t)gm * epi.ld_pre + gn) = make_float4(v[0], v[1], v[2], v[3]);
    }
    if constexpr (ACT != ACT_NONE) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = apply_act(v[j], ACT < 0 ? epi.act : ACT);
    }
    if constexpr (DACT != DACT_NONE) {
      const int dact = DACT < 0 ? epi.dact : DACT;
      if (dact != DACT_NONE) {
        const float4 x = *reinterpret_cast<const float4*>(epi.aux + (size_t)gm * epi.ld_aux + gn);
        v[0] *= apply_dact(x.x, dact); v[1] *= apply_dact(x.y, dact); v[2] *= apply_dact(x.z, dact); v[3] *= apply_dact(x.w, dact);
      }
    }
    float4* cp = reinterpret_cast<float4*>(t.C + (size_t)gm * t.ldc + gn);
    if constexpr (EXTRAS) {
      if (epi.accumulate) { const float4 o = *cp; v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w; }
    }
    *cp = make_float4(v[0], v[1], v[2], v[3]);
  };
  if (t.splits > 1 && t.peer_stride == 0 && total <= nthr * 2 * U) {
    // The whole slice fits in registers: pull it over DSMEM, tell the cluster we are done with its shared memory
    // (peers may exit), and only then do the epilogue math and the global stores.
    float4 acc[2 * U];
    if (threadIdx.x == 0) trace(9);
#pragma unroll
    for (int u = 0; u < 2 * U; ++u) {
      const int idx = threadIdx.x + u * nthr;
      if (idx < total)
        acc[u] = load_reduced(t, t.stage_addr + (((t.row_bias + (idx >> t.c4_shift)) * t.lds + (idx & c4_mask) * 4) << 2));
    }
    if (threadIdx.x == 0) { if (acc[0].x == 123.456f) trace(15); trace(10); }
    ptx::cluster_arrive_relaxed();
    if (threadIdx.x == 0) trace(11);
#pragma unroll
    for (int u = 0; u < 2 * U; ++u) {
      const int idx = threadIdx.x + u * nthr;
      if (idx < total) one(idx, acc[u]);
    }
    return true;
  }
  const int chunk = nthr * U;
  const int main_end = (total / chunk) * chunk;
  int base = threadIdx.x;
#pragma unroll 1
  for (; base < main_end; base += chunk) {
    float4 acc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int idx = base + u * nthr;
      acc[u] = load_reduced(t, t.stage_addr + (((t.row_bias + (idx >> t.c4_shift)) * t.lds + (idx & c4_mask) * 4) << 2));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) one(base + u * nthr, acc[u]);
  }
#pragma unroll 1
  for (int idx = main_end + threadIdx.x; idx < total; idx += nthr)
    one(idx, load_reduced(t, t.stage_addr + (((t.row_bias + (idx >> t.c4_shift)) * t.lds + (idx & c4_mask) * 4) << 2)));
  return false;
}

// Store phase, general path: edge tiles, ragged N, unaligned pointers.
__device__ __noinline__ void store_tile_general(const TileStore t, const Epilogue* __restrict__ ep) {
  const Epilogue& epi = *ep;
  const int total = t.rows_per << t.c4_shift;
  const int c4_mask = (1 << t.c4_shift) - 1;
#pragma unroll 1
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int rr = t.row0 + (idx >> t.c4_shift), c4 = idx & c4_mask;
    const int gm = t.m0 + rr, gn = t.n0 + c4 * 4;
    if (gm >= t.M || gn >= t.N) continue;
    const float4 acc = load_reduced(t, t.stage_addr + (((rr - t.row0 + t.row_bias) * t.lds + c4 * 4) << 2));
    float* cp = t.C + (size_t)gm * t.ldc + gn;
    const float a4[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll 1
    for (int j = 0; j < 4; ++j)
      if (gn + j < t.N) cp[j] = epilogue_apply<-1, -1>(epi, a4[j], gm, gn + j, cp + j);
  }
}

// Returns true when the cluster "done with peers' shared memory" arrive has already been issued.
__device__ __forceinline__ bool store_tile(const TileStore& t, const Epilogue* ep) {
  const Epilogue& epi = *ep;
  const bool use_aux = epi.dact != DACT_NONE;
  const bool fast = t.m0 + BM <= t.M && t.n0 + (4 << t.c4_shift) <= t.N && (t.N & 3) == 0 && (t.ldc & 3) == 0 &&
                    aligned16(t.C) && (!use_aux || ((epi.ld_aux & 3) == 0 && aligned16(epi.aux))) &&
                    (!epi.pre_out || ((epi.ld_pre & 3) == 0 && aligned16(epi.pre_out))) &&
                    (!epi.bias || aligned16(epi.bias)) && (!epi.r1_v || aligned16(epi.r1_v));
  if (!fast) {
    store_tile_general(t, ep);
    return false;
  }
  const bool extras = epi.r1_u != nullptr || epi.pre_out != nullptr || epi.accumulate != 0 || epi.scale != 1.0f;
  const bool bias = epi.bias != nullptr;
  if (extras) return store_tile_fast<-1, -1, true, true>(t, ep);  // bias pointer may be null there: checked inside
  bool arrived = false;
#define RLREP_FAST(A, D)                                             \
  do {                                                               \
    if (bias) arrived = store_tile_fast<A, D, true, false>(t, ep);   \
    else arrived = store_tile_fast<A, D, false, false>(t, ep);       \
  } while (0)
  RLREP_EPILOGUE_SWITCH(epi, RLREP_FAST);
#undef RLREP_FAST
  return arrived;
}

// Body of gemm_tf32_kernel and of its population form gemm_tf32_members_kernel (MEMBERS, GemmArgs::mb).
template <int BN, bool A_MN, bool B_MN, bool MEMBERS>
__device__ __forceinline__ void gemm_tf32_body(const CUtensorMap& tmA, const CUtensorMap& tmB, float* __restrict__ C,
                                               int ldc, int M, int N, int K, int kb_per_split, int stages, int push,
                                               int conv_w, const Epilogue& epi, long long mstride) {
  // `stages` is a launch parameter: short K-slices run with a shallow ring so that two CTAs (of this or of a
  // concurrent GEMM on another stream) fit on one SM; long ones get the deepest ring that fits.
  const int STAGES = stages;
  // bits 8..15: K groups - 1.  gridDim.z = groups x splits: every group of `splits` CTAs (one cluster) reduces its own K
  // range into its own output matrix, `group` matrices of ceil(M / 128) * 128 rows behind each other -- K-parallelism
  // beyond the 8 CTAs a cluster can hold, for the caller to sum (the implicit conv weight gradient: K ~ 1e5)
  const int groups = ((push >> 8) & 0xff) + 1;
  push &= 1;
  constexpr int A_BYTES = BM * BK * 4;
  constexpr int B_BYTES = BN * BK * 4;
  constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
  constexpr int LDS = BN + 4;  // staging row pitch in floats: 16-byte aligned rows, conflict-free float4 access
  static_assert(BN == 32 || BN == 64 || BN == 128 || BN == 256, "BN must be a power of two in [32,256]");
  static_assert(min_stages(BN) <= num_stages(BN), "staging tile must fit in the pipeline buffers");

  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B atoms must sit on 1024-byte boundaries.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * (A_BYTES + B_BYTES));
  uint64_t* empty_bar = full_bar + 8;  // barrier slots are laid out for the maximum ring depth
  uint64_t* accum_bar = empty_bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
  float* stage = reinterpret_cast<float*>(smem);  // reuses the operand ring once the accumulator is complete
  // push mode: reduction slots [splits][BM / splits][LDS] behind the barriers (16-byte aligned: the ring is 1 KB aligned)
  float* slots = reinterpret_cast<float*>(smem + STAGES * (A_BYTES + B_BYTES) + 256);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) trace(0);
  const int n0 = blockIdx.x * BN;
  // population GEMM (MEMBERS): gridDim.y = members x M-tiles, and the tensor maps have the member as their outermost
  // dimension (GemmArgs::mb)
  const int member = MEMBERS ? blockIdx.y / ((M + BM - 1) / BM) : 0;
  const int m0 = (blockIdx.y - member * ((M + BM - 1) / BM)) * BM;
  if constexpr (MEMBERS) C = member_ptr(C, member * mstride);
  const int splits = gridDim.z / groups;
  if (groups > 1) C += (size_t)(blockIdx.z / splits) * (size_t)(((M + BM - 1) / BM) * BM) * ldc;
  const int nkb_total = (K + BK - 1) / BK;
  const int kb_begin = blockIdx.z * kb_per_split;
  const int kb_end = min(nkb_total, kb_begin + kb_per_split);
  const int nkb = kb_end - kb_begin;

  // One TMA round: arm the stage's barrier and fetch the A / B boxes of k-block (kb_begin + it).
  auto produce = [&](int it) {
    const int s = it % STAGES;
    ptx::mbar_arrive_expect_tx(&full_bar[s], A_BYTES + B_BYTES);
    const int k0 = (kb_begin + it) * BK;
    uint8_t* a_dst = sA + s * A_BYTES;
    uint8_t* b_dst = sB + s * B_BYTES;
    // MN-major operands: one 3-D box {32 (m % 32), 32 (k), rows / 32 (m / 32)} lands as consecutive 4 KB sub-boxes
    // implicit convolution (conv_w > 0): k-block t is tap (t / 3, t % 3) -- the same 32 channels, rows shifted on the grid
    if constexpr (MEMBERS) {
      if (!A_MN) ptx::tma_load_3d(a_dst, &tmA, &full_bar[s], k0, m0, member);
      else ptx::tma_load_4d(a_dst, &tmA, &full_bar[s], 0, k0, m0 / 32, member);
      if (!B_MN) ptx::tma_load_3d(b_dst, &tmB, &full_bar[s], k0, n0, member);
      else ptx::tma_load_4d(b_dst, &tmB, &full_bar[s], 0, k0, n0 / 32, member);
      return;
    }
    if (!A_MN) {
      const int t = kb_begin + it;
      if (conv_w > 0) ptx::tma_load_2d(a_dst, &tmA, &full_bar[s], 0, m0 + (t / 3) * conv_w + (t % 3));
      else ptx::tma_load_2d(a_dst, &tmA, &full_bar[s], k0, m0);
    } else {
      ptx::tma_load_3d(a_dst, &tmA, &full_bar[s], 0, k0, m0 / 32);
    }
    // implicit weight gradient (conv_w < 0): n-chunk j of the (ky, q, c) view is (q, ky) = (j % 8, j / 8)
    if (!B_MN) ptx::tma_load_2d(b_dst, &tmB, &full_bar[s], k0, n0);
    else if (conv_w < 0) ptx::tma_load_4d(b_dst, &tmB, &full_bar[s], 0, k0, (n0 / 32) % 8, (n0 / 32) / 8);
    else ptx::tma_load_3d(b_dst, &tmB, &full_bar[s], 0, k0, n0 / 32);
  };
  // one stage before the setup barrier (TMA issue itself is not free)
  const int first_round = nkb < 1 ? nkb : 1;
  if (warp == 0 && lane == 0) {
    // The producer owns the barriers: it initialises them and immediately fills the ring (no empty-wait is needed
    // for the first round), so the first operands are in flight while the other warps allocate TMEM.
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(accum_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  // the operands and C may still be in use by the previous kernel (launch_variant launches with PDL)
  ptx::pdl_wait();
  if (warp == 0 && lane == 0)
    for (int it = 0; it < first_round; ++it) produce(it);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) trace(1);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {  // same lane that ran the first round before the setup barrier
      for (int it = first_round; it < nkb; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1;
        ptx::mbar_wait(&empty_bar[s], ph ^ 1);
        produce(it);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_tf32(BM, BN, A_MN, B_MN);
      for (int it = 0; it < nkb; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1;
        ptx::mbar_wait(&full_bar[s], ph);
        if (it == 0) trace(2);
        ptx::tc_fence_after_sync();
        const uint32_t a_addr = ptx::smem_u32(sA + s * A_BYTES);
        const uint32_t b_addr = ptx::smem_u32(sB + s * B_BYTES);
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t adesc = A_MN ? ptx::make_smem_desc(a_addr + k * 1024, 4096, 512, 1)
                                      : ptx::make_smem_desc(a_addr + k * UMMA_K * 4, 16, 1024, 2);
          const uint64_t bdesc = B_MN ? ptx::make_smem_desc(b_addr + k * 1024, 4096, 512, 1)
                                      : ptx::make_smem_desc(b_addr + k * UMMA_K * 4, 16, 1024, 2);
          ptx::mma_tf32_ss(tmem_base, adesc, bdesc, idesc, (it > 0 || k > 0) ? 1u : 0u);
        }
        ptx::mma_commit(&empty_bar[s]);  // frees the smem stage once these MMAs have read it
      }
      ptx::mma_commit(accum_bar);  // accumulator complete
      trace(3);
    }
  } else if (warp < 6) {
    // ------------------------------------------------------------ TMEM -> shared staging (warps 2..5)
    // accum_bar completing means every MMA has finished reading the operand ring (and every TMA write into it was
    // consumed before that), so the ring can be overwritten with the fp32 tile.
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int r = 32 * q + lane;
    ptx::mbar_wait(accum_bar, 0);
    if (threadIdx.x == 64) trace(4);
    ptx::tc_fence_after_sync();
    if (push) {
      // row r of the tile belongs to CTA r / rows_per of the cluster: write it into that CTA's slot for this source
      const int rows_per = BM / splits;
      const uint32_t owner = r / rows_per;
      const uint32_t my_rank = ptx::cluster_ctarank();
      const uint32_t dst_row = ptx::smem_u32(slots) + ((my_rank * rows_per + (r - owner * rows_per)) * LDS) * 4;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(32 * q) << 16) + c * 32, v);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j)
          ptx::st_dsmem_f4(dst_row + (c * 32 + 4 * j) * 4, owner,
                           make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                       __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])));
      }
    } else {
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(32 * q) << 16) + c * 32, v);
        ptx::tmem_ld_wait();
        float4* dst = reinterpret_cast<float4*>(stage + r * LDS + c * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                               __uint_as_float(v[4 * j + 3]));
      }
    }
    ptx::tc_fence_before_sync();
  }

  if (threadIdx.x == 64) trace(5);
  if (splits > 1) ptx::cluster_sync(); else __syncthreads();
  if (threadIdx.x == 0) trace(6);
  if (warp == 2) ptx::tmem_dealloc(tmem_base, TMEM_COLS);  // every tcgen05.ld has completed: the tile is in shared memory
  ptx::pdl_launch_dependents();  // only the reduction and the stores remain

  // ---------------------------------------------------------------- reduce + epilogue + coalesced store (all warps)
  {
    TileStore t;
    t.stage_addr = push ? ptx::smem_u32(slots) : ptx::smem_u32(stage);
    t.lds = LDS;
    t.peer_stride = push ? (uint32_t)((BM / splits) * LDS * 4) : 0u;
    t.c4_shift = BN == 32 ? 3 : (BN == 64 ? 4 : (BN == 128 ? 5 : 6));
    t.splits = splits;
    t.rows_per = BM / splits;
    t.row0 = (splits > 1 ? (int)ptx::cluster_ctarank() : 0) * t.rows_per;
    t.row_bias = push ? 0 : t.row0;
    t.m0 = m0; t.n0 = n0; t.M = M; t.N = N;
    t.C = C; t.ldc = ldc;
    bool arrived;
    if constexpr (MEMBERS) {
      const Epilogue em = member_epilogue(epi, member * mstride);
      arrived = store_tile(t, &em);
    } else {
      arrived = store_tile(t, &epi);
    }
    if (threadIdx.x == 0) trace(7);
    if (splits > 1 && !push) {  // peers may still be reading this CTA's staging tile: do not exit before they are done
      if (!arrived) ptx::cluster_arrive_relaxed();
      ptx::cluster_wait();
    }
  }

  if (threadIdx.x == 64) trace(8);
}

template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tf32_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 float* __restrict__ C, int ldc, int M, int N, int K, int kb_per_split, int stages, int push, int conv_w,
                 const Epilogue epi) {
  gemm_tf32_body<BN, A_MN, B_MN, false>(tmA, tmB, C, ldc, M, N, K, kb_per_split, stages, push, conv_w, epi, 0);
}
// mstride bytes between consecutive members' operands, output and epilogue operands; gridDim.y = members x M-tiles
template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tf32_members_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         float* __restrict__ C, int ldc, int M, int N, int K, int kb_per_split, int stages, int push,
                         int conv_w, const Epilogue epi, long long mstride) {
  gemm_tf32_body<BN, A_MN, B_MN, true>(tmA, tmB, C, ldc, M, N, K, kb_per_split, stages, push, conv_w, epi, mstride);
}

// 32 x 32 chunk of the persistent kernel's epilogue: rows come out of the warp's transpose buffer, lanes cover four rows x
// eight 16-byte pieces per store instruction.
template <int ACT, int DACT>
__device__ __forceinline__ void persist_store_rows(const Epilogue& epi, const float* tw, float* __restrict__ C, int ldc,
                                                   int M, int m_base, int gn0, int lane) {
  const int piece = lane & 7, rsub = lane >> 3;
#pragma unroll
  for (int r4 = 0; r4 < 8; ++r4) {
    const int r = r4 * 4 + rsub;
    const int om = m_base + r, on = gn0 + 4 * piece;
    if (om < M) {
      const float4 a4 = *reinterpret_cast<const float4*>(tw + r * 36 + 4 * piece);
      float* cp = C + (size_t)om * ldc + on;
      const float in[4] = {a4.x, a4.y, a4.z, a4.w};
      float o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = epilogue_apply<ACT, DACT>(epi, in[e], om, on + e, cp + e);
      *reinterpret_cast<float4*>(cp) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ persistent variant
// For GEMMs with many output tiles and no split-K (the conv lowering: 3,000+ tiles of 3..9 k-blocks; the batch-sharded
// contrastive logits: 1,024 tiles): one CTA per SM walks the tiles, so barrier setup / TMEM allocation happen once, the
// operand ring keeps streaming across tile boundaries, and the accumulator is DOUBLE-BUFFERED in TMEM -- while four
// epilogue warps drain tile i (tcgen05.ld -> epilogue math -> 128-byte global stores, one output row per thread), the MMA
// warp is already accumulating tile i + 1 into the other half of TMEM.
//   warp 0: TMA producer | warp 1: MMA issuer (owns TMEM alloc / dealloc) | warps 2..5: epilogue (TMEM lane quarter w & 3)
// make_tc_plan picks it for conv-shaped GEMMs (thousands of narrow tiles with a handful of k-blocks each).
constexpr int kPersistThreads = 192;

template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kPersistThreads, 1)
gemm_tf32_persistent_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                            float* __restrict__ C, int ldc, int M, int N, int K, int conv_w, const Epilogue epi,
                            unsigned long long* __restrict__ dbg) {
  constexpr int STAGES = num_stages(BN);
  auto stamp = [&](int role, int tile) {
    if (dbg != nullptr && blockIdx.x == 0 && tile < 16) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
      dbg[role * 16 + tile] = t;
    }
  };
  constexpr int A_BYTES = BM * BK * 4;
  constexpr int B_BYTES = BN * BK * 4;
  constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static_assert(TMEM_COLS <= 512, "two accumulators must fit in TMEM");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * (A_BYTES + B_BYTES));
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* acc_full = empty_bar + 8;   // [2] accumulator complete (MMA -> epilogue)
  uint64_t* acc_empty = acc_full + 2;   // [2] accumulator drained (epilogue -> MMA), 4 arrivals (one per epilogue warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  // per-epilogue-warp transpose buffers [4][32 rows][36 floats] behind the barriers: a thread holds one ROW of the
  // accumulator chunk, but stores want consecutive lanes on consecutive 16-byte pieces of the same output row
  float* tbuf = reinterpret_cast<float*>(smem + STAGES * (A_BYTES + B_BYTES) + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_m = (M + BM - 1) / BM, tiles_n = (N + BN - 1) / BN;
  const int total = tiles_m * tiles_n;
  const int nkb = (K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&acc_full[a], 1);
      ptx::mbar_init(&acc_empty[a], 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer: the ring runs across tile boundaries
    if (lane == 0) {
      int it = 0, tcp = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++tcp) {
        const int m0 = (t % tiles_m) * BM, n0 = (t / tiles_m) * BN;  // m fastest: concurrent CTAs share the B tile in L2
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          ptx::mbar_wait(&empty_bar[s], ((it / STAGES) & 1) ^ 1);  // fresh barrier: parity 1 passes immediately
          if (kb == 0) stamp(0, tcp);
          ptx::mbar_arrive_expect_tx(&full_bar[s], A_BYTES + B_BYTES);
          const int k0 = kb * BK;
          if (!A_MN) {
            if (conv_w > 0) ptx::tma_load_2d(sA + s * A_BYTES, &tmA, &full_bar[s], 0, m0 + (kb / 3) * conv_w + (kb % 3));
            else ptx::tma_load_2d(sA + s * A_BYTES, &tmA, &full_bar[s], k0, m0);
          } else {
            ptx::tma_load_3d(sA + s * A_BYTES, &tmA, &full_bar[s], 0, k0, m0 / 32);
          }
          if (!B_MN) ptx::tma_load_2d(sB + s * B_BYTES, &tmB, &full_bar[s], k0, n0);
          else ptx::tma_load_3d(sB + s * B_BYTES, &tmB, &full_bar[s], 0, k0, n0 / 32);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer: alternates between the two accumulators
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_tf32(BM, BN, A_MN, B_MN);
      int it = 0, tc = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++tc) {
        const int acc = tc & 1;
        ptx::mbar_wait(&acc_empty[acc], ((tc >> 1) & 1) ^ 1);  // the epilogue has drained this accumulator
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          ptx::mbar_wait(&full_bar[s], (it / STAGES) & 1);
          if (kb == 0) stamp(1, tc);
          ptx::tc_fence_after_sync();
          const uint32_t a_addr = ptx::smem_u32(sA + s * A_BYTES);
          const uint32_t b_addr = ptx::smem_u32(sB + s * B_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = A_MN ? ptx::make_smem_desc(a_addr + k * 1024, 4096, 512, 1)
                                        : ptx::make_smem_desc(a_addr + k * UMMA_K * 4, 16, 1024, 2);
            const uint64_t bdesc = B_MN ? ptx::make_smem_desc(b_addr + k * 1024, 4096, 512, 1)
                                        : ptx::make_smem_desc(b_addr + k * UMMA_K * 4, 16, 1024, 2);
            ptx::mma_tf32_ss(d_tmem, adesc, bdesc, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          ptx::mma_commit(&empty_bar[s]);
        }
        ptx::mma_commit(&acc_full[acc]);
        stamp(2, tc);
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 2..5: one output row per thread
    const int q = warp & 3;
    const bool vec_ok = (ldc & 3) == 0 && aligned16(C);
    float* tw = tbuf + q * (32 * 36);
    int tc = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++tc) {
      const int acc = tc & 1;
      const int m0 = (t % tiles_m) * BM, n0 = (t / tiles_m) * BN;
      ptx::mbar_wait(&acc_full[acc], (tc >> 1) & 1);
      if (threadIdx.x == 64) stamp(3, tc);
      ptx::tc_fence_after_sync();
      const int gm = m0 + 32 * q + lane;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(32 * q) << 16) + acc * BN + c * 32, v);
        ptx::tmem_ld_wait();
        const int gn0 = n0 + c * 32;
        if (vec_ok && gn0 + 32 <= N) {
          // transpose through shared memory: lane = row on the way in, (row group, 16-byte piece) on the way out, so
          // every store instruction writes four complete 128-byte row segments
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(tw + lane * 36 + 4 * j) =
                make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                            __uint_as_float(v[4 * j + 3]));
          __syncwarp();
          // compile-time (activation, derivative) pairs: the run-time version drags every transcendental into an
          // unrolled 32-element body that no longer fits the instruction cache (measured 5.6 us per 128 x 32 tile)
#define RLREP_PSTORE(A, D) persist_store_rows<A, D>(epi, tw, C, ldc, M, m0 + 32 * q, gn0, lane)
          RLREP_EPILOGUE_SWITCH(epi, RLREP_PSTORE);
#undef RLREP_PSTORE
          __syncwarp();
        } else if (gm < M && gn0 < N) {
          float* crow = C + (size_t)gm * ldc + gn0;
          for (int e = 0; e < 32 && gn0 + e < N; ++e)
            crow[e] = epilogue_apply<-1, -1>(epi, __uint_as_float(v[e]), gm, gn0 + e, crow + e);
        }
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[acc]);
      if (threadIdx.x == 64) stamp(4, tc);
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------ implicit 3x3 conv, halo in smem
// The persistent kernel above runs an implicit convolution (GemmArgs::conv_w) as nine k-blocks whose A tile is the same 128
// grid rows shifted by the tap: nine TMA loads of 16 KB per tile, i.e. the input map crosses L2 -> SM nine times (measured:
// 65 us for a 55 MB map, the ~12 TB/s L2 ceiling).  Here a tile's A operand is loaded ONCE, with its halo -- grid rows
// [m0, m0 + 128 + 2 conv_w + 2) as one 128B-swizzled box -- and the nine taps are nine sets of MMAs whose A descriptors
// start `shift` rows into that buffer.  Measured on B200: the 128-byte swizzle is a function of the ABSOLUTE shared-memory
// address (bits 4-6 XOR bits 7-9), so a start address that is not 1024-byte aligned needs nothing else -- the descriptor's
// base-offset field stays 0 (setting it to shift % 8 gives wrong products).  The 36 KB of weights are loaded once per CTA and stay resident.
// N <= 32 (every convolution of the pixel agents has 32 output channels), A K-major.
// Rows of a 32 x 16 accumulator chunk staged in tw[32][20]: lane = (row group of 8, 16-byte piece), four passes
// Output mapping and tap list of a halo-kernel launch (GemmArgs::compact_* / conv_tap_*), by value
struct HaloGeom {
  int wp, hy, hx, stride, oy, ox, out_w;  // wp = 0: no compaction (rows stored where they are)
  int ntaps;
  int shift[9], kb[9];
};

// wp > 0: compacting store -- grid row m = (b, y, x) on a grid wp wide goes to row (b * ho + y) * ho + x when x, y < ho and
// nowhere otherwise (the thread's first row is decomposed once per tile, the other three follow by carrying 8 columns).
// The epilogue of this kernel is bias + activation + derivative mask only (checked by the launcher); the four rows' mask
// values are fetched as float4 BEFORE the first store -- behind a store the compiler cannot hoist them (aliasing), and four
// serialised global-load latencies per tile made this epilogue the slowest stage of the pipeline.
// Split in two so that the row mapping and the mask / bias loads are issued BEFORE the thread waits for the accumulator
// (they depend on the tile index only): the loads' latency hides behind the MMAs of the tile.
struct HaloRows {
  int row_of[4];
  bool live[4];
  float4 ax[4];
  float4 bv;
  bool use_aux;
};
__device__ __forceinline__ void halo_rows_prepare(HaloRows& hr, const Epilogue& epi, int M, int m_base, int gn0, int lane,
                                                  const HaloGeom& geo) {
  const int wp = geo.wp;
  const int piece = lane & 3, rsub = lane >> 2;
  const int on = gn0 + 4 * piece;
  int gb = 0, gy = 0, gx = 0;
  if (wp > 0) {
    // m < 2^24 (checked by the launcher): quotient from a float reciprocal, corrected by one
    const int m = m_base + rsub, wp2 = wp * wp;
    gb = __float2int_rz(__int2float_rn(m) * __frcp_rn(__int2float_rn(wp2)));
    int rem = m - gb * wp2;
    if (rem < 0) { --gb; rem += wp2; } else if (rem >= wp2) { ++gb; rem -= wp2; }
    gy = __float2int_rz(__int2float_rn(rem) * __frcp_rn(__int2float_rn(wp)));
    gx = rem - gy * wp;
    if (gx < 0) { --gy; gx += wp; } else if (gx >= wp) { ++gy; gx -= wp; }
  }
#pragma unroll
  for (int r4 = 0; r4 < 4; ++r4) {
    const int om = m_base + r4 * 8 + rsub;
    hr.live[r4] = om < M;
    hr.row_of[r4] = om;
    if (wp > 0) {
      hr.live[r4] = hr.live[r4] && gx < geo.hx && gy < geo.hy;
      hr.row_of[r4] = (gb * geo.out_w + geo.stride * gy + geo.oy) * geo.out_w + geo.stride * gx + geo.ox;
      gx += 8;  // wp > 8: at most one wrap
      if (gx >= wp) { gx -= wp; ++gy; }
      if (gy >= wp) { gy -= wp; ++gb; }
    }
  }
  hr.use_aux = epi.dact != DACT_NONE;
#pragma unroll
  for (int r4 = 0; r4 < 4; ++r4)
    hr.ax[r4] = (hr.use_aux && hr.live[r4])
                    ? __ldg(reinterpret_cast<const float4*>(epi.aux + (size_t)hr.row_of[r4] * epi.ld_aux + on))
                    : make_float4(1.f, 1.f, 1.f, 1.f);
  hr.bv = epi.bias ? __ldg(reinterpret_cast<const float4*>(epi.bias + on)) : make_float4(0.f, 0.f, 0.f, 0.f);
}
template <int ACT, int DACT>
__device__ __forceinline__ void halo_rows_finish(const HaloRows& hr, const Epilogue& epi, const float* tw,
                                                 float* __restrict__ C, int ldc, int gn0, int lane) {
  const int piece = lane & 3, rsub = lane >> 2;
  const int on = gn0 + 4 * piece;
  constexpr bool kRuntime = ACT < 0 || DACT < 0;
  const int act = kRuntime ? epi.act : ACT, dact = kRuntime ? epi.dact : DACT;
#pragma unroll
  for (int r4 = 0; r4 < 4; ++r4) {
    if (!hr.live[r4]) continue;
    const float4 a4 = *reinterpret_cast<const float4*>(tw + (r4 * 8 + rsub) * 20 + 4 * piece);
    float o[4] = {fmaf(a4.x, epi.scale, hr.bv.x), fmaf(a4.y, epi.scale, hr.bv.y), fmaf(a4.z, epi.scale, hr.bv.z),
                  fmaf(a4.w, epi.scale, hr.bv.w)};
    const float h[4] = {hr.ax[r4].x, hr.ax[r4].y, hr.ax[r4].z, hr.ax[r4].w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      o[e] = apply_act(o[e], act);
      if (hr.use_aux) o[e] *= apply_dact(h[e], dact);
    }
    *reinterpret_cast<float4*>(C + (size_t)hr.row_of[r4] * ldc + on) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

constexpr int kHaloThreads = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue: two per TMEM lane quarter, 16 columns each
constexpr int kHaloStages = 4;
constexpr int kHaloMaxRows = 256;                  // TMA box limit; 128 + 2 conv_w + 2 <= 256  ->  conv_w <= 63
constexpr int kHaloBytes = kHaloMaxRows * 128;     // per stage
constexpr int kHaloSmem = kHaloStages * kHaloBytes + 9 * 32 * BK * 4 + 1024 + 256 + 8 * 32 * 20 * 4;
static_assert(kHaloSmem <= kMaxSmem, "halo kernel shared memory");

template <bool B_MN>
__global__ void __launch_bounds__(kHaloThreads, 1)
gemm_conv_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      float* __restrict__ C, int ldc, int M, int N, int halo_rows, const HaloGeom geo,
                      const Epilogue epi) {
  constexpr int BN = 32;
  constexpr int B_BYTES = BN * BK * 4;
  constexpr uint32_t TMEM_COLS = 2 * BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                  // [kHaloStages][kHaloBytes]
  uint8_t* sB = smem + kHaloStages * kHaloBytes;       // [9][B_BYTES], resident
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + 9 * B_BYTES);
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* acc_full = empty_bar + 8;
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* w_bar = acc_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_bar + 1);
  float* tbuf = reinterpret_cast<float*>(sB + 9 * B_BYTES + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = (M + BM - 1) / BM;  // one n-tile

  if (threadIdx.x == 0) {
    for (int s = 0; s < kHaloStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&acc_full[a], 1);
      ptx::mbar_init(&acc_empty[a], 8);
    }
    ptx::mbar_init(w_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      // the weights, once: nine k-blocks of [32, 32]
      ptx::mbar_arrive_expect_tx(w_bar, 9 * B_BYTES);
      for (int kb = 0; kb < 9; ++kb) {
        if (!B_MN) ptx::tma_load_2d(sB + kb * B_BYTES, &tmB, w_bar, kb * BK, 0);
        else ptx::tma_load_3d(sB + kb * B_BYTES, &tmB, w_bar, 0, kb * BK, 0);
      }
      int it = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
        const int s = it % kHaloStages;
        ptx::mbar_wait(&empty_bar[s], ((it / kHaloStages) & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(&full_bar[s], halo_rows * 128);
        ptx::tma_load_2d(sA + s * kHaloBytes, &tmA, &full_bar[s], 0, t * BM);  // rows past M read as zero
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_tf32(BM, BN, false, B_MN);
      ptx::mbar_wait(w_bar, 0);
      // the tap list in registers (static indexing of the parameter arrays): a run-time-indexed constant load per tap in
      // front of every MMA group cost the issuing thread ~20 us per launch
      uint32_t tap_a[9], tap_b[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        tap_a[tap] = (uint32_t)geo.shift[tap] * 128u;
        tap_b[tap] = (uint32_t)geo.kb[tap] * (uint32_t)B_BYTES;
      }
      const int ntaps = geo.ntaps;
      int it = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
        const int acc = it & 1, s = it % kHaloStages;
        ptx::mbar_wait(&acc_empty[acc], ((it >> 1) & 1) ^ 1);
        ptx::mbar_wait(&full_bar[s], (it / kHaloStages) & 1);
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * BN;
        const uint32_t a_base = ptx::smem_u32(sA + s * kHaloBytes), b_base = ptx::smem_u32(sB);
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          if (tap >= ntaps) break;
          const uint32_t a_addr = a_base + tap_a[tap], b_addr = b_base + tap_b[tap];
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = ptx::make_smem_desc(a_addr + k * UMMA_K * 4, 16, 1024, 2);
            const uint64_t bdesc = B_MN ? ptx::make_smem_desc(b_addr + k * 1024, 4096, 512, 1)
                                        : ptx::make_smem_desc(b_addr + k * UMMA_K * 4, 16, 1024, 2);
            ptx::mma_tf32_ss(d_tmem, adesc, bdesc, idesc, (tap > 0 || k > 0) ? 1u : 0u);
          }
        }
        ptx::mma_commit(&empty_bar[s]);
        ptx::mma_commit(&acc_full[acc]);
      }
    }
  } else {
    // epilogue warps 2..9: TMEM lane quarter warp % 4, columns [16 half, 16 half + 16) -- with one warp per quarter the
    // epilogue (1.3 us per tile) was the longest stage of the pipeline
    const int q = warp & 3, half = (warp - 2) >> 2;
    const bool vec_ok = (ldc & 3) == 0 && aligned16(C);
    float* tw = tbuf + (warp - 2) * (32 * 20);
    int tc = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++tc) {
      const int acc = tc & 1;
      const int m0 = t * BM;
      const int gm = m0 + 32 * q + lane, gn0 = 16 * half;
      const bool fast = vec_ok && N == 32;
      HaloRows hr;
      if (fast) halo_rows_prepare(hr, epi, M, m0 + 32 * q, gn0, lane, geo);  // mask / bias loads in flight during the MMAs
      ptx::mbar_wait(&acc_full[acc], (tc >> 1) & 1);
      ptx::tc_fence_after_sync();
      uint32_t v[16];
      ptx::tmem_ld_32x32b_x16(tmem_base + (static_cast<uint32_t>(32 * q) << 16) + acc * BN + gn0, v);
      ptx::tmem_ld_wait();
      if (fast) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(tw + lane * 20 + 4 * j) =
              make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                          __uint_as_float(v[4 * j + 3]));
        __syncwarp();
#define RLREP_HSTORE(A, D) halo_rows_finish<A, D>(hr, epi, tw, C, ldc, gn0, lane)
        RLREP_EPILOGUE_SWITCH(epi, RLREP_HSTORE);
#undef RLREP_HSTORE
        __syncwarp();
      } else if (gm < M) {
        int om = gm;
        bool live = true;
        if (geo.wp > 0) {
          const int gb = gm / (geo.wp * geo.wp), rem = gm - gb * geo.wp * geo.wp;
          const int gy = rem / geo.wp, gx = rem - gy * geo.wp;
          live = gx < geo.hx && gy < geo.hy;
          om = (gb * geo.out_w + geo.stride * gy + geo.oy) * geo.out_w + geo.stride * gx + geo.ox;
        }
        if (live) {
          float* crow = C + (size_t)om * ldc;
          for (int e = 0; e < 16 && gn0 + e < N; ++e)
            crow[gn0 + e] = epilogue_apply<-1, -1>(epi, __uint_as_float(v[e]), om, gn0 + e, crow + gn0 + e);
        }
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[acc]);
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, TMEM_COLS);
}

template <bool B_MN>
void launch_conv_halo(const TcGemmPlan& p, cudaStream_t stream) {
  auto kern = gemm_conv_halo_kernel<B_MN>;
  static bool attr_set = false;
  if (!attr_set) {
    RLREP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kHaloSmem));
    attr_set = true;
  }
  const GemmArgs& a = p.args;
  const int tiles = ceil_div(a.M, BM);
  HaloGeom geo;
  geo.wp = a.compact_wp;
  geo.hy = a.compact_ho;
  geo.hx = a.compact_hx > 0 ? a.compact_hx : a.compact_ho;
  geo.stride = a.compact_stride; geo.oy = a.compact_oy; geo.ox = a.compact_ox;
  geo.out_w = a.compact_out_w > 0 ? a.compact_out_w : a.compact_ho;
  geo.ntaps = a.conv_ntaps > 0 ? a.conv_ntaps : 9;
  for (int t = 0; t < 9; ++t) {
    geo.shift[t] = a.conv_ntaps > 0 ? a.conv_tap_shift[t] : (t / 3) * a.conv_w + (t % 3);
    geo.kb[t] = a.conv_ntaps > 0 ? a.conv_tap_kb[t] : t;
    RLREP_CHECK(t >= geo.ntaps || (geo.shift[t] >= 0 && geo.shift[t] + 128 <= p.halo_rows && geo.kb[t] >= 0 && geo.kb[t] < 9),
                "halo convolution: tap outside the halo buffer");
  }
  kern<<<std::min(tiles, kNumSMs), kHaloThreads, kHaloSmem, stream>>>(p.tmA, p.tmB, a.C, a.ldc, a.M, a.N, p.halo_rows, geo,
                                                                       a.epi);
  RLREP_LAUNCHED_W("gemm_conv_halo", stream, 4.0 * ((double)a.M * 32 + (double)a.N * a.K + (double)a.M * a.N),
                   2.0 * a.M * a.N * a.K);
}
template <int BN, int AMN>
void launch_conv_halo_if(const TcGemmPlan& p, cudaStream_t stream) {
  if constexpr (BN == 32 && AMN == 0) {
    if (p.args.b_mn) launch_conv_halo<true>(p, stream);
    else launch_conv_halo<false>(p, stream);
  } else {
    throw Error("the halo convolution kernel exists for BN = 32, K-major A only");
  }
}

template <int BN, bool A_MN, bool B_MN>
void launch_variant_persistent(const TcGemmPlan& p, cudaStream_t stream) {
  auto kern = gemm_tf32_persistent_kernel<BN, A_MN, B_MN>;
  static bool attr_set = false;
  if (!attr_set) {
    RLREP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(BN) + 4 * 32 * 36 * 4));
    attr_set = true;
  }
  const GemmArgs& a = p.args;
  RLREP_CHECK(a.compact_wp == 0 && a.conv_ntaps == 0, "compacting stores / tap lists exist on the halo convolution kernel only");
  const int tiles = ceil_div(a.M, BM) * ceil_div(a.N, BN);
  kern<<<std::min(tiles, kNumSMs), kPersistThreads, smem_bytes(BN) + 4 * 32 * 36 * 4, stream>>>(p.tmA, p.tmB, a.C, a.ldc, a.M, a.N, a.K, a.conv_w, a.epi, g_persist_dbg);
  RLREP_LAUNCHED_W("gemm_tf32_persistent", stream,
                   4.0 * ((double)a.M * (a.conv_w > 0 ? 32 : a.K) + (double)a.N * a.K + (double)a.M * a.N),
                   2.0 * a.M * a.N * a.K);
}

template <int BN, bool A_MN, bool B_MN>
void fill_launch_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr, dim3 grid, int split_k, int stages,
                        bool push, cudaStream_t stream) {
  static bool attr_set = false;  // per template instantiation
  if (!attr_set) {
    RLREP_CUDA(cudaFuncSetAttribute(gemm_tf32_kernel<BN, A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    RLREP_CUDA(cudaFuncSetAttribute(gemm_tf32_members_kernel<BN, A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kMaxSmem));
    attr_set = true;
  }
  cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes(BN, stages, push);
  cfg.stream = stream;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = split_k;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
}

template <int BN, bool A_MN, bool B_MN>
void launch_variant(const TcGemmPlan& p, cudaStream_t stream) {
  const GemmArgs& a = p.args;
  RLREP_CHECK(a.compact_wp == 0 && a.conv_ntaps == 0, "compacting stores / tap lists exist on the halo convolution kernel only");
  RLREP_CHECK(p.stages >= (p.push ? 2 : min_stages(BN)) && p.stages <= num_stages(BN), "bad pipeline depth");
  RLREP_CHECK(!p.push || (p.split_k > 1 && smem_bytes(BN, p.stages, true) <= kMaxSmem), "bad push-mode plan");
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  fill_launch_config<BN, A_MN, B_MN>(cfg, attr, dim3(ceil_div(a.N, BN), ceil_div(a.M, BM) * a.mb.n, p.split_k * p.k_groups),
                                     p.split_k, p.stages, p.push, stream);
  attr[1] = pdl_attribute();
  cfg.numAttrs = 2;
  const int push = (p.push ? 1 : 0) | ((p.k_groups - 1) << 8);
  if (a.mb.n > 1)
    RLREP_CUDA(cudaLaunchKernelEx(&cfg, gemm_tf32_members_kernel<BN, A_MN, B_MN>, p.tmA, p.tmB, a.C, a.ldc, a.M, a.N, a.K,
                                  p.kb_per_split, p.stages, push, a.conv_w, a.epi, a.mb.stride));
  else
    RLREP_CUDA(cudaLaunchKernelEx(&cfg, gemm_tf32_kernel<BN, A_MN, B_MN>, p.tmA, p.tmB, a.C, a.ldc, a.M, a.N, a.K,
                                  p.kb_per_split, p.stages, push, a.conv_wgrad_hi > 0 ? -1 : a.conv_w, a.epi));
  g_trace_reader = &read_trace_here;
  // implicit convolution: A is the [M, 32] pixel matrix, read once from HBM (the nine shifted re-reads hit L2)
  RLREP_LAUNCHED_W("gemm_tf32", stream,
                   4.0 * a.mb.n * ((double)a.M * (a.conv_w > 0 ? 32 : a.K) + (double)(a.conv_wgrad_hi > 0 ? 128 : a.N) * a.K +
                                   (double)a.M * a.N),
                   2.0 * a.M * a.N * a.K * a.mb.n);
}

// How many clusters of `split_k` CTAs of this variant the GPU can hold at once (occupancy API; clusters must fit in
// one GPC, so this is NOT 148 / split_k) -- the denominator of the cost model's wave count.
template <int BN, bool A_MN, bool B_MN>
int max_clusters_variant(int split_k, int stages, bool push) {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  fill_launch_config<BN, A_MN, B_MN>(cfg, attr, dim3(1, 1, split_k), split_k, stages, push, nullptr);
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, gemm_tf32_kernel<BN, A_MN, B_MN>, &cfg) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    n = kNumSMs / split_k;
  }
  return n;
}

}  // namespace

#define RLREP_TC_DEFINE(BN, AMN)                                              \
  void launch_tc_##BN##_##AMN(const TcGemmPlan& p, cudaStream_t stream) {     \
    if (p.halo_rows > 0) {                                                    \
      launch_conv_halo_if<BN, AMN>(p, stream);                                \
      return;                                                                 \
    }                                                                         \
    if (p.persistent) {                                                       \
      if (p.args.b_mn) launch_variant_persistent<BN, (AMN) != 0, true>(p, stream);   \
      else launch_variant_persistent<BN, (AMN) != 0, false>(p, stream);       \
      return;                                                                 \
    }                                                                         \
    if (p.args.b_mn) launch_variant<BN, (AMN) != 0, true>(p, stream);         \
    else launch_variant<BN, (AMN) != 0, false>(p, stream);                    \
  }                                                                           \
  int max_clusters_##BN##_##AMN(bool b_mn, int split_k, int stages, bool push) {          \
    return b_mn ? max_clusters_variant<BN, (AMN) != 0, true>(split_k, stages, push)       \
                : max_clusters_variant<BN, (AMN) != 0, false>(split_k, stages, push);     \
  }
#endif  // RLREP_TC_DEVICE_CODE

}  // namespace tc
}  // namespace rlrep

// GEMM chain kernel and its host-side planner (see gemm_chain.cuh).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "gemm_chain.cuh"
#include "ptx.cuh"

namespace rlrep {

namespace {

constexpr int kThreads = 320;           // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quarter)
constexpr int kEpiWarps = 8;
constexpr int kStages = 6;
constexpr int kCW = 16;                 // epilogue chunk width in columns (registers: 16 accumulator values per thread)
constexpr int kTwPitch = kCW + 4;       // transpose buffer row pitch in floats (16-byte aligned rows)
constexpr int kMaxBn = 128;
constexpr int kBM = 128, kBK = 32;
constexpr int kABytes = kBM * kBK * 4;  // 16 KB
constexpr int kStageBytes = kABytes + kMaxBn * kBK * 4;  // 32 KB: A tile + the widest B tile
constexpr int kTbufFloats = kEpiWarps * 32 * kTwPitch;
// Completion counters: kSub sub-counters per GEMM, each alone in its 128-byte line (same-line atomics serialise in the L2
// slice at ~27 clk each, and every waiting producer polls these lines); tile t publishes on sub-counter t % kSub.
constexpr int kSub = 4, kCtrStride = 32;
constexpr int kDbgItems = 16, kDbgEvents = 10;  // debug timeline: items per CTA x events per item
// events: 0 producer picks the item up, 1 dependencies satisfied, 2 last TMA of the item issued, 3 MMA sees the first
// operands, 4 accumulator committed, 5 epilogue sees the accumulator, 6 split-K arrival counted, 7 tile published
constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256 + kTbufFloats * 4;
static_assert(kSmemBytes <= 227 * 1024, "chain kernel shared memory");

// ------------------------------------------------------------------------------------------------ device helpers
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned atom_add_acq_rel(unsigned* p, unsigned v) {
  unsigned old;
  asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void fence_tensormap_acquire(const CUtensorMap* m) {
  asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ unsigned ld_relaxed(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Bounded spin on the kSub sub-counters of GEMM `dep`: a scheduling bug must surface as a trap (launch error), never as a
// hung GPU.  The polls are relaxed loads with a short back-off -- an acquire load would invalidate this SM's L1 on every
// iteration under the feet of the epilogue warps, and 148 producers hammering one L2 line delay the very atomics they are
// waiting for -- and ONE acquire fence follows once all counts are reached.
__device__ __forceinline__ void wait_counter(const unsigned* done, int dep, int dep_tiles) {
  const unsigned* p = done + (size_t)dep * kSub * kCtrStride;
  unsigned target[kSub];
#pragma unroll
  for (int sub = 0; sub < kSub; ++sub) target[sub] = (unsigned)((dep_tiles - sub + kSub - 1) / kSub);
  long long t0 = 0;
  while (true) {
    unsigned v[kSub];
#pragma unroll
    for (int sub = 0; sub < kSub; ++sub) v[sub] = ld_relaxed(p + sub * kCtrStride);  // all four polls in flight together
    bool ok = true;
#pragma unroll
    for (int sub = 0; sub < kSub; ++sub) ok = ok && v[sub] >= target[sub];
    if (ok) return;
    __nanosleep(20);
    if (t0 == 0) t0 = clock64();
    if (clock64() - t0 > 4000000000LL) {
      printf("rlrep: chain dependency wait timed out (block %d, gemm %d, tiles %d, counters %u %u %u %u)\n", blockIdx.x, dep,
             dep_tiles, v[0], v[1], v[2], v[3]);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_acquire_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// Named barrier of the eight epilogue warps (256 threads); barrier 0 stays with __syncthreads.
__device__ __forceinline__ void epilogue_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// ELU for the TF32 path: x > 0 -> x, else expm1(x) as a degree-7 Taylor polynomial above -ln(2)/2 (relative error < 2e-8)
// and exp(x) - 1 through ex2.approx below (relative error < 4e-7 on a result in (-1, -0.29]).  15 instructions and no
// branch instead of expm1f's 28: the epilogue is issue-bound (one warp per scheduler), every instruction counts.
__device__ __forceinline__ float elu_fast(float x) {
  const float n = fminf(x, 0.f);
  float p = 1.f / 5040.f;
  p = fmaf(p, n, 1.f / 720.f);
  p = fmaf(p, n, 1.f / 120.f);
  p = fmaf(p, n, 1.f / 24.f);
  p = fmaf(p, n, 1.f / 6.f);
  p = fmaf(p, n, 0.5f);
  p = fmaf(p, n, 1.f);
  p *= n;
  const float e = __expf(n) - 1.f;
  const float r = n < -0.34657359f ? e : p;
  return x > 0.f ? x : r;
}

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// One element of the epilogue on the general (ragged / unaligned) path.  In-chain operands are read with ld.cg: the producer
// may be another SM of this same launch, so nothing about them may come from this SM's L1.
__device__ __forceinline__ float chain_epilogue_scalar(const Epilogue& e, float acc, int m, int n, const float* cptr) {
  float v = acc * e.scale;
  if (e.r1_u) v = fmaf(__ldcg(e.r1_u + m), __ldcg(e.r1_v + n), v);
  if (e.bias) v += __ldg(e.bias + n);
  if (e.pre_out) e.pre_out[(size_t)m * e.ld_pre + n] = v;
  v = apply_act(v, e.act);
  if (e.dact != DACT_NONE) v *= apply_dact(__ldcg(e.aux + (size_t)m * e.ld_aux + n), e.dact);
  if (e.accumulate) v += __ldcg(cptr);
  return v;
}

// Global operands of one 32 x 16 epilogue chunk, fetched BEFORE the accumulator is touched: inside the store loop every
// load would sit behind the previous row's store (the compiler must assume C aliases aux / bias).  Lane mapping as in
// chain_store_rows: piece = lane & 3 (16-byte column piece), rsub = lane >> 2 (row within a group of eight).
struct ChunkOperands {
  float4 bias, r1v;
  float4 aux[4];
  float r1u[4];
};
__device__ __forceinline__ void chunk_prefetch(ChunkOperands& o, const Epilogue& epi, int M, int m_base, int gn0, int lane) {
  const int piece = lane & 3, rsub = lane >> 2;
  const int on = gn0 + 4 * piece;
  o.bias = make_float4(0.f, 0.f, 0.f, 0.f);
  o.r1v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (epi.bias) o.bias = __ldg(reinterpret_cast<const float4*>(epi.bias + on));
  if (epi.r1_u) o.r1v = __ldcg(reinterpret_cast<const float4*>(epi.r1_v + on));
#pragma unroll
  for (int r4 = 0; r4 < 4; ++r4) {
    const int om = m_base + r4 * 8 + rsub;
    o.aux[r4] = make_float4(0.f, 0.f, 0.f, 0.f);
    o.r1u[r4] = 0.f;
    if (om < M) {
      if (epi.dact != DACT_NONE) o.aux[r4] = __ldcg(reinterpret_cast<const float4*>(epi.aux + (size_t)om * epi.ld_aux + on));
      if (epi.r1_u) o.r1u[r4] = __ldcg(epi.r1_u + om);
    }
  }
}

// 32 x 16 chunk out of the warp's transpose buffer: lanes cover eight rows x four 16-byte pieces per store instruction
// (eight 64-byte row segments).  ACT / DACT are compile-time (only the transcendental code of the layer at hand is in the
// loop); the rare extras (scale, pre-activation copy, accumulate) are warp-uniform run-time branches.
template <int ACT, int DACT>
__device__ __forceinline__ void chain_store_rows(const Epilogue& epi, const ChunkOperands& o, const float* tw,
                                                 float* __restrict__ C, int ldc, int M, int m_base, int gn0, int lane) {
  const int piece = lane & 3, rsub = lane >> 2;
  const int on = gn0 + 4 * piece;
#pragma unroll
  for (int r4 = 0; r4 < 4; ++r4) {
    const int r = r4 * 8 + rsub;
    const int om = m_base + r;
    if (om < M) {
      const float4 a4 = *reinterpret_cast<const float4*>(tw + r * kTwPitch + 4 * piece);
      float v[4] = {a4.x * epi.scale, a4.y * epi.scale, a4.z * epi.scale, a4.w * epi.scale};
      if (epi.r1_u) {
        const float u = o.r1u[r4];
        v[0] = fmaf(u, o.r1v.x, v[0]); v[1] = fmaf(u, o.r1v.y, v[1]); v[2] = fmaf(u, o.r1v.z, v[2]); v[3] = fmaf(u, o.r1v.w, v[3]);
      }
      v[0] += o.bias.x; v[1] += o.bias.y; v[2] += o.bias.z; v[3] += o.bias.w;
      if (epi.pre_out)
        *reinterpret_cast<float4*>(epi.pre_out + (size_t)om * epi.ld_pre + on) = make_float4(v[0], v[1], v[2], v[3]);
      if constexpr (ACT != ACT_NONE) {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = ACT == ACT_ELU ? elu_fast(v[e]) : apply_act(v[e], ACT < 0 ? epi.act : ACT);
      }
      if constexpr (DACT != DACT_NONE) {
        const int dact = DACT < 0 ? epi.dact : DACT;
        if (dact != DACT_NONE) {
          const float4 x = o.aux[r4];
          v[0] *= apply_dact(x.x, dact); v[1] *= apply_dact(x.y, dact); v[2] *= apply_dact(x.z, dact); v[3] *= apply_dact(x.w, dact);
        }
      }
      float4* cp = reinterpret_cast<float4*>(C + (size_t)om * ldc + on);
      if (epi.accumulate) {
        const float4 c0 = __ldcg(cp);
        v[0] += c0.x; v[1] += c0.y; v[2] += c0.z; v[3] += c0.w;
      }
      *cp = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ kernel
__global__ void __launch_bounds__(kThreads, 1)
gemm_chain_kernel(const ChainGemmDesc* __restrict__ gemms, const ChainTask* __restrict__ tasks,
                  const int* __restrict__ task_begin, unsigned* __restrict__ done, unsigned* __restrict__ exit_ctr,
                  int n_gemms, unsigned long long* __restrict__ dbg) {
  // Debug timeline (rlrep_gemm_chain_set_debug): %globaltimer stamps per (CTA, item, event); see kDbg* below.
  auto stamp = [&](int item, int ev) {
    if (dbg != nullptr && item < kDbgItems) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)::"memory");
      dbg[((size_t)blockIdx.x * kDbgItems + item) * kDbgEvents + ev] = t;
    }
  };
  // debug: kernel entry / exit of every CTA in the last item row (a CTA with kDbgItems items overwrites nothing: events 2, 3)
  if (threadIdx.x == 0) stamp(kDbgItems - 1, 2);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* acc_full = empty_bar + 8;   // [2] accumulator complete (MMA -> epilogue)
  uint64_t* acc_empty = acc_full + 2;   // [2] accumulator drained (epilogue -> MMA), one arrival per epilogue warp
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  volatile unsigned* arrival = reinterpret_cast<volatile unsigned*>(tmem_slot + 1);  // split-K arrival order, CTA-wide
  float* tbuf = reinterpret_cast<float*>(smem + kStages * kStageBytes + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t_begin = task_begin[blockIdx.x], t_end = task_begin[blockIdx.x + 1];

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&acc_full[a], 1);
      ptx::mbar_init(&acc_empty[a], kEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 2 * kMaxBn);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // Everything above reads build-time data only (task lists); the completion counters, operands and outputs belong to the
  // previous kernel until it has completed.
  ptx::pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int it = 0, last_gemm = -1;
      for (int t = t_begin; t < t_end; ++t) {
        const ChainTask tk = tasks[t];
        const ChainGemmDesc* g = gemms + tk.gemm;
        // Everything that does not depend on the dependencies' DATA happens before the wait: the item's descriptor fields
        // go to registers and the tensor maps are made visible to the TMA unit, so that once the counters are reached only
        // the fences stand between this thread and the first operand load.
        const int n_deps = g->n_deps;
        const int bn = g->bn, a_mn = g->a_mn, b_mn = g->b_mn;
        const int m0 = (tk.tile % g->tiles_m) * kBM, n0 = (tk.tile / g->tiles_m) * bn;
        const int kb0 = tk.split * g->kb_per_split, kb1 = min(g->nkb, kb0 + g->kb_per_split);
        int dep_id[kChainMaxDeps], dep_tiles[kChainMaxDeps];
#pragma unroll
        for (int d = 0; d < kChainMaxDeps; ++d) {
          dep_id[d] = d < n_deps ? g->dep[d] : 0;
          dep_tiles[d] = d < n_deps ? (int)g->dep_target[d] : 0;
        }
        if (tk.gemm != last_gemm) {
          fence_tensormap_acquire(&g->tmA);
          fence_tensormap_acquire(&g->tmB);
          last_gemm = tk.gemm;
        }
        stamp(t - t_begin, 0);
        if (dbg != nullptr && t - t_begin < kDbgItems)  // slot 8: which item this is
          dbg[((size_t)blockIdx.x * kDbgItems + (t - t_begin)) * kDbgEvents + 8] =
              (unsigned long long)tk.gemm | ((unsigned long long)tk.tile << 16) | ((unsigned long long)tk.split << 40);
#pragma unroll
        for (int d = 0; d < kChainMaxDeps; ++d)
          if (d < n_deps) wait_counter(done, dep_id[d], dep_tiles[d]);
        if (n_deps > 0) {
          fence_acquire_gpu();
          // the tiles were written through the generic proxy by other SMs; TMA reads through the async proxy
          fence_proxy_async_global();
        }
        stamp(t - t_begin, 1);
        const uint32_t tx = kABytes + bn * kBK * 4;
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % kStages;
          ptx::mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);  // fresh barrier: parity 1 passes immediately
          ptx::mbar_arrive_expect_tx(&full_bar[s], tx);
          uint8_t* a_dst = smem + s * kStageBytes;
          uint8_t* b_dst = a_dst + kABytes;
          const int k0 = kb * kBK;
          if (!a_mn) ptx::tma_load_2d(a_dst, &g->tmA, &full_bar[s], k0, m0);
          else ptx::tma_load_3d(a_dst, &g->tmA, &full_bar[s], 0, k0, m0 / 32);
          if (!b_mn) ptx::tma_load_2d(b_dst, &g->tmB, &full_bar[s], k0, n0);
          else ptx::tma_load_3d(b_dst, &g->tmB, &full_bar[s], 0, k0, n0 / 32);
        }
        stamp(t - t_begin, 2);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer: alternates between the two accumulators
    if (ptx::elect_one()) {
      int it = 0, tc = 0;
      for (int t = t_begin; t < t_end; ++t, ++tc) {
        const ChainTask tk = tasks[t];
        const ChainGemmDesc* g = gemms + tk.gemm;
        const int bn = g->bn, a_mn = g->a_mn, b_mn = g->b_mn;
        const int kb0 = tk.split * g->kb_per_split, kb1 = min(g->nkb, kb0 + g->kb_per_split);
        const uint32_t idesc = ptx::make_idesc_tf32(kBM, bn, a_mn != 0, b_mn != 0);
        const int acc = tc & 1;
        ptx::mbar_wait(&acc_empty[acc], ((tc >> 1) & 1) ^ 1);  // the epilogue has drained this accumulator
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * kMaxBn;
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % kStages;
          ptx::mbar_wait(&full_bar[s], (it / kStages) & 1);
          if (kb == kb0) stamp(t - t_begin, 3);
          ptx::tc_fence_after_sync();
          const uint32_t a_addr = ptx::smem_u32(smem + s * kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
          for (int k = 0; k < kBK / 8; ++k) {
            const uint64_t adesc = a_mn ? ptx::make_smem_desc(a_addr + k * 1024, 4096, 512, 1)
                                        : ptx::make_smem_desc(a_addr + k * 32, 16, 1024, 2);
            const uint64_t bdesc = b_mn ? ptx::make_smem_desc(b_addr + k * 1024, 4096, 512, 1)
                                        : ptx::make_smem_desc(b_addr + k * 32, 16, 1024, 2);
            ptx::mma_tf32_ss(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          ptx::mma_commit(&empty_bar[s]);
        }
        ptx::mma_commit(&acc_full[acc]);
        stamp(t - t_begin, 4);
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 2..9.  A warp may touch the TMEM lanes of
    // quarter warp % 4 only; the two warps of a quarter split the tile's 32-column chunks (even / odd): the epilogue is
    // issue-bound -- ~1300 dependent instructions per chunk on a warp that has its scheduler to itself -- so twice the
    // warps is twice the speed.
    const int q = warp & 3, half = (warp - 2) >> 2;
    float* tw = tbuf + (warp - 2) * (32 * kTwPitch);
    int tc = 0;
    for (int t = t_begin; t < t_end; ++t, ++tc) {
      const ChainTask tk = tasks[t];
      const ChainGemmDesc* g = gemms + tk.gemm;
      // everything this item needs from its descriptor, read ONCE into registers: a reference into global memory would be
      // re-read behind every store (the compiler must assume the stores alias it)
      const Epilogue epi = g->epi;
      const int bn = g->bn, M = g->M, N = g->N, ldc = g->ldc, split_k = g->split_k;
      float* __restrict__ C = g->C;
      float* __restrict__ ws = g->ws;
      unsigned* __restrict__ tile_ctr = g->tile_ctr;
      const int m0 = (tk.tile % g->tiles_m) * kBM, n0 = (tk.tile / g->tiles_m) * bn;
      const int chunks = bn / kCW;
      const int acc = tc & 1;
      const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + acc * kMaxBn;
      const int row = 32 * q + lane;  // row of the tile this thread holds
      ptx::mbar_wait(&acc_full[acc], (tc >> 1) & 1);
      if (threadIdx.x == 64) stamp(t - t_begin, 5);
      ptx::tc_fence_after_sync();

      bool final = true;
      const size_t part_floats = (size_t)kBM * bn;
      float* ws_tile = split_k > 1 ? ws + (size_t)tk.tile * split_k * part_floats : nullptr;
      // Distributed reduction: the split_k CTAs of a tile each finalise the chunks c with c % split_k == their split index,
      // so the reduction reads and the epilogue run split_k-wide instead of on the last arriver alone.  Each CTA writes the
      // chunks the OTHERS own, arrives, waits until all have arrived, then reduces its own chunks in the fixed order.
      const bool dist = split_k > 1 && g->dist != 0;
      int c_first = half, c_step = 2;
      if (split_k > 1) {
        // pass 1: this CTA's partial tile goes to the workspace, element (row, c*16 + 4*j + e) at
        // ((c*4 + j) * 128 + row) * 4 + e -- 512 contiguous bytes per store instruction
        float* part = ws_tile + (size_t)tk.split * part_floats;
#pragma unroll 1
        for (int c = half; c < chunks; c += 2) {
          if (dist && c % split_k == tk.split) continue;  // nobody else reads the chunks this CTA finalises itself
          uint32_t v[kCW];
          ptx::tmem_ld_32x32b_x16(t_acc + c * kCW, v);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < kCW / 4; ++j)
            __stcg(reinterpret_cast<float4*>(part + ((size_t)(c * (kCW / 4) + j) * kBM + row) * 4),
                   make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                               __uint_as_float(v[4 * j + 3])));
        }
        // ONE arrival per item: the eight warps meet, a single thread releases the CTA's partial tile and acquires the others'
        epilogue_bar();
        if (threadIdx.x == 64) {
          unsigned* ctr = tile_ctr + tk.tile;
          const unsigned old = atom_add_acq_rel(ctr, 1u);
          if (dist) {
            // wait for the other splits' partials (they run concurrently: same dependencies, same position in their CTAs'
            // lists); the counter goes on to count departures, so it never drops while someone is still waiting here
            if (old + 1 < (unsigned)split_k) {
              unsigned long long t0 = 0;
              unsigned spins = 0;
              while (ld_relaxed(ctr) < (unsigned)split_k) {
                __nanosleep(20);
                if ((++spins & 0xfff) == 0) {
                  unsigned long long now;
                  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                  if (t0 == 0) t0 = now;
                  else if (now - t0 > 2000000000ull) __trap();  // a planning bug must not hang the GPU
                }
              }
              fence_acquire_gpu();
            }
          } else if (old == (unsigned)(split_k - 1)) {
            *ctr = 0;  // every split has arrived: re-armed for the next launch
          }
          *arrival = old;
          stamp(t - t_begin, 6);
        }
        epilogue_bar();
        final = dist || *arrival == (unsigned)(split_k - 1);
        if (dist) {
          c_first = tk.split + split_k * half;
          c_step = 2 * split_k;
        }
      }
      if (final) {
        const bool use_aux = epi.dact != DACT_NONE;
        const bool vec_ok = (ldc & 3) == 0 && aligned16(C) && (N & 3) == 0 &&
                            (!use_aux || ((epi.ld_aux & 3) == 0 && aligned16(epi.aux))) &&
                            (!epi.pre_out || ((epi.ld_pre & 3) == 0 && aligned16(epi.pre_out))) &&
                            (!epi.bias || aligned16(epi.bias)) && (!epi.r1_v || aligned16(epi.r1_v));
#pragma unroll 1
        for (int c = c_first; c < chunks; c += c_step) {
          const int gn0 = n0 + c * kCW;
          const bool fast = vec_ok && gn0 + kCW <= N;
          ChunkOperands ops;
          if (fast) chunk_prefetch(ops, epi, M, m0 + 32 * q, gn0, lane);  // in flight while the accumulator is drained
          float a[kCW];
          if (split_k == 1) {
            uint32_t v[kCW];
            ptx::tmem_ld_32x32b_x16(t_acc + c * kCW, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < kCW; ++e) a[e] = __uint_as_float(v[e]);
          } else {
            // Fixed summation order p_0 + p_1 + ... over the splits whoever arrives last: this CTA's own partial is read
            // from TMEM at its position (bit-identical to what it wrote), the others from the workspace, the loads of the
            // next remote split in flight while the current one is added.
            const float* base = ws_tile + ((size_t)(c * (kCW / 4)) * kBM + row) * 4;
            float4 nxt[kCW / 4];
            const int s_first = tk.split == 0 ? 1 : 0;
#pragma unroll
            for (int j = 0; j < kCW / 4; ++j)
              nxt[j] = __ldcg(reinterpret_cast<const float4*>(base + (size_t)s_first * part_floats + (size_t)j * kBM * 4));
#pragma unroll 1
            for (int s = 0; s < split_k; ++s) {
              if (s == tk.split) {
                uint32_t v[kCW];
                ptx::tmem_ld_32x32b_x16(t_acc + c * kCW, v);
                ptx::tmem_ld_wait();
                if (s == 0) {
#pragma unroll
                  for (int e = 0; e < kCW; ++e) a[e] = __uint_as_float(v[e]);
                } else {
#pragma unroll
                  for (int e = 0; e < kCW; ++e) a[e] += __uint_as_float(v[e]);
                }
                continue;
              }
              float4 cur[kCW / 4];
#pragma unroll
              for (int j = 0; j < kCW / 4; ++j) cur[j] = nxt[j];
              int s2 = s + 1;
              if (s2 == tk.split) ++s2;
              if (s2 < split_k) {
#pragma unroll
                for (int j = 0; j < kCW / 4; ++j)
                  nxt[j] = __ldcg(reinterpret_cast<const float4*>(base + (size_t)s2 * part_floats + (size_t)j * kBM * 4));
              }
              if (s == 0) {
#pragma unroll
                for (int j = 0; j < kCW / 4; ++j) { a[4 * j] = cur[j].x; a[4 * j + 1] = cur[j].y; a[4 * j + 2] = cur[j].z; a[4 * j + 3] = cur[j].w; }
              } else {
#pragma unroll
                for (int j = 0; j < kCW / 4; ++j) { a[4 * j] += cur[j].x; a[4 * j + 1] += cur[j].y; a[4 * j + 2] += cur[j].z; a[4 * j + 3] += cur[j].w; }
              }
            }
          }
          // transpose through the warp's shared-memory buffer: thread = row on the way in, (row group, 16-byte piece) on the
          // way out; ragged / unaligned tiles read the same buffer element-wise
#pragma unroll
          for (int j = 0; j < kCW / 4; ++j)
            *reinterpret_cast<float4*>(tw + lane * kTwPitch + 4 * j) = make_float4(a[4 * j], a[4 * j + 1], a[4 * j + 2], a[4 * j + 3]);
          __syncwarp();
          if (fast) {
#define RLREP_CSTORE(A, D) chain_store_rows<A, D>(epi, ops, tw, C, ldc, M, m0 + 32 * q, gn0, lane)
            RLREP_EPILOGUE_SWITCH(epi, RLREP_CSTORE);
#undef RLREP_CSTORE
          } else if (gn0 < N) {
            const int piece = lane & 3, rsub = lane >> 2;
#pragma unroll 1
            for (int r4 = 0; r4 < 4; ++r4) {
              const int r = r4 * 8 + rsub, om = m0 + 32 * q + r;
              if (om >= M) continue;
#pragma unroll 1
              for (int e = 0; e < 4; ++e) {
                const int on = gn0 + 4 * piece + e;
                if (on < N) {
                  float* cp = C + (size_t)om * ldc + on;
                  *cp = chain_epilogue_scalar(epi, tw[r * kTwPitch + 4 * piece + e], om, on, cp);
                }
              }
            }
          }
          __syncwarp();
        }
        // the tile is final: ONE release per item publishes it
        if (threadIdx.x == 64) stamp(t - t_begin, 9);
        epilogue_bar();
        if (threadIdx.x == 64) {
          fence_proxy_async_global();
          // a distributed reduction publishes once per (tile, split): each CTA's columns are final on their own
          const int pub = dist ? tk.tile * split_k + tk.split : tk.tile;
          red_release_add(done + ((size_t)tk.gemm * kSub + (pub % kSub)) * kCtrStride, 1u);
          stamp(t - t_begin, 7);
          if (dist) {  // departure: the last CTA to have read the others' partials re-arms the counter
            unsigned* ctr = tile_ctr + tk.tile;
            if (atomicAdd(ctr, 1u) == (unsigned)(2 * split_k - 1)) *ctr = 0;
          }
        }
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[acc]);
    }
  }
  // This thread's role is done: the tail below (TMEM release, exit counter, counter re-arm) overlaps the next kernel's start.
  ptx::pdl_launch_dependents();
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 2 * kMaxBn);
  // The last CTA to get here re-arms the completion counters for the next launch (every wait of this launch is over).
  if (threadIdx.x == 0) {
    const unsigned old = atom_add_acq_rel(exit_ctr, 1u);
    if (old == gridDim.x - 1) {
      for (int i = 0; i < n_gemms * kSub; ++i) done[(size_t)i * kCtrStride] = 0;
      *exit_ctr = 0;
      __threadfence();
    }
    stamp(kDbgItems - 1, 3);
  }
}

// ------------------------------------------------------------------------------------------------ host planner
struct Range {
  uintptr_t lo = 0, hi = 0;
  bool overlaps(const Range& o) const { return lo < o.hi && o.lo < hi && lo != hi && o.lo != o.hi; }
};
Range range_of(const float* p, long long rows, long long ld, long long cols) {
  Range r;
  if (p == nullptr || rows <= 0 || cols <= 0) return r;
  r.lo = reinterpret_cast<uintptr_t>(p);
  r.hi = r.lo + (size_t)((rows - 1) * ld + cols) * sizeof(float);
  return r;
}
struct Footprint {
  std::vector<Range> reads, writes;
};
Footprint footprint(const GemmArgs& a) {
  Footprint f;
  f.reads.push_back(a.a_mn ? range_of(a.A, a.K, a.lda, a.M) : range_of(a.A, a.M, a.lda, a.K));
  f.reads.push_back(a.b_mn ? range_of(a.B, a.K, a.ldb, a.N) : range_of(a.B, a.N, a.ldb, a.K));
  f.reads.push_back(range_of(a.epi.bias, 1, 0, a.N));
  f.reads.push_back(range_of(a.epi.r1_u, 1, 0, a.M));
  f.reads.push_back(range_of(a.epi.r1_v, 1, 0, a.N));
  if (a.epi.dact != DACT_NONE) f.reads.push_back(range_of(a.epi.aux, a.M, a.epi.ld_aux, a.N));
  f.writes.push_back(range_of(a.C, a.M, a.ldc, a.N));
  if (a.epi.accumulate) f.reads.push_back(f.writes.back());
  f.writes.push_back(range_of(a.epi.pre_out, a.M, a.epi.ld_pre, a.N));
  return f;
}
bool conflicts(const Footprint& earlier, const Footprint& later) {
  for (const Range& w : earlier.writes) {
    for (const Range& r : later.reads)
      if (w.overlaps(r)) return true;  // read after write
    for (const Range& r : later.writes)
      if (w.overlaps(r)) return true;  // write after write
  }
  for (const Range& w : later.writes)
    for (const Range& r : earlier.reads)
      if (w.overlaps(r)) return true;  // write after read
  return false;
}

unsigned long long* g_chain_dbg = nullptr;

int env_int(const char* name, int dflt) {
  const char* e = std::getenv(name);
  return e ? std::atoi(e) : dflt;
}

// Estimated microseconds for one GEMM laid out as tiles x split items over `share` SMs.  Calibrated on the in-kernel
// timeline (tests/gpu_chain_probe.py): operands stream at ~150 KB/us into one SM until the chip-wide L2 -> SM rate
// (~12 TB/s) binds; every item pays ~1.5 us of dependency propagation, TMA latency and publish; an epilogue chunk pair
// (2 x 32 columns, one per epilogue warp group) ~1 us; split-K adds the partial's round trip through L2 and the last
// arriver's reads.
// A distributed reduction (dist) finalises bn / split columns per CTA after one wait for the other splits.
bool dist_possible(int bn, int split) { return split > 1 && (bn / kCW) % split == 0; }
double plan_cost(int tiles, int nkb, int bn, int split, int share, bool dist) {
  const int kb_per = ceil_div(nkb, split);
  const double kb_bytes = kABytes + bn * kBK * 4;
  const double waves = std::ceil((double)tiles * split / share);
  const double stream = waves * kb_per * kb_bytes / 150e3;
  const double chip = (double)tiles * split * kb_per * kb_bytes / 12e6;
  if (dist) {
    // partial tile out (bn / 64 * 0.25 us), one arrival + wait (~1 us when the splits run in the same wave), the other
    // splits' slices back in and the epilogue on bn / split columns
    return 1.5 + std::max(stream, chip) + waves * (0.25 * ceil_div(bn, 64) + 1.0 + 1.0 * ceil_div(bn / split, 64)) +
           0.1 * (split - 1);
  }
  double t = 1.5 + std::max(stream, chip) + waves * 1.0 * ceil_div(bn, 64);
  if (split > 1) t += 1.5 + 0.3 * (split - 1) * ceil_div(bn, 64);
  return t;
}

}  // namespace

void set_chain_debug_buffer(unsigned long long* dev) { g_chain_dbg = dev; }

bool chain_eligible(const GemmArgs& a) {
  return tc_eligible(a) && a.conv_w == 0 && a.M >= 32 && a.N >= 32 && a.K >= 8;
}

GemmChain::~GemmChain() {
  if (dev_) cudaFree(dev_);
}

bool GemmChain::matches(const std::vector<GemmArgs>& seq) const {
  if (seq.size() != seq_.size()) return false;
  for (size_t i = 0; i < seq.size(); ++i) {
    const GemmArgs &x = seq[i], &y = seq_[i];
    if (x.M != y.M || x.N != y.N || x.K != y.K || x.A != y.A || x.B != y.B || x.C != y.C || x.lda != y.lda ||
        x.ldb != y.ldb || x.ldc != y.ldc || x.a_mn != y.a_mn || x.b_mn != y.b_mn || x.epi.bias != y.epi.bias ||
        x.epi.r1_u != y.epi.r1_u || x.epi.r1_v != y.epi.r1_v || x.epi.aux != y.epi.aux || x.epi.pre_out != y.epi.pre_out ||
        x.epi.ld_aux != y.epi.ld_aux || x.epi.ld_pre != y.epi.ld_pre || x.epi.act != y.epi.act || x.epi.dact != y.epi.dact ||
        x.epi.accumulate != y.epi.accumulate || x.epi.scale != y.epi.scale)
      return false;
  }
  return true;
}

void GemmChain::build(const std::vector<GemmArgs>& seq, int force_bn, int force_split) {
  RLREP_CHECK(dev_ == nullptr, "chain already built");
  RLREP_CHECK(!seq.empty(), "empty chain");
  const int n = (int)seq.size();
  for (const GemmArgs& a : seq) RLREP_CHECK(chain_eligible(a), "GEMM cannot be a member of a chain");
  seq_ = seq;
  int n_sm = kNumSMs;
  {
    int dev = 0;
    RLREP_CUDA(cudaGetDevice(&dev));
    RLREP_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  static bool attr_set = false;
  if (!attr_set) {
    RLREP_CUDA(cudaFuncSetAttribute(gemm_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  int per_sm = 0;
  RLREP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gemm_chain_kernel, kThreads, kSmemBytes));
  RLREP_CHECK(per_sm >= 1, "chain kernel does not fit on an SM");
  const int n_cta = n_sm;  // one resident CTA per SM: the dependency spins rely on every CTA being scheduled

  // ---- dependency DAG from address ranges, transitively reduced, and levels (longest path)
  std::vector<Footprint> fp(n);
  for (int i = 0; i < n; ++i) fp[i] = footprint(seq[i]);
  std::vector<std::vector<int>> deps(n);
  std::vector<std::vector<char>> reach(n, std::vector<char>(n, 0));  // reach[j][i]: i is an ancestor of j
  std::vector<int> level(n, 0);
  for (int j = 0; j < n; ++j) {
    std::vector<int> direct;
    for (int i = 0; i < j; ++i)
      if (conflicts(fp[i], fp[j])) direct.push_back(i);
    for (int i : direct) {
      reach[j][i] = 1;
      for (int k = 0; k < n; ++k)
        if (reach[i][k]) reach[j][k] = 1;
    }
    for (int i : direct) {  // drop edges implied by another direct dependency
      bool implied = false;
      for (int k : direct)
        if (k != i && reach[k][i]) implied = true;
      if (!implied) deps[j].push_back(i);
      level[j] = std::max(level[j], level[i] + 1);
    }
    RLREP_CHECK((int)deps[j].size() <= kChainMaxDeps, "a chain GEMM has too many direct dependencies");
  }
  levels_ = 1 + *std::max_element(level.begin(), level.end());

  // ---- per level: SM share by work among the level's GEMMs, tile width / K-split per GEMM (K-split until it fills its share)
  std::vector<int> bn(n), split(n), share(n), first_cta(n), dist(n, 0);
  const int dist_mode = env_int("RLREP_CHAIN_DIST", 1);  // 0: last-arriver reductions only, 1: cost model, 2: wherever possible
  auto work_of = [&](int i) {
    return (double)ceil_div(seq[i].M, kBM) * ceil_div(seq[i].N, kMaxBn) * ceil_div(seq[i].K, kBK);
  };
  // items (= publishes on its completion counter) of chain member i
  auto items_of = [&](int i) { return ceil_div(seq[i].M, kBM) * ceil_div(seq[i].N, bn[i]) * (dist[i] ? split[i] : 1); };
  for (int L = 0; L < levels_; ++L) {
    std::vector<int> members;
    for (int i = 0; i < n; ++i)
      if (level[i] == L) members.push_back(i);
    double total = 0.0;
    for (int i : members) total += work_of(i);
    int cursor = 0, seen = 0;
    for (int i : members) {
      const GemmArgs& a = seq[i];
      const int nkb = ceil_div(a.K, kBK);
      ++seen;
      int sh = std::max(4, (int)std::floor(n_cta * work_of(i) / total));
      if (seen == (int)members.size()) sh = std::max(sh, n_cta - cursor);  // the last member takes what is left
      sh = std::min(sh, n_cta);
      first_cta[i] = cursor % n_cta;
      cursor += sh;
      share[i] = sh;
      double best = 1e300;
      for (int cbn : {32, 64, 128}) {
        if (force_bn && cbn != force_bn) continue;
        if (!force_bn && cbn > 32 && cbn / 2 >= a.N) continue;  // tile mostly out of bounds
        const int tiles = ceil_div(a.M, kBM) * ceil_div(a.N, cbn);
        for (int s : {1, 2, 4, 8, 16}) {
          if (force_split && s != force_split) continue;
          if (s > 1 && (s - 1) * ceil_div(nkb, s) >= nkb) continue;  // would leave an empty split
          for (int d = 0; d < 2; ++d) {
            if (d == 1 && (dist_mode == 0 || !dist_possible(cbn, s) || tiles * s > sh)) continue;  // the splits must share a wave
            if (d == 0 && dist_mode == 2 && dist_possible(cbn, s) && tiles * s <= sh) continue;
            const double c = plan_cost(tiles, nkb, cbn, s, sh, d == 1);
            if (c < best - 1e-9) {
              best = c;
              bn[i] = cbn;
              split[i] = s;
              dist[i] = d;
            }
          }
        }
      }
      if (best > 1e299) {  // forced values not realisable for this GEMM
        bn[i] = force_bn ? force_bn : 32;
        split[i] = 1;
        dist[i] = 0;
      }
    }
  }

  // ---- items -> per-CTA lists (level order), device image
  std::vector<std::vector<ChainTask>> per_cta(n_cta);
  std::vector<int> order(n);
  for (int i = 0; i < n; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return level[x] < level[y]; });
  size_t ws_floats = 0, ctr_count = 0;
  std::vector<size_t> ws_off(n, 0), ctr_off(n, 0);
  std::vector<ChainGemmDesc> descs(n);
  bytes_ = flops_ = 0.0;
  for (int i : order) {
    const GemmArgs& a = seq[i];
    const int tiles_m = ceil_div(a.M, kBM), tiles_n = ceil_div(a.N, bn[i]);
    const int tiles = tiles_m * tiles_n;
    int item = 0;
    for (int t = 0; t < tiles; ++t)
      for (int s = 0; s < split[i]; ++s, ++item)
        per_cta[(first_cta[i] + item % share[i]) % n_cta].push_back(ChainTask{i, t, s, 0});
    ChainGemmDesc& d = descs[i];
    std::memset(&d, 0, sizeof(d));
    d.tmA = make_operand_map(a.A, a.a_mn, a.M, a.K, a.lda, kBM);
    d.tmB = make_operand_map(a.B, a.b_mn, a.N, a.K, a.ldb, bn[i]);
    d.epi = a.epi;
    d.C = a.C;
    d.ldc = a.ldc; d.M = a.M; d.N = a.N; d.K = a.K;
    d.bn = bn[i]; d.a_mn = a.a_mn; d.b_mn = a.b_mn; d.nkb = ceil_div(a.K, kBK);
    d.split_k = split[i]; d.kb_per_split = ceil_div(d.nkb, split[i]);
    d.dist = dist[i];
    d.tiles_m = tiles_m; d.tiles_n = tiles_n;
    d.n_deps = (int)deps[i].size();
    for (int k = 0; k < d.n_deps; ++k) {
      const int j = deps[i][k];
      d.dep[k] = j;
      d.dep_target[k] = (unsigned)items_of(j);  // tiles of the dependency
    }
    ctr_off[i] = ctr_count;
    ctr_count += (size_t)tiles;
    if (split[i] > 1) {
      ws_off[i] = ws_floats;
      ws_floats += (size_t)tiles * split[i] * kBM * bn[i];
    }
    bytes_ += 4.0 * ((double)a.M * a.K + (double)a.N * a.K + (double)a.M * a.N);
    flops_ += 2.0 * a.M * a.N * a.K;
  }
  std::vector<ChainTask> tasks;
  std::vector<int> begin(n_cta + 1, 0);
  for (int c = 0; c < n_cta; ++c) {
    begin[c] = (int)tasks.size();
    tasks.insert(tasks.end(), per_cta[c].begin(), per_cta[c].end());
  }
  begin[n_cta] = (int)tasks.size();
  grid_ = n_cta;

  auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
  const size_t o_desc = 0;
  const size_t o_tasks = up(o_desc + sizeof(ChainGemmDesc) * n);
  const size_t o_begin = up(o_tasks + sizeof(ChainTask) * tasks.size());
  const size_t o_done = up(o_begin + sizeof(int) * begin.size());
  const size_t o_exit = up(o_done + sizeof(unsigned) * n * kSub * kCtrStride);
  const size_t o_ctr = up(o_exit + sizeof(unsigned));
  const size_t o_ws = up(o_ctr + sizeof(unsigned) * ctr_count);
  const size_t total_bytes = o_ws + sizeof(float) * ws_floats + 256;
  RLREP_CUDA(cudaMalloc(&dev_, total_bytes));
  RLREP_CUDA(cudaMemset(dev_, 0, o_ws));
  char* base = static_cast<char*>(dev_);
  d_gemms_ = reinterpret_cast<ChainGemmDesc*>(base + o_desc);
  d_tasks_ = reinterpret_cast<ChainTask*>(base + o_tasks);
  d_task_begin_ = reinterpret_cast<int*>(base + o_begin);
  d_done_ = reinterpret_cast<unsigned*>(base + o_done);
  d_exit_ = reinterpret_cast<unsigned*>(base + o_exit);
  for (int i = 0; i < n; ++i) {
    descs[i].tile_ctr = reinterpret_cast<unsigned*>(base + o_ctr) + ctr_off[i];
    descs[i].ws = split[i] > 1 ? reinterpret_cast<float*>(base + o_ws) + ws_off[i] : nullptr;
  }
  RLREP_CUDA(cudaMemcpy(d_gemms_, descs.data(), sizeof(ChainGemmDesc) * n, cudaMemcpyHostToDevice));
  RLREP_CUDA(cudaMemcpy(d_tasks_, tasks.data(), sizeof(ChainTask) * tasks.size(), cudaMemcpyHostToDevice));
  RLREP_CUDA(cudaMemcpy(d_task_begin_, begin.data(), sizeof(int) * begin.size(), cudaMemcpyHostToDevice));
  RLREP_CUDA(cudaDeviceSynchronize());
  if (env_int("RLREP_CHAIN_VERBOSE", 0)) {
    std::fprintf(stderr, "rlrep chain: %d GEMMs, %d levels, %zu items, ws %.1f MB\n", n, levels_, tasks.size(),
                 ws_floats * 4 / 1e6);
    for (int i = 0; i < n; ++i)
      std::fprintf(stderr, "  [%d] L%d M=%d N=%d K=%d a_mn=%d b_mn=%d bn=%d split=%d%s share=%d deps=%d\n", i, level[i],
                   seq[i].M, seq[i].N, seq[i].K, (int)seq[i].a_mn, (int)seq[i].b_mn, bn[i], split[i],
                   dist[i] ? " (distributed)" : "", share[i], (int)deps[i].size());
  }
}

void GemmChain::launch(cudaStream_t stream) {
  RLREP_CHECK(dev_ != nullptr, "chain not built");
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid_);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = stream;
  // cooperative: all CTAs are co-scheduled or none is, so two chains launched on different streams can never hold part of
  // the GPU each while spinning on tiles of CTAs that are not resident
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  attr[1] = pdl_attribute();
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  RLREP_CUDA(cudaLaunchKernelEx(&cfg, gemm_chain_kernel, (const ChainGemmDesc*)d_gemms_, (const ChainTask*)d_tasks_,
                                (const int*)d_task_begin_, d_done_, d_exit_, (int)seq_.size(), g_chain_dbg));
  RLREP_LAUNCHED_W("gemm_chain", stream, bytes_, flops_);
}

}  // namespace rlrep

// GEMM chain: a whole DAG of dependent tcgen05 GEMMs (the forward or backward pass of a few small MLPs) executed by ONE
// persistent kernel.
//
// Why: at batch 256 every linear layer of the update is a 0.1-1 GFLOP GEMM whose tensor time is under a microsecond; run as
// one kernel per layer each costs 6-20 us of launch, pipeline fill, split-K cluster reduction and drain, and ~60 of them are
// chained behind each other (DESIGN.md section 5).  Here one CTA per SM stays resident for the whole DAG: barriers, the TMEM
// allocation and the instruction cache are set up once, every CTA walks a STATIC list of (GEMM, tile, K-split) items that the
// host laid out level by level over the 148 SMs, and a dependent item starts the moment the tiles it reads are complete -- a
// per-GEMM completion counter in global memory (release by the epilogue warps, acquire by the TMA producer) replaces the
// kernel boundary.
//
//   warp 0      TMA producer: waits on the item's dependency counters, then streams its k-blocks through the operand ring
//   warp 1      MMA issuer: tcgen05.mma kind::tf32 into one of two TMEM accumulators (tile i+1 accumulates while tile i drains)
//   warps 2..5  epilogue: TMEM -> registers -> (split-K: partial tile to an L2-resident workspace; the LAST arriver of a
//               (tile, row-quarter) sums all partials in split order -- deterministic -- and goes on) -> transpose through
//               shared memory -> fused bias / activation / derivative epilogue -> 128-byte row stores -> release the counter
//
// Tile width (32 / 64 / 128) and K-split are per GEMM and run-time; operands may be K- or MN-major like the one-GEMM kernels
// (gemm_tc_kernel.cuh), so forward, data-gradient and weight-gradient GEMMs share a chain.
#pragma once
#include <vector>

#include "gemm.cuh"

namespace rlrep {

constexpr int kChainMaxDeps = 6;

struct alignas(128) ChainGemmDesc {
  CUtensorMap tmA;  // 128 bytes each; TMA reads them from global memory
  CUtensorMap tmB;
  Epilogue epi;
  int dist;            // split-K reduction distributed over the tile's split CTAs (each finalises bn / split_k columns)
  float* C;
  float* ws;           // split-K partial tiles [tile][split][bn / 4][128 rows][4]; nullptr when split_k == 1
  unsigned* tile_ctr;  // [tiles] split-K arrivals per tile; self-resetting
  int ldc, M, N, K;
  int bn, a_mn, b_mn, nkb;
  int split_k, kb_per_split, tiles_m, tiles_n;
  int n_deps;
  int dep[kChainMaxDeps];              // GEMMs of this chain whose output (or operands) this one must wait for
  unsigned dep_target[kChainMaxDeps];  // their tile counts (completion = every tile published)
};

struct ChainTask {
  int gemm, tile, split, pad;
};

class GemmChain {
 public:
  GemmChain() = default;
  GemmChain(const GemmChain&) = delete;
  GemmChain& operator=(const GemmChain&) = delete;
  ~GemmChain();
  // True when `seq` is the GEMM sequence this chain was built for (same shapes, pointers and epilogues).
  bool matches(const std::vector<GemmArgs>& seq) const;
  // Infers the dependency DAG from the operands' address ranges, picks tile width / K-split per GEMM, lays the items out
  // over the SMs level by level and uploads the program.  `force_bn` / `force_split` (0 = automatic) are test hooks.
  void build(const std::vector<GemmArgs>& seq, int force_bn = 0, int force_split = 0);
  void launch(cudaStream_t stream);
  int size() const { return (int)seq_.size(); }
  int levels() const { return levels_; }

 private:
  std::vector<GemmArgs> seq_;
  void* dev_ = nullptr;
  ChainGemmDesc* d_gemms_ = nullptr;
  ChainTask* d_tasks_ = nullptr;
  int* d_task_begin_ = nullptr;
  unsigned* d_done_ = nullptr;
  unsigned* d_exit_ = nullptr;
  int grid_ = 0, levels_ = 0;
  double bytes_ = 0.0, flops_ = 0.0;
};

// Debug aid: device buffer of grid x 16 items x 10 slots uint64 %globaltimer stamps (nullptr = off); see gemm_chain.cu.
void set_chain_debug_buffer(unsigned long long* dev);

// True when `a` can be a member of a chain (tensor-core eligible, no implicit-convolution addressing).
bool chain_eligible(const GemmArgs& a);

}  // namespace rlrep

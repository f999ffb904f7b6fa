// Host side of the tcgen05 TF32 GEMM (see gemm_tc_kernel.cuh for the kernel): tensor-map construction, the tile /
// split-K cost model and the dispatch to the per-variant launchers.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "gemm.cuh"
#include "gemm_tc_kernel.cuh"

namespace rlrep {

namespace tc {
void (*g_trace_reader)(unsigned long long*) = nullptr;
unsigned long long* g_persist_dbg = nullptr;
}

namespace {
using tc::BK;
using tc::BM;

// ------------------------------------------------------------------ host side
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  RLREP_CHECK(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  return fn;
}

// K-major operand: tensor map over a row-major fp32 matrix [rows, K] with leading dimension ld; box = box_rows x 32.
CUtensorMap make_map_kmajor(const float* base, int rows, int cols, int ld, int box_rows) {
  CUtensorMap m;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 2, const_cast<float*>(base), gdim, gstride, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RLREP_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return m;
}

// MN-major operand: the row-major matrix [K, mn] viewed as a 3-D tensor (mn % 32, k, mn / 32) so that ONE TMA
// instruction fetches all the 32-wide boxes of a tile: box = {32, 32, tile_mn / 32}.  Elements with mn >= the real
// extent alias the next k-row (never out of the allocation as long as K*ld floats are readable plus the arena's
// padding); they only feed output rows / columns that are never stored.
CUtensorMap make_map_mnmajor(const float* base, int K, int mn, int ld, int tile_mn) {
  CUtensorMap m;
  cuuint64_t gdim[3] = {32u, (cuuint64_t)K, (cuuint64_t)((mn + 31) / 32)};
  cuuint64_t gstride[2] = {(cuuint64_t)ld * 4, 128u};
  cuuint32_t box[3] = {32u, 32u, (cuuint32_t)(tile_mn / 32)};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 3, const_cast<float*>(base), gdim, gstride, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RLREP_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (3-D) failed with CUresult " + std::to_string((int)r));
  return m;
}

// Implicit conv weight gradient (GemmArgs::conv_wgrad_hi): the convolution's input X [rows, 32] on a grid Hi wide as the
// 4-D tensor (c, k, q, ky) -> X[4 k + q + ky * Hi, c], q = 0..7 (6 and 7 are padding: a ky row of the view is 256 columns, so
// that 128- and 256-wide tiles never straddle two ky rows); box {32, 32, tile_n / 32, 1} lands exactly like the 3-D
// MN-major box.  The largest shift (q = 7, ky = 2) reads 2 Hi + 7 rows past the map: the caller keeps that many readable rows of
// finite values behind it (they meet zeros of the folded gradient).
CUtensorMap make_map_conv_wgrad(const float* base, long long rows, int hi, int tile_n) {
  CUtensorMap m;
  cuuint64_t gdim[4] = {32u, (cuuint64_t)(rows / 4), 8u, 3u};
  cuuint64_t gstride[3] = {512u, 128u, (cuuint64_t)hi * 128u};
  cuuint32_t box[4] = {32u, 32u, (cuuint32_t)(tile_n / 32), 1u};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 4, const_cast<float*>(base), gdim, gstride, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RLREP_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (4-D) failed with CUresult " + std::to_string((int)r));
  return m;
}

int max_clusters(int bn, bool a_mn, bool b_mn, int s, int stages, bool push) {
  static std::mutex mu;
  static std::unordered_map<int, int> cache;
  const int key = (bn << 13) | (push << 12) | (a_mn << 11) | (b_mn << 10) | (s << 5) | stages;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  int n = 0;
  switch (bn) {
    case 32: n = a_mn ? tc::max_clusters_32_1(b_mn, s, stages, push) : tc::max_clusters_32_0(b_mn, s, stages, push); break;
    case 64: n = a_mn ? tc::max_clusters_64_1(b_mn, s, stages, push) : tc::max_clusters_64_0(b_mn, s, stages, push); break;
    case 128: n = a_mn ? tc::max_clusters_128_1(b_mn, s, stages, push) : tc::max_clusters_128_0(b_mn, s, stages, push); break;
    default: n = a_mn ? tc::max_clusters_256_1(b_mn, s, stages, push) : tc::max_clusters_256_0(b_mn, s, stages, push); break;
  }
  cache[key] = n;
  return n;
}

// Ring depth.  A short K-slice is one burst of loads: a ring that fits twice into an SM (2 x ~113 KB) lets two CTAs
// -- of this GEMM or of one running concurrently on another stream -- share the SM; long slices get the deepest ring.
bool use_push(int bn, int s) { return s > 1 && tc::push_possible(bn); }

int pick_stages(int bn, int kb_per, bool push) {
  if (push) return std::max(2, std::min(kb_per, tc::max_stages_push(bn)));
  const int deepest = tc::num_stages(bn), fewest = tc::min_stages(bn);
  const int shallow = (113 * 1024 - 1280) / tc::stage_bytes(bn);
  if (shallow < fewest || kb_per > 2 * shallow) return deepest;
  return std::max(fewest, std::min(shallow, kb_per));
}

// Cost model (cycles through one SM) used to pick the tile width and the split-K cluster size: operand bytes from
// L2 at ~48 B/clk, the cluster reduction over DSMEM at ~16 B/clk, stores at ~32 B/clk and a fixed per-CTA cost that
// grows with the cluster size, times the number of waves.  The wave count uses the occupancy API's answer for how
// many clusters of this shape the GPU holds at once (8-CTA clusters must fit in a GPC: far fewer than 148 / 8), scaled
// by the share of the GPU the caller expects to have.
double plan_cost(const GemmArgs& a, int nkb, int bn, int s, double sm_share, int* kb_per_out, int* stages_out,
                 int groups = 1) {
  const int kb_per = ceil_div(nkb, s);
  const bool push = use_push(bn, s);
  const int stages = pick_stages(bn, kb_per, push);
  *kb_per_out = kb_per;
  *stages_out = stages;
  const int clusters = ceil_div(a.M, BM) * ceil_div(a.N, bn) * groups;
  const double cap = std::max(1.0, max_clusters(bn, a.a_mn, a.b_mn, s, stages, push) * sm_share);
  const double waves = std::ceil(clusters / cap);
  const double load = (double)(BM + bn) * BK * 4 * kb_per / 48.0;
  const double tile = (double)BM * bn * 4;
  // pull: every CTA reads its rows from all peers over DSMEM (dependent loads, ~16 B/clk); push: posted remote
  // stores overlapped with the TMEM drain (~2x cheaper end to end, measured)
  const double reduce = s > 1 ? tile / (push ? 32.0 : 16.0) : 0.0;
  const double store = tile / s / 32.0;
  const double fixed = 1500.0 + (s == 2 ? 300.0 : s == 4 ? 600.0 : s == 8 ? 900.0 : 0.0);
  return waves * (load + reduce + store + fixed);
}

}  // namespace

void set_gemm_debug_buffer(unsigned long long* dev80) { tc::g_persist_dbg = dev80; }

CUtensorMap make_operand_map(const float* base, bool mn_major, int mn, int K, int ld, int box_mn) {
  return mn_major ? make_map_mnmajor(base, K, mn, ld, box_mn) : make_map_kmajor(base, mn, K, ld, box_mn);
}

void read_gemm_trace(unsigned long long* out16) {
  RLREP_CHECK(tc::g_trace_reader != nullptr, "no tcgen05 GEMM has been launched yet");
  tc::g_trace_reader(out16);
}

bool tc_eligible(const GemmArgs& a) {
  auto ok = [](const float* p, int ld) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (ld & 3) == 0 && ld > 0; };
  // MN-major operands are fetched through a (mn % 32, k, mn / 32) view: keep mn a multiple of 32 so the view never
  // reaches past the last row of the matrix.
  if (a.a_mn && (a.M & 31) != 0) return false;
  if (a.b_mn && (a.N & 31) != 0) return false;
  if (a.conv_w > 0 && (a.a_mn || a.K != 9 * 32)) return false;
  if (a.conv_wgrad_hi > 0 && (!a.a_mn || !a.b_mn || a.N != 768 || a.conv_w > 0 || a.ldb != 128)) return false;
  return a.A2 == nullptr && ok(a.A, a.lda) && ok(a.B, a.ldb) && a.M > 0 && a.N > 0 && a.K > 0;
}

TcGemmPlan make_tc_plan(const GemmArgs& a, int bn, int split_k, float* /*ws*/, size_t /*ws_floats*/, double sm_share) {
  RLREP_CHECK(tc_eligible(a), "operands violate TMA alignment (16-byte base, ld % 4 == 0)");
  RLREP_CHECK(bn == 0 || bn == 32 || bn == 64 || bn == 128 || bn == 256, "bn must be 32/64/128/256");
  RLREP_CHECK(split_k == 0 || split_k == 1 || split_k == 2 || split_k == 4 || split_k == 8,
              "split_k is the cluster size along K: 1, 2, 4 or 8");
  TcGemmPlan p;
  p.args = a;
  const int nkb_all = ceil_div(a.K, BK);
  // K groups (GemmArgs::k_groups): each group is planned like a GEMM over its share of K
  const int groups = (a.k_groups > 1 && nkb_all >= 64 * a.k_groups) ? a.k_groups : 1;
  RLREP_CHECK(a.k_groups == 1 || (a.conv_w == 0 && !a.epi.accumulate), "K groups: plain GEMMs only");
  p.k_groups = groups;
  const int nkb = ceil_div(nkb_all, groups);
  double best = 1e300;
  for (int cand_bn : {32, 64, 128, 256}) {
    if (bn != 0 && cand_bn != bn) continue;
    if (bn == 0 && cand_bn > 32 && cand_bn / 2 >= a.N) continue;  // tile mostly out of bounds
    for (int s : {1, 2, 4, 8}) {
      if (split_k != 0 && s != split_k) continue;
      int kb_per = 0, stages = 0;
      if (s > 1 && (s - 1) * ceil_div(nkb, s) >= nkb) continue;  // would leave an empty split
      if (groups > 1 && (s * groups - 1) * ceil_div(nkb, s) >= nkb_all) continue;
      const double c = plan_cost(a, nkb, cand_bn, s, sm_share, &kb_per, &stages, groups);
      if (c < best) {
        best = c;
        p.bn = cand_bn;
        p.split_k = s;
        p.kb_per_split = kb_per;
        p.stages = stages;
        p.push = use_push(cand_bn, s);
      }
    }
  }
  if (p.bn == 0) {  // requested split not realisable (K too short): fall back to no split
    p.bn = bn ? bn : 32;
    p.split_k = 1;
    p.k_groups = 1;
    p.kb_per_split = nkb_all;
    p.stages = pick_stages(p.bn, nkb, false);
    p.push = false;
  }
  {
    // Persistent variant (one CTA per SM walks the tiles, double-buffered TMEM accumulator): used for the conv-shaped
    // GEMMs -- thousands of narrow tiles with a handful of k-blocks each -- where one tile per CTA pays the whole
    // setup -> TMA -> MMA -> epilogue latency for almost no work (measured at M = 430k: K=288, N=32 150 -> 87 us, now
    // L2-bandwidth bound; K=32, N=288 570 -> 309 us).  Wide tiles keep the one-tile-per-CTA kernel: two or three
    // co-resident CTAs overlap each other there, and the persistent epilogue (1.3 us per 128 x 32 chunk) would dominate
    // -- except for one- or two-k-block GEMMs (the stride-2 transposed conv's K = 32), where any tile width wins.
    const int tiles = ceil_div(a.M, BM) * ceil_div(a.N, p.bn);
    p.persistent = p.split_k == 1 && tiles >= 4 * kNumSMs && ((p.bn <= 64 && nkb <= 16) || nkb <= 2);
  }
  // K-major operand: matrix [rows = M|N, cols = K]; MN-major: matrix [rows = K, cols = M|N].
  // implicit convolution: A is the [M, 32] pixel matrix itself (rows past M zero-fill), not an [M, 288] column matrix
  {
    // implicit convolution, many tiles, 32 output channels: the halo kernel (one A load per tile instead of nine)
    const int rows = (128 + 2 * a.conv_w + 2 + 7) & ~7;
    // its epilogue is bias + activation + derivative mask (16-byte aligned, dense 32-column operands)
    const bool plain = a.epi.r1_u == nullptr && a.epi.pre_out == nullptr && !a.epi.accumulate &&
                       (a.epi.bias == nullptr || (reinterpret_cast<uintptr_t>(a.epi.bias) & 15) == 0) &&
                       (a.epi.dact == DACT_NONE || ((reinterpret_cast<uintptr_t>(a.epi.aux) & 15) == 0 && (a.epi.ld_aux & 3) == 0));
    if (plain && a.conv_w > 0 && p.persistent && p.bn == 32 && a.N <= 32 && rows <= 256) p.halo_rows = rows;
  }
  // (a compacting GEMM whose plan has no halo is refused by GemmRunner::run_compact before anything is launched)
  p.tmA = a.a_mn ? make_map_mnmajor(a.A, a.K, a.M, a.lda, BM)
                 : make_map_kmajor(a.A, a.M, a.conv_w > 0 ? 32 : a.K, a.lda, p.halo_rows > 0 ? p.halo_rows : BM);
  {
    static const bool verbose = [] {
      const char* e = std::getenv("RLREP_TC_VERBOSE");
      return e != nullptr && std::atoi(e) != 0;
    }();
    if (verbose)
      std::fprintf(stderr, "rlrep tc plan: M=%d N=%d K=%d a_mn=%d b_mn=%d conv_w=%d wgrad=%d -> bn=%d split=%d groups=%d stages=%d%s%s%s\n",
                   a.M, a.N, a.K, (int)a.a_mn, (int)a.b_mn, a.conv_w, a.conv_wgrad_hi, p.bn, p.split_k, p.k_groups, p.stages,
                   p.push ? " push" : "", p.persistent ? " persistent" : "", p.halo_rows > 0 ? " halo" : "");
  }
  if (a.conv_wgrad_hi > 0) {
    RLREP_CHECK(!p.persistent, "implicit weight gradient: one tile per CTA");
    p.tmB = make_map_conv_wgrad(a.B, 4LL * a.K, a.conv_wgrad_hi, p.bn);
  } else {
    p.tmB = a.b_mn ? make_map_mnmajor(a.B, a.K, a.N, a.ldb, p.bn) : make_map_kmajor(a.B, a.N, a.K, a.ldb, p.bn);
  }
  return p;
}

void launch_tc(const TcGemmPlan& p, cudaStream_t stream) {
  const bool a = p.args.a_mn;
  switch (p.bn) {
    case 32: a ? tc::launch_tc_32_1(p, stream) : tc::launch_tc_32_0(p, stream); break;
    case 64: a ? tc::launch_tc_64_1(p, stream) : tc::launch_tc_64_0(p, stream); break;
    case 128: a ? tc::launch_tc_128_1(p, stream) : tc::launch_tc_128_0(p, stream); break;
    case 256: a ? tc::launch_tc_256_1(p, stream) : tc::launch_tc_256_0(p, stream); break;
    default: throw Error("bad bn");
  }
}

}  // namespace rlrep

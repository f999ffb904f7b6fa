// Host runtime: replay ring, GEMM dispatch with cached TMA plans, linear-layer pass helpers, graph replay.
#include <algorithm>
#include <atomic>

#include "agent.cuh"

namespace rlrep {

namespace {
thread_local long long g_launches = 0;
thread_local bool g_profiling = false;
thread_local std::vector<cudaEvent_t> g_events;       // g_events[0] = start, then one per launch
thread_local std::vector<const char*> g_names;
thread_local std::vector<double> g_bytes, g_flops;
}  // namespace

long long launch_count() { return g_launches; }

void note_launch(const char* name, cudaStream_t stream, double bytes, double flops) {
  if (std::strncmp(name, "nccl_", 5) != 0) ++g_launches;  // NCCL's kernels are recorded in profiles but are not ours
  if (g_profiling) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) == cudaSuccess) {
      cudaEventRecord(e, stream);
      g_events.push_back(e);
      g_names.push_back(name);
      g_bytes.push_back(bytes);
      g_flops.push_back(flops);
    }
  }
}

void profile_begin(cudaStream_t stream) {
  for (cudaEvent_t e : g_events) cudaEventDestroy(e);
  g_events.clear();
  g_names.clear();
  g_bytes.clear();
  g_flops.clear();
  cudaEvent_t e;
  RLREP_CUDA(cudaEventCreate(&e));
  RLREP_CUDA(cudaEventRecord(e, stream));
  g_events.push_back(e);
  g_profiling = true;
}

std::vector<ProfileEntry> profile_end(cudaStream_t stream) {
  g_profiling = false;
  RLREP_CUDA(cudaStreamSynchronize(stream));
  std::vector<ProfileEntry> out;
  for (size_t i = 0; i + 1 < g_events.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, g_events[i], g_events[i + 1]);
    out.push_back({g_names[i], ms, g_bytes[i], g_flops[i]});
  }
  for (cudaEvent_t e : g_events) cudaEventDestroy(e);
  g_events.clear();
  g_names.clear();
  return out;
}

// ================================================================================================ Ring
namespace {
constexpr size_t kStageRows = 8192;
}  // namespace

namespace {
std::atomic<unsigned long long> g_ring_generation{0};
}  // namespace

Ring::Ring(int state_dim, int action_dim, long long cap)
    : S(state_dim), A(action_dim), capacity(cap), generation(++g_ring_generation) {
  RLREP_CHECK(S > 0 && A > 0 && cap > 0, "bad ring dimensions");
  const RecordLayout l = RecordLayout::of(S, A);
  off_a = l.off_a;
  off_r = l.off_r;
  off_d = l.off_d;
  off_s2 = l.off_s2;
  R = l.R;
  RLREP_CUDA(cudaMalloc(&data, (size_t)capacity * R * sizeof(float)));
  RLREP_CUDA(cudaMemset(data, 0, (size_t)capacity * R * sizeof(float)));
  RLREP_CUDA(cudaDeviceSynchronize());  // see DeviceArena::commit: the null-stream memset must not race later stream work
  stage_rows_ = kStageRows;
  RLREP_CUDA(cudaMallocHost(&stage_host_, stage_rows_ * R * sizeof(float)));
  RLREP_CUDA(cudaMalloc(&stage_dev_, stage_rows_ * R * sizeof(float)));
  idx_cap_ = 1 << 16;
  RLREP_CUDA(cudaMallocHost(&idx_host_, idx_cap_ * sizeof(long long)));
  RLREP_CUDA(cudaMalloc(&idx_dev_, idx_cap_ * sizeof(long long)));
}

Ring::~Ring() {
  cudaFree(data);
  cudaFreeHost(stage_host_);
  cudaFree(stage_dev_);
  cudaFreeHost(idx_host_);
  cudaFree(idx_dev_);
}

void Ring::add_packed(const float* rows_host, int n, cudaStream_t s) {
  int done = 0;
  while (done < n) {
    // One launch writes slot (ptr + b) % capacity for every staged row b: a chunk longer than the ring would map several
    // rows to one slot inside ONE launch (a race; the reference keeps the newest row, utils/buffer.py:28-36), so chunks
    // never exceed the capacity and consecutive chunks are stream-ordered.
    const int chunk = (int)std::min<size_t>(std::min<size_t>(stage_rows_, (size_t)capacity), (size_t)(n - done));
    RLREP_CUDA(cudaStreamSynchronize(s));  // staging buffers are reused
    std::memcpy(stage_host_, rows_host + (size_t)done * R, (size_t)chunk * R * sizeof(float));
    RLREP_CUDA(cudaMemcpyAsync(stage_dev_, stage_host_, (size_t)chunk * R * sizeof(float), cudaMemcpyHostToDevice, s));
    launch_ring_write(data, R / 4, capacity, ptr, stage_dev_, chunk, s);
    ptr = (ptr + chunk) % capacity;
    size = std::min(size + chunk, capacity);
    done += chunk;
  }
  RLREP_CUDA(cudaStreamSynchronize(s));
}

void Ring::load_columns(const void* state, const void* action, const void* next_state, const void* reward,
                        const void* done, long long n, int is_f64, cudaStream_t s) {
  RLREP_CHECK(n <= capacity, "more rows than ring capacity");
  auto get = [is_f64](const void* base, long long i) -> float {
    return is_f64 ? (float)static_cast<const double*>(base)[i] : static_cast<const float*>(base)[i];
  };
  ptr = 0;
  size = 0;
  long long row = 0;
  while (row < n) {
    const int chunk = (int)std::min<long long>((long long)stage_rows_, n - row);
    RLREP_CUDA(cudaStreamSynchronize(s));
    std::memset(stage_host_, 0, (size_t)chunk * R * sizeof(float));
    for (int i = 0; i < chunk; ++i) {
      float* rec = stage_host_ + (size_t)i * R;
      const long long r = row + i;
      for (int j = 0; j < S; ++j) rec[j] = get(state, r * S + j);
      for (int j = 0; j < A; ++j) rec[off_a + j] = get(action, r * A + j);
      rec[off_r] = get(reward, r);
      rec[off_d] = get(done, r);
      for (int j = 0; j < S; ++j) rec[off_s2 + j] = get(next_state, r * S + j);
    }
    RLREP_CUDA(cudaMemcpyAsync(stage_dev_, stage_host_, (size_t)chunk * R * sizeof(float), cudaMemcpyHostToDevice, s));
    launch_ring_write(data, R / 4, capacity, ptr, stage_dev_, chunk, s);
    ptr = (ptr + chunk) % capacity;
    size = std::min(size + chunk, capacity);
    row += chunk;
  }
  RLREP_CUDA(cudaStreamSynchronize(s));
}

void Ring::gather_from_host_idx(const long long* idx_host, int B, float* out_dev, cudaStream_t s) {
  RLREP_CHECK(B > 0 && B <= idx_cap_, "batch too large for the ring's index staging");
  for (int i = 0; i < B; ++i) RLREP_CHECK(idx_host[i] >= 0 && idx_host[i] < size, "replay index out of range");
  RLREP_CUDA(cudaStreamSynchronize(s));
  std::memcpy(idx_host_, idx_host, (size_t)B * sizeof(long long));
  RLREP_CUDA(cudaMemcpyAsync(idx_dev_, idx_host_, (size_t)B * sizeof(long long), cudaMemcpyHostToDevice, s));
  launch_gather(data, R / 4, idx_dev_, B, out_dev, s);
}

// ================================================================================================ GemmRunner
void GemmRunner::init(Precision prec, size_t ws_floats) {
  prec_ = prec;
  ws_floats_ = ws_floats;
  if (ws_floats_) RLREP_CUDA(cudaMalloc(&ws_, ws_floats_ * sizeof(float)));
}
GemmRunner::~GemmRunner() {
  if (ws_) cudaFree(ws_);
  if (kg_ws_) cudaFree(kg_ws_);
}

void GemmRunner::begin_chain(cudaStream_t s) {
  RLREP_CHECK(!recording_, "begin_chain inside a chain");
  if (!chains_enabled()) return;
  recording_ = true;
  chain_stream_ = s;
  pending_.clear();
}

void GemmRunner::flush_chain() {
  if (pending_.empty()) return;
  if (pending_.size() == 1) {  // nothing to chain: the one-GEMM kernels do this better
    const GemmArgs a = pending_[0];
    pending_.clear();
    const bool rec = recording_;
    recording_ = false;
    run(a, chain_stream_);
    recording_ = rec;
    return;
  }
  GemmChain* chain = nullptr;
  for (auto& c : chains_)
    if (c->matches(pending_)) chain = c.get();
  if (chain == nullptr) {
    chains_.emplace_back(new GemmChain());
    chain = chains_.back().get();
    chain->build(pending_);
  }
  chain->launch(chain_stream_);
  pending_.clear();
}

void GemmRunner::end_chain() {
  if (!recording_) return;
  flush_chain();
  recording_ = false;
}

bool GemmRunner::compact_supported(GemmArgs a, int wp, int ho) {
  if (recording_ || prec_ != PREC_TF32 || !tc_eligible(a) || a.conv_w <= 0 || a.M < 32 || a.N != 32 || wp <= 8 ||
      a.M >= (1 << 24))
    return false;
  a.compact_wp = wp;
  a.compact_ho = ho;
  const TcGemmPlan probe = make_tc_plan(a, 0, 0, ws_, ws_floats_, sm_share_);  // cheap: cost model + two tensor maps
  return probe.halo_rows > 0;
}
bool GemmRunner::run_compact(GemmArgs a, int wp, int ho, cudaStream_t s) {
  if (!compact_supported(a, wp, ho)) return false;
  a.compact_wp = wp;
  a.compact_ho = ho;
  run(a, s);
  return true;
}

void GemmRunner::run(const GemmArgs& a, cudaStream_t s) {
  RLREP_CHECK(a.mb.n == 1 || !recording_, "population GEMMs do not join GEMM chains");
  if (recording_) {
    if (chain_eligible(a)) {
      pending_.push_back(a);
      return;
    }
    flush_chain();  // program order on the chain's stream
    s = chain_stream_;
  }
  // Short-K layers (K = 17 / 23 inputs) also go to the tensor cores: the tensor maps carry the LOGICAL K, so TMA
  // zero-fills the rest of the 32-wide k-block whatever sits behind the operands in memory.
  const bool tc = prec_ == PREC_TF32 && tc_eligible(a) && a.M >= 32 && a.N >= 32 && a.K >= 8;
  RLREP_CHECK(a.compact_wp == 0 || tc, "compacting stores exist on the tensor-core halo kernel only");
  if (!tc) {
    launch_simt(a, s);
    return;
  }
  // Deep and skinny (the pixel agents' 39,200-wide linears at batch 256: K = 39,200 and 2 x 1..4 tiles): a split-K cluster
  // holds 8 CTAs, so such a GEMM runs on 16-64 CTAs that stream ~5 MB each.  Cut K into groups (GemmArgs::k_groups: own
  // cluster and raw partial output each), then one elementwise pass adds the groups and applies the epilogue.
  if (a.k_groups == 1 && a.conv_w == 0 && a.conv_wgrad_hi == 0 && !recording_ && a.mb.n == 1) {
    const int tiles = ceil_div(a.M, 128) * ceil_div(a.N, 128), nkb = ceil_div(a.K, 32);
    int groups = 1;
    constexpr int kCtaCap = 296;  // up to two waves of CTAs (measured on the muLV update: 148 -> 5.82 ms, 296 -> 5.77 ms)
    while (groups < 8 && tiles * 8 * groups * 2 <= kCtaCap && nkb >= 256 * groups * 2) groups *= 2;
    if (groups > 1 && nkb >= 1024) {
      const int ldw = (a.N + 3) & ~3, m_pad = ceil_div(a.M, 128) * 128;
      const size_t need = (size_t)groups * m_pad * ldw;
      if (need > kg_ws_floats_) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        RLREP_CUDA(cudaStreamIsCapturing(s, &cap));
        RLREP_CHECK(cap == cudaStreamCaptureStatusNone, "K-group workspace must be sized before a graph capture");
        if (kg_ws_) RLREP_CUDA(cudaFree(kg_ws_));
        RLREP_CUDA(cudaMalloc(&kg_ws_, need * sizeof(float)));
        kg_ws_floats_ = need;
        plans_.clear();  // plans hold the old workspace address as their C
      }
      GemmArgs g = a;
      g.C = kg_ws_; g.ldc = ldw;
      g.epi = Epilogue();
      g.k_groups = groups;
      run(g, s);
      launch_kgroup_finish(kg_ws_, groups, a.M, a.N, ldw, (size_t)m_pad * ldw, a.C, a.ldc, a.epi, s);
      return;
    }
  }
  std::string key(sizeof(GemmArgs), '\0');
  {
    // field-wise copy into a zeroed buffer so padding bytes never differ
    GemmArgs* k = reinterpret_cast<GemmArgs*>(&key[0]);
    k->M = a.M; k->N = a.N; k->K = a.K;
    k->A = a.A; k->lda = a.lda; k->a_mn = a.a_mn;
    k->B = a.B; k->ldb = a.ldb; k->b_mn = a.b_mn;
    k->C = a.C; k->ldc = a.ldc; k->conv_w = a.conv_w; k->conv_wgrad_hi = a.conv_wgrad_hi;
    k->compact_wp = a.compact_wp; k->compact_ho = a.compact_ho; k->k_groups = a.k_groups;
    k->compact_hx = a.compact_hx; k->compact_stride = a.compact_stride; k->compact_oy = a.compact_oy;
    k->compact_ox = a.compact_ox; k->compact_out_w = a.compact_out_w; k->conv_ntaps = a.conv_ntaps;
    for (int t = 0; t < 9; ++t) { k->conv_tap_shift[t] = a.conv_tap_shift[t]; k->conv_tap_kb[t] = a.conv_tap_kb[t]; }
    k->epi.bias = a.epi.bias; k->epi.r1_u = a.epi.r1_u; k->epi.r1_v = a.epi.r1_v; k->epi.aux = a.epi.aux;
    k->epi.pre_out = a.epi.pre_out; k->epi.ld_aux = a.epi.ld_aux; k->epi.ld_pre = a.epi.ld_pre;
    k->epi.act = a.epi.act; k->epi.dact = a.epi.dact; k->epi.accumulate = a.epi.accumulate;
    k->epi.scale = a.epi.scale;
    k->mb.n = a.mb.n; k->mb.stride = a.mb.stride;
    k->K1 = sm_share_ < 0.75 ? 1 : 0;  // (K1 is unused on this path) plans differ with the share of the GPU
  }
  auto it = plans_.find(key);
  if (it == plans_.end()) it = plans_.emplace(key, make_tc_plan(a, 0, 0, ws_, ws_floats_, sm_share_)).first;
  launch_tc(it->second, s);
}

// ================================================================================================ linear passes
void linear_fwd(GemmRunner& g, cudaStream_t s, int rows, Mat x, const Linear& l, int act, float* y, int ldy, Mat x2,
                int k1, float* pre_out) {
  GemmArgs a;
  // Narrow heads (N = 2A = 12 ...) run over the padded extent when the output pitch has room for it: the padding rows
  // of W and b are zero and stay zero (their gradients are exactly zero), so the extra columns are written as zeros.
  const bool pad_n = l.out < 32 && l.out_alloc >= 32 && ldy >= l.out_alloc && rows >= 64 && pre_out == nullptr;
  a.M = rows; a.N = pad_n ? l.out_alloc : l.out; a.K = l.in;
  a.A = x.p; a.lda = x.ld;
  if (x2.p) { a.A2 = x2.p; a.lda2 = x2.ld; a.K1 = k1; }
  a.B = l.W; a.ldb = l.ld;
  a.C = y; a.ldc = ldy;
  a.epi.bias = l.b;
  a.epi.act = act;
  if (pre_out) { a.epi.pre_out = pre_out; a.epi.ld_pre = ldy; }
  a.mb = g.members();
  g.run(a, s);
}

void linear_dgrad(GemmRunner& g, cudaStream_t s, int rows, Mat dy, const Linear& l, int dact, Mat aux, float* dx,
                  int lddx, int col0, int n_cols) {
  GemmArgs a;
  a.M = rows; a.N = n_cols < 0 ? l.in : n_cols; a.K = l.out;
  a.A = dy.p; a.lda = dy.ld;
  a.B = l.W + col0; a.ldb = l.ld; a.b_mn = true;  // W[out, in] read as B(n = in, k = out)
  a.C = dx; a.ldc = lddx;
  a.epi.dact = dact;
  a.epi.aux = aux.p; a.epi.ld_aux = aux.ld;
  a.mb = g.members();
  g.run(a, s);
}

void linear_wgrad(GemmRunner& g, cudaStream_t s, int rows, Mat dy, Mat x, const Linear& l, Mat x2, int k1,
                  bool bias_grad) {
  // dW[out, in] = sum_b dy[b, out] x[b, in]:  A = dy (MN-major, k = batch), B = x (MN-major)
  if (x2.p == nullptr) {
    GemmArgs a;
    // MN-major operands need extents that are multiples of 32 on the tensor-core path: run over the padded extents
    // when the buffers are wide enough.  Whatever sits in the padding columns of dy / x only lands in the padding
    // rows / columns of dW, which no pass ever reads as data (K extents are always the logical ones).
    a.M = (l.out % 32 != 0 && dy.ld >= l.out_alloc && l.out_alloc % 32 == 0) ? l.out_alloc : l.out;
    a.N = (l.in % 32 != 0 && x.ld >= l.ld && l.ld % 32 == 0) ? l.ld : l.in;
    a.K = rows;
    a.A = dy.p; a.lda = dy.ld; a.a_mn = true;
    a.B = x.p; a.ldb = x.ld; a.b_mn = true;
    a.C = l.dW; a.ldc = l.ld;
    a.mb = g.members();
    g.run(a, s);
  } else {
    // two input segments -> two column blocks of dW
    GemmArgs a;
    a.M = l.out; a.N = k1; a.K = rows;
    a.A = dy.p; a.lda = dy.ld; a.a_mn = true;
    a.B = x.p; a.ldb = x.ld; a.b_mn = true;
    a.C = l.dW; a.ldc = l.ld;
    a.mb = g.members();
    g.run(a, s);
    GemmArgs b = a;
    b.N = l.in - k1;
    b.B = x2.p; b.ldb = x2.ld;
    b.C = l.dW + k1;
    g.run(b, s);
  }
  if (bias_grad) launch_colreduce(dy.p, dy.ld, rows, l.out, nullptr, l.db, 0, s, g.members());
}

// ================================================================================================ GraphReplay
void GraphReplay::reset() {
  if (exec_) cudaGraphExecDestroy(exec_);
  if (graph_) cudaGraphDestroy(graph_);
  exec_ = nullptr;
  graph_ = nullptr;
  calls_ = 0;
}

void GraphReplay::run(cudaStream_t s, bool enabled, const std::function<void()>& body) {
  if (!enabled) {
    body();
    return;
  }
  if (exec_ != nullptr) {
    RLREP_CUDA(cudaGraphLaunch(exec_, s));
    return;
  }
  if (calls_ == 0) {
    ++calls_;
    body();
    return;
  }
  RLREP_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  try {
    body();
  } catch (...) {
    cudaGraph_t g = nullptr;
    cudaStreamEndCapture(s, &g);
    if (g) cudaGraphDestroy(g);
    throw;
  }
  RLREP_CUDA(cudaStreamEndCapture(s, &graph_));
  RLREP_CUDA(cudaGraphInstantiate(&exec_, graph_, 0));
  RLREP_CUDA(cudaGraphLaunch(exec_, s));
}

bool GraphReplay::stats(int* kernel_nodes, int* programmatic_edges) const {
  if (exec_ == nullptr) return false;
  size_t n_nodes = 0;
  RLREP_CUDA(cudaGraphGetNodes(graph_, nullptr, &n_nodes));
  std::vector<cudaGraphNode_t> nodes(n_nodes);
  RLREP_CUDA(cudaGraphGetNodes(graph_, nodes.data(), &n_nodes));
  int kernels = 0;
  for (cudaGraphNode_t n : nodes) {
    cudaGraphNodeType t;
    RLREP_CUDA(cudaGraphNodeGetType(n, &t));
    if (t == cudaGraphNodeTypeKernel) ++kernels;
  }
  size_t n_edges = 0;
  RLREP_CUDA(cudaGraphGetEdges_v2(graph_, nullptr, nullptr, nullptr, &n_edges));
  std::vector<cudaGraphNode_t> from(n_edges), to(n_edges);
  std::vector<cudaGraphEdgeData> data(n_edges);
  RLREP_CUDA(cudaGraphGetEdges_v2(graph_, from.data(), to.data(), data.data(), &n_edges));
  int programmatic = 0;
  for (size_t i = 0; i < n_edges; ++i)
    if (data[i].type == cudaGraphDependencyTypeProgrammatic) ++programmatic;
  *kernel_nodes = kernels;
  *programmatic_edges = programmatic;
  return true;
}

}  // namespace rlrep

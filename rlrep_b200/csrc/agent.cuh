// Host-side runtime shared by the agent handles: device arena, parameter groups laid out for the fused
// optimiser kernel, the replay ring, GEMM dispatch with cached TMA plans, and CUDA-graph replay of train().
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>
#include <functional>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "gemm.cuh"
#include "gemm_chain.cuh"
#include "kernels.cuh"

namespace rlrep {

// ---------------------------------------------------------------------------------------------- memory
// One cudaMalloc per arena.  Buffers are registered first (`want`), then `commit` allocates once and fills in the
// registered pointers at 256-byte aligned offsets (TMA bases need 16 bytes, float4 kernels 16).
class DeviceArena {
 public:
  DeviceArena() = default;
  DeviceArena(const DeviceArena&) = delete;
  DeviceArena& operator=(const DeviceArena&) = delete;
  ~DeviceArena() { release(); }
  template <typename T>
  void want(T** slot, size_t count) {
    Req r;
    r.slot = reinterpret_cast<void**>(slot);
    r.offset = total_;
    reqs_.push_back(r);
    total_ += (count * sizeof(T) + 255) & ~size_t(255);
  }
  void commit() {
    RLREP_CHECK(base_ == nullptr, "arena already committed");
    RLREP_CUDA(cudaMalloc(&base_, total_ ? total_ : 256));
    RLREP_CUDA(cudaMemset(base_, 0, total_ ? total_ : 256));
    // The memset runs on the legacy default stream and is asynchronous with respect to the agents' NON-BLOCKING
    // streams: without this wait it can still be zeroing the arena when the first copies into it (control block,
    // weights) have already landed.
    RLREP_CUDA(cudaDeviceSynchronize());
    for (const Req& r : reqs_) *r.slot = static_cast<char*>(base_) + r.offset;
  }
  void release() {
    if (base_) cudaFree(base_);
    base_ = nullptr;
    total_ = 0;
    reqs_.clear();
  }
  size_t bytes() const { return total_; }

 private:
  struct Req {
    void** slot;
    size_t offset;
  };
  void* base_ = nullptr;
  size_t total_ = 0;
  std::vector<Req> reqs_;
};

// ---------------------------------------------------------------------------------------------- parameters
struct ParamTensor {
  std::string name;  // reference state_dict name, e.g. "phi.l1.weight"
  int rows = 0, cols = 0;  // logical shape (what state_dict sees)
  int ld = 0;              // row pitch in floats (>= cols); the padding is zero-initialised and never exported
  size_t offset = 0;       // floats from the start of the group
};

// A contiguous optimiser group: p | g | m | v (+ target copy of a prefix).  Elementwise Adam/Polyak do not care
// about tensor boundaries, so one kernel launch updates the whole group.
struct ParamGroup {
  std::string name;
  std::vector<ParamTensor> tensors;
  size_t n = 0;         // floats, each tensor padded to a multiple of 4
  size_t n_target = 0;  // prefix [0, n_target) has a Polyak target
  float *p = nullptr, *g = nullptr, *m = nullptr, *v = nullptr, *target = nullptr;
  std::string target_prefix_from, target_prefix_to;  // e.g. "phi." -> "phi_target."

  // ld = row pitch (0 -> cols), alloc_rows = rows actually allocated (0 -> rows); both only ever add zero padding.
  // exact = true does not round the tensor up to 4 floats (for tensors that must abut the next one; call align4()
  // after the last of them).
  size_t add(const std::string& nm, int rows, int cols, int ld = 0, int alloc_rows = 0, bool exact = false) {
    ParamTensor t;
    t.name = nm;
    t.rows = rows;
    t.cols = cols;
    t.ld = ld > 0 ? ld : cols;
    t.offset = n;
    tensors.push_back(t);
    const size_t sz = (size_t)(alloc_rows > 0 ? alloc_rows : rows) * t.ld;
    n += exact ? sz : ((sz + 3) & ~size_t(3));
    return t.offset;
  }
  void align4() { n = (n + 3) & ~size_t(3); }
  // `this` must stay at a fixed address until the arena is committed.
  void want(DeviceArena& a, bool with_opt = true) {
    a.want(&p, n);
    if (with_opt) { a.want(&g, n); a.want(&m, n); a.want(&v, n); }
    if (n_target) a.want(&target, n_target);
  }
};

// View of one nn.Linear inside a group.
struct Linear {
  float *W = nullptr, *b = nullptr, *dW = nullptr, *db = nullptr;
  int out = 0, in = 0;    // logical shape of W[out, in]
  int ld = 0;             // row pitch of W / dW in floats
  int out_alloc = 0;      // rows allocated (>= out)
};

struct LinearSlot {  // offsets resolved to pointers after the arena is committed
  size_t w_off = 0, b_off = 0;
  int out = 0, in = 0, ld = 0, out_alloc = 0;
  Linear view(const ParamGroup& g, bool target = false) const {
    Linear l;
    const float* base = target ? g.target : g.p;
    l.W = const_cast<float*>(base) + w_off;
    l.b = const_cast<float*>(base) + b_off;
    if (!target && g.g) { l.dW = g.g + w_off; l.db = g.g + b_off; }
    l.out = out;
    l.in = in;
    l.ld = ld > 0 ? ld : in;
    l.out_alloc = out_alloc > 0 ? out_alloc : out;
    return l;
  }
};

inline int round_up32(int x) { return (x + 31) & ~31; }

// pad = true stores W as [round_up32(out), round_up32(in)] (zero padding) so that every pass of the layer -- also
// the ones that read W or its input MN-major -- satisfies the tensor-core path's TMA constraints (16-byte row pitch,
// MN extents that are multiples of 32).  N = 1 heads are stored unpadded (they run on the row-dot kernels).
inline LinearSlot add_linear(ParamGroup& g, const std::string& name, int out, int in, bool pad = true) {
  LinearSlot s;
  s.out = out;
  s.in = in;
  s.ld = pad ? round_up32(in) : in;
  s.out_alloc = pad ? round_up32(out) : out;
  s.w_off = g.add(name + ".weight", out, in, s.ld, s.out_alloc);
  s.b_off = g.add(name + ".bias", out, 1, 1, s.out_alloc);
  return s;
}

// Two linears that share their input, stored back to back so they run as ONE GEMM: weights [out_a + out_b, in],
// biases [out_a + out_b].  Rows are padded up to a multiple of 32 after the second block.
inline LinearSlot add_stacked(ParamGroup& g, const std::string& a, int out_a, const std::string& b, int out_b, int in) {
  RLREP_CHECK(in % 32 == 0, "stacked heads need an input width that is a multiple of 32");
  LinearSlot s;
  s.out = out_a + out_b;
  s.in = in;
  s.ld = in;
  s.out_alloc = round_up32(s.out);
  s.w_off = g.add(a + ".weight", out_a, in);
  g.add(b + ".weight", out_b, in, in, s.out_alloc - out_a);
  s.b_off = g.add(a + ".bias", out_a, 1, 1, out_a, /*exact=*/true);
  g.add(b + ".bias", out_b, 1, 1, s.out_alloc - out_a, /*exact=*/true);
  g.align4();
  return s;
}

// ---------------------------------------------------------------------------------------------- replay ring
// Device-resident fp32 ring of packed records  [ s (S) | a (A) | r | d | pad | s' (S) | pad ]  with the s' block
// and the record size rounded up to 4 floats, so gathers are whole 128-bit loads and cat(s, a) is contiguous.
// Reference: utils/buffer.py:13-48 (fp64 host arrays; the fp32 cast happens at sample time -- casting at add
// time is bit-equivalent, SURVEY.md A.6 #8).
struct RecordLayout {
  int R, off_a, off_r, off_d, off_s2;
  static RecordLayout of(int S, int A) {
    RecordLayout l;
    l.off_a = S;
    l.off_r = S + A;
    l.off_d = S + A + 1;
    l.off_s2 = (S + A + 2 + 3) & ~3;
    l.R = (l.off_s2 + S + 3) & ~3;
    return l;
  }
};

class Ring {
 public:
  Ring(int state_dim, int action_dim, long long capacity);
  ~Ring();
  Ring(const Ring&) = delete;
  Ring& operator=(const Ring&) = delete;

  int S, A, R;            // record width in floats
  int off_a, off_r, off_d, off_s2;
  long long capacity, size = 0, ptr = 0;
  float* data = nullptr;  // [capacity, R]
  // Unique per Ring object for the life of the process: captured graphs bake `data` in, and a new ring can be allocated
  // at the address of a destroyed one, so agents key their graph on this id rather than on the object's address.
  const unsigned long long generation;

  // rows_host: n packed records (already laid out [n, R]); written at ptr.. with wrap-around.
  void add_packed(const float* rows_host, int n, cudaStream_t s);
  // fills the ring from five host arrays in the reference's layout (float64 or float32), n rows from slot 0
  void load_columns(const void* state, const void* action, const void* next_state, const void* reward,
                    const void* done, long long n, int is_f64, cudaStream_t s);
  void gather_from_host_idx(const long long* idx_host, int B, float* out_dev, cudaStream_t s);

 private:
  float* stage_host_ = nullptr;  // pinned
  float* stage_dev_ = nullptr;
  long long* idx_host_ = nullptr;  // pinned
  long long* idx_dev_ = nullptr;
  size_t stage_rows_ = 0;
  int idx_cap_ = 0;
};

// ---------------------------------------------------------------------------------------------- GEMM dispatch
enum Precision : int { PREC_TF32 = 0, PREC_FP32 = 1 };

class GemmRunner {
 public:
  void init(Precision prec, size_t ws_floats);
  ~GemmRunner();
  // Chooses the tcgen05 path when the operands allow it and the shape is worth a 128-row tile, else CUDA cores.
  void run(const GemmArgs& a, cudaStream_t s);
  // Implicit convolution (a.conv_w > 0) whose valid rows go straight to their compact positions (GemmArgs::compact_*):
  // true when the GEMM ran that way (the halo kernel), false when this GEMM does not qualify -- nothing was launched and
  // the caller runs it on the grid and compacts afterwards.
  bool run_compact(GemmArgs a, int wp, int ho, cudaStream_t s);
  bool compact_supported(GemmArgs a, int wp, int ho);  // the same decision without launching anything
  // Share of the GPU the next GEMMs should plan for: 0.5 inside fork()/join() sections where two independent kernel
  // chains run on two streams, 1.0 elsewhere.  Part of the plan-cache key.
  void set_sm_share(double share) { sm_share_ = share; }

  // GEMM chains (gemm_chain.cuh): between begin_chain(s) and end_chain() every run() is RECORDED instead of launched --
  // whatever stream it names -- and end_chain() executes the recorded DAG as one persistent kernel on `s` (dependencies are
  // inferred from the operands' addresses; the program is built on first use and cached by GEMM sequence).  A GEMM that
  // cannot join a chain (CUDA-core shapes) closes the chain recorded so far and runs on `s` in program order.  Callers
  // must not launch kernels that consume a recorded GEMM's output before end_chain().
  bool chains_enabled() const { return prec_ == PREC_TF32; }
  void begin_chain(cudaStream_t s);
  void end_chain();
  bool recording() const { return recording_; }

 private:
  void flush_chain();
  bool recording_ = false;
  cudaStream_t chain_stream_ = nullptr;
  std::vector<GemmArgs> pending_;
  std::vector<std::unique_ptr<GemmChain>> chains_;
  Precision prec_ = PREC_TF32;
  double sm_share_ = 1.0;
  float* ws_ = nullptr;
  size_t ws_floats_ = 0;
  // K-group partial outputs of GEMMs with a huge K and a handful of tiles (run(): "deep and skinny"); grown on first use of a
  // shape -- the first call of every update path runs eagerly, so never inside a graph capture
  float* kg_ws_ = nullptr;
  size_t kg_ws_floats_ = 0;
  std::unordered_map<std::string, TcGemmPlan> plans_;
};

// Convenience wrappers over GemmRunner for the three passes of y = act(x W^T + b).
struct Mat {
  const float* p = nullptr;
  int ld = 0;
};
void linear_fwd(GemmRunner& g, cudaStream_t s, int rows, Mat x, const Linear& l, int act, float* y, int ldy,
                Mat x2 = Mat(), int k1 = 0, float* pre_out = nullptr);
// dx = (dy W) * dact(aux);  n_cols selects the leading columns [col0, col0+n_cols) of the input gradient.
void linear_dgrad(GemmRunner& g, cudaStream_t s, int rows, Mat dy, const Linear& l, int dact, Mat aux, float* dx,
                  int lddx, int col0 = 0, int n_cols = -1);
// dW = dy^T x (x may be two K-major segments); db = colsum(dy) is launched here unless `bias_grad` is false (the
// caller then batches it with other bias gradients through bias_job + launch_colreduce_multi).
void linear_wgrad(GemmRunner& g, cudaStream_t s, int rows, Mat dy, Mat x, const Linear& l, Mat x2 = Mat(), int k1 = 0,
                  bool bias_grad = true);
inline ColJob bias_job(int rows, Mat dy, const Linear& l) {
  ColJob j;
  j.X = dy.p; j.ld = dy.ld; j.rows = rows; j.cols = l.out; j.u = nullptr; j.out = l.db;
  return j;
}

// ---------------------------------------------------------------------------------------------- graph replay
// Captures a launch sequence once and replays it; the sequence must only depend on device-resident state.
class GraphReplay {
 public:
  ~GraphReplay() { reset(); }
  void reset();
  // First call runs `body` eagerly (creates TMA plans, sets kernel attributes); the second captures it into a
  // graph; later calls replay.  `enabled = false` always runs eagerly.
  void run(cudaStream_t s, bool enabled, const std::function<void()>& body);
  bool captured() const { return exec_ != nullptr; }
  // Kernel nodes of the captured graph and its edges of type programmatic (PDL); false while nothing is captured.
  bool stats(int* kernel_nodes, int* programmatic_edges) const;

 private:
  int calls_ = 0;
  cudaGraph_t graph_ = nullptr;
  cudaGraphExec_t exec_ = nullptr;
};

// ---------------------------------------------------------------------------------------------- agent interface
struct AgentConfig {
  int alg = 0;
  int state_dim = 0, action_dim = 0, batch = 256;
  int hidden_dim = 256, feature_dim = 256, actor_hidden_dim = 256;
  int k_feat = 0;  // feature iterations per train() (extra_feature_steps + 1)
  double lr = 3e-4, lr_feat = 1e-4, lr_actor = 1e-4, lr_alpha = 1e-4;
  float discount = 0.99f, tau = 0.005f, feature_tau = 0.005f;
  double alpha0 = 0.1;
  int target_update_period = 2, learn_alpha = 1, use_feature_target = 1;
  int precision = PREC_TF32;
  int use_graph = 1;
  // algorithm-specific extras
  int phi_hidden_dim = 0, phi_hidden_depth = 0, mu_hidden_dim = 0, mu_hidden_depth = 0;
  int nabla_hidden_dim = 0, nabla_hidden_depth = 0, num_noise = 20, num_noises = 1000;
  float sigma_scale = 0.449f;
};

class Agent {
 public:
  virtual ~Agent() = default;
  virtual void train(Ring& ring, const long long* idx_host, int n_idx, const float* eps_host, int n_eps,
                     float* metrics_host, int n_metrics) = 0;
  // Benchmark aid: `n_steps` updates back to back with every input already resident in HBM (indices / noise for
  // all steps uploaded before the timed region, staged per step by device-to-device copies); returns the CUDA-event
  // time of the whole loop in milliseconds.  State advances exactly as n_steps train() calls would.
  virtual float train_resident(Ring& ring, const long long* idx_host, const float* eps_host, int n_steps) = 0;
  // One eager (non-graph) train() with an event behind every launch -> per-launch (kernel name, ms).
  virtual std::vector<ProfileEntry> profile_train(Ring& ring, const long long* idx_host, const float* eps_host) = 0;
  virtual int idx_per_train() const = 0;  // replay indices consumed per train()
  virtual int eps_per_train() const = 0;  // floats of host-drawn noise consumed per train()
  virtual const std::vector<std::string>& metric_names() const = 0;
  virtual std::vector<ParamGroup*> groups() = 0;
  virtual void act(const float* state_host, const float* eps_host, float* action_host) = 0;
  // `rows` observations [rows, S] (and noise [rows, A] or nullptr) -> actions [rows, A]: batched policy evaluation
  virtual void act_batch(const float* states_host, const float* eps_host, int rows, float* actions_host) = 0;
  virtual void sync_targets_from_params() = 0;  // target <- param copies (after loading weights)
  // Shape of the captured train() graph (GraphReplay::stats); false before the graph has been captured.
  virtual bool graph_stats(int* kernel_nodes, int* programmatic_edges) const = 0;

  AgentConfig cfg;
  cudaStream_t stream = nullptr;
  Control* ctl = nullptr;
  int last_launches = 0;
};

std::unique_ptr<Agent> make_sac_agent(const AgentConfig& cfg, cudaStream_t s);
std::unique_ptr<Agent> make_ctrlsac_agent(const AgentConfig& cfg, cudaStream_t s);
std::unique_ptr<Agent> make_vlsac_agent(const AgentConfig& cfg, cudaStream_t s);
std::unique_ptr<Agent> make_spedersac_agent(const AgentConfig& cfg, cudaStream_t s);
std::unique_ptr<Agent> make_diffsrsac_agent(const AgentConfig& cfg, cudaStream_t s);
class Comm;
// cfg.batch = rows per rank; the global batch is cfg.batch * comm->world (agent_ctrlsac_dp.cu)
std::unique_ptr<Agent> make_ctrlsac_sharded_agent(const AgentConfig& cfg, cudaStream_t s, Comm* comm);

}  // namespace rlrep

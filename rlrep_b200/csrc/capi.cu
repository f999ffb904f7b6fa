// extern "C" surface of librlrep_b200.so (declared in include/rlrep_b200.h).
#include <algorithm>
#include <cmath>
#include <memory>
#include <string>
#include <vector>

#include "agent.cuh"
#include "gemm_chain.cuh"
#include "comm.cuh"
#include "common.cuh"
#include "conv.cuh"
#include "deconv.cuh"
#include "drq.cuh"
#include "layout.cuh"
#include "mulv.cuh"
#include "pixel_replay.cuh"
#include "ldiffsr.cuh"
#include "gemm.cuh"
#include "rlrep_b200.h"

namespace rlrep {
namespace {
thread_local std::string g_last_error;
}
void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* get_last_error() { return g_last_error.c_str(); }

Epilogue to_epilogue(const rlrep_epilogue* e) {
  Epilogue o;
  if (e == nullptr) return o;
  o.bias = e->bias_dev;
  o.r1_u = e->r1_u_dev;
  o.r1_v = e->r1_v_dev;
  o.aux = e->aux_dev;
  o.pre_out = e->pre_out_dev;
  o.ld_aux = e->ld_aux;
  o.ld_pre = e->ld_pre;
  o.act = e->act;
  o.dact = e->dact;
  o.accumulate = e->accumulate;
  o.scale = e->scale;
  return o;
}
}  // namespace rlrep

using namespace rlrep;

// The TF32 GemmRunner behind rlrep_gemm's path 2 (one per thread, like the chain recorder below): it dispatches exactly as an
// agent's runner does -- tensor cores or CUDA cores by shape, K groups plus their finishing pass for deep and skinny GEMMs --
// and keeps its plans and K-group workspace between calls.
static GemmRunner& gemm_runner() {
  thread_local std::unique_ptr<GemmRunner> r;
  if (!r) {
    r.reset(new GemmRunner());
    r->init(PREC_TF32, 0);
  }
  return *r;
}

// Calibration kernels for rlrep_gemm_bench (path 2 / 3): an empty kernel, plain and with programmatic dependent
// launch, to measure the per-launch floor of a dependent kernel chain on this GPU.
__global__ void null_kernel(float* p) {
  if (p == reinterpret_cast<float*>(1)) *p = 0.f;
}
__global__ void null_pdl_kernel(float* p) {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (p == reinterpret_cast<float*>(1)) *p = 0.f;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// Every handle remembers the CUDA device it was created on, and every entry point that takes a handle runs on that device
// whatever the calling thread's current device is (worker threads of a population start on device 0): scoped
// cudaSetDevice, restored on exit.
static int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return d;
}
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int want) {
    if (want < 0) return;
    int cur = 0;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != want && cudaSetDevice(want) == cudaSuccess) prev = cur;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define RLREP_API_BEGIN_ON(h) RLREP_API_BEGIN DeviceGuard _device_guard((h) != nullptr ? (h)->device : -1);

struct rlrep_ring {
  int device = current_device();
  std::unique_ptr<Ring> impl;
};

struct rlrep_comm {
  int device = current_device();
  std::unique_ptr<Comm> impl;
};

struct TensorRef {
  std::string name;
  float* ptr;
  int rows, cols, ld;
};

// The tensor index of a handle: entry i by index, its description, and synchronous copies between its [rows, cols]
// (row pitch ld) and a dense host array.
static const TensorRef& tensor_at(const std::vector<TensorRef>& ts, int i) {
  RLREP_CHECK(i >= 0 && i < (int)ts.size(), "tensor index out of range");
  return ts[i];
}
static void tensor_info(const std::vector<TensorRef>& ts, int i, const char** name, float** ptr_dev, int* rows,
                        int* cols) {
  const TensorRef& t = tensor_at(ts, i);
  if (name) *name = t.name.c_str();
  if (ptr_dev) *ptr_dev = t.ptr;
  if (rows) *rows = t.rows;
  if (cols) *cols = t.cols;
}
static void tensor_read(const TensorRef& t, float* out_host, cudaStream_t st) {
  RLREP_CHECK(out_host != nullptr, "null argument");
  RLREP_CUDA(cudaMemcpy2DAsync(out_host, (size_t)t.cols * 4, t.ptr, (size_t)t.ld * 4, (size_t)t.cols * 4, t.rows,
                               cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
}
static void tensor_read(const std::vector<TensorRef>& ts, int i, float* out_host, cudaStream_t st) {
  tensor_read(tensor_at(ts, i), out_host, st);
}
static void tensor_write(const TensorRef& t, const float* in_host, cudaStream_t st) {
  RLREP_CHECK(in_host != nullptr, "null argument");
  RLREP_CUDA(cudaMemcpy2DAsync(t.ptr, (size_t)t.ld * 4, in_host, (size_t)t.cols * 4, (size_t)t.cols * 4, t.rows,
                               cudaMemcpyHostToDevice, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
}
static void tensor_write(const std::vector<TensorRef>& ts, int i, const float* in_host, cudaStream_t st) {
  tensor_write(tensor_at(ts, i), in_host, st);
}

struct rlrep_agent {
  int device = current_device();
  std::unique_ptr<Agent> impl;
  std::vector<TensorRef> tensors;
  cudaStream_t owned_stream = nullptr;  // created when the caller passed the (uncapturable) legacy default stream
};

static void index_tensors(rlrep_agent* a) {
  a->tensors.clear();
  for (ParamGroup* g : a->impl->groups()) {
    for (const ParamTensor& t : g->tensors) a->tensors.push_back({t.name, g->p + t.offset, t.rows, t.cols, t.ld});
    // Adam moments under "optim.m/<name>" / "optim.v/<name>": with rlrep_agent_get/set_optim_state they make a checkpoint
    // resume bit-identically to an uninterrupted run (torch.optim.Adam's exp_avg / exp_avg_sq of the same parameter)
    if (g->m && g->v)
      for (const ParamTensor& t : g->tensors) {
        a->tensors.push_back({"optim.m/" + t.name, g->m + t.offset, t.rows, t.cols, t.ld});
        a->tensors.push_back({"optim.v/" + t.name, g->v + t.offset, t.rows, t.cols, t.ld});
      }
    if (g->target) {
      for (const ParamTensor& t : g->tensors) {
        if (t.offset >= g->n_target) continue;
        if (t.name.compare(0, g->target_prefix_from.size(), g->target_prefix_from) != 0) continue;
        a->tensors.push_back({g->target_prefix_to + t.name.substr(g->target_prefix_from.size()), g->target + t.offset,
                              t.rows, t.cols, t.ld});
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ pixel agent handles
struct PixelHandle {
  int device = current_device();
  std::unique_ptr<PixelAgent> impl;
  std::vector<TensorRef> tensors;
  cudaStream_t owned_stream = nullptr;  // created when the caller passed the (uncapturable) legacy default stream
  virtual ~PixelHandle() {
    if (impl) cudaStreamSynchronize(impl->stream());
    impl.reset();
    if (owned_stream) cudaStreamDestroy(owned_stream);
  }
};
struct rlrep_drq : PixelHandle {
  DrqV2& agent() { return static_cast<DrqV2&>(*impl); }
};
struct rlrep_mulv : PixelHandle {
  MulvDrq& agent() { return static_cast<MulvDrq&>(*impl); }
};
struct rlrep_ldiff : PixelHandle {
  LatentDiffSR& agent() { return static_cast<LatentDiffSR&>(*impl); }
};

// The agent runs on `stream`, or on a stream of its own when that is null.  Its tensors are indexed group by group under
// the reference's names: the parameters, their gradients of the most recent update ("grad/<name>", for gradient-level
// parity tests), the Adam moments of groups that have an optimiser ("optim.m/<name>", "optim.v/<name>": with
// rlrep_<agent>_get/set_optim_state they make a checkpoint resume bit-identically), then the target copies.
template <class Handle, class Impl, class Config>
static Handle* create_pixel(const Config& c, void* stream) {
  std::unique_ptr<Handle> h(new Handle);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (st == nullptr) {
    RLREP_CUDA(cudaStreamCreateWithFlags(&h->owned_stream, cudaStreamNonBlocking));
    st = h->owned_stream;
  }
  h->impl.reset(new Impl(c, st));
  for (ParamGroup* g : h->impl->groups()) {
    auto add = [&](float* base, const std::string& from, const std::string& to) {
      for (const ParamTensor& t : g->tensors) {
        const std::string name = h->impl->tensor_name(*g, t.name);
        RLREP_CHECK(name.compare(0, from.size(), from) == 0, name + " does not start with " + from);
        h->tensors.push_back({to + name.substr(from.size()), base + t.offset, t.rows, t.cols, t.ld});
      }
    };
    add(g->p, "", "");
    if (g->g) add(g->g, "", "grad/");
    if (g->m && g->v) {
      add(g->m, "", "optim.m/");
      add(g->v, "", "optim.v/");
    }
    if (g->target) add(g->target, g->target_prefix_from, g->target_prefix_to);
  }
  return h.release();
}

static int pixel_destroy(PixelHandle* h) {
  RLREP_API_BEGIN_ON(h)
  delete h;
  RLREP_API_END
}
static int pixel_num_tensors(PixelHandle* h, int* n) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && n, "null argument");
  *n = (int)h->tensors.size();
  RLREP_API_END
}
static int pixel_tensor_info(PixelHandle* h, int i, const char** name, float** ptr_dev, int* rows, int* cols) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h, "null argument");
  tensor_info(h->tensors, i, name, ptr_dev, rows, cols);
  RLREP_API_END
}
static int pixel_tensor_read(PixelHandle* h, int i, float* out_host) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h, "null argument");
  tensor_read(h->tensors, i, out_host, h->impl->stream());
  RLREP_API_END
}
static int pixel_tensor_write(PixelHandle* h, int i, const float* in_host) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h, "null argument");
  tensor_write(h->tensors, i, in_host, h->impl->stream());
  RLREP_API_END
}
static int pixel_sync_targets(PixelHandle* h) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h, "null argument");
  h->impl->sync_targets_from_params();
  RLREP_API_END
}
static int pixel_update_resident(PixelHandle* h, int n_steps, float stddev, float* total_ms) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && total_ms, "null argument");
  *total_ms = h->impl->update_resident(n_steps, stddev);
  RLREP_API_END
}
static int pixel_profile_update(PixelHandle* h, float stddev, int max_entries, const char** names, float* ms,
                                double* bytes, double* flops, int* n_entries) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && n_entries && (max_entries == 0 || (names && ms)), "null argument");
  std::vector<ProfileEntry> prof = h->impl->profile_update(stddev);
  const int n = (int)std::min<size_t>(prof.size(), (size_t)max_entries);
  for (int i = 0; i < n; ++i) {
    names[i] = prof[i].name;  // string literals with static storage
    ms[i] = prof[i].ms;
    if (bytes) bytes[i] = prof[i].bytes;
    if (flops) flops[i] = prof[i].flops;
  }
  *n_entries = (int)prof.size();
  RLREP_API_END
}
static int pixel_last_launches(PixelHandle* h, int* launches) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && launches, "null argument");
  *launches = h->impl->last_launches;
  RLREP_API_END
}
// The pixel agents' optimiser counters are the three Adam step counters of the control block; they have no `steps`
// gate and no temperature, so those fields read as 0 and a non-zero value for them is refused.
static int pixel_get_optim_state(PixelHandle* h, rlrep_optim_state* out) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && out, "null argument");
  Control c;
  cudaStream_t st = h->impl->stream();
  RLREP_CUDA(cudaMemcpyAsync(&c, h->impl->control(), sizeof(c), cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  *out = rlrep_optim_state{};
  out->t_feature = c.t_feat; out->t_critic = c.t_critic; out->t_actor = c.t_actor;
  RLREP_API_END
}
static int pixel_set_optim_state(PixelHandle* h, const rlrep_optim_state* in) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && in, "null argument");
  RLREP_CHECK(in->steps == 0 && in->t_alpha == 0 && in->log_alpha == 0.0 && in->log_alpha_m == 0.0 &&
                  in->log_alpha_v == 0.0,
              "pixel agents have no steps gate and no temperature: steps, t_alpha and log_alpha* must be 0");
  RLREP_CHECK(in->t_feature >= 0 && in->t_critic >= 0 && in->t_actor >= 0, "Adam step counters must be non-negative");
  Control c;
  cudaStream_t st = h->impl->stream();
  RLREP_CUDA(cudaMemcpyAsync(&c, h->impl->control(), sizeof(c), cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  c.t_feat = in->t_feature; c.t_critic = in->t_critic; c.t_actor = in->t_actor;
  RLREP_CUDA(cudaMemcpyAsync(h->impl->control(), &c, sizeof(c), cudaMemcpyHostToDevice, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_API_END
}

extern "C" {

int rlrep_abi_version(void) { return RLREP_ABI_VERSION; }
const char* rlrep_last_error(void) { return get_last_error(); }

int rlrep_gemm(void* stream, int path, int M, int N, int K, const float* A, int lda, int a_mn, const float* A2,
               int lda2, int K1, const float* B, int ldb, int b_mn, float* C, int ldc, const rlrep_epilogue* epi,
               int bn, int split_k, float* ws, size_t ws_floats) {
  RLREP_API_BEGIN
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.lda = lda; g.a_mn = a_mn != 0;
  g.A2 = A2; g.lda2 = lda2; g.K1 = K1;
  g.B = B; g.ldb = ldb; g.b_mn = b_mn != 0;
  g.C = C; g.ldc = ldc;
  g.epi = to_epilogue(epi);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (path == 0) {
    TcGemmPlan p = make_tc_plan(g, bn, split_k, ws, ws_floats);
    launch_tc(p, st);
  } else if (path == 2) {
    RLREP_CHECK(A2 == nullptr && bn == 0 && split_k == 0, "path 2 plans the GEMM itself: no A2, bn or split_k");
    gemm_runner().run(g, st);
  } else {
    launch_simt(g, st);
  }
  RLREP_API_END
}

namespace {
thread_local std::vector<GemmArgs> g_chain_seq;
}

int rlrep_gemm_chain_set_debug(unsigned long long* dev) {
  RLREP_API_BEGIN
  set_chain_debug_buffer(dev);
  RLREP_API_END
}

int rlrep_gemm_chain_begin(void) {
  RLREP_API_BEGIN
  g_chain_seq.clear();
  RLREP_API_END
}

int rlrep_gemm_chain_add(int M, int N, int K, const float* A, int lda, int a_mn, const float* B, int ldb, int b_mn,
                         float* C, int ldc, const rlrep_epilogue* epi) {
  RLREP_API_BEGIN
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.lda = lda; g.a_mn = a_mn != 0;
  g.B = B; g.ldb = ldb; g.b_mn = b_mn != 0;
  g.C = C; g.ldc = ldc;
  g.epi = to_epilogue(epi);
  RLREP_CHECK(chain_eligible(g), "operands violate the tensor-core path's constraints (see rlrep_gemm, path 0)");
  g_chain_seq.push_back(g);
  RLREP_API_END
}

int rlrep_gemm_chain_run(void* stream, int bn, int split_k, int iters, float* ms_out, int* levels_out) {
  RLREP_API_BEGIN
  RLREP_CHECK(!g_chain_seq.empty() && iters >= 1, "empty chain");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GemmChain chain;
  chain.build(g_chain_seq, bn, split_k);
  if (levels_out) *levels_out = chain.levels();
  cudaEvent_t e0, e1;
  RLREP_CUDA(cudaEventCreate(&e0));
  RLREP_CUDA(cudaEventCreate(&e1));
  chain.launch(st);  // the first launch also warms the instruction cache; it is part of the result, not of the timing
  RLREP_CUDA(cudaEventRecord(e0, st));
  for (int i = 1; i < iters; ++i) chain.launch(st);
  RLREP_CUDA(cudaEventRecord(e1, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  float ms = 0.f;
  RLREP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (ms_out) *ms_out = iters > 1 ? ms / (iters - 1) : 0.f;
  g_chain_seq.clear();
  RLREP_API_END
}

// Times `iters` back-to-back launches of one planned GEMM with CUDA events on `stream` (tensor maps encoded
// once, as the agent handles do).  Tuning/benchmark aid; ms_out = average milliseconds per GEMM.
int rlrep_gemm_bench(void* stream, int path, int M, int N, int K, const float* A, int lda, int a_mn, const float* B,
                     int ldb, int b_mn, float* C, int ldc, const rlrep_epilogue* epi, int bn, int split_k, float* ws,
                     size_t ws_floats, int iters, float* ms_out, int* bn_out, int* split_out) {
  RLREP_API_BEGIN
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.lda = lda; g.a_mn = a_mn != 0;
  g.B = B; g.ldb = ldb; g.b_mn = b_mn != 0;
  g.C = C; g.ldc = ldc;
  g.epi = to_epilogue(epi);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaEvent_t e0, e1;
  RLREP_CUDA(cudaEventCreate(&e0));
  RLREP_CUDA(cudaEventCreate(&e1));
  TcGemmPlan p;
  if (path == 0) {
    p = make_tc_plan(g, bn, split_k, ws, ws_floats);
    if (bn_out) *bn_out = p.bn;
    if (split_out) *split_out = p.split_k;
  }
  auto launch_once = [&](cudaStream_t s) {
    if (path == 0) launch_tc(p, s);
    else if (path == 1) launch_simt(g, s);
    else if (path == 2) null_kernel<<<M, 128, 0, s>>>(C);
    else {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(M);
      cfg.blockDim = dim3(128);
      cfg.stream = s;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      RLREP_CUDA(cudaLaunchKernelEx(&cfg, null_pdl_kernel, C));
    }
  };
  for (int i = 0; i < 3; ++i) launch_once(st);
  // Replay through a CUDA graph so the number is device time, not the host's launch rate.
  cudaStream_t cs;
  RLREP_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
  for (int i = 0; i < iters; ++i) launch_once(cs);
  RLREP_CUDA(cudaStreamEndCapture(cs, &graph));
  RLREP_CUDA(cudaGraphInstantiate(&exec, graph, 0));
  RLREP_CUDA(cudaGraphLaunch(exec, cs));
  RLREP_CUDA(cudaEventRecord(e0, cs));
  RLREP_CUDA(cudaGraphLaunch(exec, cs));
  RLREP_CUDA(cudaEventRecord(e1, cs));
  RLREP_CUDA(cudaStreamSynchronize(cs));
  cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  cudaStreamDestroy(cs);
  RLREP_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  RLREP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  *ms_out = ms / iters;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  RLREP_API_END
}

int rlrep_gemm_set_debug_buffer(unsigned long long* dev80) {
  RLREP_API_BEGIN
  set_gemm_debug_buffer(dev80);
  RLREP_API_END
}
int rlrep_gemm_trace(unsigned long long* out16_host) {
  RLREP_API_BEGIN
  RLREP_CUDA(cudaDeviceSynchronize());
  read_gemm_trace(out16_host);
  RLREP_API_END
}

// ------------------------------------------------------------------------------------------------ ring
int rlrep_ring_create(int state_dim, int action_dim, long long capacity, rlrep_ring** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(out != nullptr, "null out pointer");
  std::unique_ptr<rlrep_ring> r(new rlrep_ring);
  r->impl.reset(new Ring(state_dim, action_dim, capacity));
  *out = r.release();
  RLREP_API_END
}
int rlrep_ring_destroy(rlrep_ring* ring) {
  RLREP_API_BEGIN_ON(ring)
  delete ring;
  RLREP_API_END
}
int rlrep_ring_layout(const rlrep_ring* ring, int* record_floats, int* off_action, int* off_reward, int* off_done,
                      int* off_next_state) {
  RLREP_API_BEGIN_ON(ring)
  const Ring& r = *ring->impl;
  *record_floats = r.R; *off_action = r.off_a; *off_reward = r.off_r; *off_done = r.off_d; *off_next_state = r.off_s2;
  RLREP_API_END
}
int rlrep_ring_state(const rlrep_ring* ring, long long* size, long long* ptr, long long* capacity) {
  RLREP_API_BEGIN_ON(ring)
  *size = ring->impl->size; *ptr = ring->impl->ptr; *capacity = ring->impl->capacity;
  RLREP_API_END
}
int rlrep_ring_add_packed(rlrep_ring* ring, const float* rows_host, int n, void* stream) {
  RLREP_API_BEGIN_ON(ring)
  ring->impl->add_packed(rows_host, n, static_cast<cudaStream_t>(stream));
  RLREP_API_END
}
int rlrep_ring_load(rlrep_ring* ring, const void* state, const void* action, const void* next_state,
                    const void* reward, const void* done, long long n, int is_f64, void* stream) {
  RLREP_API_BEGIN_ON(ring)
  ring->impl->load_columns(state, action, next_state, reward, done, n, is_f64, static_cast<cudaStream_t>(stream));
  RLREP_API_END
}
int rlrep_ring_gather(rlrep_ring* ring, const int64_t* idx_host, int B, float* out_dev, void* stream) {
  RLREP_API_BEGIN_ON(ring)
  ring->impl->gather_from_host_idx(reinterpret_cast<const long long*>(idx_host), B, out_dev,
                                   static_cast<cudaStream_t>(stream));
  RLREP_API_END
}

// ------------------------------------------------------------------------------------------------ agents
// ------------------------------------------------------------------------------------------------ pixel encoder
struct rlrep_conv_encoder {
  int device = current_device();
  std::unique_ptr<ConvEncoder> impl;
  cudaStream_t owned_stream = nullptr;
};

// Reference layout [32, C, 3, 3] <-> stored layout: layer 0 as is, layers 1-3 as [32, (ky, kx, c)].
static void conv_layout(int layer, int k, bool to_stored, const float* in, float* out) {
  if (layer == 0) {
    std::copy(in, in + (size_t)32 * k, out);
    return;
  }
  for (int o = 0; o < 32; ++o)
    for (int c = 0; c < 32; ++c)
      for (int t = 0; t < 9; ++t) {
        const size_t ref = ((size_t)o * 32 + c) * 9 + t, st = (size_t)o * 288 + (size_t)t * 32 + c;
        if (to_stored) out[st] = in[ref];
        else out[ref] = in[st];
      }
}

int rlrep_conv_encoder_create(int batch, int in_channels, int height, int precision, void* stream,
                              rlrep_conv_encoder** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(out != nullptr, "null out pointer");
  std::unique_ptr<rlrep_conv_encoder> h(new rlrep_conv_encoder);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (st == nullptr) {
    RLREP_CUDA(cudaStreamCreateWithFlags(&h->owned_stream, cudaStreamNonBlocking));
    st = h->owned_stream;
  }
  h->impl.reset(new ConvEncoder(batch, in_channels, height, static_cast<Precision>(precision), st));
  *out = h.release();
  RLREP_API_END
}
int rlrep_conv_encoder_destroy(rlrep_conv_encoder* enc) {
  RLREP_API_BEGIN_ON(enc)
  if (enc) {
    if (enc->impl) cudaStreamSynchronize(enc->impl->stream());
    enc->impl.reset();
    if (enc->owned_stream) cudaStreamDestroy(enc->owned_stream);
  }
  delete enc;
  RLREP_API_END
}
int rlrep_conv_encoder_read(rlrep_conv_encoder* enc, int layer, int what, float* out_host) {
  RLREP_API_BEGIN_ON(enc)
  RLREP_CHECK(enc && out_host && layer >= 0 && layer < 4 && what >= 0 && what < 4, "bad argument");
  const Linear l = enc->impl->layer(layer);
  const int k = enc->impl->layer_k(layer);
  cudaStream_t st = enc->impl->stream();
  if (what == 1 || what == 3) {
    RLREP_CUDA(cudaMemcpyAsync(out_host, what == 1 ? l.b : l.db, 32 * sizeof(float), cudaMemcpyDeviceToHost, st));
    RLREP_CUDA(cudaStreamSynchronize(st));
  } else {
    std::vector<float> tmp((size_t)32 * k);
    RLREP_CUDA(cudaMemcpy2DAsync(tmp.data(), (size_t)k * 4, what == 0 ? l.W : l.dW, (size_t)l.ld * 4, (size_t)k * 4, 32,
                                 cudaMemcpyDeviceToHost, st));
    RLREP_CUDA(cudaStreamSynchronize(st));
    conv_layout(layer, k, false, tmp.data(), out_host);
  }
  RLREP_API_END
}
int rlrep_conv_encoder_write(rlrep_conv_encoder* enc, int layer, int what, const float* in_host) {
  RLREP_API_BEGIN_ON(enc)
  RLREP_CHECK(enc && in_host && layer >= 0 && layer < 4 && (what == 0 || what == 1), "bad argument");
  const Linear l = enc->impl->layer(layer);
  const int k = enc->impl->layer_k(layer);
  cudaStream_t st = enc->impl->stream();
  if (what == 1) {
    RLREP_CUDA(cudaMemcpyAsync(l.b, in_host, 32 * sizeof(float), cudaMemcpyHostToDevice, st));
  } else {
    std::vector<float> tmp((size_t)32 * k);
    conv_layout(layer, k, true, in_host, tmp.data());
    RLREP_CUDA(cudaMemcpy2DAsync(l.W, (size_t)l.ld * 4, tmp.data(), (size_t)k * 4, (size_t)k * 4, 32,
                                 cudaMemcpyHostToDevice, st));
    RLREP_CUDA(cudaStreamSynchronize(st));
  }
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_API_END
}
int rlrep_conv_encoder_forward_pitched(rlrep_conv_encoder* enc, const unsigned char* obs_dev, const int* shifts_dev,
                                       float* feat_dev, int ld_feat, int no_grad) {
  RLREP_API_BEGIN_ON(enc)
  RLREP_CHECK(enc && obs_dev && feat_dev, "null argument");
  RLREP_CHECK(ld_feat == 0 || ld_feat >= enc->impl->feature_dim(), "feature row pitch narrower than a feature row");
  enc->impl->forward(obs_dev, shifts_dev, feat_dev, ld_feat, /*target=*/false, no_grad != 0);
  RLREP_API_END
}
int rlrep_conv_encoder_forward(rlrep_conv_encoder* enc, const unsigned char* obs_dev, const int* shifts_dev,
                               float* feat_dev) {
  return rlrep_conv_encoder_forward_pitched(enc, obs_dev, shifts_dev, feat_dev, 0, 0);
}
int rlrep_conv_encoder_backward_pitched(rlrep_conv_encoder* enc, const float* dfeat_dev, int ld_dfeat) {
  RLREP_API_BEGIN_ON(enc)
  RLREP_CHECK(enc && dfeat_dev, "null argument");
  RLREP_CHECK(ld_dfeat == 0 || ld_dfeat >= enc->impl->feature_dim(), "gradient row pitch narrower than a feature row");
  enc->impl->backward(dfeat_dev, ld_dfeat);
  RLREP_API_END
}
int rlrep_conv_encoder_backward(rlrep_conv_encoder* enc, const float* dfeat_dev) {
  return rlrep_conv_encoder_backward_pitched(enc, dfeat_dev, 0);
}
int rlrep_conv_encoder_read_map(rlrep_conv_encoder* enc, int which, int layer, float* out_dev) {
  RLREP_API_BEGIN_ON(enc)
  RLREP_CHECK(enc && out_dev && (which == 0 || which == 1) && layer >= 0 && layer < 4, "bad argument");
  ConvEncoder& e = *enc->impl;
  const int P = e.hw(layer) * e.hw(layer);
  launch_nhwc_to_cp(which == 0 ? e.act(layer) : e.dact(layer), e.batch(), P, out_dev, (long long)P * 32, e.stream());
  RLREP_LAUNCHED("nhwc_to_nchw", e.stream());
  RLREP_API_END
}
int rlrep_conv_encoder_feature_dim(rlrep_conv_encoder* enc, int* dim) {
  RLREP_API_BEGIN_ON(enc)
  RLREP_CHECK(enc && dim, "null argument");
  *dim = enc->impl->feature_dim();
  RLREP_API_END
}

// ------------------------------------------------------------------------------------------------ pixel decoder
struct rlrep_conv_decoder {
  int device = current_device();
  std::unique_ptr<ConvDecoder> impl;
  cudaStream_t owned_stream = nullptr;
};

// Reference layout [ci, co, 3, 3] of a transposed layer (0-3) <-> stored [(ky, kx, co), ci]; the output conv (layer 4) is
// stored in the reference's [3, 32, k, k] as is.
static void deconv_layout(int layer, size_t n, bool to_stored, const float* in, float* out) {
  if (layer == 4) {
    std::copy(in, in + n, out);
    return;
  }
  for (int ci = 0; ci < 32; ++ci)
    for (int co = 0; co < 32; ++co)
      for (int t = 0; t < 9; ++t) {
        const size_t ref = ((size_t)ci * 32 + co) * 9 + t, st = ((size_t)t * 32 + co) * 32 + ci;
        if (to_stored) out[st] = in[ref];
        else out[ref] = in[st];
      }
}
static size_t deconv_param_size(const ConvDecoder& d, int layer, bool bias) {
  if (layer == 4) return bias ? 3 : (size_t)3 * 32 * d.out_kernel() * d.out_kernel();
  return bias ? 32 : 288 * 32;
}

int rlrep_conv_decoder_create(int batch, int out_kernel, int precision, void* stream, rlrep_conv_decoder** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(out != nullptr, "null out pointer");
  std::unique_ptr<rlrep_conv_decoder> h(new rlrep_conv_decoder);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (st == nullptr) {
    RLREP_CUDA(cudaStreamCreateWithFlags(&h->owned_stream, cudaStreamNonBlocking));
    st = h->owned_stream;
  }
  h->impl.reset(new ConvDecoder(batch, static_cast<Precision>(precision), st, out_kernel));
  *out = h.release();
  RLREP_API_END
}
int rlrep_conv_decoder_destroy(rlrep_conv_decoder* dec) {
  RLREP_API_BEGIN_ON(dec)
  if (dec) {
    if (dec->impl) cudaStreamSynchronize(dec->impl->stream());
    dec->impl.reset();
    if (dec->owned_stream) cudaStreamDestroy(dec->owned_stream);
  }
  delete dec;
  RLREP_API_END
}
int rlrep_conv_decoder_read(rlrep_conv_decoder* dec, int layer, int what, float* out_host) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && out_host && layer >= 0 && layer < 5 && what >= 0 && what < 4, "bad argument");
  ConvDecoder& d = *dec->impl;
  const bool bias = what == 1 || what == 3;
  const size_t n = deconv_param_size(d, layer, bias);
  const float* src = (what < 2 ? d.group().p : d.group().g) + (bias ? d.bias_offset(layer) : d.weight_offset(layer));
  std::vector<float> tmp(n);
  cudaStream_t st = d.stream();
  RLREP_CUDA(cudaMemcpyAsync(tmp.data(), src, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  if (bias) std::copy(tmp.begin(), tmp.end(), out_host);
  else deconv_layout(layer, n, false, tmp.data(), out_host);
  RLREP_API_END
}
int rlrep_conv_decoder_write(rlrep_conv_decoder* dec, int layer, int what, const float* in_host) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && in_host && layer >= 0 && layer < 5 && (what == 0 || what == 1), "bad argument");
  ConvDecoder& d = *dec->impl;
  const bool bias = what == 1;
  const size_t n = deconv_param_size(d, layer, bias);
  std::vector<float> tmp(in_host, in_host + n);
  if (!bias) deconv_layout(layer, n, true, in_host, tmp.data());
  cudaStream_t st = d.stream();
  RLREP_CUDA(cudaMemcpyAsync(d.group().p + (bias ? d.bias_offset(layer) : d.weight_offset(layer)), tmp.data(),
                             n * sizeof(float), cudaMemcpyHostToDevice, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_API_END
}
int rlrep_conv_decoder_forward(rlrep_conv_decoder* dec, const float* x_dev, int ld_x) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && x_dev && ld_x >= 0, "bad argument");
  dec->impl->forward(x_dev, ld_x);
  RLREP_API_END
}
int rlrep_conv_decoder_l1_loss(rlrep_conv_decoder* dec, const unsigned char* target_dev, float grad_scale,
                               float* loss_dev) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && target_dev && loss_dev, "null argument");
  dec->impl->l1_loss(target_dev, grad_scale, loss_dev);
  RLREP_API_END
}
int rlrep_conv_decoder_mse_sum_loss(rlrep_conv_decoder* dec, const unsigned char* target_dev, const int* shifts_dev,
                                    float grad_scale, float* loss_dev) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && target_dev && loss_dev, "null argument");
  dec->impl->mse_sum_loss(target_dev, shifts_dev, grad_scale, loss_dev);
  RLREP_API_END
}
int rlrep_conv_decoder_backward(rlrep_conv_decoder* dec, float* dx_dev, int ld_dx) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && dx_dev && ld_dx >= 0, "bad argument");
  dec->impl->backward(dx_dev, ld_dx);
  RLREP_API_END
}
int rlrep_conv_decoder_read_map(rlrep_conv_decoder* dec, int which, int i, float* out_dev) {
  RLREP_API_BEGIN_ON(dec)
  RLREP_CHECK(dec && out_dev && which >= 0 && which < 4 && (which >= 2 || (i >= 0 && i < 5)), "bad argument");
  ConvDecoder& d = *dec->impl;
  if (which >= 2) {
    d.copy_pred(out_dev, which == 3);
  } else {
    const int P = d.hw(i) * d.hw(i);
    launch_nhwc_to_cp(which == 0 ? d.act(i) : d.dact(i), d.batch(), P, out_dev, (long long)P * 32, d.stream());
    RLREP_LAUNCHED("nhwc_to_nchw", d.stream());
  }
  RLREP_API_END
}

// ------------------------------------------------------------------------------------------------ pixel agents
// rlrep_drq, rlrep_mulv and rlrep_ldiff are one handle over a PixelAgent: only create, update and act differ.
int rlrep_drq_create(const rlrep_drq_config* c, void* stream, rlrep_drq** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(c != nullptr && out != nullptr, "null argument");
  DrqConfig d;
  d.batch = c->batch_size; d.channels = c->channels; d.height = c->height; d.action_dim = c->action_dim;
  d.bn_dim = c->bn_dim; d.hidden_dim = c->hidden_dim;
  d.encoder_lr = c->encoder_lr; d.actor_lr = c->actor_lr; d.critic_lr = c->critic_lr;
  d.tau = c->tau; d.stddev_clip = c->stddev_clip; d.precision = c->precision;
  *out = create_pixel<rlrep_drq, DrqV2>(d, stream);
  RLREP_API_END
}
int rlrep_drq_destroy(rlrep_drq* drq) { return pixel_destroy(drq); }
int rlrep_drq_num_tensors(rlrep_drq* drq, int* n) { return pixel_num_tensors(drq, n); }
int rlrep_drq_tensor_info(rlrep_drq* drq, int i, const char** name, float** ptr_dev, int* rows, int* cols) {
  return pixel_tensor_info(drq, i, name, ptr_dev, rows, cols);
}
int rlrep_drq_tensor_read(rlrep_drq* drq, int i, float* out_host) { return pixel_tensor_read(drq, i, out_host); }
int rlrep_drq_tensor_write(rlrep_drq* drq, int i, const float* in_host) { return pixel_tensor_write(drq, i, in_host); }
int rlrep_drq_sync_targets(rlrep_drq* drq) { return pixel_sync_targets(drq); }
int rlrep_drq_update(rlrep_drq* drq, const unsigned char* img, const float* action, const float* reward,
                     const float* discount, const unsigned char* next_img, const int* shifts, const float* eps,
                     float stddev, float* metrics_host) {
  RLREP_API_BEGIN_ON(drq)
  RLREP_CHECK(drq && img && action && reward && discount && next_img && shifts && eps && metrics_host, "null argument");
  drq->agent().update(img, action, reward, discount, next_img, shifts, eps, stddev, metrics_host);
  RLREP_API_END
}
int rlrep_drq_act(rlrep_drq* drq, const unsigned char* obs_host, const float* eps_host, float stddev, float* action_host) {
  return rlrep_drq_act_batch(drq, obs_host, eps_host, stddev, 1, action_host);
}
int rlrep_drq_act_batch(rlrep_drq* drq, const unsigned char* obs, const float* eps_host, float stddev, int n,
                        float* actions_host) {
  RLREP_API_BEGIN_ON(drq)
  RLREP_CHECK(drq && obs && actions_host, "null argument");
  RLREP_CHECK(n > 0, "n must be positive");
  drq->agent().act_batch(obs, eps_host, stddev, n, actions_host);
  RLREP_API_END
}
int rlrep_drq_update_resident(rlrep_drq* drq, int n_steps, float stddev, float* total_ms) {
  return pixel_update_resident(drq, n_steps, stddev, total_ms);
}
int rlrep_drq_profile_update(rlrep_drq* drq, float stddev, int max_entries, const char** names, float* ms, double* bytes,
                             double* flops, int* n_entries) {
  return pixel_profile_update(drq, stddev, max_entries, names, ms, bytes, flops, n_entries);
}
int rlrep_drq_last_launches(rlrep_drq* drq, int* launches) { return pixel_last_launches(drq, launches); }
int rlrep_drq_get_optim_state(rlrep_drq* drq, rlrep_optim_state* out) { return pixel_get_optim_state(drq, out); }
int rlrep_drq_set_optim_state(rlrep_drq* drq, const rlrep_optim_state* in) {
  return pixel_set_optim_state(drq, in);
}

int rlrep_mulv_create(const rlrep_mulv_config* c, void* stream, rlrep_mulv** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(c != nullptr && out != nullptr, "null argument");
  MulvConfig d;
  d.batch = c->batch_size; d.channels = c->channels; d.height = c->height; d.action_dim = c->action_dim;
  d.feat_dim = c->feat_dim; d.hidden_dim = c->hidden_dim; d.num_noise = c->num_noise;
  d.lr = c->lr; d.tau = c->tau; d.stddev_clip = c->stddev_clip; d.vae_w = c->vae_w; d.mse_w = c->mse_w;
  d.c_noise = c->c_noise; d.precision = c->precision;
  *out = create_pixel<rlrep_mulv, MulvDrq>(d, stream);
  RLREP_API_END
}
int rlrep_mulv_destroy(rlrep_mulv* h) { return pixel_destroy(h); }
int rlrep_mulv_num_tensors(rlrep_mulv* h, int* n) { return pixel_num_tensors(h, n); }
int rlrep_mulv_tensor_info(rlrep_mulv* h, int i, const char** name, float** ptr_dev, int* rows, int* cols) {
  return pixel_tensor_info(h, i, name, ptr_dev, rows, cols);
}
int rlrep_mulv_tensor_read(rlrep_mulv* h, int i, float* out_host) { return pixel_tensor_read(h, i, out_host); }
int rlrep_mulv_tensor_write(rlrep_mulv* h, int i, const float* in_host) { return pixel_tensor_write(h, i, in_host); }
int rlrep_mulv_sync_targets(rlrep_mulv* h) { return pixel_sync_targets(h); }
int rlrep_mulv_update(rlrep_mulv* h, const unsigned char* img, const float* action, const float* reward,
                      const float* discount, const unsigned char* next_img, const unsigned char* img_step1,
                      const int* shifts, const float* eps_z, const float* eps_act, const float* noise, float stddev,
                      float* metrics_host) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && img && action && reward && discount && next_img && img_step1 && shifts && eps_z && eps_act && noise &&
                  metrics_host, "null argument");
  h->agent().update(img, action, reward, discount, next_img, img_step1, shifts, eps_z, eps_act, noise, stddev,
                    metrics_host);
  RLREP_API_END
}
int rlrep_mulv_act(rlrep_mulv* h, const unsigned char* obs_host, const float* eps_host, float stddev, float* action_host) {
  return rlrep_mulv_act_batch(h, obs_host, eps_host, stddev, 1, action_host);
}
int rlrep_mulv_act_batch(rlrep_mulv* h, const unsigned char* obs, const float* eps_host, float stddev, int n,
                         float* actions_host) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && obs && actions_host, "null argument");
  RLREP_CHECK(n > 0, "n must be positive");
  h->agent().act_batch(obs, eps_host, stddev, n, actions_host);
  RLREP_API_END
}
int rlrep_mulv_update_resident(rlrep_mulv* h, int n_steps, float stddev, float* total_ms) {
  return pixel_update_resident(h, n_steps, stddev, total_ms);
}
int rlrep_mulv_profile_update(rlrep_mulv* h, float stddev, int max_entries, const char** names, float* ms, double* bytes,
                              double* flops, int* n_entries) {
  return pixel_profile_update(h, stddev, max_entries, names, ms, bytes, flops, n_entries);
}
int rlrep_mulv_last_launches(rlrep_mulv* h, int* launches) { return pixel_last_launches(h, launches); }
int rlrep_mulv_get_optim_state(rlrep_mulv* h, rlrep_optim_state* out) { return pixel_get_optim_state(h, out); }
int rlrep_mulv_set_optim_state(rlrep_mulv* h, const rlrep_optim_state* in) {
  return pixel_set_optim_state(h, in);
}

int rlrep_ldiff_create(const rlrep_ldiff_config* c, void* stream, rlrep_ldiff** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(c != nullptr && out != nullptr, "null argument");
  LdiffConfig d;
  d.batch = c->batch_size; d.action_dim = c->action_dim; d.latent = c->latent_dim; d.feat = c->feature_dim; d.bn = c->bn_dim;
  d.psi_h = c->psi_hidden_dim; d.psi_d = c->psi_hidden_depth; d.zeta_h = c->zeta_hidden_dim; d.zeta_d = c->zeta_hidden_depth;
  d.hidden = c->hidden_dim; d.ae_lr = c->ae_lr; d.score_lr = c->score_lr; d.actor_lr = c->actor_lr; d.critic_lr = c->critic_lr;
  d.weight_decay = c->weight_decay; d.tau = c->tau; d.kl_coef = c->kl_coef; d.ae_coef = c->ae_coef;
  d.stddev_clip = c->stddev_clip; d.precision = c->precision;
  *out = create_pixel<rlrep_ldiff, LatentDiffSR>(d, stream);
  RLREP_API_END
}
int rlrep_ldiff_destroy(rlrep_ldiff* h) { return pixel_destroy(h); }
int rlrep_ldiff_num_tensors(rlrep_ldiff* h, int* n) { return pixel_num_tensors(h, n); }
int rlrep_ldiff_tensor_info(rlrep_ldiff* h, int i, const char** name, float** ptr_dev, int* rows, int* cols) {
  return pixel_tensor_info(h, i, name, ptr_dev, rows, cols);
}
int rlrep_ldiff_tensor_read(rlrep_ldiff* h, int i, float* out_host) { return pixel_tensor_read(h, i, out_host); }
int rlrep_ldiff_tensor_write(rlrep_ldiff* h, int i, const float* in_host) { return pixel_tensor_write(h, i, in_host); }
int rlrep_ldiff_sync_targets(rlrep_ldiff* h) { return pixel_sync_targets(h); }
int rlrep_ldiff_update(rlrep_ldiff* h, const rlrep_ldiff_inputs* in, float* metrics_host) {
  RLREP_API_BEGIN_ON(h)
  RLREP_CHECK(h && in && metrics_host, "null argument");
  LatentDiffSR::Inputs x;
  x.frames = in->frames; x.next_frames = in->next_frames; x.shifts = in->shifts; x.next_shifts = in->next_shifts;
  x.action = in->action; x.reward = in->reward; x.discount = in->discount; x.eps_post = in->eps_post;
  x.alphabar = in->alphabar; x.temb = in->temb; x.noise = in->noise; x.psi_masks = in->psi_masks;
  x.zeta_masks = in->zeta_masks; x.eps_act = in->eps_act; x.stddev = in->stddev;
  RLREP_CHECK(x.frames && x.next_frames && x.shifts && x.next_shifts && x.action && x.reward && x.discount && x.eps_post &&
                  x.alphabar && x.temb && x.noise && x.psi_masks && x.zeta_masks && x.eps_act, "null input pointer");
  h->agent().update(x, metrics_host);
  RLREP_API_END
}
int rlrep_ldiff_update_resident(rlrep_ldiff* h, int n_steps, float stddev, float* total_ms) {
  return pixel_update_resident(h, n_steps, stddev, total_ms);
}
int rlrep_ldiff_profile_update(rlrep_ldiff* h, float stddev, int max_entries, const char** names, float* ms, double* bytes,
                               double* flops, int* n_entries) {
  return pixel_profile_update(h, stddev, max_entries, names, ms, bytes, flops, n_entries);
}
int rlrep_ldiff_last_launches(rlrep_ldiff* h, int* launches) { return pixel_last_launches(h, launches); }
int rlrep_ldiff_get_optim_state(rlrep_ldiff* h, rlrep_optim_state* out) { return pixel_get_optim_state(h, out); }
int rlrep_ldiff_set_optim_state(rlrep_ldiff* h, const rlrep_optim_state* in) {
  return pixel_set_optim_state(h, in);
}

// ------------------------------------------------------------------------------------------------ communicator
// ------------------------------------------------------------------------------------------------ pixel replay ring
struct rlrep_pixring {
  int device = current_device();
  std::unique_ptr<PixelRing> impl;
  cudaStream_t stream = nullptr;
};

int rlrep_pixring_create(long long capacity, int frame_bytes, int action_dim, int frame_stack, int nstep, rlrep_pixring** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(out != nullptr, "null argument");
  std::unique_ptr<rlrep_pixring> h(new rlrep_pixring);
  RLREP_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  h->impl.reset(new PixelRing(capacity, frame_bytes, action_dim, frame_stack, nstep));
  *out = h.release();
  RLREP_API_END
}
int rlrep_pixring_destroy(rlrep_pixring* ring) {
  RLREP_API_BEGIN_ON(ring)
  if (ring) {
    ring->impl.reset();
    if (ring->stream) cudaStreamDestroy(ring->stream);
    delete ring;
  }
  RLREP_API_END
}
int rlrep_pixring_write(rlrep_pixring* ring, long long slot, int copies, const unsigned char* frame_host,
                        const float* action_host, float reward, float discount, int has_step) {
  RLREP_API_BEGIN_ON(ring)
  RLREP_CHECK(ring, "null argument");
  ring->impl->write(slot, copies, frame_host, action_host, reward, discount, has_step != 0, ring->stream);
  RLREP_API_END
}
int rlrep_pixring_flush(rlrep_pixring* ring) {
  RLREP_API_BEGIN_ON(ring)
  RLREP_CHECK(ring, "null argument");
  ring->impl->flush(ring->stream);
  RLREP_API_END
}
int rlrep_pixring_gather(rlrep_pixring* ring, const int64_t* idx_host, int n, const float* discount_vec_host, float next_dis,
                         unsigned char* obs_dev, float* act_dev, float* rew_dev, float* dis_dev, unsigned char* nobs_dev,
                         unsigned char* sobs_dev) {
  RLREP_API_BEGIN_ON(ring)
  RLREP_CHECK(ring, "null argument");
  ring->impl->gather(reinterpret_cast<const long long*>(idx_host), n, discount_vec_host, next_dis, obs_dev, act_dev, rew_dev,
                     dis_dev, nobs_dev, sobs_dev, ring->stream);
  RLREP_CUDA(cudaStreamSynchronize(ring->stream));  // the batch is complete when the call returns, whatever stream reads it
  RLREP_API_END
}

int rlrep_comm_unique_id(unsigned char* out128) {
  RLREP_API_BEGIN
  RLREP_CHECK(out128 != nullptr, "null argument");
  Comm::unique_id(out128);
  RLREP_API_END
}
int rlrep_comm_create(const unsigned char* id128, int rank, int world, rlrep_comm** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(id128 != nullptr && out != nullptr, "null argument");
  std::unique_ptr<rlrep_comm> c(new rlrep_comm);
  c->impl.reset(new Comm(id128, rank, world));
  *out = c.release();
  RLREP_API_END
}
int rlrep_comm_destroy(rlrep_comm* comm) {
  RLREP_API_BEGIN_ON(comm)
  delete comm;
  RLREP_API_END
}
int rlrep_comm_info(rlrep_comm* comm, int* rank, int* world, int* nccl_version, long long* collectives) {
  RLREP_API_BEGIN_ON(comm)
  RLREP_CHECK(comm != nullptr, "null argument");
  if (rank) *rank = comm->impl->rank;
  if (world) *world = comm->impl->world;
  if (nccl_version) *nccl_version = Comm::version();
  if (collectives) *collectives = comm->impl->collectives;
  RLREP_API_END
}

static int create_agent(const rlrep_agent_config* c, rlrep_comm* comm, void* stream, rlrep_agent** out);

int rlrep_agent_create(const rlrep_agent_config* c, void* stream, rlrep_agent** out) {
  return create_agent(c, nullptr, stream, out);
}
int rlrep_agent_create_sharded(const rlrep_agent_config* c, rlrep_comm* comm, void* stream, rlrep_agent** out) {
  if (comm == nullptr) {
    set_last_error("rlrep_agent_create_sharded: null communicator");
    return 1;
  }
  return create_agent(c, comm, stream, out);
}

static AgentConfig agent_config(const rlrep_agent_config* c) {
  AgentConfig a;
  a.alg = c->alg;
  a.state_dim = c->state_dim; a.action_dim = c->action_dim; a.batch = c->batch_size;
  a.hidden_dim = c->hidden_dim; a.feature_dim = c->feature_dim; a.actor_hidden_dim = c->actor_hidden_dim;
  a.k_feat = c->feature_steps;
  a.lr = c->lr_critic; a.lr_feat = c->lr_feature; a.lr_actor = c->lr_actor; a.lr_alpha = c->lr_alpha;
  a.discount = c->discount; a.tau = c->tau; a.feature_tau = c->feature_tau;
  a.alpha0 = c->alpha;
  a.target_update_period = c->target_update_period;
  a.learn_alpha = c->auto_entropy_tuning;
  a.use_feature_target = c->use_feature_target;
  a.precision = c->precision;
  a.use_graph = c->use_cuda_graph;
  a.phi_hidden_dim = c->phi_hidden_dim; a.phi_hidden_depth = c->phi_hidden_depth;
  a.mu_hidden_dim = c->mu_hidden_dim; a.mu_hidden_depth = c->mu_hidden_depth;
  a.nabla_hidden_dim = c->nabla_mu_hidden_dim; a.nabla_hidden_depth = c->nabla_mu_hidden_depth;
  a.num_noise = c->num_noise; a.num_noises = c->num_noises;
  a.sigma_scale = c->sigma_scale_factor;
  RLREP_CHECK(a.target_update_period > 0, "target_update_period must be positive");
  return a;
}

// The handle runs on `stream`; the legacy default stream cannot be captured into a CUDA graph, so for a null `stream` the
// handle gets a private one.  Every entry point that hands results back to the host synchronises it, so callers never
// observe the difference.
static cudaStream_t handle_stream(rlrep_agent* h, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (st == nullptr) {
    RLREP_CUDA(cudaStreamCreateWithFlags(&h->owned_stream, cudaStreamNonBlocking));
    st = h->owned_stream;
  }
  return st;
}

static int create_agent(const rlrep_agent_config* c, rlrep_comm* comm, void* stream, rlrep_agent** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(c != nullptr && out != nullptr, "null argument");
  const AgentConfig a = agent_config(c);
  std::unique_ptr<rlrep_agent> h(new rlrep_agent);
  cudaStream_t st = handle_stream(h.get(), stream);
  if (comm != nullptr) {
    RLREP_CHECK(a.alg == RLREP_ALG_CTRLSAC, "batch sharding is implemented for ctrlsac (the path with a B x B exchange)");
    h->impl = make_ctrlsac_sharded_agent(a, st, comm->impl.get());
  } else switch (a.alg) {
    case RLREP_ALG_SAC: h->impl = make_sac_agent(a, st); break;
    case RLREP_ALG_CTRLSAC: h->impl = make_ctrlsac_agent(a, st); break;
    case RLREP_ALG_VLSAC: h->impl = make_vlsac_agent(a, st); break;
    case RLREP_ALG_SPEDERSAC: h->impl = make_spedersac_agent(a, st); break;
    case RLREP_ALG_DIFFSRSAC: h->impl = make_diffsrsac_agent(a, st); break;
    default: throw Error("algorithm not implemented in this build");
  }
  index_tensors(h.get());
  *out = h.release();
  RLREP_API_END
}
int rlrep_agent_destroy(rlrep_agent* agent) {
  RLREP_API_BEGIN_ON(agent)
  if (agent && agent->impl) cudaStreamSynchronize(agent->impl->stream);
  if (agent) {
    agent->impl.reset();
    if (agent->owned_stream) cudaStreamDestroy(agent->owned_stream);
  }
  delete agent;
  RLREP_API_END
}
int rlrep_agent_num_tensors(rlrep_agent* agent, int* n) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && n, "null argument");
  *n = (int)agent->tensors.size();
  RLREP_API_END
}
int rlrep_agent_tensor_info(rlrep_agent* agent, int i, const char** name, float** ptr_dev, int* rows, int* cols) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent, "null argument");
  tensor_info(agent->tensors, i, name, ptr_dev, rows, cols);
  RLREP_API_END
}
int rlrep_agent_tensor_read(rlrep_agent* agent, int i, float* out_host) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent, "null argument");
  tensor_read(agent->tensors, i, out_host, agent->impl->stream);
  RLREP_API_END
}
int rlrep_agent_tensor_write(rlrep_agent* agent, int i, const float* in_host) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent, "null argument");
  tensor_write(agent->tensors, i, in_host, agent->impl->stream);
  RLREP_API_END
}
int rlrep_agent_get_log_alpha(rlrep_agent* agent, double* log_alpha) {
  RLREP_API_BEGIN_ON(agent)
  Control h;
  RLREP_CUDA(cudaMemcpyAsync(&h, agent->impl->ctl, sizeof(h), cudaMemcpyDeviceToHost, agent->impl->stream));
  RLREP_CUDA(cudaStreamSynchronize(agent->impl->stream));
  *log_alpha = h.log_alpha;
  RLREP_API_END
}
int rlrep_agent_set_log_alpha(rlrep_agent* agent, double log_alpha) {
  RLREP_API_BEGIN_ON(agent)
  Control h;
  cudaStream_t st = agent->impl->stream;
  RLREP_CUDA(cudaMemcpyAsync(&h, agent->impl->ctl, sizeof(h), cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  h.log_alpha = log_alpha;
  h.alpha = (float)std::exp(log_alpha);
  RLREP_CUDA(cudaMemcpyAsync(agent->impl->ctl, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_API_END
}
int rlrep_agent_get_optim_state(rlrep_agent* agent, rlrep_optim_state* out) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && out, "null argument");
  Control h;
  RLREP_CUDA(cudaMemcpyAsync(&h, agent->impl->ctl, sizeof(h), cudaMemcpyDeviceToHost, agent->impl->stream));
  RLREP_CUDA(cudaStreamSynchronize(agent->impl->stream));
  out->steps = h.steps;
  out->t_feature = h.t_feat; out->t_critic = h.t_critic; out->t_actor = h.t_actor; out->t_alpha = h.t_alpha;
  out->log_alpha = h.log_alpha; out->log_alpha_m = h.la_m; out->log_alpha_v = h.la_v;
  RLREP_API_END
}
int rlrep_agent_set_optim_state(rlrep_agent* agent, const rlrep_optim_state* in) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && in, "null argument");
  Control h;
  cudaStream_t st = agent->impl->stream;
  RLREP_CUDA(cudaMemcpyAsync(&h, agent->impl->ctl, sizeof(h), cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  h.steps = in->steps;
  h.t_feat = in->t_feature; h.t_critic = in->t_critic; h.t_actor = in->t_actor; h.t_alpha = in->t_alpha;
  h.log_alpha = in->log_alpha; h.la_m = in->log_alpha_m; h.la_v = in->log_alpha_v;
  h.alpha = (float)std::exp(in->log_alpha);
  RLREP_CUDA(cudaMemcpyAsync(agent->impl->ctl, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_API_END
}
int rlrep_agent_get_steps(rlrep_agent* agent, int* steps) {
  RLREP_API_BEGIN_ON(agent)
  Control h;
  RLREP_CUDA(cudaMemcpyAsync(&h, agent->impl->ctl, sizeof(h), cudaMemcpyDeviceToHost, agent->impl->stream));
  RLREP_CUDA(cudaStreamSynchronize(agent->impl->stream));
  *steps = h.steps;
  RLREP_API_END
}
int rlrep_agent_train_counts(rlrep_agent* agent, int* n_idx, int* n_eps, int* n_metrics) {
  RLREP_API_BEGIN_ON(agent)
  *n_idx = agent->impl->idx_per_train();
  *n_eps = agent->impl->eps_per_train();
  *n_metrics = (int)agent->impl->metric_names().size();
  RLREP_API_END
}
const char* rlrep_agent_metric_name(rlrep_agent* agent, int i) {
  const auto& names = agent->impl->metric_names();
  if (i < 0 || i >= (int)names.size()) return nullptr;
  return names[i].c_str();
}
int rlrep_agent_train(rlrep_agent* agent, rlrep_ring* ring, const int64_t* idx_host, int n_idx, const float* eps_host,
                      int n_eps, float* metrics_host, int n_metrics) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && ring && idx_host && eps_host && metrics_host, "null argument");
  agent->impl->train(*ring->impl, reinterpret_cast<const long long*>(idx_host), n_idx, eps_host, n_eps, metrics_host,
                     n_metrics);
  RLREP_API_END
}
int rlrep_agent_act(rlrep_agent* agent, const float* state_host, const float* eps_host, float* action_host) {
  RLREP_API_BEGIN_ON(agent)
  agent->impl->act(state_host, eps_host, action_host);
  RLREP_API_END
}
int rlrep_agent_act_batch(rlrep_agent* agent, const float* states_host, const float* eps_host, int rows,
                          float* actions_host) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && states_host && actions_host && rows >= 0, "bad arguments");
  agent->impl->act_batch(states_host, eps_host, rows, actions_host);
  RLREP_API_END
}
int rlrep_agent_last_launches(rlrep_agent* agent, int* launches) {
  RLREP_API_BEGIN_ON(agent)
  *launches = agent->impl->last_launches;
  RLREP_API_END
}
int rlrep_agent_graph_stats(rlrep_agent* agent, int* kernel_nodes, int* programmatic_edges) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && kernel_nodes && programmatic_edges, "null argument");
  RLREP_CHECK(agent->impl->graph_stats(kernel_nodes, programmatic_edges),
              "no captured graph yet (train() captures it on its second call, with use_graph on)");
  RLREP_API_END
}
int rlrep_agent_train_resident(rlrep_agent* agent, rlrep_ring* ring, const int64_t* idx_host, const float* eps_host,
                               int n_steps, float* total_ms) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && ring && idx_host && eps_host && total_ms, "null argument");
  *total_ms = agent->impl->train_resident(*ring->impl, reinterpret_cast<const long long*>(idx_host), eps_host, n_steps);
  RLREP_API_END
}
int rlrep_agent_profile_train(rlrep_agent* agent, rlrep_ring* ring, const int64_t* idx_host, const float* eps_host,
                              int max_entries, const char** names, float* ms, double* bytes, double* flops,
                              int* n_entries) {
  RLREP_API_BEGIN_ON(agent)
  RLREP_CHECK(agent && ring && idx_host && eps_host && n_entries && (max_entries == 0 || (names && ms)), "null argument");
  std::vector<ProfileEntry> prof =
      agent->impl->profile_train(*ring->impl, reinterpret_cast<const long long*>(idx_host), eps_host);
  const int n = (int)std::min<size_t>(prof.size(), (size_t)max_entries);
  for (int i = 0; i < n; ++i) {
    names[i] = prof[i].name;  // string literals with static storage
    ms[i] = prof[i].ms;
    if (bytes) bytes[i] = prof[i].bytes;
    if (flops) flops[i] = prof[i].flops;
  }
  *n_entries = (int)prof.size();
  RLREP_API_END
}
int rlrep_agent_sync_targets(rlrep_agent* agent) {
  RLREP_API_BEGIN_ON(agent)
  agent->impl->sync_targets_from_params();
  RLREP_API_END
}

// ------------------------------------------------------------------------------------------------ SAC populations
struct rlrep_sacpop : rlrep_agent {};

static Members pop_members(rlrep_sacpop* p) { return p->impl->mb; }
static void check_member(rlrep_sacpop* p, int member) {
  RLREP_CHECK(member >= 0 && member < pop_members(p).n, "member index out of range");
}
static TensorRef member_tensor(rlrep_sacpop* p, int member, int i) {
  check_member(p, member);
  TensorRef t = tensor_at(p->tensors, i);
  t.ptr = member_ptr(t.ptr, member * pop_members(p).stride);
  return t;
}
static Control* member_control(rlrep_sacpop* p, int member) {
  check_member(p, member);
  return member_ptr(p->impl->ctl, member * pop_members(p).stride);
}
static std::vector<Ring*> member_rings(rlrep_sacpop* p, rlrep_ring* const* rings, int n_rings) {
  RLREP_CHECK(n_rings == pop_members(p).n, "one ring per member");
  std::vector<Ring*> out(n_rings);
  for (int m = 0; m < n_rings; ++m) {
    RLREP_CHECK(rings[m] != nullptr, "null argument");
    out[m] = rings[m]->impl.get();
  }
  return out;
}

int rlrep_sacpop_create(const rlrep_agent_config* c, int members, void* stream, rlrep_sacpop** out) {
  RLREP_API_BEGIN
  RLREP_CHECK(c != nullptr && out != nullptr, "null argument");
  RLREP_CHECK(c->alg == RLREP_ALG_SAC, "populations are implemented for sac");
  RLREP_CHECK(members >= 1, "a population needs at least one member");
  const AgentConfig a = agent_config(c);
  std::unique_ptr<rlrep_sacpop> h(new rlrep_sacpop);
  cudaStream_t st = handle_stream(h.get(), stream);
  h->impl = make_sac_population(a, st, members);
  index_tensors(h.get());
  *out = h.release();
  RLREP_API_END
}
int rlrep_sacpop_destroy(rlrep_sacpop* pop) {
  RLREP_API_BEGIN_ON(pop)
  if (pop && pop->impl) cudaStreamSynchronize(pop->impl->stream);
  if (pop) {
    pop->impl.reset();
    if (pop->owned_stream) cudaStreamDestroy(pop->owned_stream);
  }
  delete pop;
  RLREP_API_END
}
int rlrep_sacpop_members(rlrep_sacpop* pop, int* members) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && members, "null argument");
  *members = pop_members(pop).n;
  RLREP_API_END
}
int rlrep_sacpop_num_tensors(rlrep_sacpop* pop, int* n) { return rlrep_agent_num_tensors(pop, n); }
int rlrep_sacpop_tensor_info(rlrep_sacpop* pop, int member, int i, const char** name, float** ptr_dev, int* rows,
                             int* cols) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop, "null argument");
  const TensorRef t = member_tensor(pop, member, i);
  if (name) *name = tensor_at(pop->tensors, i).name.c_str();
  if (ptr_dev) *ptr_dev = t.ptr;
  if (rows) *rows = t.rows;
  if (cols) *cols = t.cols;
  RLREP_API_END
}
int rlrep_sacpop_tensor_read(rlrep_sacpop* pop, int member, int i, float* out_host) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && out_host, "null argument");
  tensor_read(member_tensor(pop, member, i), out_host, pop->impl->stream);
  RLREP_API_END
}
int rlrep_sacpop_tensor_write(rlrep_sacpop* pop, int member, int i, const float* in_host) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && in_host, "null argument");
  tensor_write(member_tensor(pop, member, i), in_host, pop->impl->stream);
  RLREP_API_END
}
int rlrep_sacpop_sync_targets(rlrep_sacpop* pop) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop, "null argument");
  pop->impl->sync_targets_from_params();
  RLREP_API_END
}
int rlrep_sacpop_get_optim_state(rlrep_sacpop* pop, int member, rlrep_optim_state* out) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && out, "null argument");
  Control h;
  RLREP_CUDA(cudaMemcpyAsync(&h, member_control(pop, member), sizeof(h), cudaMemcpyDeviceToHost, pop->impl->stream));
  RLREP_CUDA(cudaStreamSynchronize(pop->impl->stream));
  out->steps = h.steps;
  out->t_feature = h.t_feat; out->t_critic = h.t_critic; out->t_actor = h.t_actor; out->t_alpha = h.t_alpha;
  out->log_alpha = h.log_alpha; out->log_alpha_m = h.la_m; out->log_alpha_v = h.la_v;
  RLREP_API_END
}
int rlrep_sacpop_set_optim_state(rlrep_sacpop* pop, int member, const rlrep_optim_state* in) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && in, "null argument");
  Control* c = member_control(pop, member);
  cudaStream_t st = pop->impl->stream;
  Control h;
  RLREP_CUDA(cudaMemcpyAsync(&h, c, sizeof(h), cudaMemcpyDeviceToHost, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  h.steps = in->steps;
  h.t_feat = in->t_feature; h.t_critic = in->t_critic; h.t_actor = in->t_actor; h.t_alpha = in->t_alpha;
  h.log_alpha = in->log_alpha; h.la_m = in->log_alpha_m; h.la_v = in->log_alpha_v;
  h.alpha = (float)std::exp(in->log_alpha);
  RLREP_CUDA(cudaMemcpyAsync(c, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  RLREP_CUDA(cudaStreamSynchronize(st));
  RLREP_API_END
}
int rlrep_sacpop_train_counts(rlrep_sacpop* pop, int* n_idx, int* n_eps, int* n_metrics) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && n_idx && n_eps && n_metrics, "null argument");
  *n_idx = pop->impl->idx_per_train();
  *n_eps = pop->impl->eps_per_train();
  *n_metrics = (int)pop->impl->metric_names().size();
  RLREP_API_END
}
const char* rlrep_sacpop_metric_name(rlrep_sacpop* pop, int i) {
  if (pop == nullptr) {
    set_last_error("null argument");
    return nullptr;
  }
  return rlrep_agent_metric_name(pop, i);
}
int rlrep_sacpop_train(rlrep_sacpop* pop, rlrep_ring* const* rings, int n_rings, const int64_t* idx_host, int n_idx,
                       const float* eps, int n_eps, float* metrics_host, int n_metrics) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && rings && idx_host && eps && metrics_host, "null argument");
  const std::vector<Ring*> r = member_rings(pop, rings, n_rings);
  pop->impl->train_members(r.data(), reinterpret_cast<const long long*>(idx_host), n_idx, eps, n_eps, metrics_host,
                           n_metrics);
  RLREP_API_END
}
int rlrep_sacpop_act(rlrep_sacpop* pop, const float* states_host, const float* eps_host, float* actions_host) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && states_host && actions_host, "null argument");
  pop->impl->act_members(states_host, eps_host, actions_host);
  RLREP_API_END
}
int rlrep_sacpop_train_resident(rlrep_sacpop* pop, rlrep_ring* const* rings, int n_rings, const int64_t* idx_host,
                                const float* eps_host, int n_steps, float* total_ms) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && rings && idx_host && eps_host && total_ms, "null argument");
  const std::vector<Ring*> r = member_rings(pop, rings, n_rings);
  *total_ms = pop->impl->train_resident_members(r.data(), reinterpret_cast<const long long*>(idx_host), eps_host, n_steps);
  RLREP_API_END
}
int rlrep_sacpop_last_launches(rlrep_sacpop* pop, int* launches) {
  RLREP_API_BEGIN_ON(pop)
  RLREP_CHECK(pop && launches, "null argument");
  *launches = pop->impl->last_launches;
  RLREP_API_END
}

}  // extern "C"

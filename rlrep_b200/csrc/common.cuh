// Shared host-side helpers: error propagation (every C-ABI call returns int, 0 = ok) and launch checks.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

namespace rlrep {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

struct Error : std::runtime_error {
  using std::runtime_error::runtime_error;
};

void set_last_error(const std::string& msg);
const char* get_last_error();

#define RLREP_CUDA(expr)                                                                              \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess) {                                                                          \
      throw ::rlrep::Error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" __FILE__ \
                           ":" + std::to_string(__LINE__) + ")");                                     \
    }                                                                                                 \
  } while (0)

#define RLREP_CHECK(cond, msg)                                                                           \
  do {                                                                                                   \
    if (!(cond)) {                                                                                       \
      throw ::rlrep::Error(std::string("check failed: " #cond " -- ") + (msg) + " (" __FILE__ ":" +    \
                           std::to_string(__LINE__) + ")");                                              \
    }                                                                                                    \
  } while (0)

// Every kernel launch goes through this: checks the launch, counts it (bench.py reports gpu_launches) and, when a
// profile is being recorded, drops a CUDA event behind it so per-kernel device time can be read back.
// `bytes` / `flops` = ALGORITHMIC work of the launch (operands read once, results written once; 2 flop per MAC), 0 when
// the kernel is latency-bound bookkeeping; bench.py turns them into per-kernel roofline fractions.
void note_launch(const char* name, cudaStream_t stream, double bytes = 0.0, double flops = 0.0);
long long launch_count();
#define RLREP_LAUNCHED(name, stream)          \
  do {                                        \
    RLREP_CUDA(cudaGetLastError());           \
    ::rlrep::note_launch(name, stream);       \
  } while (0)
#define RLREP_LAUNCHED_W(name, stream, bytes, flops)            \
  do {                                                          \
    RLREP_CUDA(cudaGetLastError());                             \
    ::rlrep::note_launch(name, stream, (bytes), (flops));       \
  } while (0)

// Programmatic dependent launch: the kernel may be scheduled while the previous kernel in `stream` is still running
// and must call ptx::pdl_wait() before it touches memory that kernel may read or write (ptx.cuh).  In a captured graph
// the edge from the previous kernel becomes a programmatic edge.
inline cudaLaunchAttribute pdl_attribute() {
  cudaLaunchAttribute a = {};
  a.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  a.val.programmaticStreamSerializationAllowed = 1;
  return a;
}
template <typename... KernelArgs, typename... Args>
void launch_pdl(void (*kernel)(KernelArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1] = {pdl_attribute()};
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  RLREP_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
}

// Per-kernel timing of an eager (non-graph) launch sequence: begin, run the launches, end -> (name, ms) per launch.
void profile_begin(cudaStream_t stream);
struct ProfileEntry {
  const char* name;
  float ms;
  double bytes, flops;
};
std::vector<ProfileEntry> profile_end(cudaStream_t stream);

// Wrap a C-ABI body: exceptions become error code + message.
#define RLREP_API_BEGIN try {
#define RLREP_API_END                              \
  return 0;                                        \
  }                                                \
  catch (const std::exception& ex) {               \
    ::rlrep::set_last_error(ex.what());            \
    return 1;                                      \
  }                                                \
  catch (...) {                                    \
    ::rlrep::set_last_error("unknown exception");  \
    return 2;                                      \
  }

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

}  // namespace rlrep

// Element-wise epilogue shared by the tcgen05 GEMM, its split-K reducer and the CUDA-core GEMM.
//
// For an accumulator value acc at (m, n) the epilogue computes, in this order:
//   v = acc * scale
//   v += r1_u[m] * r1_v[n]              (rank-1 term; reward-head gradient folded into d z_phi)
//   v += bias[n]
//   pre_out[m, n] = v                   (optional: keep the pre-activation, needed by sin layers)
//   v = act(v)                          (ELU / ReLU / tanh / sin -- reference: F.elu, F.relu, F.tanh, torch.sin)
//   v *= dact(aux[m, n])                (backward: multiply by the activation derivative of the layer below)
//   v += C[m, n]                        (optional accumulate)
#pragma once
#include <cuda_runtime.h>

#include "members.cuh"

namespace rlrep {

enum Act : int { ACT_NONE = 0, ACT_ELU = 1, ACT_RELU = 2, ACT_TANH = 3, ACT_SIN = 4 };
// Derivative selectors. *_OUT variants take the layer's OUTPUT as aux (ELU: y>0 ? 1 : y+1; ReLU: y>0;
// tanh: 1-y^2); DACT_COS_PRE takes the saved pre-activation of a sin layer.
enum DAct : int { DACT_NONE = 0, DACT_ELU_OUT = 1, DACT_RELU_OUT = 2, DACT_TANH_OUT = 3, DACT_COS_PRE = 4 };

struct Epilogue {
  const float* bias = nullptr;
  const float* r1_u = nullptr;
  const float* r1_v = nullptr;
  const float* aux = nullptr;
  float* pre_out = nullptr;
  int ld_aux = 0;
  int ld_pre = 0;
  int act = ACT_NONE;
  int dact = DACT_NONE;
  int accumulate = 0;
  float scale = 1.0f;
};

// The epilogue of a population member: every operand pointer moved by `off` bytes (members.cuh).
__host__ __device__ __forceinline__ Epilogue member_epilogue(Epilogue e, long long off) {
  e.bias = member_ptr(e.bias, off);
  e.r1_u = member_ptr(e.r1_u, off);
  e.r1_v = member_ptr(e.r1_v, off);
  e.aux = member_ptr(e.aux, off);
  e.pre_out = member_ptr(e.pre_out, off);
  return e;
}

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    // branch-free: behind a per-element branch the elements a thread holds cannot interleave their ~28-instruction
    // expm1f chains and the epilogue becomes latency-bound
    case ACT_ELU: {
      const float e = expm1f(fminf(v, 0.f));
      return v > 0.f ? v : e;
    }
    case ACT_RELU: return v > 0.f ? v : 0.f;
    case ACT_TANH: return tanhf(v);
    case ACT_SIN: return sinf(v);
    default: return v;
  }
}
__device__ __forceinline__ float apply_dact(float h, int dact) {
  switch (dact) {
    case DACT_ELU_OUT: return h > 0.f ? 1.f : h + 1.f;
    case DACT_RELU_OUT: return h > 0.f ? 1.f : 0.f;
    case DACT_TANH_OUT: return 1.f - h * h;
    case DACT_COS_PRE: return cosf(h);
    default: return 1.f;
  }
}

// One element. `cptr` points at C[m, n]; used only for accumulate.
// ACT / DACT >= 0 fix the activation / derivative at compile time (tight store loops: the transcendental code of
// the other cases is not even instantiated); -1 selects them at run time from the struct.
template <int ACT = -1, int DACT = -1>
__device__ __forceinline__ float epilogue_apply(const Epilogue& e, float acc, int m, int n, const float* cptr) {
  float v = acc * e.scale;
  if (e.r1_u) v = fmaf(__ldg(e.r1_u + m), __ldg(e.r1_v + n), v);
  if (e.bias) v += __ldg(e.bias + n);
  if (e.pre_out) e.pre_out[(size_t)m * e.ld_pre + n] = v;
  if constexpr (ACT < 0) v = apply_act(v, e.act);
  else if constexpr (ACT != ACT_NONE) v = apply_act(v, ACT);
  if constexpr (DACT < 0) {
    if (e.dact != DACT_NONE) v *= apply_dact(e.aux[(size_t)m * e.ld_aux + n], e.dact);
  } else if constexpr (DACT != DACT_NONE) {
    v *= apply_dact(e.aux[(size_t)m * e.ld_aux + n], DACT);
  }
  if (e.accumulate) v += *cptr;
  return v;
}

// Expands CALL(ACT, DACT) for the (activation, derivative) pair of `e`: the pairs the update step uses get a
// specialised instantiation, anything else the run-time version CALL(-1, -1).
#define RLREP_EPILOGUE_SWITCH(e, CALL)                                      \
  do {                                                                      \
    switch ((e).act * 8 + (e).dact) {                                       \
      case ACT_NONE * 8 + DACT_NONE: CALL(ACT_NONE, DACT_NONE); break;      \
      case ACT_ELU * 8 + DACT_NONE: CALL(ACT_ELU, DACT_NONE); break;        \
      case ACT_RELU * 8 + DACT_NONE: CALL(ACT_RELU, DACT_NONE); break;      \
      case ACT_TANH * 8 + DACT_NONE: CALL(ACT_TANH, DACT_NONE); break;      \
      case ACT_SIN * 8 + DACT_NONE: CALL(ACT_SIN, DACT_NONE); break;        \
      case ACT_NONE * 8 + DACT_ELU_OUT: CALL(ACT_NONE, DACT_ELU_OUT); break;    \
      case ACT_NONE * 8 + DACT_RELU_OUT: CALL(ACT_NONE, DACT_RELU_OUT); break;  \
      case ACT_NONE * 8 + DACT_TANH_OUT: CALL(ACT_NONE, DACT_TANH_OUT); break;  \
      case ACT_NONE * 8 + DACT_COS_PRE: CALL(ACT_NONE, DACT_COS_PRE); break;    \
      default: CALL(-1, -1); break;                                         \
    }                                                                       \
  } while (0)

}  // namespace rlrep

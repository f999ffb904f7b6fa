// Populations: N agents of one configuration (different seeds) in one handle, trained by one launch sequence.  Every
// member owns an identical copy of the agent's device arena, and the copies sit at a fixed byte stride in one
// allocation, so member m's copy of any buffer is the pointer member 0 uses plus m * stride.  A kernel launched for a
// population gets grid dimension z = members and offsets every arena pointer it is given by blockIdx.z * stride; a lone
// agent is the population of one (n = 1, stride = 0) and its kernels compute exactly what they computed before.
#pragma once
#include <cstdint>

namespace rlrep {

struct Members {
  int n = 1;
  long long stride = 0;  // bytes between consecutive members' arenas
};

// Byte offset of population member blockIdx.z.  Kernel bodies that take a member dimension are templates on MEMBERS:
// the lone-agent instantiation (MEMBERS = false) sees a compile-time 0 and compiles to the code without members.  (The
// GEMMs keep their lone kernels under their names and add separately named population kernels over the same body.)
template <bool MEMBERS>
__device__ __forceinline__ long long member_offset(long long stride) {
  if constexpr (MEMBERS) return blockIdx.z * stride;
  else return 0;
}

// p + off bytes; a null (absent optional operand) stays null.
template <typename T>
__host__ __device__ __forceinline__ T* member_ptr(T* p, long long off) {
  return p == nullptr ? p : reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(p) + off);
}

}  // namespace rlrep

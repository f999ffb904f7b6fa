// Small-batch policy of the pixel agents (see pixel_act.cu): encoder -> actor trunk -> policy MLP -> sample, for
// 1..kPixelActRows observations per pass, in IEEE fp32 whatever precision the owning handle trains in.
#pragma once
#include "agent.cuh"

namespace rlrep {

constexpr int kPixelActRows = 64;  // observations per pass (fewer only for frames far above 84 px); larger batches run
                                   // in chunks of this many

// Views of the owner's parameters, read in place at every act (so acting always sees the latest update).
struct PixelPolicyWeights {
  Linear conv[4];            // ConvEncoder::layer(l): layer 1 [32, C*9] (reference layout), layers 2-4 [32, (ky, kx, c)]
  Linear trunk;              // actor.trunk.0 [bn, F], rows zero-padded to out_alloc
  const float* ln_w = nullptr;  // actor.trunk.1 (LayerNorm, eps 1e-5) + tanh
  const float* ln_b = nullptr;
  Linear policy[3];          // actor.policy.0 / .2 / .4
};

class PixelPolicy {
 public:
  PixelPolicy(int channels, int height, int action_dim, const PixelPolicyWeights& w, cudaStream_t s);
  ~PixelPolicy();
  PixelPolicy(const PixelPolicy&) = delete;
  PixelPolicy& operator=(const PixelPolicy&) = delete;

  // obs uint8 [n, C, H, H] in host or device memory; eps_host [n, A] standard normal draws, or nullptr for the mean
  // (deterministic); stddev = schedule(step).  actions_host [n, A] = TruncatedNormal(mu, stddev).sample(clip=None).
  // Each observation's action depends on that observation (and its eps row) only, bit for bit: not on n, nor on its
  // position in the batch.
  void act(const unsigned char* obs, const float* eps_host, float stddev, int n, float* actions_host);

 private:
  void reserve(int rows);
  void forward(int rows, float stddev);

  int C_, H_, A_, LA_, bn_, LB_, hid_;
  int hw_[4] = {0, 0, 0, 0};
  size_t frame_bytes_;
  PixelPolicyWeights w_;
  cudaStream_t stream_;
  GemmRunner gemm_;  // PREC_FP32: the policy MLP runs on the exact-fp32 SIMT GEMMs
  int chunk_ = kPixelActRows;  // observations per pass
  int jg_ = 0;                 // trunk weight rows per shared-memory pass
  int cap_ = 0;                // rows the arena holds (0 until the first act)
  DeviceArena arena_;
  unsigned char* frames_ = nullptr;
  float *act_a_ = nullptr, *act_b_ = nullptr, *feat_ = nullptr, *partial_ = nullptr, *th_ = nullptr;
  float *h1_ = nullptr, *h2_ = nullptr, *raw_ = nullptr, *mu_ = nullptr, *eps_ = nullptr, *action_ = nullptr;
  unsigned char* stage_host_ = nullptr;  // pinned: frames then eps of one chunk
  float* out_host_ = nullptr;            // pinned: actions of one chunk
};

}  // namespace rlrep

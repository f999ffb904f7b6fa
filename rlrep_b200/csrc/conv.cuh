// DrQ-v2 pixel encoder handle (see conv.cu).
#pragma once
#include "agent.cuh"
#include "conv_implicit.cuh"

namespace rlrep {

class ConvEncoder {
 public:
  // with_target: the group also carries a Polyak target copy of all four layers (muLV-Rep's encoder_target)
  ConvEncoder(int batch, int in_channels, int height, Precision prec, cudaStream_t s, bool with_target = false);
  // obs uint8 [B, C, H, H] (device), shifts int32 [B, 2] = (x, y) in [0, 8] or nullptr (no augmentation);
  // feat fp32 [B, 32 * 35 * 35] in the reference's flatten order (channel, row, column), row pitch ld_feat (0 = dense);
  // target = true runs the target copy of the weights; no_grad = true promises that no backward() follows this
  // forward (layers 2-4 then run as implicit convolutions, without column matrices)
  void forward(const unsigned char* obs_dev, const int* shifts_dev, float* feat_dev, int ld_feat = 0, bool target = false,
               bool no_grad = false);
  // dfeat [B, 32 * 35 * 35] (row pitch ld_dfeat) -> dW / db of the four layers (activations of the last forward are
  // reused, so that forward must have run with target = false and no_grad = false; anything else is refused)
  void backward(const float* dfeat_dev, int ld_dfeat = 0);

  // Read-only views of the internal maps, for kernel-level tests: act(l) [B, hw(l), hw(l), 32] is the post-ReLU output
  // of layer l (last forward), dact(l) the gradient with respect to its pre-activation, ReLU mask applied (last backward).
  int hw(int l) const { return hw_[l]; }
  const float* act(int l) const { return act_[l]; }
  const float* dact(int l) const { return dact_[l]; }

  int batch() const { return B_; }
  int feature_dim() const { return 32 * hw_[3] * hw_[3]; }
  int layer_k(int l) const { return l == 0 ? K1_ : 288; }
  Linear layer(int l) const { return conv_[l].view(g_); }
  cudaStream_t stream() const { return stream_; }
  ParamGroup& group() { return g_; }  // p | g | m | v of the four conv layers (the owner runs Adam over it)
  long long rows(int l) const { return (long long)B_ * hw_[l] * hw_[l]; }

 private:
  int B_, C_, H_, K1_ = 0, ldk1_ = 0;
  int hw_[4] = {0, 0, 0, 0};
  cudaStream_t stream_;
  DeviceArena arena_;
  GemmRunner gemm_;
  ParamGroup g_;
  LinearSlot conv_[4];
  float* col_[4] = {nullptr, nullptr, nullptr, nullptr};
  float* act_[4] = {nullptr, nullptr, nullptr, nullptr};
  float* dact_[4] = {nullptr, nullptr, nullptr, nullptr};
  // layers 2-4 without column matrices at all (TF32 path, B % 4 == 0): implicit forward convolution and the implicit
  // weight gradient of GemmArgs::conv_wgrad_hi; otherwise explicit im2col + folded GEMM
  bool implicit_wgrad_ = false;
  // the last forward ran the online weights with gradients: act_ (and on the explicit path every col_) hold the maps of
  // the input backward() differentiates.  A target / no_grad forward overwrites them with another input's.
  bool backward_ready_ = false;
  FullCorrScratch corr_;
  static constexpr int kBiasChunks = 296;  // 2 x 148 SMs
  float* bias_partial_ = nullptr;
  static constexpr int kFold = 4;  // rows folded per GEMM row in the weight-gradient GEMMs (conv.cu backward())
  float* wfold_ = nullptr;
};

}  // namespace rlrep

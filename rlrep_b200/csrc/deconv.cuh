// muLV-Rep pixel decoder handle (see deconv.cu).
#pragma once
#include "agent.cuh"
#include "conv_implicit.cuh"

namespace rlrep {

class ConvDecoder {
 public:
  // out_kernel 2: muLV-Rep (..., ConvT s2 41 -> 83, Conv2d k2 p1); 3: latent Diff-SR VAE (ConvT s2 + output_padding 1
  // 41 -> 84, Conv2d k3 p1).  with_target: the group also carries a Polyak target copy (vae_target.decoder).
  ConvDecoder(int batch, Precision prec, cudaStream_t s, int out_kernel = 2, bool with_target = false);
  // x fp32 [B, 32 * 35 * 35] in the reference's (channel, row, column) order, row pitch ld_x -> prediction [B, 3, 84, 84]
  // kept inside the handle (read it with copy_pred)
  void forward(const float* x_dev, int ld_x);
  // s_loss = 10 * mean |pred - (target / 255 - 0.5)| (drqv2.py:359-362); target uint8 [B, 3, 84, 84].  Leaves
  // d loss / d pred * grad_scale inside the handle for backward(); loss_out[0] = s_loss.
  void l1_loss(const unsigned char* target_dev, float grad_scale, float* loss_out_dev);
  // recon_loss = sum((pred - (frame / 255 - 0.5))^2) / B (latent_diff_sr.py:242); frame = uint8 [B, 3, 84, 84] looked up
  // through the per-frame augmentation shift (int32 [B, 2], (x, y) in [0, 8]; nullptr = none)
  void mse_sum_loss(const unsigned char* target_dev, const int* shifts_dev, float grad_scale, float* loss_out_dev);
  // parameter gradients of the five layers and dx [B, 32 * 35 * 35] (row pitch ld_dx)
  void backward(float* dx_dev, int ld_dx);
  void copy_pred(float* pred_nchw_dev, bool grad = false);  // [B, 3, 84, 84]; grad: d loss / d pred * grad_scale instead

  ParamGroup& group() { return g_; }
  int batch() const { return B_; }
  int out_kernel() const { return ks_; }
  cudaStream_t stream() const { return stream_; }

  // Read-only views of the internal maps, for kernel-level tests: act(i) [B, hw(i), hw(i), 32] is layer i's input
  // (i = 0: the decoder input); dact(i) the gradient with respect to it, ReLU mask applied for i > 0.  Weight / bias
  // offsets l = 0..4 index group().p and group().g.
  int hw(int i) const { return hw_[i]; }
  const float* act(int i) const { return act_[i]; }
  const float* dact(int i) const { return dact_[i]; }
  size_t weight_offset(int l) const { return w_off_[l]; }
  size_t bias_offset(int l) const { return b_off_[l]; }

 private:
  long long rows(int i) const { return (long long)B_ * hw_[i] * hw_[i]; }
  Linear layer(int l) const;

  static constexpr int kLossBlocks = 592;  // 4 x 148 SMs
  int B_, ks_ = 2;
  int hw_[6] = {35, 37, 39, 41, 83, 84};  // act_[i] is [B, hw_[i], hw_[i], 32]; the prediction is [B, 84, 84, 3(+1)]
  cudaStream_t stream_;
  DeviceArena arena_;
  GemmRunner gemm_;
  ParamGroup g_;
  size_t w_off_[5] = {0, 0, 0, 0, 0}, b_off_[5] = {0, 0, 0, 0, 0};
  float* act_[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  float* dact_[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  float *col_ = nullptr, *pred_ = nullptr, *dpred_ = nullptr, *loss_partial_ = nullptr, *wg_partial_ = nullptr;
  float* bias_partial_ = nullptr;
  static constexpr int kBiasChunks = 296;
  // CTAs of the output layer's weight-gradient pass: 6 per SM for the 3x3 kernel (two waves of the 3 CTAs an SM holds,
  // measured 1253 -> 762 us at 1024 frames), 4 per SM for the 2x2 kernel (fewer rows per warp there: 134 vs 184 us)
  static constexpr int kWgBlocks = 888, kWgBlocks2 = 592;
  static constexpr int kFold = 4;  // rows folded per GEMM row in the weight-gradient GEMMs (deconv.cu backward())
  float* wfold_ = nullptr;
  bool implicit_bwd_ = false;
  FullCorrScratch corr_;
};

}  // namespace rlrep

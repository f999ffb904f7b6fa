// Plain DrQ-v2 pixel agent handle (see agent_drqv2.cu).
#pragma once
#include <memory>

#include "pixel_agent.cuh"

namespace rlrep {

struct DrqConfig {
  int batch = 256, channels = 9, height = 84, action_dim = 4, bn_dim = 50, hidden_dim = 1024;
  double encoder_lr = 1e-4, actor_lr = 1e-4, critic_lr = 1e-4;
  float tau = 0.01f, stddev_clip = 0.3f;
  int precision = PREC_TF32;
};

class DrqV2 : public PixelAgent {
 public:
  DrqV2(const DrqConfig& c, cudaStream_t s);

  // One `train_step` that updates (the caller implements `update_every`).  Host buffers: img / next_img uint8
  // [B, C, H, H]; action [B, A]; reward, discount [B]; shifts int32 [2][B][2] (img then next_img; (x, y) in [0, 8]);
  // eps [2][B][A] standard normal draws (next action, actor step); stddev = schedule(step).
  // metrics_out[5] = {critic_loss, mean(q_pred), mean(q_target), mean(reward), actor_loss}.
  void update(const unsigned char* img, const float* action, const float* reward, const float* discount,
              const unsigned char* next_img, const int* shifts, const float* eps, float stddev, float* metrics_out);
  // select_action on n observations (PixelPolicy::act): obs uint8 [n, C, H, H] host or device; eps [n, A] standard normal
  // or nullptr (deterministic: the mean); actions [n, A].  Reads the current weights and no update buffer.
  // The policy's buffers are allocated by the first call: a handle that never acts allocates nothing for it.
  void act_batch(const unsigned char* obs, const float* eps_host, float stddev, int n, float* actions_host);
  std::vector<ParamGroup*> groups() override { return {&enc_->group(), &actor_g_, &crit_g_}; }
  std::string tensor_name(const ParamGroup& g, const std::string& t) const override {
    return &g == &enc_->group() ? "encoder." + t : t;
  }

 private:
  void launch_update(float stddev) override;
  void trunk_forward(const LinearSlot& t, const ParamGroup& g, bool target, size_t ln_w, size_t ln_b, const float* x,
                     float* pre, float* out, int ld_out, float* xhat, float* rstd);
  void q_forward(bool target, int set);
  void q_backward(int set, bool wgrad);
  void actor_forward(const float* latent, const float* eps, float stddev, int set, bool keep);

  DrqConfig cfg_;
  int B_, A_, bn_, H_, F_ = 0, LB_ = 0, LC_ = 0, LA_ = 0;
  std::unique_ptr<ConvEncoder> enc_;
  DeviceArena arena_;
  GemmRunner gemm_;
  ParamGroup crit_g_, actor_g_;
  LinearSlot ct_, q0_, q1a_, q1b_, q2a_, q2b_, at_, p0_, p1_, p2_;
  size_t cln_w_ = 0, cln_b_ = 0, aln_w_ = 0, aln_b_ = 0;
  unsigned char *img_dev_ = nullptr, *next_img_dev_ = nullptr;
  int* shifts_dev_ = nullptr;
  float *eps_dev_ = nullptr, *action_dev_ = nullptr, *reward_dev_ = nullptr, *discount_dev_ = nullptr;
  float *latent_ = nullptr, *next_latent_ = nullptr, *dlatent_ = nullptr;
  float *tpre_[2] = {nullptr, nullptr}, *cat_[2] = {nullptr, nullptr}, *hid0_[2] = {nullptr, nullptr};
  float *hid1_[2] = {nullptr, nullptr}, *q_[2] = {nullptr, nullptr};
  float *xhat_c_ = nullptr, *rstd_c_ = nullptr, *xhat_a_ = nullptr, *rstd_a_ = nullptr, *th_ = nullptr;
  float *ap1_ = nullptr, *ap2_ = nullptr, *raw_ = nullptr, *mu_ = nullptr, *dq_ = nullptr;
  float *dhid1_ = nullptr, *dhid0_ = nullptr, *dcat_ = nullptr, *dtpre_ = nullptr, *gb_ = nullptr, *gg_ = nullptr;
  float *draw_ = nullptr, *dap2_ = nullptr, *dap1_ = nullptr, *dth_ = nullptr;
  std::unique_ptr<PixelPolicy> policy_;
};

}  // namespace rlrep

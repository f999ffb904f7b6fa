// muLV-Rep DrQ-v2 pixel agent handle (see agent_mulvdrq.cu).
#pragma once
#include <memory>

#include "deconv.cuh"
#include "pixel_agent.cuh"

namespace rlrep {

struct MulvConfig {
  int batch = 256, channels = 9, height = 84, action_dim = 4, feat_dim = 100, hidden_dim = 1024, num_noise = 20;
  double lr = 1e-4;
  float tau = 0.01f, stddev_clip = 0.3f, vae_w = 0.5f, mse_w = 1.0f, c_noise = 0.1f;
  int precision = PREC_TF32;
};

// Stacked Gaussian head: [mean_linear.0 ; log_std_linear.0] as one [2 LF, in] matrix (each half padded to LF rows) plus
// the two LayerNorms.
struct GaussHead {
  LinearSlot lin;
  size_t g_mean = 0, b_mean = 0, g_ls = 0, b_ls = 0;
};
// Activations of one evaluation of a Gaussian head that will be differentiated.
struct GaussActs {
  float *pre = nullptr, *m = nullptr, *raw = nullptr, *xhat_m = nullptr, *xhat_s = nullptr, *rstd_m = nullptr,
        *rstd_s = nullptr;
};

class MulvDrq : public PixelAgent {
 public:
  MulvDrq(const MulvConfig& c, cudaStream_t s);

  // One `update` that steps (the caller implements `up_every`).  Host buffers: img / next_img uint8 [B, C, H, H];
  // img_step1 uint8 [B, 3, H, H] (the last frame of the one-step-ahead observation); action [B, A]; reward, discount [B];
  // shifts int32 [2][B][2] (img, next_img); eps_z [B, F]; eps_act [2][B][A] (next action, actor step);
  // noise [3][NN][F] (critic_target, critic, critic of the actor step); stddev = schedule(step).
  // metrics_out[8] = {critic_loss, mean(q1), mean(q2), mean(target_q), s_loss, r_loss, kl_loss, actor_loss}.
  void update(const unsigned char* img, const float* action, const float* reward, const float* discount,
              const unsigned char* next_img, const unsigned char* img_step1, const int* shifts, const float* eps_z,
              const float* eps_act, const float* noise, float stddev, float* metrics_out);
  // act (drqv2.py:270-282) on n observations (PixelPolicy::act): obs uint8 [n, C, H, H] host or device; eps [n, A]
  // standard normal or nullptr (eval_mode: the mean); actions [n, A].  Reads the current weights and no update buffer.
  // The policy's buffers are allocated by the first call: a handle that never acts allocates nothing for it.
  void act_batch(const unsigned char* obs, const float* eps_host, float stddev, int n, float* actions_host);
  std::vector<ParamGroup*> groups() override {
    return {&enc_->group(), &penc_->group(), &dec_->group(), &actor_g_, &crit_g_, &fe_g_, &fd_g_, &ff_g_};
  }
  std::string tensor_name(const ParamGroup& g, const std::string& t) const override {
    const bool conv_stack = &g == &enc_->group() || &g == &penc_->group() || &g == &dec_->group();
    return conv_stack ? g.name + "." + t : t;
  }

 private:
  void launch_update(float stddev) override;
  void gauss_forward(const GaussHead& h, const ParamGroup& g, bool target, Mat x, GaussActs& a, bool keep);
  void gauss_backward(const GaussHead& h, ParamGroup& g, Mat x, const GaussActs& a, const float* dm, const float* draw,
                      bool wgrad);
  void critic_forward(bool target, int slot, const float* m, const float* raw, const float* noise);
  void critic_backward(int slot, const float* raw, const float* noise, bool wgrad, float* dm, float* draw);
  void actor_forward(const float* latent, int ld_latent, const float* eps, float stddev, float* action_out, int ld_action,
                     bool keep);

  MulvConfig cfg_;
  int B_, A_, D_, H_, NN_, F_ = 0, LF_ = 0, LA_ = 0, LDE_ = 0, LDS_ = 0;
  std::unique_ptr<ConvEncoder> enc_, penc_;
  std::unique_ptr<ConvDecoder> dec_;
  DeviceArena arena_;
  GemmRunner gemm_;
  ParamGroup actor_g_, crit_g_, fe_g_, fd_g_, ff_g_;
  GaussHead fe_, ff_;
  LinearSlot at_, p0_, p1_, p2_, c14_, c2_, c5_, c3_, c6_, d1_, d2_, ds_, dr_;
  size_t aln_w_ = 0, aln_b_ = 0;
  unsigned char *img_dev_ = nullptr, *next_img_dev_ = nullptr, *step1_dev_ = nullptr;
  int* shifts_dev_ = nullptr;
  float *eps_z_dev_ = nullptr, *eps_act_dev_ = nullptr, *noise_dev_ = nullptr, *action_dev_ = nullptr;
  float *reward_dev_ = nullptr, *discount_dev_ = nullptr;
  float *enc_in_ = nullptr, *nsa_ = nullptr, *dstate_ = nullptr, *dstep1_ = nullptr;
  GaussActs ge_, gf_, gn_;
  float *z_ = nullptr, *dz_ = nullptr, *fh1_ = nullptr, *fh2_ = nullptr, *s_hat_ = nullptr, *ds_hat_ = nullptr;
  float *r_hat_ = nullptr, *dr_hat_ = nullptr, *dfh2_ = nullptr, *dfh1_ = nullptr, *kl_partial_ = nullptr;
  float *dm1_ = nullptr, *draw1_ = nullptr, *dm2_ = nullptr, *draw2_ = nullptr, *dcm_ = nullptr, *dcraw_ = nullptr;
  float *dpre_ = nullptr, *gb_ = nullptr, *gg_ = nullptr, *gb2_ = nullptr, *gg2_ = nullptr;
  float *xs_[2] = {nullptr, nullptr}, *hid1_[2] = {nullptr, nullptr}, *m20_[2] = {nullptr, nullptr};
  float *hid2_[2] = {nullptr, nullptr}, *q_[2] = {nullptr, nullptr};
  float *dq_ = nullptr, *dhid2_ = nullptr, *dm20_ = nullptr, *dhid1_ = nullptr, *bpart_ = nullptr, *dxs_ = nullptr;
  float *tpre_ = nullptr, *th_ = nullptr, *xhat_a_ = nullptr, *rstd_a_ = nullptr, *ap1_ = nullptr, *ap2_ = nullptr;
  float *raw_a_ = nullptr, *mu_ = nullptr, *daction_ = nullptr, *draw_a_ = nullptr, *dap2_ = nullptr, *dap1_ = nullptr;
  float *dth_ = nullptr, *dtpre_ = nullptr;
  static constexpr int kKlBlocks = 64;
  std::unique_ptr<PixelPolicy> policy_;
};

}  // namespace rlrep

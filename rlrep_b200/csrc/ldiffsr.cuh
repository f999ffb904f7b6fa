// Latent Diff-SR DrQ-v2 pixel agent handle (see agent_ldiffsr.cu).
#pragma once
#include <memory>

#include "deconv.cuh"
#include "nets.cuh"
#include "pixel_agent.cuh"

namespace rlrep {

struct LdiffConfig {
  int batch = 256, action_dim = 4, latent = 256, feat = 2048, bn = 512, psi_h = 512, psi_d = 2, zeta_h = 512, zeta_d = 4,
      hidden = 1024;
  double ae_lr = 3e-4, score_lr = 3e-4, actor_lr = 1e-4, critic_lr = 1e-4, weight_decay = 0.01;
  float tau = 0.01f, kl_coef = 1.0f, ae_coef = 1.0f, stddev_clip = 0.3f, dropout = 0.1f;
  int precision = PREC_TF32;
};

struct ResBlockSlots {
  size_t ln_w = 0, ln_b = 0;
  LinearSlot fc1, fc2;
};
struct ResNetSlots {  // score_idql.MLPResNet (:45-70)
  LinearSlot fc, out_fc;
  std::vector<ResBlockSlots> blocks;
  int in = 0, h = 0, out = 0;
};
struct ResNetActs {  // one evaluation that will be differentiated
  float *x = nullptr, *m = nullptr;  // residual stream (input of the final Mish after the last block), Mish output
  std::vector<float*> hm, hn, xhat, rstd, pre1, a1;  // per block: masked input, LN output, LN stats, fc1 output, Mish
  void want(DeviceArena& a, const ResNetSlots& n, int rows);
};
struct BottleneckSlots {  // psi_bottleneck1 / 2: Linear -> LayerNorm -> tanh on the state and on the action
  LinearSlot s_lin, a_lin;
  size_t s_lnw = 0, s_lnb = 0, a_lnw = 0, a_lnb = 0;
};
struct BottleneckActs {
  float *pre_s = nullptr, *pre_a = nullptr, *cat = nullptr, *xhat_s = nullptr, *xhat_a = nullptr, *rstd_s = nullptr,
        *rstd_a = nullptr;
};

class LatentDiffSR : public PixelAgent {
 public:
  LatentDiffSR(const LdiffConfig& c, cudaStream_t s);

  struct Inputs {  // all host pointers; N = 4 * batch frames
    const unsigned char* frames;       // [N, 3, 84, 84]: the 3B frames of img_stack, then the B newest next frames
    const unsigned char* next_frames;  // [3B, 3, 84, 84]: the frames of next_img_stack
    const int* shifts;                 // [N, 2] per-frame augmentation shift ((4, 4) = none for the last B)
    const int* next_shifts;            // [3B, 2]
    const float *action, *reward, *discount;  // [B, A], [B], [B]
    const float* eps_post;             // [N, L] posterior noise
    const float *alphabar, *temb, *noise;  // [B], [B, L/2], [B, L]
    const float* psi_masks;            // [psi_d][2B, psi_h]: rows [0, B) score step, rows [B, 2B) critic step
    const float* zeta_masks;           // [zeta_d][B, zeta_h]
    const float* eps_act;              // [2][B][A]
    float stddev;
  };
  // metrics_out[8] = {recon_loss, kl_loss, score_loss, critic_loss, mean(q_pred), mean(q_target), mean(reward), actor_loss}
  void update(const Inputs& in, float* metrics_out);
  std::vector<ParamGroup*> groups() override {
    return {&enc_->group(), &vh_g_, &dec_->group(), &score_g_, &dead_g_, &actor_g_, &crit_g_};
  }
  // the conv stacks' "convnet.<i>.*" / "deconvnet.<i>.*" are the VAE's "vae.encoder.convs.<i>.*" /
  // "vae.decoder.deconvs.<i>.*"
  std::string tensor_name(const ParamGroup& g, const std::string& t) const override {
    if (&g == &enc_->group()) return "vae.encoder.convs." + t.substr(std::string("convnet.").size());
    if (&g == &dec_->group()) return "vae.decoder.deconvs." + t.substr(std::string("deconvnet.").size());
    return t;
  }

 private:
  void launch_update(float stddev) override;
  ResNetSlots add_resnet(const std::string& prefix, int depth, int in, int out, int h);
  void resnet_forward(const ResNetSlots& n, bool target, int rows, Mat in, const float* masks, size_t mask_stride,
                      ResNetActs& a, float* out, int ld_out);
  void resnet_backward(const ResNetSlots& n, bool target, int rows, Mat in, const float* masks, size_t mask_stride,
                       ResNetActs& a, Mat dout, bool wgrad, float* din);
  void bottleneck_forward(bool target, int rows, Mat state, Mat action, BottleneckActs& a);
  void bottleneck_backward(bool target, int rows, Mat state, Mat action, BottleneckActs& a, const float* dcat, bool wgrad,
                           float* dstate, float* daction);
  void head_forward(bool target, const float* feat, bool keep, float* h2);
  void critic_forward(bool target, int slot, const float* feature, bool keep);
  void critic_backward(int slot, bool wgrad, float* dfeature);
  void actor_forward(Mat latent, const float* eps, float stddev, float* action_out, int ld_action, bool keep);

  LdiffConfig cfg_;
  int B_, N_, A_, L_, F_ = 0, feat_, bn_, H_, LA_ = 0, LZ_ = 0, T_ = 0;
  std::unique_ptr<ConvEncoder> enc_;
  std::unique_ptr<ConvDecoder> dec_;
  DeviceArena arena_;
  GemmRunner gemm_;
  ParamGroup vh_g_, score_g_, dead_g_, actor_g_, crit_g_;
  LinearSlot efc_, eout_, dfc_, at_, p0_, p1_, p2_;
  size_t eln_w_ = 0, eln_b_ = 0, aln_w_ = 0, aln_b_ = 0, cln_w_ = 0, cln_b_ = 0;
  BottleneckSlots bneck_;
  ResNetSlots psi_, zeta_;
  RffCritic rff_;
  unsigned char *frames_dev_ = nullptr, *next_frames_dev_ = nullptr;
  int *shifts_dev_ = nullptr, *next_shifts_dev_ = nullptr;
  float *action_dev_ = nullptr, *reward_dev_ = nullptr, *discount_dev_ = nullptr, *eps_post_dev_ = nullptr, *ab_dev_ = nullptr;
  float *temb_dev_ = nullptr, *noise_dev_ = nullptr, *psi_masks_dev_ = nullptr, *zeta_masks_dev_ = nullptr, *eps_act_dev_ = nullptr;
  // VAE
  float *feat_buf_ = nullptr, *tfeat_ = nullptr, *hpre_ = nullptr, *hs_ = nullptr, *hxhat_ = nullptr, *hrstd_ = nullptr;
  float *h2_ = nullptr, *h2t_ = nullptr, *mean_ = nullptr, *tmean_ = nullptr, *z_ = nullptr, *kl_partial_ = nullptr;
  float *dec_in_ = nullptr, *ddec_in_ = nullptr, *dz_ = nullptr, *dh2_ = nullptr, *dhs_ = nullptr, *dhpre_ = nullptr;
  float* dfeat_ = nullptr;
  // score
  float *psi_in_ = nullptr, *act2_ = nullptr, *psi_out_ = nullptr, *dpsi_out_ = nullptr, *dpsi_in_ = nullptr, *dcat_ = nullptr;
  float *zin_ = nullptr, *dzin_ = nullptr, *flat_ = nullptr, *dflat_ = nullptr, *target_ = nullptr, *coef_ = nullptr;
  float *dscore_ = nullptr, *loss_rows_ = nullptr;
  BottleneckActs bn_on_, bn_t_;
  ResNetActs psi_on_, psi_t_, zeta_on_;
  float *feat_t_ = nullptr, *dfeat_t_ = nullptr, *dcat_t_ = nullptr;
  float *dx_ = nullptr, *dtmp_h_ = nullptr, *dhm_ = nullptr, *d4_ = nullptr, *gb_ = nullptr, *gg_ = nullptr, *dpre_s_ = nullptr;
  // critic / actor
  float *cn_[2] = {nullptr, nullptr}, *cxhat_ = nullptr, *crstd_ = nullptr, *dcn_ = nullptr, *dq_ = nullptr;
  float *act_t_ = nullptr, *acta_ = nullptr, *dacta_ = nullptr;
  float *tpre_ = nullptr, *th_ = nullptr, *xhat_a_ = nullptr, *rstd_a_ = nullptr, *ap1_ = nullptr, *ap2_ = nullptr;
  float *raw_a_ = nullptr, *mu_ = nullptr, *draw_a_ = nullptr, *dap2_ = nullptr, *dap1_ = nullptr, *dth_ = nullptr;
  float* dtpre_ = nullptr;
  static constexpr int kKlBlocks = 64;
};

}  // namespace rlrep

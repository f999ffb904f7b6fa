// Plain DrQ-v2 pixel update (reference: agent/diffsrdrq/drqv2.py:93-148 `DrQv2.train_step`, networks in
// agent/diffsrdrq/network_arch/drqv2.py) -- SURVEY.md 8a row a17, second symbol; the first pixel agent assembled on the
// conv-encoder building block (conv.cu).
//
// Per update: encoder(aug(next_img)) [no grad] -> encoder(aug(img)) -> target: actor(next) + TruncatedNormal sample,
// critic_target -> q_target = r + discount * min;  critic(latent, action) -> MSE over the stacked twin Q -> backward
// through the Q MLPs, the LayerNorm/tanh trunk and the encoder -> Adam(critic) (+ Polyak of critic_target, tau) and
// Adam(encoder);  actor step on the detached latent: actor -> sample -> critic (new weights) -> -mean(min Q) ->
// dgrad through the critic to the action, backward through the actor -> Adam(actor).
// Randomness (two shift draws, two [B, A] normal draws) and the std-dev schedule value come from the host.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "agent.cuh"
#include "conv.cuh"
#include "drq.cuh"
#include "staging.cuh"

namespace rlrep {

DrqV2::DrqV2(const DrqConfig& c, cudaStream_t s)
    : PixelAgent(s), cfg_(c), B_(c.batch), A_(c.action_dim), bn_(c.bn_dim), H_(c.hidden_dim) {
  RLREP_CHECK(B_ > 0 && A_ > 0 && bn_ > 0 && H_ % 32 == 0, "bad DrQ-v2 dimensions (hidden_dim must be a multiple of 32)");
  enc_.reset(new ConvEncoder(B_, c.channels, c.height, static_cast<Precision>(c.precision), s));
  F_ = enc_->feature_dim();
  RLREP_CHECK(F_ % 32 == 0, "encoder feature width must be a multiple of 32");
  LB_ = round_up32(bn_);
  LC_ = round_up32(bn_ + A_);
  LA_ = round_up32(A_);

  crit_g_.name = "critic";
  ct_ = add_linear(crit_g_, "critic.trunk.0", bn_, F_);
  cln_w_ = crit_g_.add("critic.trunk.1.weight", bn_, 1, 1, LB_);
  cln_b_ = crit_g_.add("critic.trunk.1.bias", bn_, 1, 1, LB_);
  q0_.out = 2 * H_;
  q0_.in = bn_ + A_;
  q0_.ld = LC_;
  q0_.out_alloc = 2 * H_;
  q0_.w_off = crit_g_.add("critic.Q1.0.weight", H_, bn_ + A_, LC_);
  crit_g_.add("critic.Q2.0.weight", H_, bn_ + A_, LC_);
  q0_.b_off = crit_g_.add("critic.Q1.0.bias", H_, 1);
  crit_g_.add("critic.Q2.0.bias", H_, 1);
  q1a_ = add_linear(crit_g_, "critic.Q1.2", H_, H_);
  q1b_ = add_linear(crit_g_, "critic.Q2.2", H_, H_);
  q2a_ = add_linear(crit_g_, "critic.Q1.4", 1, H_, false);
  q2b_ = add_linear(crit_g_, "critic.Q2.4", 1, H_, false);
  crit_g_.n_target = crit_g_.n;
  crit_g_.target_prefix_from = "critic.";
  crit_g_.target_prefix_to = "critic_target.";
  crit_g_.want(arena_);

  actor_g_.name = "actor";
  at_ = add_linear(actor_g_, "actor.trunk.0", bn_, F_);
  aln_w_ = actor_g_.add("actor.trunk.1.weight", bn_, 1, 1, LB_);
  aln_b_ = actor_g_.add("actor.trunk.1.bias", bn_, 1, 1, LB_);
  p0_ = add_linear(actor_g_, "actor.policy.0", H_, bn_);
  p1_ = add_linear(actor_g_, "actor.policy.2", H_, H_);
  p2_ = add_linear(actor_g_, "actor.policy.4", A_, H_);
  actor_g_.want(arena_);

  const size_t BF = (size_t)B_ * F_, BH = (size_t)B_ * H_;
  arena_.want(&ctl_, 1);
  arena_.want(&metrics_dev_, 8);
  arena_.want(&img_dev_, (size_t)B_ * c.channels * c.height * c.height);
  arena_.want(&next_img_dev_, (size_t)B_ * c.channels * c.height * c.height);
  arena_.want(&shifts_dev_, 4 * B_);
  arena_.want(&eps_dev_, (size_t)2 * B_ * A_);
  arena_.want(&action_dev_, (size_t)B_ * A_);
  arena_.want(&reward_dev_, B_);
  arena_.want(&discount_dev_, B_);
  arena_.want(&latent_, BF);
  arena_.want(&next_latent_, BF);
  arena_.want(&dlatent_, BF);
  for (int i = 0; i < 2; ++i) {
    arena_.want(&tpre_[i], (size_t)B_ * LB_);
    arena_.want(&cat_[i], (size_t)B_ * LC_);
    arena_.want(&hid0_[i], 2 * BH);
    arena_.want(&hid1_[i], 2 * BH);
    arena_.want(&q_[i], 2 * B_);
  }
  arena_.want(&xhat_c_, (size_t)B_ * LB_);
  arena_.want(&rstd_c_, B_);
  arena_.want(&xhat_a_, (size_t)B_ * LB_);
  arena_.want(&rstd_a_, B_);
  arena_.want(&th_, (size_t)B_ * LB_);
  arena_.want(&ap1_, BH);
  arena_.want(&ap2_, BH);
  arena_.want(&raw_, (size_t)B_ * LA_);
  arena_.want(&mu_, (size_t)B_ * A_);
  arena_.want(&dq_, 2 * B_);
  arena_.want(&dhid1_, 2 * BH);
  arena_.want(&dhid0_, 2 * BH);
  arena_.want(&dcat_, (size_t)B_ * LC_);
  arena_.want(&dtpre_, (size_t)B_ * LB_);
  arena_.want(&gb_, (size_t)B_ * LB_);
  arena_.want(&gg_, (size_t)B_ * LB_);
  arena_.want(&draw_, (size_t)B_ * LA_);
  arena_.want(&dap2_, BH);
  arena_.want(&dap1_, BH);
  arena_.want(&dth_, (size_t)B_ * LB_);
  arena_.commit();
  gemm_.init(static_cast<Precision>(c.precision), 0);
  const size_t img_bytes = (size_t)B_ * c.channels * c.height * c.height;
  alloc_host(2 * img_bytes + (size_t)4 * B_ * sizeof(int) + ((size_t)2 * B_ * A_ + (size_t)B_ * A_ + 2 * B_) * sizeof(float));
  Control h;
  std::memset(&h, 0, sizeof(h));
  RLREP_CUDA(cudaMemcpyAsync(ctl_, &h, sizeof(h), cudaMemcpyHostToDevice, stream_));
  RLREP_CUDA(cudaStreamSynchronize(stream_));
}

// Linear(F -> bn) -> LayerNorm -> tanh; y goes to out[:, 0:bn] (pitch ld_out)
void DrqV2::trunk_forward(const LinearSlot& t, const ParamGroup& g, bool target, size_t ln_w, size_t ln_b, const float* x,
                          float* pre, float* out, int ld_out, float* xhat, float* rstd) {
  const Linear l = t.view(g, target);
  const float* base = target ? g.target : g.p;
  // N runs over the padded width LB (zero weight rows / bias): the padding columns of `pre` come out as exact zeros
  Linear lp = l;
  lp.out = LB_;
  linear_fwd(gemm_, stream_, B_, Mat{x, F_}, lp, ACT_NONE, pre, LB_);
  launch_ln_tanh_fwd(pre, LB_, B_, bn_, base + ln_w, base + ln_b, out, ld_out, xhat, LB_, rstd, stream_);
}

// twin Q MLPs on cat = [h | action | 0] (pitch LC); q1 -> q[0:B], q2 -> q[B:2B]
void DrqV2::q_forward(bool target, int set) {
  const Linear l0 = q0_.view(crit_g_, target), l1a = q1a_.view(crit_g_, target), l1b = q1b_.view(crit_g_, target);
  const Linear l2a = q2a_.view(crit_g_, target), l2b = q2b_.view(crit_g_, target);
  const size_t BH = (size_t)B_ * H_;
  linear_fwd(gemm_, stream_, B_, Mat{cat_[set], LC_}, l0, ACT_RELU, hid0_[set], 2 * H_);
  linear_fwd(gemm_, stream_, B_, Mat{hid0_[set], 2 * H_}, l1a, ACT_RELU, hid1_[set], H_);
  linear_fwd(gemm_, stream_, B_, Mat{hid0_[set] + H_, 2 * H_}, l1b, ACT_RELU, hid1_[set] + BH, H_);
  launch_rowdot_pair(RowDotJob{hid1_[set], l2a.W, l2a.b, q_[set], H_, H_},
                     RowDotJob{hid1_[set] + BH, l2b.W, l2b.b, q_[set] + B_, H_, H_}, B_, stream_);
}

// (dq1 | dq2) -> dcat [B, LC] (gradient w.r.t. [h | action]); wgrad: also the critic's parameter gradients
void DrqV2::q_backward(int set, bool wgrad) {
  const Linear l0 = q0_.view(crit_g_), l1a = q1a_.view(crit_g_), l1b = q1b_.view(crit_g_);
  const Linear l2a = q2a_.view(crit_g_), l2b = q2b_.view(crit_g_);
  const size_t BH = (size_t)B_ * H_;
  float* d1a = dhid1_;
  float* d1b = dhid1_ + BH;
  launch_outer_dact(dq_, l2a.W, B_, H_, hid1_[set], H_, DACT_RELU_OUT, d1a, H_, stream_);
  launch_outer_dact(dq_ + B_, l2b.W, B_, H_, hid1_[set] + BH, H_, DACT_RELU_OUT, d1b, H_, stream_);
  if (wgrad) {
    linear_wgrad(gemm_, stream_, B_, Mat{d1a, H_}, Mat{hid0_[set], 2 * H_}, l1a, Mat(), 0, false);
    linear_wgrad(gemm_, stream_, B_, Mat{d1b, H_}, Mat{hid0_[set] + H_, 2 * H_}, l1b, Mat(), 0, false);
  }
  linear_dgrad(gemm_, stream_, B_, Mat{d1a, H_}, l1a, DACT_RELU_OUT, Mat{hid0_[set], 2 * H_}, dhid0_, 2 * H_);
  linear_dgrad(gemm_, stream_, B_, Mat{d1b, H_}, l1b, DACT_RELU_OUT, Mat{hid0_[set] + H_, 2 * H_}, dhid0_ + H_, 2 * H_);
  if (wgrad) {
    linear_wgrad(gemm_, stream_, B_, Mat{dhid0_, 2 * H_}, Mat{cat_[set], LC_}, l0, Mat(), 0, false);
    const ColJob jobs[7] = {ColJob{hid1_[set], dq_, l2a.dW, H_, B_, H_},           ColJob{dq_, nullptr, l2a.db, 1, B_, 1},
                            ColJob{hid1_[set] + BH, dq_ + B_, l2b.dW, H_, B_, H_}, ColJob{dq_ + B_, nullptr, l2b.db, 1, B_, 1},
                            bias_job(B_, Mat{d1a, H_}, l1a),                       bias_job(B_, Mat{d1b, H_}, l1b),
                            bias_job(B_, Mat{dhid0_, 2 * H_}, l0)};
    launch_colreduce_multi(jobs, 7, stream_);
  }
  // all (padded) input columns on the tensor-core path; [0, bn) is d h, [bn, bn + A) is d action
  linear_dgrad(gemm_, stream_, B_, Mat{dhid0_, 2 * H_}, l0, DACT_NONE, Mat(), dcat_, LC_, 0, LC_);
}

// actor(latent): trunk -> policy MLP -> raw [B, LA]; sample -> action into cat_[set][:, bn : bn + A]
void DrqV2::actor_forward(const float* latent, const float* eps, float stddev, int set, bool keep) {
  const Linear l0 = p0_.view(actor_g_), l1 = p1_.view(actor_g_), l2 = p2_.view(actor_g_);
  trunk_forward(at_, actor_g_, false, aln_w_, aln_b_, latent, tpre_[set], th_, LB_, keep ? xhat_a_ : nullptr,
                keep ? rstd_a_ : nullptr);
  linear_fwd(gemm_, stream_, B_, Mat{th_, LB_}, l0, ACT_RELU, ap1_, H_);
  linear_fwd(gemm_, stream_, B_, Mat{ap1_, H_}, l1, ACT_RELU, ap2_, H_);
  linear_fwd(gemm_, stream_, B_, Mat{ap2_, H_}, l2, ACT_NONE, raw_, LA_);
  launch_trunc_normal_sample(raw_, LA_, B_, A_, eps, stddev, cfg_.stddev_clip, mu_, cat_[set] + bn_, LC_, stream_);
}

// select_action (drqv2.py:74-82) on n observations: the small-batch policy (pixel_act.cu) over this handle's
// parameters, created on first use
void DrqV2::act_batch(const unsigned char* obs, const float* eps_host, float stddev, int n, float* actions_host) {
  if (!policy_)
    policy_.reset(new PixelPolicy(cfg_.channels, cfg_.height, A_,
                                  actor_policy_weights(*enc_, actor_g_, at_, aln_w_, aln_b_, p0_, p1_, p2_), stream_));
  policy_->act(obs, eps_host, stddev, n, actions_host);
}

void DrqV2::update(const unsigned char* img, const float* action, const float* reward, const float* discount,
                   const unsigned char* next_img, const int* shifts, const float* eps, float stddev, float* metrics_out) {
  cudaStream_t s = stream_;
  const size_t img_bytes = (size_t)B_ * cfg_.channels * cfg_.height * cfg_.height;
  // ---- stage the step's inputs through one pinned buffer (H2D inside the step, like the reference's .to(device))
  RLREP_CUDA(cudaStreamSynchronize(s));
  unsigned char* st = stage_host_;
  auto put = [&](void* dev, const void* src, size_t bytes) { stage_h2d(st, dev, src, bytes, s); };
  put(img_dev_, img, img_bytes);
  put(next_img_dev_, next_img, img_bytes);
  put(shifts_dev_, shifts, (size_t)4 * B_ * sizeof(int));
  put(eps_dev_, eps, (size_t)2 * B_ * A_ * sizeof(float));
  put(action_dev_, action, (size_t)B_ * A_ * sizeof(float));
  put(reward_dev_, reward, B_ * sizeof(float));
  put(discount_dev_, discount, B_ * sizeof(float));
  finish_update(stddev, metrics_out, 5);
}

// Every launch of one update on the batch currently resident in the device buffers.
void DrqV2::launch_update(float stddev) {
  cudaStream_t s = stream_;

  TickParams t;
  t.k_feat = 1;  // the encoder's Adam step uses the "feature" slot of the control block
  t.period = 1;
  t.lr_feat = cfg_.encoder_lr;
  t.lr_critic = cfg_.critic_lr;
  t.lr_actor = cfg_.actor_lr;
  t.lr_alpha = 0.0;
  t.critic_steps = 1;
  launch_tick(ctl_, t, s);

  // ---- critic step (drqv2.py:112-133).  next_img first: its activations are not needed again, img's are.
  enc_->forward(next_img_dev_, shifts_dev_ + 2 * B_, next_latent_, 0, false, /*no_grad=*/true);
  enc_->forward(img_dev_, shifts_dev_, latent_);
  actor_forward(next_latent_, eps_dev_, stddev, /*set=*/0, /*keep=*/false);
  trunk_forward(ct_, crit_g_, /*target=*/true, cln_w_, cln_b_, next_latent_, tpre_[0], cat_[0], LC_, nullptr, nullptr);
  q_forward(/*target=*/true, 0);
  trunk_forward(ct_, crit_g_, false, cln_w_, cln_b_, latent_, tpre_[1], cat_[1], LC_, xhat_c_, rstd_c_);
  {
    const ColSegment seg{0, bn_, A_};  // the batch's action behind h
    launch_pack_columns(action_dev_, A_, cat_[1], LC_, B_, &seg, 1, s);
  }
  q_forward(false, 1);
  launch_drq_critic_loss(reward_dev_, discount_dev_, q_[0], q_[0] + B_, q_[1], q_[1] + B_, B_, dq_, dq_ + B_,
                         metrics_dev_ + 0, s);
  q_backward(1, /*wgrad=*/true);
  {
    const Linear lt = ct_.view(crit_g_);
    launch_ln_tanh_bwd(dcat_, LC_, cat_[1], LC_, xhat_c_, LB_, rstd_c_, B_, bn_, crit_g_.p + cln_w_, dtpre_, LB_, gb_, gg_,
                       LB_, s);
    Linear lp = lt;
    lp.out = LB_;  // padded rows: their gradient is exactly zero (dtpre padding columns are zero)
    linear_wgrad(gemm_, s, B_, Mat{dtpre_, LB_}, Mat{latent_, F_}, lp, Mat(), 0, false);
    const ColJob jobs[3] = {bias_job(B_, Mat{dtpre_, LB_}, lt), ColJob{gg_, nullptr, crit_g_.g + cln_w_, LB_, B_, bn_},
                            ColJob{gb_, nullptr, crit_g_.g + cln_b_, LB_, B_, bn_}};
    launch_colreduce_multi(jobs, 3, s);
    linear_dgrad(gemm_, s, B_, Mat{dtpre_, LB_}, lp, DACT_NONE, Mat(), dlatent_, F_);
  }
  enc_->backward(dlatent_);
  launch_adam_polyak(crit_g_.p, crit_g_.g, crit_g_.m, crit_g_.v, crit_g_.n, &ctl_->critic, crit_g_.target,
                     crit_g_.n_target, cfg_.tau, nullptr, s);
  {
    ParamGroup& eg = enc_->group();
    launch_adam_polyak(eg.p, eg.g, eg.m, eg.v, eg.n, &ctl_->feat[0], nullptr, 0, 0.f, nullptr, s);
  }

  // ---- actor step (drqv2.py:135-148) on the detached latent, against the just-updated critic
  actor_forward(latent_, eps_dev_ + (size_t)B_ * A_, stddev, 0, /*keep=*/true);
  trunk_forward(ct_, crit_g_, false, cln_w_, cln_b_, latent_, tpre_[1], cat_[0], LC_, nullptr, nullptr);
  q_forward(false, 0);
  launch_drq_actor_loss(q_[0], q_[0] + B_, B_, dq_, dq_ + B_, metrics_dev_ + 4, s);
  q_backward(0, /*wgrad=*/false);
  {
    const Linear l0 = p0_.view(actor_g_), l1 = p1_.view(actor_g_), l2 = p2_.view(actor_g_), lt = at_.view(actor_g_);
    launch_trunc_normal_bwd(dcat_ + bn_, LC_, mu_, B_, A_, draw_, LA_, s);
    linear_wgrad(gemm_, s, B_, Mat{draw_, LA_}, Mat{ap2_, H_}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{draw_, LA_}, l2, DACT_RELU_OUT, Mat{ap2_, H_}, dap2_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dap2_, H_}, Mat{ap1_, H_}, l1, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dap2_, H_}, l1, DACT_RELU_OUT, Mat{ap1_, H_}, dap1_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dap1_, H_}, Mat{th_, LB_}, l0, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dap1_, H_}, l0, DACT_NONE, Mat(), dth_, LB_, 0, LB_);
    launch_ln_tanh_bwd(dth_, LB_, th_, LB_, xhat_a_, LB_, rstd_a_, B_, bn_, actor_g_.p + aln_w_, dtpre_, LB_, gb_, gg_, LB_,
                       s);
    Linear lp = lt;
    lp.out = LB_;
    linear_wgrad(gemm_, s, B_, Mat{dtpre_, LB_}, Mat{latent_, F_}, lp, Mat(), 0, false);
    const ColJob jobs[6] = {bias_job(B_, Mat{draw_, LA_}, l2),  bias_job(B_, Mat{dap2_, H_}, l1),
                            bias_job(B_, Mat{dap1_, H_}, l0),   bias_job(B_, Mat{dtpre_, LB_}, lt),
                            ColJob{gg_, nullptr, actor_g_.g + aln_w_, LB_, B_, bn_},
                            ColJob{gb_, nullptr, actor_g_.g + aln_b_, LB_, B_, bn_}};
    launch_colreduce_multi(jobs, 6, s);
  }
  launch_adam_polyak(actor_g_.p, actor_g_.g, actor_g_.m, actor_g_.v, actor_g_.n, &ctl_->actor, nullptr, 0, 0.f, nullptr, s);
}

}  // namespace rlrep

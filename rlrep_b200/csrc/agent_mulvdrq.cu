// muLV-Rep DrQ-v2 pixel update (reference: agent/mulvdrq/drqv2.py:313-461 `DrQV2Agent.update`, :284-311 `update_actor`;
// networks drqv2.py:52-196, vae.py:13-124) -- SURVEY.md 8a row a16, with `mulv_config.py`'s defaults: aug, no pre_aug,
// back_q2feat, tanh heads, ReLU critic, Huber critic loss, soft target updates (tau) of critic / encoder / feat_f.
//
// Per update (single stream, eager):
//   no grad:  next_state = encoder_target(aug(next_img)); a' = actor(next_state) + clipped noise;
//             (m', ls') = feat_f_target(next_state, a'); target_Q = r + discount * min critic_target(m', ls' ; noise 0)
//   forward:  state = encoder(aug(img)); state1 = predict_encoder(last frame of the next observation);
//             (m1, ls1) = feat_encoder(state, a, state1); z = m1 + exp(ls1) eps; (x, r_hat) = feat_decoder(z);
//             pred = decoder(x); s_loss = 10 L1(pred, frame); r_loss = mse; (m2, ls2) = feat_f(state, a);
//             kl = KL(1 || 2).mean(); Q = critic(m2, ls2 ; noise 1); critic_loss = Huber
//   backward of critic_loss + (s_loss + r_loss + kl) * vae_w through everything, Adam on the seven groups
//   actor:    a = actor(state.detach()); Q = critic(feat_f(state, a) ; noise 2) with the NEW weights; -mean(min Q);
//             dgrad only through critic and feat_f to the action; Adam(actor);  then the three soft updates.
// The reference evaluates feat_encoder and feat_f twice on identical inputs (sample + KL, KL + critic); here each is ONE
// forward whose head gradients are summed before a single backward.  Wide inputs live in one [B, 2F + A] matrix
// (state | action | state1): feat_encoder reads all of it, feat_f and the actor trunk read its leading columns.
#include "mulv.cuh"

#include "staging.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace rlrep {

namespace {

GaussHead add_gauss(ParamGroup& g, const std::string& prefix, int D, int in) {
  GaussHead h;
  const int LF = round_up32(D), ld = round_up32(in);
  h.lin.out = 2 * LF;
  h.lin.in = in;
  h.lin.ld = ld;
  h.lin.out_alloc = 2 * LF;
  h.lin.w_off = g.add(prefix + ".mean_linear.0.weight", D, in, ld, LF);
  g.add(prefix + ".log_std_linear.0.weight", D, in, ld, LF);
  h.lin.b_off = g.add(prefix + ".mean_linear.0.bias", D, 1, 1, LF);
  g.add(prefix + ".log_std_linear.0.bias", D, 1, 1, LF);
  h.g_mean = g.add(prefix + ".mean_linear.1.weight", D, 1, 1, LF);
  h.b_mean = g.add(prefix + ".mean_linear.1.bias", D, 1, 1, LF);
  h.g_ls = g.add(prefix + ".log_std_linear.1.weight", D, 1, 1, LF);
  h.b_ls = g.add(prefix + ".log_std_linear.1.bias", D, 1, 1, LF);
  return h;
}

void want_gauss(DeviceArena& a, GaussActs& g, int B, int LF) {
  a.want(&g.pre, (size_t)B * 2 * LF);
  a.want(&g.m, (size_t)B * LF);
  a.want(&g.raw, (size_t)B * LF);
  a.want(&g.xhat_m, (size_t)B * LF);
  a.want(&g.xhat_s, (size_t)B * LF);
  a.want(&g.rstd_m, B);
  a.want(&g.rstd_s, B);
}

}  // namespace

MulvDrq::MulvDrq(const MulvConfig& c, cudaStream_t s)
    : PixelAgent(s), cfg_(c), B_(c.batch), A_(c.action_dim), D_(c.feat_dim), H_(c.hidden_dim), NN_(c.num_noise) {
  RLREP_CHECK(B_ > 0 && A_ > 0 && D_ > 0 && NN_ > 0 && H_ % 32 == 0,
              "bad muLV-DrQ dimensions (hidden_dim must be a multiple of 32)");
  RLREP_CHECK(c.height == 84, "the pixel decoder is built for 84 x 84 frames (35 -> 37 -> 39 -> 41 -> 83 -> 84)");
  const Precision prec = static_cast<Precision>(c.precision);
  enc_.reset(new ConvEncoder(B_, c.channels, c.height, prec, s, /*with_target=*/true));
  enc_->group().name = "encoder";
  enc_->group().target_prefix_from = "encoder.";
  enc_->group().target_prefix_to = "encoder_target.";
  penc_.reset(new ConvEncoder(B_, 3, c.height, prec, s));
  penc_->group().name = "predict_encoder";
  dec_.reset(new ConvDecoder(B_, prec, s));
  F_ = enc_->feature_dim();
  LF_ = round_up32(D_);
  LA_ = round_up32(A_);
  LDE_ = round_up32(2 * F_ + A_);
  LDS_ = round_up32(F_ + A_);

  actor_g_.name = "actor";
  at_ = add_linear(actor_g_, "actor.trunk.0", D_, F_);
  aln_w_ = actor_g_.add("actor.trunk.1.weight", D_, 1, 1, LF_);
  aln_b_ = actor_g_.add("actor.trunk.1.bias", D_, 1, 1, LF_);
  p0_ = add_linear(actor_g_, "actor.policy.0", H_, D_);
  p1_ = add_linear(actor_g_, "actor.policy.2", H_, H_);
  p2_ = add_linear(actor_g_, "actor.policy.4", A_, H_);
  actor_g_.want(arena_);

  crit_g_.name = "critic";
  c14_.out = 2 * H_;
  c14_.in = D_;
  c14_.ld = LF_;
  c14_.out_alloc = 2 * H_;
  c14_.w_off = crit_g_.add("critic.l1.weight", H_, D_, LF_);
  crit_g_.add("critic.l4.weight", H_, D_, LF_);
  c14_.b_off = crit_g_.add("critic.l1.bias", H_, 1);
  crit_g_.add("critic.l4.bias", H_, 1);
  c2_ = add_linear(crit_g_, "critic.l2", H_, H_);
  c5_ = add_linear(crit_g_, "critic.l5", H_, H_);
  c3_ = add_linear(crit_g_, "critic.l3", 1, H_, false);
  c6_ = add_linear(crit_g_, "critic.l6", 1, H_, false);
  crit_g_.n_target = crit_g_.n;
  crit_g_.target_prefix_from = "critic.";
  crit_g_.target_prefix_to = "critic_target.";
  crit_g_.want(arena_);

  fe_g_.name = "feat_encoder";
  fe_ = add_gauss(fe_g_, "feat_encoder", D_, 2 * F_ + A_);
  fe_g_.want(arena_);
  fd_g_.name = "feat_decoder";
  d1_ = add_linear(fd_g_, "feat_decoder.l1", H_, D_);
  d2_ = add_linear(fd_g_, "feat_decoder.l2", H_, H_);
  ds_ = add_linear(fd_g_, "feat_decoder.state_linear", F_, H_);
  dr_ = add_linear(fd_g_, "feat_decoder.reward_linear", 1, H_, false);
  fd_g_.want(arena_);
  ff_g_.name = "feat_f";
  ff_ = add_gauss(ff_g_, "feat_f", D_, F_ + A_);
  ff_g_.n_target = ff_g_.n;
  ff_g_.target_prefix_from = "feat_f.";
  ff_g_.target_prefix_to = "feat_f_target.";
  ff_g_.want(arena_);

  const size_t img_bytes = (size_t)B_ * c.channels * c.height * c.height;
  const size_t step1_bytes = (size_t)B_ * 3 * c.height * c.height;
  const size_t BH = (size_t)B_ * H_, BL = (size_t)B_ * LF_, BF = (size_t)B_ * F_, BN = (size_t)B_ * NN_;
  arena_.want(&ctl_, 1);
  arena_.want(&metrics_dev_, 8);
  arena_.want(&img_dev_, img_bytes);
  arena_.want(&next_img_dev_, img_bytes);
  arena_.want(&step1_dev_, step1_bytes);
  arena_.want(&shifts_dev_, 4 * B_);
  arena_.want(&eps_z_dev_, (size_t)B_ * D_);
  arena_.want(&eps_act_dev_, (size_t)2 * B_ * A_);
  arena_.want(&noise_dev_, (size_t)3 * NN_ * D_);
  arena_.want(&action_dev_, (size_t)B_ * A_);
  arena_.want(&reward_dev_, B_);
  arena_.want(&discount_dev_, B_);
  arena_.want(&enc_in_, (size_t)B_ * LDE_);
  arena_.want(&nsa_, (size_t)B_ * LDS_);
  arena_.want(&dstate_, BF);
  arena_.want(&dstep1_, BF);
  want_gauss(arena_, ge_, B_, LF_);
  want_gauss(arena_, gf_, B_, LF_);
  want_gauss(arena_, gn_, B_, LF_);
  arena_.want(&z_, BL); arena_.want(&dz_, BL);
  arena_.want(&fh1_, BH); arena_.want(&fh2_, BH); arena_.want(&dfh1_, BH); arena_.want(&dfh2_, BH);
  arena_.want(&s_hat_, BF); arena_.want(&ds_hat_, BF);
  arena_.want(&r_hat_, B_); arena_.want(&dr_hat_, B_);
  arena_.want(&kl_partial_, kKlBlocks);
  arena_.want(&dm1_, BL); arena_.want(&draw1_, BL); arena_.want(&dm2_, BL); arena_.want(&draw2_, BL);
  arena_.want(&dcm_, BL); arena_.want(&dcraw_, BL);
  arena_.want(&dpre_, 2 * BL);
  arena_.want(&gb_, BL); arena_.want(&gg_, BL); arena_.want(&gb2_, BL); arena_.want(&gg2_, BL);
  for (int i = 0; i < 2; ++i) {
    arena_.want(&xs_[i], BN * LF_);
    arena_.want(&hid1_[i], BN * 2 * H_);
    arena_.want(&m20_[i], 2 * BH);
    arena_.want(&hid2_[i], 2 * BH);
    arena_.want(&q_[i], 2 * B_);
  }
  arena_.want(&dq_, 2 * B_);
  arena_.want(&dhid2_, 2 * BH);
  arena_.want(&dm20_, 2 * BH);
  arena_.want(&dhid1_, BN * 2 * H_);
  arena_.want(&bpart_, 2 * BH);
  arena_.want(&dxs_, BN * LF_);
  arena_.want(&tpre_, BL); arena_.want(&th_, BL); arena_.want(&xhat_a_, BL); arena_.want(&rstd_a_, B_);
  arena_.want(&ap1_, BH); arena_.want(&ap2_, BH); arena_.want(&dap1_, BH); arena_.want(&dap2_, BH);
  arena_.want(&raw_a_, (size_t)B_ * LA_); arena_.want(&mu_, (size_t)B_ * A_);
  arena_.want(&daction_, (size_t)B_ * LA_); arena_.want(&draw_a_, (size_t)B_ * LA_);
  arena_.want(&dth_, BL); arena_.want(&dtpre_, BL);
  arena_.commit();
  gemm_.init(prec, 0);

  alloc_host(2 * img_bytes + step1_bytes + (size_t)4 * B_ * sizeof(int) +
             ((size_t)B_ * D_ + (size_t)2 * B_ * A_ + (size_t)3 * NN_ * D_ + (size_t)B_ * A_ + 2 * B_) * sizeof(float));
  Control h;
  std::memset(&h, 0, sizeof(h));
  RLREP_CUDA(cudaMemcpyAsync(ctl_, &h, sizeof(h), cudaMemcpyHostToDevice, stream_));
  RLREP_CUDA(cudaStreamSynchronize(stream_));
}

// vae.Encoder.forward / GaussianFeature.forward (vae.py:40-48, :118-124): mean = tanh(LN(W_m x)), raw = LN(W_s x); the
// two first layers are one [2 LF, in] GEMM
void MulvDrq::gauss_forward(const GaussHead& h, const ParamGroup& g, bool target, Mat x, GaussActs& a, bool keep) {
  const Linear l = h.lin.view(g, target);
  const float* base = target ? g.target : g.p;
  linear_fwd(gemm_, stream_, B_, x, l, ACT_NONE, a.pre, 2 * LF_);
  launch_ln_act_fwd(a.pre, 2 * LF_, B_, D_, base + h.g_mean, base + h.b_mean, true, a.m, LF_, LF_,
                    keep ? a.xhat_m : nullptr, LF_, keep ? a.rstd_m : nullptr, stream_);
  launch_ln_act_fwd(a.pre + LF_, 2 * LF_, B_, D_, base + h.g_ls, base + h.b_ls, false, a.raw, LF_, LF_,
                    keep ? a.xhat_s : nullptr, LF_, keep ? a.rstd_s : nullptr, stream_);
}

// (dm, draw) -> dpre_ [B, 2 LF] (gradient of the stacked first layer's output); wgrad: every parameter gradient of the head
void MulvDrq::gauss_backward(const GaussHead& h, ParamGroup& g, Mat x, const GaussActs& a, const float* dm,
                             const float* draw, bool wgrad) {
  cudaStream_t s = stream_;
  launch_ln_act_bwd(dm, LF_, a.m, LF_, a.xhat_m, LF_, a.rstd_m, B_, D_, g.p + h.g_mean, true, dpre_, 2 * LF_, LF_, gb_, gg_,
                    LF_, s);
  launch_ln_act_bwd(draw, LF_, a.raw, LF_, a.xhat_s, LF_, a.rstd_s, B_, D_, g.p + h.g_ls, false, dpre_ + LF_, 2 * LF_, LF_,
                    gb2_, gg2_, LF_, s);
  if (!wgrad) return;
  const Linear l = h.lin.view(g);
  linear_wgrad(gemm_, s, B_, Mat{dpre_, 2 * LF_}, x, l, Mat(), 0, false);
  const ColJob jobs[5] = {bias_job(B_, Mat{dpre_, 2 * LF_}, l),
                          ColJob{gg_, nullptr, g.g + h.g_mean, LF_, B_, D_},
                          ColJob{gb_, nullptr, g.g + h.b_mean, LF_, B_, D_},
                          ColJob{gg2_, nullptr, g.g + h.g_ls, LF_, B_, D_},
                          ColJob{gb2_, nullptr, g.g + h.b_ls, LF_, B_, D_}};
  launch_colreduce_multi(jobs, 5, s);
}

// Critic.forward (drqv2.py:177-196): x = m + exp(ls) * noise * c_noise over NN draws; relu(l1 x) averaged over the
// draws; relu(l2 .); l3.  l1 | l4 are one stacked GEMM over B * NN rows.  q1 -> q_[slot][0:B], q2 -> [B:2B]
void MulvDrq::critic_forward(bool target, int slot, const float* m, const float* raw, const float* noise) {
  cudaStream_t s = stream_;
  const Linear l14 = c14_.view(crit_g_, target), l2 = c2_.view(crit_g_, target), l5 = c5_.view(crit_g_, target);
  const Linear l3 = c3_.view(crit_g_, target), l6 = c6_.view(crit_g_, target);
  const size_t BH = (size_t)B_ * H_;
  launch_gauss_noise_expand(m, raw, LF_, B_, D_, noise, NN_, cfg_.c_noise, xs_[slot], LF_, s);
  linear_fwd(gemm_, s, B_ * NN_, Mat{xs_[slot], LF_}, l14, ACT_RELU, hid1_[slot], 2 * H_);
  launch_group_mean(hid1_[slot], 2 * H_, B_, NN_, 2 * H_, m20_[slot], s);
  linear_fwd(gemm_, s, B_, Mat{m20_[slot], 2 * H_}, l2, ACT_RELU, hid2_[slot], H_);
  linear_fwd(gemm_, s, B_, Mat{m20_[slot] + H_, 2 * H_}, l5, ACT_RELU, hid2_[slot] + BH, H_);
  launch_rowdot_pair(RowDotJob{hid2_[slot], l3.W, l3.b, q_[slot], H_, H_},
                     RowDotJob{hid2_[slot] + BH, l6.W, l6.b, q_[slot] + B_, H_, H_}, B_, s);
}

// (dq1 | dq2) in dq_ -> gradient w.r.t. the Gaussian head (dm, draw); wgrad: also the critic's parameter gradients
void MulvDrq::critic_backward(int slot, const float* raw, const float* noise, bool wgrad, float* dm, float* draw) {
  cudaStream_t s = stream_;
  const Linear l14 = c14_.view(crit_g_), l2 = c2_.view(crit_g_), l5 = c5_.view(crit_g_);
  const Linear l3 = c3_.view(crit_g_), l6 = c6_.view(crit_g_);
  const size_t BH = (size_t)B_ * H_;
  float* d2a = dhid2_;
  float* d2b = dhid2_ + BH;
  const float* h2a = hid2_[slot];
  const float* h2b = hid2_[slot] + BH;
  launch_outer_dact(dq_, l3.W, B_, H_, h2a, H_, DACT_RELU_OUT, d2a, H_, s);
  launch_outer_dact(dq_ + B_, l6.W, B_, H_, h2b, H_, DACT_RELU_OUT, d2b, H_, s);
  if (wgrad) {
    linear_wgrad(gemm_, s, B_, Mat{d2a, H_}, Mat{m20_[slot], 2 * H_}, l2, Mat(), 0, false);
    linear_wgrad(gemm_, s, B_, Mat{d2b, H_}, Mat{m20_[slot] + H_, 2 * H_}, l5, Mat(), 0, false);
  }
  linear_dgrad(gemm_, s, B_, Mat{d2a, H_}, l2, DACT_NONE, Mat(), dm20_, 2 * H_);
  linear_dgrad(gemm_, s, B_, Mat{d2b, H_}, l5, DACT_NONE, Mat(), dm20_ + H_, 2 * H_);
  launch_group_mean_bwd_dact(dm20_, hid1_[slot], 2 * H_, B_, NN_, 2 * H_, DACT_RELU_OUT, dhid1_, bpart_, s);
  if (wgrad) {
    linear_wgrad(gemm_, s, B_ * NN_, Mat{dhid1_, 2 * H_}, Mat{xs_[slot], LF_}, l14, Mat(), 0, false);
    const ColJob jobs[7] = {ColJob{h2a, dq_, l3.dW, H_, B_, H_},       ColJob{dq_, nullptr, l3.db, 1, B_, 1},
                            ColJob{h2b, dq_ + B_, l6.dW, H_, B_, H_},  ColJob{dq_ + B_, nullptr, l6.db, 1, B_, 1},
                            bias_job(B_, Mat{d2a, H_}, l2),            bias_job(B_, Mat{d2b, H_}, l5),
                            bias_job(B_, Mat{bpart_, 2 * H_}, l14)};
    launch_colreduce_multi(jobs, 7, s);
  }
  linear_dgrad(gemm_, s, B_ * NN_, Mat{dhid1_, 2 * H_}, l14, DACT_NONE, Mat(), dxs_, LF_, 0, LF_);
  launch_gauss_noise_expand_bwd(dxs_, LF_, raw, LF_, B_, D_, noise, NN_, cfg_.c_noise, dm, draw, s);
}

// Actor.forward (drqv2.py:134-150) + TruncatedNormal.sample(clip): trunk (Linear, LayerNorm, tanh) -> policy MLP -> tanh
void MulvDrq::actor_forward(const float* latent, int ld_latent, const float* eps, float stddev, float* action_out,
                            int ld_action, bool keep) {
  cudaStream_t s = stream_;
  const Linear l0 = p0_.view(actor_g_), l1 = p1_.view(actor_g_), l2 = p2_.view(actor_g_);
  Linear lt = at_.view(actor_g_);
  lt.out = LF_;  // padded rows are zero: the padding columns of tpre_ come out as exact zeros
  linear_fwd(gemm_, s, B_, Mat{latent, ld_latent}, lt, ACT_NONE, tpre_, LF_);
  launch_ln_act_fwd(tpre_, LF_, B_, D_, actor_g_.p + aln_w_, actor_g_.p + aln_b_, true, th_, LF_, LF_,
                    keep ? xhat_a_ : nullptr, LF_, keep ? rstd_a_ : nullptr, s);
  linear_fwd(gemm_, s, B_, Mat{th_, LF_}, l0, ACT_RELU, ap1_, H_);
  linear_fwd(gemm_, s, B_, Mat{ap1_, H_}, l1, ACT_RELU, ap2_, H_);
  linear_fwd(gemm_, s, B_, Mat{ap2_, H_}, l2, ACT_NONE, raw_a_, LA_);
  launch_trunc_normal_sample(raw_a_, LA_, B_, A_, eps, stddev, cfg_.stddev_clip, mu_, action_out, ld_action, s);
}

// act (drqv2.py:270-282) on n observations: the small-batch policy (pixel_act.cu) over this handle's parameters,
// created on first use
void MulvDrq::act_batch(const unsigned char* obs, const float* eps_host, float stddev, int n, float* actions_host) {
  if (!policy_)
    policy_.reset(new PixelPolicy(cfg_.channels, cfg_.height, A_,
                                  actor_policy_weights(*enc_, actor_g_, at_, aln_w_, aln_b_, p0_, p1_, p2_), stream_));
  policy_->act(obs, eps_host, stddev, n, actions_host);
}

void MulvDrq::update(const unsigned char* img, const float* action, const float* reward, const float* discount,
                     const unsigned char* next_img, const unsigned char* img_step1, const int* shifts, const float* eps_z,
                     const float* eps_act, const float* noise, float stddev, float* metrics_out) {
  cudaStream_t s = stream_;
  const size_t img_bytes = (size_t)B_ * cfg_.channels * cfg_.height * cfg_.height;
  const size_t step1_bytes = (size_t)B_ * 3 * cfg_.height * cfg_.height;
  RLREP_CUDA(cudaStreamSynchronize(s));
  unsigned char* st = stage_host_;
  auto put = [&](void* dev, const void* src, size_t bytes) { stage_h2d(st, dev, src, bytes, s); };
  put(img_dev_, img, img_bytes);
  put(next_img_dev_, next_img, img_bytes);
  put(step1_dev_, img_step1, step1_bytes);
  put(shifts_dev_, shifts, (size_t)4 * B_ * sizeof(int));
  put(eps_z_dev_, eps_z, (size_t)B_ * D_ * sizeof(float));
  put(eps_act_dev_, eps_act, (size_t)2 * B_ * A_ * sizeof(float));
  put(noise_dev_, noise, (size_t)3 * NN_ * D_ * sizeof(float));
  put(action_dev_, action, (size_t)B_ * A_ * sizeof(float));
  put(reward_dev_, reward, B_ * sizeof(float));
  put(discount_dev_, discount, B_ * sizeof(float));
  finish_update(stddev, metrics_out, 8);
}

// Every launch of one update on the batch currently resident in the device buffers.
void MulvDrq::launch_update(float stddev) {
  cudaStream_t s = stream_;
  const float w = cfg_.vae_w * cfg_.mse_w;
  const float* noise_t = noise_dev_;
  const float* noise_c = noise_dev_ + (size_t)NN_ * D_;
  const float* noise_a = noise_dev_ + (size_t)2 * NN_ * D_;

  TickParams t;
  t.k_feat = 1;
  t.period = 1;
  t.lr_feat = t.lr_critic = t.lr_actor = cfg_.lr;  // eight Adam optimisers, one learning rate, one step count
  t.lr_alpha = 0.0;
  t.critic_steps = 1;
  launch_tick(ctl_, t, s);

  // ---- target_Q (drqv2.py:379-388, no grad).  next_img first: its encoder activations are not needed again.
  enc_->forward(next_img_dev_, shifts_dev_ + 2 * B_, nsa_, LDS_, /*target=*/true);
  actor_forward(nsa_, LDS_, eps_act_dev_, stddev, nsa_ + F_, LDS_, /*keep=*/false);
  gauss_forward(ff_, ff_g_, /*target=*/true, Mat{nsa_, LDS_}, gn_, false);
  critic_forward(/*target=*/true, 0, gn_.m, gn_.raw, noise_t);

  // ---- model forward (drqv2.py:343-377)
  enc_->forward(img_dev_, shifts_dev_, enc_in_, LDE_, false);
  {
    const ColSegment seg{0, F_, A_};
    launch_pack_columns(action_dev_, A_, enc_in_, LDE_, B_, &seg, 1, s);
  }
  penc_->forward(step1_dev_, nullptr, enc_in_ + F_ + A_, LDE_, false);
  const Mat xe{enc_in_, LDE_};  // feat_encoder reads [state | action | state1]; feat_f and the actor the leading columns
  gauss_forward(fe_, fe_g_, false, xe, ge_, true);
  launch_gauss_sample(ge_.m, ge_.raw, LF_, B_, D_, eps_z_dev_, z_, LF_, s);
  const Linear d1 = d1_.view(fd_g_), d2 = d2_.view(fd_g_), ds = ds_.view(fd_g_), dr = dr_.view(fd_g_);
  linear_fwd(gemm_, s, B_, Mat{z_, LF_}, d1, ACT_RELU, fh1_, H_);
  linear_fwd(gemm_, s, B_, Mat{fh1_, H_}, d2, ACT_RELU, fh2_, H_);
  linear_fwd(gemm_, s, B_, Mat{fh2_, H_}, ds, ACT_NONE, s_hat_, F_);
  launch_rowdot(fh2_, H_, B_, H_, dr.W, dr.b, r_hat_, s);
  dec_->forward(s_hat_, F_);
  dec_->l1_loss(step1_dev_, w, metrics_dev_ + 4);
  launch_reward_mse(r_hat_, reward_dev_, B_, w, dr_hat_, metrics_dev_ + 5, s);
  gauss_forward(ff_, ff_g_, false, xe, gf_, true);
  critic_forward(false, 1, gf_.m, gf_.raw, noise_c);
  launch_huber_critic_loss(reward_dev_, discount_dev_, q_[0], q_[0] + B_, q_[1], q_[1] + B_, B_, dq_, dq_ + B_,
                           metrics_dev_ + 0, s);

  // ---- backward: critic -> feat_f head;  decoder -> feat_decoder -> z;  KL joins both heads
  critic_backward(1, gf_.raw, noise_c, /*wgrad=*/true, dcm_, dcraw_);
  dec_->backward(ds_hat_, F_);
  linear_wgrad(gemm_, s, B_, Mat{ds_hat_, F_}, Mat{fh2_, H_}, ds, Mat(), 0, false);
  {  // d fh2 = (d s_hat W_s + d r_hat (x) w_r) * relu'(fh2)
    GemmArgs a;
    a.M = B_; a.N = H_; a.K = F_;
    a.A = ds_hat_; a.lda = F_;
    a.B = ds.W; a.ldb = ds.ld; a.b_mn = true;
    a.C = dfh2_; a.ldc = H_;
    a.epi.r1_u = dr_hat_; a.epi.r1_v = dr.W;
    a.epi.dact = DACT_RELU_OUT; a.epi.aux = fh2_; a.epi.ld_aux = H_;
    gemm_.run(a, s);
  }
  linear_wgrad(gemm_, s, B_, Mat{dfh2_, H_}, Mat{fh1_, H_}, d2, Mat(), 0, false);
  linear_dgrad(gemm_, s, B_, Mat{dfh2_, H_}, d2, DACT_RELU_OUT, Mat{fh1_, H_}, dfh1_, H_);
  linear_wgrad(gemm_, s, B_, Mat{dfh1_, H_}, Mat{z_, LF_}, d1, Mat(), 0, false);
  linear_dgrad(gemm_, s, B_, Mat{dfh1_, H_}, d1, DACT_NONE, Mat(), dz_, LF_, 0, LF_);
  {
    const ColJob jobs[5] = {bias_job(B_, Mat{ds_hat_, F_}, ds), ColJob{fh2_, dr_hat_, dr.dW, H_, B_, H_},
                            ColJob{dr_hat_, nullptr, dr.db, 1, B_, 1}, bias_job(B_, Mat{dfh2_, H_}, d2),
                            bias_job(B_, Mat{dfh1_, H_}, d1)};
    launch_colreduce_multi(jobs, 5, s);
  }
  launch_gauss_kl_bwd(ge_.m, ge_.raw, gf_.m, gf_.raw, LF_, B_, D_, eps_z_dev_, dz_, cfg_.vae_w, dcm_, dcraw_, dm1_, draw1_,
                      dm2_, draw2_, kl_partial_, kKlBlocks, s);
  launch_sum_scaled(kl_partial_, kKlBlocks, 1.f / ((float)B_ * (float)D_), metrics_dev_ + 6, s);

  // ---- feat_encoder backward -> d state, d state1;  feat_f backward accumulates into d state
  gauss_backward(fe_, fe_g_, xe, ge_, dm1_, draw1_, true);
  {
    const Linear le = fe_.lin.view(fe_g_);
    linear_dgrad(gemm_, s, B_, Mat{dpre_, 2 * LF_}, le, DACT_NONE, Mat(), dstate_, F_, 0, F_);
    linear_dgrad(gemm_, s, B_, Mat{dpre_, 2 * LF_}, le, DACT_NONE, Mat(), dstep1_, F_, F_ + A_, F_);
  }
  penc_->backward(dstep1_, F_);
  gauss_backward(ff_, ff_g_, xe, gf_, dm2_, draw2_, true);
  {
    const Linear lf = ff_.lin.view(ff_g_);
    GemmArgs a;
    a.M = B_; a.N = F_; a.K = lf.out;
    a.A = dpre_; a.lda = 2 * LF_;
    a.B = lf.W; a.ldb = lf.ld; a.b_mn = true;
    a.C = dstate_; a.ldc = F_;
    a.epi.accumulate = 1;
    gemm_.run(a, s);
  }
  enc_->backward(dstate_, F_);

  // ---- the seven optimisers (drqv2.py:403-423); soft updates (:441-451) ride on the Adam kernels
  auto adam = [&](ParamGroup& g, const AdamHyper* h) {
    launch_adam_polyak(g.p, g.g, g.m, g.v, g.n, h, g.n_target ? g.target : nullptr, g.n_target, cfg_.tau, nullptr, s);
  };
  adam(enc_->group(), &ctl_->critic);
  adam(penc_->group(), &ctl_->critic);
  adam(dec_->group(), &ctl_->critic);
  adam(fe_g_, &ctl_->critic);
  adam(fd_g_, &ctl_->critic);
  adam(ff_g_, &ctl_->critic);
  adam(crit_g_, &ctl_->critic);

  // ---- actor step (drqv2.py:284-311) on the detached state, against the just-updated feat_f and critic
  actor_forward(enc_in_, LDE_, eps_act_dev_ + (size_t)B_ * A_, stddev, enc_in_ + F_, LDE_, /*keep=*/true);
  gauss_forward(ff_, ff_g_, false, xe, gf_, true);
  critic_forward(false, 0, gf_.m, gf_.raw, noise_a);
  launch_drq_actor_loss(q_[0], q_[0] + B_, B_, dq_, dq_ + B_, metrics_dev_ + 7, s);
  critic_backward(0, gf_.raw, noise_a, /*wgrad=*/false, dcm_, dcraw_);
  gauss_backward(ff_, ff_g_, xe, gf_, dcm_, dcraw_, /*wgrad=*/false);
  {
    const Linear lf = ff_.lin.view(ff_g_);
    linear_dgrad(gemm_, s, B_, Mat{dpre_, 2 * LF_}, lf, DACT_NONE, Mat(), daction_, LA_, F_, A_);
    const Linear l0 = p0_.view(actor_g_), l1 = p1_.view(actor_g_), l2 = p2_.view(actor_g_), lt = at_.view(actor_g_);
    launch_trunc_normal_bwd(daction_, LA_, mu_, B_, A_, draw_a_, LA_, s);
    linear_wgrad(gemm_, s, B_, Mat{draw_a_, LA_}, Mat{ap2_, H_}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{draw_a_, LA_}, l2, DACT_RELU_OUT, Mat{ap2_, H_}, dap2_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dap2_, H_}, Mat{ap1_, H_}, l1, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dap2_, H_}, l1, DACT_RELU_OUT, Mat{ap1_, H_}, dap1_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dap1_, H_}, Mat{th_, LF_}, l0, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dap1_, H_}, l0, DACT_NONE, Mat(), dth_, LF_, 0, LF_);
    launch_ln_act_bwd(dth_, LF_, th_, LF_, xhat_a_, LF_, rstd_a_, B_, D_, actor_g_.p + aln_w_, true, dtpre_, LF_, LF_, gb_,
                      gg_, LF_, s);
    Linear lp = lt;
    lp.out = LF_;
    linear_wgrad(gemm_, s, B_, Mat{dtpre_, LF_}, Mat{enc_in_, LDE_}, lp, Mat(), 0, false);
    const ColJob jobs[6] = {bias_job(B_, Mat{draw_a_, LA_}, l2), bias_job(B_, Mat{dap2_, H_}, l1),
                            bias_job(B_, Mat{dap1_, H_}, l0),    bias_job(B_, Mat{dtpre_, LF_}, lt),
                            ColJob{gg_, nullptr, actor_g_.g + aln_w_, LF_, B_, D_},
                            ColJob{gb_, nullptr, actor_g_.g + aln_b_, LF_, B_, D_}};
    launch_colreduce_multi(jobs, 6, s);
  }
  launch_adam_polyak(actor_g_.p, actor_g_.g, actor_g_.m, actor_g_.v, actor_g_.n, &ctl_->actor, nullptr, 0, 0.f, nullptr, s);
}

}  // namespace rlrep

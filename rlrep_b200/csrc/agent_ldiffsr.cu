// Latent Diff-SR DrQ-v2 pixel update (reference: agent/diffsrdrq/latent_diff_sr.py:306-390 `train_step` with `ae_step`
// :234-259, `score_step` :275-304, `critic_step` :355-379, `actor_step` :381-390, `update_target` :135-139) on
// configs/latent_diff_sr.yaml's path: use_repr_target, back_critic_grad, critic_loss mse, reg_coef 0, grad_norm null,
// extra_repr_step 1, do_scale false, repr_coef 1.  The checker is oracle/ldiffsr_oracle.py (bit-identical to the
// reference class on tests/golden/ldiffsr_b4.npz).
//
// Per update: target branch (vae_target on next_img_stack's frames -> actor -> psi_target -> critic_target) ->
// per-frame VAE on the 3B + B frames (conv encoder, LayerNorm+swish head, posterior sample, transposed-conv decoder,
// MSE-sum + KL) -> factored score matching: psi on [latent ; latent_mode] as ONE 2B-row pass (rows [0, B) feed the
// score loss, rows [B, 2B) are the critic's features; both run the online weights in training mode with their own
// host-drawn dropout masks), zeta on the perturbed next latent, score = psi . zeta / feat through the Diff-SR-SAC
// kernels -> RFF critic (LayerNorm in front) with the TD loss, gradient into psi and the VAE mean -> one backward ->
// Adam(vae), AdamW(score), Adam(critic) -> actor step through the FROZEN psi target (still the pre-update target) and the
// new critic -> Adam(actor) -> soft updates.
#include "ldiffsr.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

#include "staging.cuh"

namespace rlrep {

void ResNetActs::want(DeviceArena& a, const ResNetSlots& n, int rows) {
  const size_t R = (size_t)rows;
  a.want(&x, R * n.h);
  a.want(&m, R * n.h);
  const size_t nb = n.blocks.size();
  hm.assign(nb, nullptr); hn.assign(nb, nullptr); xhat.assign(nb, nullptr); rstd.assign(nb, nullptr);
  pre1.assign(nb, nullptr); a1.assign(nb, nullptr);
  for (size_t b = 0; b < nb; ++b) {
    a.want(&hm[b], R * n.h); a.want(&hn[b], R * n.h); a.want(&xhat[b], R * n.h); a.want(&rstd[b], R);
    a.want(&pre1[b], R * 4 * n.h); a.want(&a1[b], R * 4 * n.h);
  }
}

ResNetSlots LatentDiffSR::add_resnet(const std::string& prefix, int depth, int in, int out, int h) {
  RLREP_CHECK(in % 32 == 0 && h % 32 == 0 && out % 32 == 0, "MLP-ResNet widths must be multiples of 32");
  ResNetSlots n;
  n.in = in; n.h = h; n.out = out;
  n.fc = add_linear(score_g_, prefix + ".fc", h, in);
  for (int b = 0; b < depth; ++b) {
    const std::string bp = prefix + ".blocks." + std::to_string(b);
    ResBlockSlots s;
    s.ln_w = score_g_.add(bp + ".layer_norm.weight", h, 1);
    s.ln_b = score_g_.add(bp + ".layer_norm.bias", h, 1);
    s.fc1 = add_linear(score_g_, bp + ".fc1", 4 * h, h);
    s.fc2 = add_linear(score_g_, bp + ".fc2", h, 4 * h);
    // the block's `residual` Linear is never reached (input and output widths agree, score_idql.py:38-39): it has no
    // gradient, so torch's AdamW skips it entirely -- kept outside the optimiser group, exported like any weight
    add_linear(dead_g_, bp + ".residual", h, h);
    n.blocks.push_back(s);
  }
  n.out_fc = add_linear(score_g_, prefix + ".out_fc", out, h);
  return n;
}

LatentDiffSR::LatentDiffSR(const LdiffConfig& c, cudaStream_t s)
    : PixelAgent(s), cfg_(c), B_(c.batch), N_(4 * c.batch), A_(c.action_dim), L_(c.latent), feat_(c.feat), bn_(c.bn),
      H_(c.hidden) {
  RLREP_CHECK(B_ > 0 && A_ > 0 && L_ % 64 == 0 && feat_ % 32 == 0 && bn_ % 32 == 0 && H_ % 32 == 0,
              "bad latent Diff-SR dimensions (latent % 64, feature / bn / hidden % 32)");
  RLREP_CHECK(c.ae_lr == c.score_lr, "vae and score optimisers share one Adam step-size slot: ae_lr must equal score_lr");
  const Precision prec = static_cast<Precision>(c.precision);
  enc_.reset(new ConvEncoder(N_, 3, 84, prec, s, /*with_target=*/true));
  enc_->group().name = "vae.encoder";
  enc_->group().target_prefix_from = "vae.";
  enc_->group().target_prefix_to = "vae_target.";
  dec_.reset(new ConvDecoder(N_, prec, s, /*out_kernel=*/3, /*with_target=*/true));
  dec_->group().name = "vae.decoder";
  dec_->group().target_prefix_from = "vae.";
  dec_->group().target_prefix_to = "vae_target.";
  F_ = enc_->feature_dim();
  LA_ = round_up32(A_);
  T_ = L_ / 2;
  LZ_ = L_ + T_;

  vh_g_.name = "vae_head";
  efc_ = add_linear(vh_g_, "vae.encoder.fc", L_, F_);
  eln_w_ = vh_g_.add("vae.encoder.ln.weight", L_, 1);
  eln_b_ = vh_g_.add("vae.encoder.ln.bias", L_, 1);
  eout_ = add_linear(vh_g_, "vae.encoder.out", 2 * L_, L_);
  dfc_ = add_linear(vh_g_, "vae.decoder.fc", F_, L_);
  vh_g_.n_target = vh_g_.n;
  vh_g_.target_prefix_from = "vae.";
  vh_g_.target_prefix_to = "vae_target.";
  vh_g_.want(arena_);

  score_g_.name = "score";
  dead_g_.name = "score_dead";
  bneck_.s_lin = add_linear(score_g_, "score.psi_bottleneck1.0", bn_, 3 * L_);
  bneck_.s_lnw = score_g_.add("score.psi_bottleneck1.1.weight", bn_, 1);
  bneck_.s_lnb = score_g_.add("score.psi_bottleneck1.1.bias", bn_, 1);
  bneck_.a_lin = add_linear(score_g_, "score.psi_bottleneck2.0", bn_, A_);
  bneck_.a_lnw = score_g_.add("score.psi_bottleneck2.1.weight", bn_, 1);
  bneck_.a_lnb = score_g_.add("score.psi_bottleneck2.1.bias", bn_, 1);
  psi_ = add_resnet("score.psi", c.psi_d, 2 * bn_, feat_, c.psi_h);
  zeta_ = add_resnet("score.zeta", c.zeta_d, LZ_, L_ * feat_, c.zeta_h);
  for (ParamGroup* g : {&score_g_, &dead_g_}) {
    g->n_target = g->n;
    g->target_prefix_from = "score.";
    g->target_prefix_to = "score_target.";
  }
  score_g_.want(arena_);
  dead_g_.want(arena_, /*with_opt=*/false);

  actor_g_.name = "actor";
  at_ = add_linear(actor_g_, "actor.trunk.0", bn_, 3 * L_);
  aln_w_ = actor_g_.add("actor.trunk.1.weight", bn_, 1);
  aln_b_ = actor_g_.add("actor.trunk.1.bias", bn_, 1);
  p0_ = add_linear(actor_g_, "actor.policy.0", H_, bn_);
  p1_ = add_linear(actor_g_, "actor.policy.2", H_, H_);
  p2_ = add_linear(actor_g_, "actor.policy.4", A_, H_);
  actor_g_.want(arena_);

  crit_g_.name = "critic";
  cln_w_ = crit_g_.add("critic.ln.weight", feat_, 1);
  cln_b_ = crit_g_.add("critic.ln.bias", feat_, 1);
  rff_.plan(crit_g_, arena_, feat_, H_, B_);
  crit_g_.n_target = crit_g_.n;
  crit_g_.target_prefix_from = "critic.";
  crit_g_.target_prefix_to = "critic_target.";
  crit_g_.want(arena_);

  const size_t frame = (size_t)3 * 84 * 84, NL = (size_t)N_ * L_, NF = (size_t)N_ * F_, B2 = 2 * (size_t)B_;
  arena_.want(&ctl_, 1);
  arena_.want(&metrics_dev_, 8);
  arena_.want(&frames_dev_, N_ * frame);
  arena_.want(&next_frames_dev_, N_ * frame);  // 3B valid frames; the encoder handle runs N-frame batches
  arena_.want(&shifts_dev_, 2 * N_);
  arena_.want(&next_shifts_dev_, 2 * N_);
  arena_.want(&action_dev_, (size_t)B_ * A_); arena_.want(&reward_dev_, B_); arena_.want(&discount_dev_, B_);
  arena_.want(&eps_post_dev_, NL); arena_.want(&ab_dev_, B_); arena_.want(&temb_dev_, (size_t)B_ * T_);
  arena_.want(&noise_dev_, (size_t)B_ * L_);
  arena_.want(&psi_masks_dev_, (size_t)c.psi_d * B2 * c.psi_h);
  arena_.want(&zeta_masks_dev_, (size_t)c.zeta_d * B_ * c.zeta_h);
  arena_.want(&eps_act_dev_, (size_t)2 * B_ * A_);
  arena_.want(&feat_buf_, NF); arena_.want(&tfeat_, NF); arena_.want(&dfeat_, NF);
  arena_.want(&hpre_, NL); arena_.want(&hs_, NL); arena_.want(&hxhat_, NL); arena_.want(&hrstd_, N_);
  arena_.want(&h2_, 2 * NL); arena_.want(&h2t_, 2 * NL); arena_.want(&mean_, NL); arena_.want(&tmean_, NL);
  arena_.want(&z_, NL); arena_.want(&kl_partial_, kKlBlocks);
  arena_.want(&dec_in_, NF); arena_.want(&ddec_in_, NF);
  arena_.want(&dz_, NL); arena_.want(&dh2_, 2 * NL); arena_.want(&dhs_, NL); arena_.want(&dhpre_, NL);
  arena_.want(&psi_in_, B2 * 3 * L_); arena_.want(&act2_, B2 * LA_);
  arena_.want(&psi_out_, B2 * feat_); arena_.want(&dpsi_out_, B2 * feat_);
  arena_.want(&dpsi_in_, B2 * 3 * L_); arena_.want(&dcat_, B2 * 2 * bn_);
  arena_.want(&zin_, (size_t)B_ * LZ_); arena_.want(&dzin_, (size_t)B_ * LZ_);
  arena_.want(&flat_, (size_t)B_ * feat_ * L_); arena_.want(&dflat_, (size_t)B_ * feat_ * L_);
  arena_.want(&target_, (size_t)B_ * L_); arena_.want(&coef_, B_); arena_.want(&dscore_, (size_t)B_ * L_);
  arena_.want(&loss_rows_, B_);
  for (BottleneckActs* a : {&bn_on_, &bn_t_}) {
    const size_t R = a == &bn_on_ ? B2 : (size_t)B_;
    arena_.want(&a->pre_s, R * bn_); arena_.want(&a->pre_a, R * bn_); arena_.want(&a->cat, R * 2 * bn_);
    arena_.want(&a->xhat_s, R * bn_); arena_.want(&a->xhat_a, R * bn_); arena_.want(&a->rstd_s, R); arena_.want(&a->rstd_a, R);
  }
  psi_on_.want(arena_, psi_, (int)B2);
  psi_t_.want(arena_, psi_, B_);
  zeta_on_.want(arena_, zeta_, B_);
  arena_.want(&feat_t_, (size_t)B_ * feat_); arena_.want(&dfeat_t_, (size_t)B_ * feat_);
  arena_.want(&dcat_t_, (size_t)B_ * 2 * bn_);
  const int hmax = std::max(c.psi_h, c.zeta_h);
  arena_.want(&dx_, B2 * hmax); arena_.want(&dtmp_h_, B2 * hmax); arena_.want(&dhm_, B2 * hmax);
  arena_.want(&d4_, B2 * 4 * hmax); arena_.want(&gb_, B2 * std::max(hmax, bn_)); arena_.want(&gg_, B2 * std::max(hmax, bn_));
  arena_.want(&dpre_s_, B2 * bn_);
  for (int i = 0; i < 2; ++i) arena_.want(&cn_[i], (size_t)B_ * feat_);
  arena_.want(&cxhat_, (size_t)B_ * feat_); arena_.want(&crstd_, B_); arena_.want(&dcn_, (size_t)B_ * feat_);
  arena_.want(&dq_, 2 * B_);
  arena_.want(&act_t_, (size_t)B_ * LA_); arena_.want(&acta_, (size_t)B_ * LA_); arena_.want(&dacta_, (size_t)B_ * LA_);
  const size_t Bb = (size_t)B_ * bn_, BH = (size_t)B_ * H_;
  arena_.want(&tpre_, Bb); arena_.want(&th_, Bb); arena_.want(&xhat_a_, Bb); arena_.want(&rstd_a_, B_);
  arena_.want(&ap1_, BH); arena_.want(&ap2_, BH); arena_.want(&dap1_, BH); arena_.want(&dap2_, BH);
  arena_.want(&raw_a_, (size_t)B_ * LA_); arena_.want(&mu_, (size_t)B_ * A_); arena_.want(&draw_a_, (size_t)B_ * LA_);
  arena_.want(&dth_, Bb); arena_.want(&dtpre_, Bb);
  arena_.commit();
  gemm_.init(prec, 0);

  alloc_host(2 * N_ * frame + (size_t)4 * N_ * sizeof(int) +
             ((size_t)B_ * A_ + 2 * B_ + NL + B_ + (size_t)B_ * T_ + (size_t)B_ * L_ + (size_t)c.psi_d * B2 * c.psi_h +
              (size_t)c.zeta_d * B_ * c.zeta_h + (size_t)2 * B_ * A_) * sizeof(float));
  Control h;
  std::memset(&h, 0, sizeof(h));
  RLREP_CUDA(cudaMemcpyAsync(ctl_, &h, sizeof(h), cudaMemcpyHostToDevice, stream_));
  RLREP_CUDA(cudaStreamSynchronize(stream_));
}

// ---------------------------------------------------------------------------------------------- MLP-ResNet (psi / zeta)
// masks: [depth][rows, h] host-drawn Bernoulli(1 - p) masks (nullptr = eval mode: no dropout)
void LatentDiffSR::resnet_forward(const ResNetSlots& n, bool target, int rows, Mat in, const float* masks, size_t mask_stride,
                                  ResNetActs& a, float* out, int ld_out) {
  cudaStream_t s = stream_;
  const float* base = target ? score_g_.target : score_g_.p;
  const float inv_keep = 1.f / (1.f - cfg_.dropout);
  const size_t Rh = (size_t)rows * n.h;
  linear_fwd(gemm_, s, rows, in, n.fc.view(score_g_, target), ACT_NONE, a.x, n.h);
  for (size_t b = 0; b < n.blocks.size(); ++b) {
    const ResBlockSlots& k = n.blocks[b];
    const float* ln_in = a.x;
    if (masks != nullptr) {
      launch_mask_scale(a.x, masks + b * mask_stride, inv_keep, Rh, 0, a.hm[b], s);
      ln_in = a.hm[b];
    }
    launch_ln_act2_fwd(ln_in, n.h, rows, n.h, base + k.ln_w, base + k.ln_b, 0, a.hn[b], n.h, n.h, a.xhat[b], n.h, a.rstd[b], s);
    linear_fwd(gemm_, s, rows, Mat{a.hn[b], n.h}, k.fc1.view(score_g_, target), ACT_NONE, a.pre1[b], 4 * n.h);
    launch_mish_fwd(a.pre1[b], Rh * 4, a.a1[b], s);
    const Linear l2 = k.fc2.view(score_g_, target);
    GemmArgs g;  // x += mish(.) W2^T + b2   (the residual add rides on the epilogue)
    g.M = rows; g.N = n.h; g.K = 4 * n.h;
    g.A = a.a1[b]; g.lda = 4 * n.h;
    g.B = l2.W; g.ldb = l2.ld;
    g.C = a.x; g.ldc = n.h;
    g.epi.bias = l2.b;
    g.epi.accumulate = 1;
    gemm_.run(g, s);
  }
  launch_mish_fwd(a.x, Rh, a.m, s);
  linear_fwd(gemm_, s, rows, Mat{a.m, n.h}, n.out_fc.view(score_g_, target), ACT_NONE, out, ld_out);
}

// dout -> parameter gradients (wgrad) and / or din [rows, n.in]
void LatentDiffSR::resnet_backward(const ResNetSlots& n, bool target, int rows, Mat in, const float* masks, size_t mask_stride,
                                   ResNetActs& a, Mat dout, bool wgrad, float* din) {
  cudaStream_t s = stream_;
  const float* base = target ? score_g_.target : score_g_.p;
  const float inv_keep = 1.f / (1.f - cfg_.dropout);
  const size_t Rh = (size_t)rows * n.h;
  const Linear lo = n.out_fc.view(score_g_, target);
  if (wgrad) {
    linear_wgrad(gemm_, s, rows, dout, Mat{a.m, n.h}, lo, Mat(), 0, false);
    const ColJob j = bias_job(rows, dout, lo);
    launch_colreduce_multi(&j, 1, s);
  }
  linear_dgrad(gemm_, s, rows, dout, lo, DACT_NONE, Mat(), dtmp_h_, n.h);
  launch_mish_bwd(dtmp_h_, a.x, Rh, dx_, s);  // a.x still holds the input of the final Mish
  for (int b = (int)n.blocks.size() - 1; b >= 0; --b) {
    const ResBlockSlots& k = n.blocks[b];
    const Linear l1 = k.fc1.view(score_g_, target), l2 = k.fc2.view(score_g_, target);
    if (wgrad) linear_wgrad(gemm_, s, rows, Mat{dx_, n.h}, Mat{a.a1[b], 4 * n.h}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, s, rows, Mat{dx_, n.h}, l2, DACT_NONE, Mat(), d4_, 4 * n.h);
    launch_mish_bwd(d4_, a.pre1[b], Rh * 4, d4_, s);
    if (wgrad) linear_wgrad(gemm_, s, rows, Mat{d4_, 4 * n.h}, Mat{a.hn[b], n.h}, l1, Mat(), 0, false);
    linear_dgrad(gemm_, s, rows, Mat{d4_, 4 * n.h}, l1, DACT_NONE, Mat(), dtmp_h_, n.h);
    launch_ln_act2_bwd(dtmp_h_, n.h, nullptr, n.h, a.xhat[b], n.h, a.rstd[b], rows, n.h, base + k.ln_w, base + k.ln_b, 0, dhm_,
                       n.h, n.h, gb_, gg_, n.h, s);
    if (wgrad) {  // before dx_ changes: fc2's bias gradient is the column sum of the block's OUTPUT gradient
      const ColJob jobs[4] = {bias_job(rows, Mat{dx_, n.h}, l2), bias_job(rows, Mat{d4_, 4 * n.h}, l1),
                              ColJob{gg_, nullptr, score_g_.g + k.ln_w, n.h, rows, n.h},
                              ColJob{gb_, nullptr, score_g_.g + k.ln_b, n.h, rows, n.h}};
      launch_colreduce_multi(jobs, 4, s);
    }
    // dx += d(masked input) * mask / keep   (the residual path passes dx through unchanged)
    launch_mask_scale(dhm_, masks ? masks + (size_t)b * mask_stride : nullptr, inv_keep, Rh, 1, dx_, s);
  }
  const Linear lf = n.fc.view(score_g_, target);
  if (wgrad) {
    linear_wgrad(gemm_, s, rows, Mat{dx_, n.h}, in, lf, Mat(), 0, false);
    const ColJob j = bias_job(rows, Mat{dx_, n.h}, lf);
    launch_colreduce_multi(&j, 1, s);
  }
  if (din != nullptr) linear_dgrad(gemm_, s, rows, Mat{dx_, n.h}, lf, DACT_NONE, Mat(), din, n.in);
}

// psi_bottleneck1 / 2 (score_idql.py:150-160, :172-176): cat = [tanh(LN(W1 state)) | tanh(LN(W2 action))]
void LatentDiffSR::bottleneck_forward(bool target, int rows, Mat state, Mat action, BottleneckActs& a) {
  cudaStream_t s = stream_;
  const float* base = target ? score_g_.target : score_g_.p;
  linear_fwd(gemm_, s, rows, state, bneck_.s_lin.view(score_g_, target), ACT_NONE, a.pre_s, bn_);
  launch_ln_act2_fwd(a.pre_s, bn_, rows, bn_, base + bneck_.s_lnw, base + bneck_.s_lnb, 1, a.cat, 2 * bn_, bn_, a.xhat_s, bn_,
                     a.rstd_s, s);
  linear_fwd(gemm_, s, rows, action, bneck_.a_lin.view(score_g_, target), ACT_NONE, a.pre_a, bn_);
  launch_ln_act2_fwd(a.pre_a, bn_, rows, bn_, base + bneck_.a_lnw, base + bneck_.a_lnb, 1, a.cat + bn_, 2 * bn_, bn_, a.xhat_a,
                     bn_, a.rstd_a, s);
}

void LatentDiffSR::bottleneck_backward(bool target, int rows, Mat state, Mat action, BottleneckActs& a, const float* dcat,
                                       bool wgrad, float* dstate, float* daction) {
  cudaStream_t s = stream_;
  const float* base = target ? score_g_.target : score_g_.p;
  const Linear ls = bneck_.s_lin.view(score_g_, target), la = bneck_.a_lin.view(score_g_, target);
  // state half
  launch_ln_act2_bwd(dcat, 2 * bn_, a.cat, 2 * bn_, a.xhat_s, bn_, a.rstd_s, rows, bn_, base + bneck_.s_lnw, base + bneck_.s_lnb,
                     1, dpre_s_, bn_, bn_, gb_, gg_, bn_, s);
  if (wgrad) {
    linear_wgrad(gemm_, s, rows, Mat{dpre_s_, bn_}, state, ls, Mat(), 0, false);
    const ColJob jobs[3] = {bias_job(rows, Mat{dpre_s_, bn_}, ls), ColJob{gg_, nullptr, score_g_.g + bneck_.s_lnw, bn_, rows, bn_},
                            ColJob{gb_, nullptr, score_g_.g + bneck_.s_lnb, bn_, rows, bn_}};
    launch_colreduce_multi(jobs, 3, s);
  }
  if (dstate != nullptr) linear_dgrad(gemm_, s, rows, Mat{dpre_s_, bn_}, ls, DACT_NONE, Mat(), dstate, 3 * L_);
  // action half
  launch_ln_act2_bwd(dcat + bn_, 2 * bn_, a.cat + bn_, 2 * bn_, a.xhat_a, bn_, a.rstd_a, rows, bn_, base + bneck_.a_lnw,
                     base + bneck_.a_lnb, 1, dpre_s_, bn_, bn_, gb_, gg_, bn_, s);
  if (wgrad) {
    linear_wgrad(gemm_, s, rows, Mat{dpre_s_, bn_}, action, la, Mat(), 0, false);
    const ColJob jobs[3] = {bias_job(rows, Mat{dpre_s_, bn_}, la), ColJob{gg_, nullptr, score_g_.g + bneck_.a_lnw, bn_, rows, bn_},
                            ColJob{gb_, nullptr, score_g_.g + bneck_.a_lnb, bn_, rows, bn_}};
    launch_colreduce_multi(jobs, 3, s);
  }
  if (daction != nullptr) linear_dgrad(gemm_, s, rows, Mat{dpre_s_, bn_}, la, DACT_NONE, Mat(), daction, LA_, 0, A_);
}

// vae_1d.Encoder.forward after the convolutions (:124-131): fc -> LayerNorm -> swish -> out;  h2 [N, 2L]
void LatentDiffSR::head_forward(bool target, const float* feat, bool keep, float* h2) {
  cudaStream_t s = stream_;
  const float* base = target ? vh_g_.target : vh_g_.p;
  linear_fwd(gemm_, s, N_, Mat{feat, F_}, efc_.view(vh_g_, target), ACT_NONE, hpre_, L_);
  launch_ln_act2_fwd(hpre_, L_, N_, L_, base + eln_w_, base + eln_b_, 2, hs_, L_, L_, keep ? hxhat_ : nullptr, L_,
                     keep ? hrstd_ : nullptr, s);
  linear_fwd(gemm_, s, N_, Mat{hs_, L_}, eout_.view(vh_g_, target), ACT_NONE, h2, 2 * L_);
}

// RFFCritic (network_arch/latent_diff_sr.py:117-141): LayerNorm, then the sin -> ELU -> linear twin heads
void LatentDiffSR::critic_forward(bool target, int slot, const float* feature, bool keep) {
  const float* base = target ? crit_g_.target : crit_g_.p;
  launch_ln_act2_fwd(feature, feat_, B_, feat_, base + cln_w_, base + cln_b_, 0, cn_[slot], feat_, feat_,
                     keep ? cxhat_ : nullptr, feat_, keep ? crstd_ : nullptr, stream_);
  rff_.forward(gemm_, stream_, crit_g_, target, slot, cn_[slot]);
}
// (dq1 | dq2) in dq_ -> dfeature [B, feat]; wgrad: also the critic's parameter gradients (online weights)
void LatentDiffSR::critic_backward(int slot, bool wgrad, float* dfeature) {
  cudaStream_t s = stream_;
  rff_.backward(gemm_, s, crit_g_, slot, cn_[slot], dq_, wgrad, dcn_);
  launch_ln_act2_bwd(dcn_, feat_, nullptr, feat_, cxhat_, feat_, crstd_, B_, feat_, crit_g_.p + cln_w_, crit_g_.p + cln_b_, 0,
                     dfeature, feat_, feat_, cn_[1 - slot], dcn_, feat_, s);  // g_beta -> cn_[1 - slot], g_gamma -> dcn_ (scratch)
  if (wgrad) {
    const ColJob jobs[2] = {ColJob{dcn_, nullptr, crit_g_.g + cln_w_, feat_, B_, feat_},
                            ColJob{cn_[1 - slot], nullptr, crit_g_.g + cln_b_, feat_, B_, feat_}};
    launch_colreduce_multi(jobs, 2, s);
  }
}

void LatentDiffSR::actor_forward(Mat latent, const float* eps, float stddev, float* action_out, int ld_action, bool keep) {
  cudaStream_t s = stream_;
  const Linear l0 = p0_.view(actor_g_), l1 = p1_.view(actor_g_), l2 = p2_.view(actor_g_), lt = at_.view(actor_g_);
  linear_fwd(gemm_, s, B_, latent, lt, ACT_NONE, tpre_, bn_);
  launch_ln_act2_fwd(tpre_, bn_, B_, bn_, actor_g_.p + aln_w_, actor_g_.p + aln_b_, 1, th_, bn_, bn_, keep ? xhat_a_ : nullptr,
                     bn_, keep ? rstd_a_ : nullptr, s);
  linear_fwd(gemm_, s, B_, Mat{th_, bn_}, l0, ACT_RELU, ap1_, H_);
  linear_fwd(gemm_, s, B_, Mat{ap1_, H_}, l1, ACT_RELU, ap2_, H_);
  linear_fwd(gemm_, s, B_, Mat{ap2_, H_}, l2, ACT_NONE, raw_a_, LA_);
  launch_trunc_normal_sample(raw_a_, LA_, B_, A_, eps, stddev, cfg_.stddev_clip, mu_, action_out, ld_action, s);
}

void LatentDiffSR::update(const Inputs& in, float* metrics_out) {
  cudaStream_t s = stream_;
  const size_t frame = (size_t)3 * 84 * 84, B2 = 2 * (size_t)B_;
  RLREP_CUDA(cudaStreamSynchronize(s));
  unsigned char* st = stage_host_;
  auto put = [&](void* dev, const void* src, size_t bytes) { stage_h2d(st, dev, src, bytes, s); };
  put(frames_dev_, in.frames, N_ * frame);
  put(next_frames_dev_, in.next_frames, 3 * B_ * frame);
  put(shifts_dev_, in.shifts, (size_t)2 * N_ * sizeof(int));
  put(next_shifts_dev_, in.next_shifts, (size_t)6 * B_ * sizeof(int));
  put(action_dev_, in.action, (size_t)B_ * A_ * 4);
  put(reward_dev_, in.reward, B_ * 4);
  put(discount_dev_, in.discount, B_ * 4);
  put(eps_post_dev_, in.eps_post, (size_t)N_ * L_ * 4);
  put(ab_dev_, in.alphabar, B_ * 4);
  put(temb_dev_, in.temb, (size_t)B_ * T_ * 4);
  put(noise_dev_, in.noise, (size_t)B_ * L_ * 4);
  put(psi_masks_dev_, in.psi_masks, (size_t)cfg_.psi_d * B2 * cfg_.psi_h * 4);
  put(zeta_masks_dev_, in.zeta_masks, (size_t)cfg_.zeta_d * B_ * cfg_.zeta_h * 4);
  put(eps_act_dev_, in.eps_act, (size_t)2 * B_ * A_ * 4);
  finish_update(in.stddev, metrics_out, 8);
}

void LatentDiffSR::launch_update(float stddev) {
  cudaStream_t s = stream_;
  const size_t B2 = 2 * (size_t)B_, BL3 = (size_t)B_ * 3 * L_;
  const Mat latent_mode{mean_, 3 * L_};  // rows 3b .. 3b + 2 of the [N, L] posterior means ARE row b of the [B, 3L] latent

  TickParams t;
  t.k_feat = 1;
  t.period = 1;
  t.lr_feat = cfg_.ae_lr;  // vae and score (equal learning rates, checked in the constructor)
  t.lr_critic = cfg_.critic_lr;
  t.lr_actor = cfg_.actor_lr;
  t.lr_alpha = 0.0;
  t.critic_steps = 1;
  launch_tick(ctl_, t, s);

  // ---- q_target (critic_step's no_grad block, :363-370): vae_target modes of next_img_stack's frames
  enc_->forward(next_frames_dev_, next_shifts_dev_, tfeat_, 0, /*target=*/true);
  head_forward(true, tfeat_, false, h2t_);
  {
    const ColSegment seg{0, 0, L_};
    launch_pack_columns(h2t_, 2 * L_, tmean_, L_, N_, &seg, 1, s);
  }
  actor_forward(Mat{tmean_, 3 * L_}, eps_act_dev_, stddev, act_t_, LA_, false);
  bottleneck_forward(true, B_, Mat{tmean_, 3 * L_}, Mat{act_t_, LA_}, bn_t_);
  resnet_forward(psi_, true, B_, Mat{bn_t_.cat, 2 * bn_}, nullptr, 0, psi_t_, feat_t_, feat_);
  critic_forward(true, 0, feat_t_, false);

  // ---- ae_step (:234-259)
  enc_->forward(frames_dev_, shifts_dev_, feat_buf_, 0, false);
  head_forward(false, feat_buf_, true, h2_);
  launch_posterior_fwd(h2_, N_, L_, eps_post_dev_, mean_, z_, kl_partial_, kKlBlocks, s);
  launch_sum_scaled(kl_partial_, kKlBlocks, 1.f / (float)N_, metrics_dev_ + 1, s);
  const Linear dfc = dfc_.view(vh_g_);
  linear_fwd(gemm_, s, N_, Mat{z_, L_}, dfc, ACT_RELU, dec_in_, F_);
  dec_->forward(dec_in_, F_);
  dec_->mse_sum_loss(frames_dev_, shifts_dev_, cfg_.ae_coef, metrics_dev_ + 0);

  // ---- score_step (:275-304) and the critic's feature: psi over [latent ; latent_mode], zeta on the perturbed next latent
  launch_ldiff_perturb(z_ + (size_t)3 * B_ * L_, noise_dev_, ab_dev_, temb_dev_, B_, L_, T_, 1.f / (float)feat_, zin_, LZ_,
                       target_, coef_, s);
  RLREP_CUDA(cudaMemcpyAsync(psi_in_, z_, BL3 * 4, cudaMemcpyDeviceToDevice, s));
  RLREP_CUDA(cudaMemcpyAsync(psi_in_ + BL3, mean_, BL3 * 4, cudaMemcpyDeviceToDevice, s));
  {
    const ColSegment seg{0, 0, A_};
    launch_pack_columns(action_dev_, A_, act2_, LA_, B_, &seg, 1, s);
    launch_pack_columns(action_dev_, A_, act2_ + (size_t)B_ * LA_, LA_, B_, &seg, 1, s);
  }
  const Mat psi_state{psi_in_, 3 * L_}, psi_action{act2_, LA_};
  bottleneck_forward(false, (int)B2, psi_state, psi_action, bn_on_);
  const size_t psi_ms = B2 * cfg_.psi_h, zeta_ms = (size_t)B_ * cfg_.zeta_h;
  resnet_forward(psi_, false, (int)B2, Mat{bn_on_.cat, 2 * bn_}, psi_masks_dev_, psi_ms, psi_on_, psi_out_, feat_);
  resnet_forward(zeta_, false, B_, Mat{zin_, LZ_}, zeta_masks_dev_, zeta_ms, zeta_on_, flat_, feat_ * L_);
  launch_diffsr_score(psi_out_, flat_, feat_, L_, target_, coef_, B_, dscore_, loss_rows_, s);
  launch_sum_scaled(loss_rows_, B_, 1.f / (float)B_, metrics_dev_ + 2, s);

  // ---- critic_step (:355-379) with back_critic_grad: features = psi(latent_mode, action), rows [B, 2B) of the pass above
  float* feature = psi_out_ + (size_t)B_ * feat_;
  critic_forward(false, 1, feature, true);
  launch_drq_critic_loss(reward_dev_, discount_dev_, rff_.q[0], rff_.q[0] + B_, rff_.q[1], rff_.q[1] + B_, B_, dq_, dq_ + B_,
                         metrics_dev_ + 3, s);
  critic_backward(1, /*wgrad=*/true, dpsi_out_ + (size_t)B_ * feat_);

  // ---- backward of the score loss and of the critic's features through psi / zeta
  launch_diffsr_score_bwd(psi_out_, flat_, feat_, L_, B_, dscore_, dflat_, dpsi_out_, s);
  resnet_backward(zeta_, false, B_, Mat{zin_, LZ_}, zeta_masks_dev_, zeta_ms, zeta_on_, Mat{dflat_, feat_ * L_}, true, dzin_);
  resnet_backward(psi_, false, (int)B2, Mat{bn_on_.cat, 2 * bn_}, psi_masks_dev_, psi_ms, psi_on_, Mat{dpsi_out_, feat_}, true,
                  dcat_);
  bottleneck_backward(false, (int)B2, psi_state, psi_action, bn_on_, dcat_, true, dpsi_in_, nullptr);

  // ---- backward of the VAE: decoder -> z, plus the score / critic gradients into the sample and the mean
  dec_->backward(ddec_in_, F_);
  launch_mul_dact(ddec_in_, dec_in_, (size_t)N_ * F_, DACT_RELU_OUT, s);
  linear_wgrad(gemm_, s, N_, Mat{ddec_in_, F_}, Mat{z_, L_}, dfc, Mat(), 0, false);
  {
    const ColJob j = bias_job(N_, Mat{ddec_in_, F_}, dfc);
    launch_colreduce_multi(&j, 1, s);
  }
  linear_dgrad(gemm_, s, N_, Mat{ddec_in_, F_}, dfc, DACT_NONE, Mat(), dz_, L_);
  launch_add_inplace(dz_, dpsi_in_, BL3, s);                                        // d latent (sampled), rows [0, 3B)
  launch_ldiff_perturb_bwd(dzin_, LZ_, ab_dev_, B_, L_, dz_ + (size_t)3 * B_ * L_, s);  // d next_latent_step, rows [3B, 4B)
  launch_posterior_bwd(h2_, N_, L_, eps_post_dev_, dz_, dpsi_in_ + BL3, (int)BL3, cfg_.kl_coef * cfg_.ae_coef / (float)N_, dh2_, s);
  {
    const Linear lo = eout_.view(vh_g_), lf = efc_.view(vh_g_);
    linear_wgrad(gemm_, s, N_, Mat{dh2_, 2 * L_}, Mat{hs_, L_}, lo, Mat(), 0, false);
    linear_dgrad(gemm_, s, N_, Mat{dh2_, 2 * L_}, lo, DACT_NONE, Mat(), dhs_, L_);
    launch_ln_act2_bwd(dhs_, L_, nullptr, L_, hxhat_, L_, hrstd_, N_, L_, vh_g_.p + eln_w_, vh_g_.p + eln_b_, 2, dhpre_, L_, L_,
                       hs_, dhs_, L_, s);  // g_beta -> hs_, g_gamma -> dhs_ (both dead after this point)
    linear_wgrad(gemm_, s, N_, Mat{dhpre_, L_}, Mat{feat_buf_, F_}, lf, Mat(), 0, false);
    const ColJob jobs[4] = {bias_job(N_, Mat{dh2_, 2 * L_}, lo), bias_job(N_, Mat{dhpre_, L_}, lf),
                            ColJob{dhs_, nullptr, vh_g_.g + eln_w_, L_, N_, L_}, ColJob{hs_, nullptr, vh_g_.g + eln_b_, L_, N_, L_}};
    launch_colreduce_multi(jobs, 4, s);
    linear_dgrad(gemm_, s, N_, Mat{dhpre_, L_}, lf, DACT_NONE, Mat(), dfeat_, F_);
  }
  enc_->backward(dfeat_, F_);

  // ---- optimisers: Adam(vae), AdamW(score: decoupled decay first, torch/optim/adamw.py), Adam(critic).  The Polyak of
  // vae / critic rides on the Adam kernels; the score target is still needed by the actor step and is updated after it.
  auto adam = [&](ParamGroup& g, const AdamHyper* h, bool polyak) {
    launch_adam_polyak(g.p, g.g, g.m, g.v, g.n, h, polyak ? g.target : nullptr, polyak ? g.n_target : 0, cfg_.tau, nullptr, s);
  };
  adam(enc_->group(), &ctl_->feat[0], true);
  adam(vh_g_, &ctl_->feat[0], true);
  adam(dec_->group(), &ctl_->feat[0], true);
  launch_scale_inplace(score_g_.p, score_g_.n, (float)(1.0 - cfg_.score_lr * cfg_.weight_decay), s);
  adam(score_g_, &ctl_->feat[0], false);
  adam(crit_g_, &ctl_->critic, true);

  // ---- actor_step (:381-390) on the detached posterior mode, through the frozen psi target and the new critic
  actor_forward(latent_mode, eps_act_dev_ + (size_t)B_ * A_, stddev, acta_, LA_, true);
  bottleneck_forward(true, B_, latent_mode, Mat{acta_, LA_}, bn_t_);
  resnet_forward(psi_, true, B_, Mat{bn_t_.cat, 2 * bn_}, nullptr, 0, psi_t_, feat_t_, feat_);
  critic_forward(false, 0, feat_t_, true);
  launch_drq_actor_loss(rff_.q[0], rff_.q[0] + B_, B_, dq_, dq_ + B_, metrics_dev_ + 7, s);
  critic_backward(0, /*wgrad=*/false, dfeat_t_);
  resnet_backward(psi_, true, B_, Mat{bn_t_.cat, 2 * bn_}, nullptr, 0, psi_t_, Mat{dfeat_t_, feat_}, false, dcat_t_);
  bottleneck_backward(true, B_, latent_mode, Mat{acta_, LA_}, bn_t_, dcat_t_, false, nullptr, dacta_);
  {
    const Linear l0 = p0_.view(actor_g_), l1 = p1_.view(actor_g_), l2 = p2_.view(actor_g_), lt = at_.view(actor_g_);
    launch_trunc_normal_bwd(dacta_, LA_, mu_, B_, A_, draw_a_, LA_, s);
    linear_wgrad(gemm_, s, B_, Mat{draw_a_, LA_}, Mat{ap2_, H_}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{draw_a_, LA_}, l2, DACT_RELU_OUT, Mat{ap2_, H_}, dap2_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dap2_, H_}, Mat{ap1_, H_}, l1, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dap2_, H_}, l1, DACT_RELU_OUT, Mat{ap1_, H_}, dap1_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dap1_, H_}, Mat{th_, bn_}, l0, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dap1_, H_}, l0, DACT_NONE, Mat(), dth_, bn_);
    launch_ln_act2_bwd(dth_, bn_, th_, bn_, xhat_a_, bn_, rstd_a_, B_, bn_, actor_g_.p + aln_w_, actor_g_.p + aln_b_, 1, dtpre_,
                       bn_, bn_, gb_, gg_, bn_, s);
    linear_wgrad(gemm_, s, B_, Mat{dtpre_, bn_}, latent_mode, lt, Mat(), 0, false);
    const ColJob jobs[6] = {bias_job(B_, Mat{draw_a_, LA_}, l2), bias_job(B_, Mat{dap2_, H_}, l1),
                            bias_job(B_, Mat{dap1_, H_}, l0),    bias_job(B_, Mat{dtpre_, bn_}, lt),
                            ColJob{gg_, nullptr, actor_g_.g + aln_w_, bn_, B_, bn_},
                            ColJob{gb_, nullptr, actor_g_.g + aln_b_, bn_, B_, bn_}};
    launch_colreduce_multi(jobs, 6, s);
  }
  launch_adam_polyak(actor_g_.p, actor_g_.g, actor_g_.m, actor_g_.v, actor_g_.n, &ctl_->actor, nullptr, 0, 0.f, nullptr, s);
  launch_polyak(score_g_.p, score_g_.target, score_g_.n_target, cfg_.tau, nullptr, s);
  launch_polyak(dead_g_.p, dead_g_.target, dead_g_.n_target, cfg_.tau, nullptr, s);  // sync_target walks ALL parameters
}

}  // namespace rlrep

// CTRL-SAC update step (reference: agent/ctrlsac/ctrlsac_agent.py:213-362) as one stream of sm_100a kernels.
//
// Per train(): K x [gather -> phi/mu forward -> contrastive logits (tcgen05) -> row LSE/CE -> backward ->
// fused Adam(+Polyak of phi_target)] -> critic step -> actor/alpha step -> critic Polyak (fused into the critic
// Adam launch, gated by the control block).  All of it is captured into a CUDA graph after the first call.
//
// Reference quirks kept (SURVEY.md A.6): frozen_phi == frozen_phi_target == phi after the feature loop (they are
// aliases here, not copies); phi_target is Polyak-updated but never read; critic/actor reuse the last feature
// batch; the actor backward skips the dW of the frozen phi / critic (never consumed by the reference either).
#include "agent_base.cuh"

namespace rlrep {

namespace {

class CtrlSacAgent final : public SacBase {
 public:
  CtrlSacAgent(const AgentConfig& c, cudaStream_t s) : SacBase(c, s) {
    H_ = c.hidden_dim;
    D_ = c.feature_dim;
    K_ = c.k_feat;
    RLREP_CHECK(K_ >= 1 && K_ <= kMaxFeatureSteps, "extra_feature_steps out of range");
    const RecordLayout probe_layout = RecordLayout::of(S_, A_);
    off_r_ = probe_layout.off_r;
    off_d_ = probe_layout.off_d;
    off_s2_ = probe_layout.off_s2;
    plan_common(K_ * B_, 2 * B_ * A_, probe_layout.R);

    // feature group: phi first so that its Polyak target is a prefix (ctrlsac_agent.py:163-178)
    feat_g_.name = "feature";
    p1_ = add_linear(feat_g_, "phi.l1", H_, S_ + A_);
    p2_ = add_linear(feat_g_, "phi.l2", H_, H_);
    p3_ = add_linear(feat_g_, "phi.l3", D_, H_);
    feat_g_.n_target = feat_g_.n;
    feat_g_.target_prefix_from = "phi.";
    feat_g_.target_prefix_to = "phi_target.";
    m1_ = add_linear(feat_g_, "mu.l1", H_, S_);
    m2_ = add_linear(feat_g_, "mu.l2", H_, H_);
    m3_ = add_linear(feat_g_, "mu.l3", D_, H_);
    th_ = add_linear(feat_g_, "theta.l", 1, D_, /*pad=*/false);
    feat_g_.want(arena_);

    // critic group: l1 | l4 stacked so both heads' hidden layers are ONE [2H, D] GEMM (ctrlsac_agent.py:18-52)
    crit_g_.name = "critic";
    c14_.out = 2 * H_;
    c14_.in = D_;
    c14_.w_off = crit_g_.add("critic.l1.weight", H_, D_);
    crit_g_.add("critic.l4.weight", H_, D_);
    c14_.b_off = crit_g_.add("critic.l1.bias", H_, 1);
    crit_g_.add("critic.l4.bias", H_, 1);
    c2_ = add_linear(crit_g_, "critic.l2", 1, H_, false);
    c5_ = add_linear(crit_g_, "critic.l5", 1, H_, false);
    RLREP_CHECK(H_ % 32 == 0 && D_ % 32 == 0, "hidden_dim and feature_dim must be multiples of 32");
    crit_g_.n_target = crit_g_.n;
    crit_g_.target_prefix_from = "critic.";
    crit_g_.target_prefix_to = "critic_target.";
    crit_g_.want(arena_);

    const size_t BH = (size_t)B_ * H_, BD = (size_t)B_ * D_;
    arena_.want(&h1_, BH);
    arena_.want(&h2_, BH);
    arena_.want(&g1_, BH);
    arena_.want(&g2_, BH);
    arena_.want(&zphi_, BD);
    arena_.want(&zmu_, BD);
    arena_.want(&dzphi_, BD);
    arena_.want(&dzmu_, BD);
    arena_.want(&dh2_, BH);
    arena_.want(&dh1_, BH);
    arena_.want(&dg2_, BH);
    arena_.want(&dg1_, BH);
    arena_.want(&hb1_, BH);
    arena_.want(&hb2_, BH);
    arena_.want(&hc1_, BH);
    arena_.want(&hc2_, BH);
    arena_.want(&zpi_, BD);
    arena_.want(&logits_, (size_t)B_ * B_);
    arena_.want(&loss_rows_, B_);
    arena_.want(&rpred_, B_);
    arena_.want(&drp_, B_);
    arena_.want(&hid_, 2 * BH);
    arena_.want(&hid_t_, 2 * BH);
    arena_.want(&dhid_, 2 * BH);
    arena_.want(&q1_, B_);
    arena_.want(&q2_, B_);
    arena_.want(&nq1_, B_);
    arena_.want(&nq2_, B_);
    arena_.want(&dq1_, B_);
    arena_.want(&dq2_, B_);
    arena_.want(&logp2_, B_);
    arena_.want(&head_ctr_, 4);
    finish_setup((size_t)8 << 20);

    names_ = {"total_loss", "model_loss", "r_loss", "q1_loss", "q2_loss", "q1", "q2", "actor_loss", "alpha_loss",
              "alpha"};
  }

  int idx_per_train() const override { return K_ * B_; }
  int eps_per_train() const override { return 2 * B_ * A_; }
  const std::vector<std::string>& metric_names() const override { return names_; }
  std::vector<ParamGroup*> groups() override { return {&feat_g_, &actor_g_, &crit_g_}; }

  void sync_targets_from_params() override {
    RLREP_CUDA(cudaMemcpyAsync(feat_g_.target, feat_g_.p, feat_g_.n_target * 4, cudaMemcpyDeviceToDevice, stream));
    RLREP_CUDA(cudaMemcpyAsync(crit_g_.target, crit_g_.p, crit_g_.n_target * 4, cudaMemcpyDeviceToDevice, stream));
    RLREP_CUDA(cudaStreamSynchronize(stream));
  }

 protected:
  void update(Ring& ring) override {
    begin_update();
    launch_tick(ctl, base_tick(), stream);
    const bool chain = chained();
    for (int k = 0; k < K_; ++k) {
      if (chain) {
        feature_step_chained(k, ring);
      } else {
        launch_gather(ring.data, R_ / 4, idx_dev_ + (size_t)k * B_, B_, batch_, stream);
        feature_step(k);
      }
    }
    if (chain) {
      critic_step_chained();
      actor_step_chained();
    } else {
      critic_step();
      actor_step();
    }
  }

 private:
  Mat sa() const { return Mat{batch_, R_}; }             // cat(s, a): the first S+A floats of each record
  Mat s2() const { return Mat{batch_ + off_s2_, R_}; }   // next_state
  const float* reward() const { return batch_ + off_r_; }
  const float* done() const { return batch_ + off_d_; }

  // phi(x) with x = cat of one or two segments, on stream `s`; hidden activations go to (h1, h2) -- h1_/h2_ when a
  // backward pass follows -- and the features to z [B, D].
  void phi_forward(cudaStream_t s, Mat x, Mat x2, int k1, float* z, float* h1, float* h2) {
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    linear_fwd(gemm_, s, B_, x, l1, ACT_ELU, h1, H_, x2, k1);
    linear_fwd(gemm_, s, B_, Mat{h1, H_}, l2, ACT_ELU, h2, H_);
    linear_fwd(gemm_, s, B_, Mat{h2, H_}, l3, ACT_NONE, z, D_);
  }

  void feature_step(int k) {  // ctrlsac_agent.py:213-251
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    const Linear n1 = m1_.view(feat_g_), n2 = m2_.view(feat_g_), n3 = m3_.view(feat_g_);
    const Linear th = th_.view(feat_g_);
    const float inv_b = 1.f / (float)B_;
    cudaStream_t s0 = stream, s1 = side();
    // ---- forward: phi on the main stream, mu on the side stream
    fork();
    phi_forward(s0, sa(), Mat(), 0, zphi_, h1_, h2_);
    linear_fwd(gemm_, s1, B_, s2(), n1, ACT_ELU, g1_, H_);
    linear_fwd(gemm_, s1, B_, Mat{g1_, H_}, n2, ACT_ELU, g2_, H_);
    linear_fwd(gemm_, s1, B_, Mat{g2_, H_}, n3, ACT_TANH, zmu_, D_);
    join();
    {  // logits[i, j] = <phi_i, mu_j>  (the reference's [B,1,D]*[1,B,D] broadcast, :229, as a tensor-core GEMM)
      GemmArgs a;
      a.M = B_; a.N = B_; a.K = D_;
      a.A = zphi_; a.lda = D_;
      a.B = zmu_; a.ldb = D_;
      a.C = logits_; a.ldc = B_;
      gemm_.run(a, s0);
    }
    launch_ce_rows(logits_, B_, B_, B_, 0, inv_b, loss_rows_, s0);  // logits_ now holds dL/dlogits
    launch_rowdot(zphi_, D_, B_, D_, th.W, th.b, rpred_, s0);
    launch_feature_loss_finalize(loss_rows_, B_, rpred_, reward(), R_, inv_b, drp_, metrics_dev_ + 0, s0);
    // ---- backward: the phi branch (with theta) on the main stream, the mu branch on the side stream
    fork();
    {  // d z_phi = G mu + drp (x) theta.w
      GemmArgs a;
      a.M = B_; a.N = D_; a.K = B_;
      a.A = logits_; a.lda = B_;
      a.B = zmu_; a.ldb = D_; a.b_mn = true;
      a.C = dzphi_; a.ldc = D_;
      a.epi.r1_u = drp_; a.epi.r1_v = th.W;
      gemm_.run(a, s0);
    }
    // the dgrad chain is the critical path; weight / bias gradients trail it on an aux stream
    cudaStream_t w0 = aux(0), w1 = aux(1);
    const double share = dual_share_, wshare = kAuxShare;
    wait_for(w0, mark(s0));
    gemm_.set_sm_share(wshare);
    linear_wgrad(gemm_, w0, B_, Mat{dzphi_, D_}, Mat{h2_, H_}, l3, Mat(), 0, false);
    gemm_.set_sm_share(share);
    linear_dgrad(gemm_, s0, B_, Mat{dzphi_, D_}, l3, DACT_ELU_OUT, Mat{h2_, H_}, dh2_, H_);
    wait_for(w0, mark(s0));
    gemm_.set_sm_share(wshare);
    linear_wgrad(gemm_, w0, B_, Mat{dh2_, H_}, Mat{h1_, H_}, l2, Mat(), 0, false);
    gemm_.set_sm_share(share);
    linear_dgrad(gemm_, s0, B_, Mat{dh2_, H_}, l2, DACT_ELU_OUT, Mat{h1_, H_}, dh1_, H_);
    linear_wgrad(gemm_, s0, B_, Mat{dh1_, H_}, sa(), l1, Mat(), 0, false);
    wait_for(w0, mark(s0));
    {
      ColJob jobs[5] = {bias_job(B_, Mat{dzphi_, D_}, l3), bias_job(B_, Mat{dh2_, H_}, l2),
                        bias_job(B_, Mat{dh1_, H_}, l1), ColJob{zphi_, drp_, th.dW, D_, B_, D_},  // d theta.w
                        ColJob{drp_, nullptr, th.db, 1, B_, 1}};                                  // d theta.b
      launch_colreduce_multi(jobs, 5, w0);
    }
    {  // d (pre-tanh mu) = (G^T phi) * (1 - mu^2)
      GemmArgs a;
      a.M = B_; a.N = D_; a.K = B_;
      a.A = logits_; a.lda = B_; a.a_mn = true;
      a.B = zphi_; a.ldb = D_; a.b_mn = true;
      a.C = dzmu_; a.ldc = D_;
      a.epi.dact = DACT_TANH_OUT; a.epi.aux = zmu_; a.epi.ld_aux = D_;
      gemm_.run(a, s1);
    }
    wait_for(w1, mark(s1));
    gemm_.set_sm_share(wshare);
    linear_wgrad(gemm_, w1, B_, Mat{dzmu_, D_}, Mat{g2_, H_}, n3, Mat(), 0, false);
    gemm_.set_sm_share(share);
    linear_dgrad(gemm_, s1, B_, Mat{dzmu_, D_}, n3, DACT_ELU_OUT, Mat{g2_, H_}, dg2_, H_);
    wait_for(w1, mark(s1));
    gemm_.set_sm_share(wshare);
    linear_wgrad(gemm_, w1, B_, Mat{dg2_, H_}, Mat{g1_, H_}, n2, Mat(), 0, false);
    gemm_.set_sm_share(share);
    linear_dgrad(gemm_, s1, B_, Mat{dg2_, H_}, n2, DACT_ELU_OUT, Mat{g1_, H_}, dg1_, H_);
    linear_wgrad(gemm_, s1, B_, Mat{dg1_, H_}, s2(), n1, Mat(), 0, false);
    wait_for(w1, mark(s1));
    {
      ColJob jobs[3] = {bias_job(B_, Mat{dzmu_, D_}, n3), bias_job(B_, Mat{dg2_, H_}, n2),
                        bias_job(B_, Mat{dg1_, H_}, n1)};
      launch_colreduce_multi(jobs, 3, w1);
    }
    join_aux(0, s0);
    join_aux(1, s0);
    join();
    // ---- one fused Adam over phi | mu | theta, plus Polyak of phi_target (:242-244, :253-255)
    launch_adam_polyak(feat_g_.p, feat_g_.g, feat_g_.m, feat_g_.v, feat_g_.n, &ctl->feat[k],
                       cfg.use_feature_target ? feat_g_.target : nullptr, feat_g_.n_target, cfg.feature_tau, nullptr,
                       s0);
  }

  // ---------------------------------------------------------------------------------------------- chained variants
  // Same arithmetic, same kernels for everything that is not a GEMM; every group of GEMMs between two elementwise kernels
  // runs as ONE persistent chain kernel (gemm_chain.cuh) on the main stream instead of one launch per GEMM on up to four
  // streams: 38 launches per update instead of 149, and a dependent GEMM starts when its input tiles are complete.  Every
  // kernel of this path is a programmatic dependent launch (launch_pdl): its CTAs start while the kernel before it finishes.
  // The feature step is two chains: both towers and the logits, then the whole backward pass; the replay gather runs before
  // the first and the contrastive head between the two as stand-alone kernels.
  void feature_step_chained(int k, Ring& ring) {  // ctrlsac_agent.py:213-251
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    const Linear n1 = m1_.view(feat_g_), n2 = m2_.view(feat_g_), n3 = m3_.view(feat_g_);
    const Linear th = th_.view(feat_g_);
    const float inv_b = 1.f / (float)B_;
    cudaStream_t s0 = stream;
    launch_gather(ring.data, R_ / 4, idx_dev_ + (size_t)k * B_, B_, batch_, s0);
    gemm_.begin_chain(s0);
    phi_forward(s0, sa(), Mat(), 0, zphi_, h1_, h2_);
    linear_fwd(gemm_, s0, B_, s2(), n1, ACT_ELU, g1_, H_);
    linear_fwd(gemm_, s0, B_, Mat{g1_, H_}, n2, ACT_ELU, g2_, H_);
    linear_fwd(gemm_, s0, B_, Mat{g2_, H_}, n3, ACT_TANH, zmu_, D_);
    {  // logits[i, j] = <phi_i, mu_j>
      GemmArgs a;
      a.M = B_; a.N = B_; a.K = D_;
      a.A = zphi_; a.lda = D_;
      a.B = zmu_; a.ldb = D_;
      a.C = logits_; a.ldc = B_;
      gemm_.run(a, s0);
    }
    if (k == K_ - 1) {
      // The critic step's actor trunks, a' ~ pi(s') and a_pi ~ pi(s): they read only the actor, which the feature loop
      // does not touch, and this last batch, so they share this chain's levels with phi and mu instead of running as a
      // chain of their own on the critical path.
      actor_trunk(s2(), /*set=*/1, s0);
      actor_trunk(Mat{batch_, R_}, /*set=*/0, s0);
    }
    gemm_.end_chain();
    // row log-sum-exp / CE gradient (logits_ then holds dL/dlogits), reward head and the loss metrics
    launch_contrastive_head(logits_, B_, B_, B_, 0, inv_b, zphi_, D_, D_, th.W, th.b, reward(), R_, loss_rows_, rpred_, drp_,
                            metrics_dev_ + 0, head_ctr_, s0);
    gemm_.begin_chain(s0);
    {  // d z_phi = G mu + drp (x) theta.w
      GemmArgs a;
      a.M = B_; a.N = D_; a.K = B_;
      a.A = logits_; a.lda = B_;
      a.B = zmu_; a.ldb = D_; a.b_mn = true;
      a.C = dzphi_; a.ldc = D_;
      a.epi.r1_u = drp_; a.epi.r1_v = th.W;
      gemm_.run(a, s0);
    }
    {  // d (pre-tanh mu) = (G^T phi) * (1 - mu^2)
      GemmArgs a;
      a.M = B_; a.N = D_; a.K = B_;
      a.A = logits_; a.lda = B_; a.a_mn = true;
      a.B = zphi_; a.ldb = D_; a.b_mn = true;
      a.C = dzmu_; a.ldc = D_;
      a.epi.dact = DACT_TANH_OUT; a.epi.aux = zmu_; a.epi.ld_aux = D_;
      gemm_.run(a, s0);
    }
    linear_dgrad(gemm_, s0, B_, Mat{dzphi_, D_}, l3, DACT_ELU_OUT, Mat{h2_, H_}, dh2_, H_);
    linear_dgrad(gemm_, s0, B_, Mat{dzmu_, D_}, n3, DACT_ELU_OUT, Mat{g2_, H_}, dg2_, H_);
    linear_wgrad(gemm_, s0, B_, Mat{dzphi_, D_}, Mat{h2_, H_}, l3, Mat(), 0, false);
    linear_wgrad(gemm_, s0, B_, Mat{dzmu_, D_}, Mat{g2_, H_}, n3, Mat(), 0, false);
    linear_dgrad(gemm_, s0, B_, Mat{dh2_, H_}, l2, DACT_ELU_OUT, Mat{h1_, H_}, dh1_, H_);
    linear_dgrad(gemm_, s0, B_, Mat{dg2_, H_}, n2, DACT_ELU_OUT, Mat{g1_, H_}, dg1_, H_);
    linear_wgrad(gemm_, s0, B_, Mat{dh2_, H_}, Mat{h1_, H_}, l2, Mat(), 0, false);
    linear_wgrad(gemm_, s0, B_, Mat{dg2_, H_}, Mat{g1_, H_}, n2, Mat(), 0, false);
    linear_wgrad(gemm_, s0, B_, Mat{dh1_, H_}, sa(), l1, Mat(), 0, false);
    linear_wgrad(gemm_, s0, B_, Mat{dg1_, H_}, s2(), n1, Mat(), 0, false);
    gemm_.end_chain();
    {
      ColJob jobs[8] = {bias_job(B_, Mat{dzphi_, D_}, l3), bias_job(B_, Mat{dh2_, H_}, l2),
                        bias_job(B_, Mat{dh1_, H_}, l1), ColJob{zphi_, drp_, th.dW, D_, B_, D_},  // d theta.w
                        ColJob{drp_, nullptr, th.db, 1, B_, 1},                                   // d theta.b
                        bias_job(B_, Mat{dzmu_, D_}, n3), bias_job(B_, Mat{dg2_, H_}, n2),
                        bias_job(B_, Mat{dg1_, H_}, n1)};
      launch_colreduce_multi(jobs, 8, s0);
    }
    launch_adam_polyak(feat_g_.p, feat_g_.g, feat_g_.m, feat_g_.v, feat_g_.n, &ctl->feat[k],
                       cfg.use_feature_target ? feat_g_.target : nullptr, feat_g_.n_target, cfg.feature_tau, nullptr,
                       s0);
  }

  void critic_step_chained() {  // ctrlsac_agent.py:257-293
    cudaStream_t s0 = stream;
    const float* eps_next = eps_dev_;
    const float* eps_pi = eps_dev_ + (size_t)B_ * A_;
    const Linear l14t = c14_.view(crit_g_, true), l14 = c14_.view(crit_g_), l2 = c2_.view(crit_g_), l5 = c5_.view(crit_g_);
    const Linear l2t = c2_.view(crit_g_, true), l5t = c5_.view(crit_g_, true);
    // a' ~ pi(s') for the TD target and a_pi ~ pi(s) for the actor step; their trunks ran in the last feature step's
    // forward chain
    actor_sample_cat_pair(s2(), eps_next, logp2_, Mat{batch_, R_}, eps_pi, s0);
    const Mat s2a{cat_next_, LDSA_}, spi{cat_pi_, LDSA_};
    gemm_.begin_chain(s0);
    phi_forward(s0, s2a, Mat(), 0, zmu_, h1_, h2_);  // frozen_phi_target(s', a'); zmu_ is free after the feature loop
    linear_fwd(gemm_, s0, B_, Mat{zmu_, D_}, l14t, ACT_ELU, hid_t_, 2 * H_);
    phi_forward(s0, sa(), Mat(), 0, zphi_, hb1_, hb2_);  // frozen_phi_target(s, a)
    linear_fwd(gemm_, s0, B_, Mat{zphi_, D_}, l14, ACT_ELU, hid_, 2 * H_);
    phi_forward(s0, spi, Mat(), 0, zpi_, hc1_, hc2_);  // frozen_phi(s, a_pi), consumed by the actor step
    gemm_.end_chain();
    {  // the four N = 1 heads, the TD loss and the way back to the hidden layer: one launch, a CTA per row
      CriticHeadArgs a;
      a.hid_t = hid_t_; a.hid = hid_; a.ldh = 2 * H_; a.H = H_; a.B = B_;
      a.w2t = l2t.W; a.b2t = l2t.b; a.w5t = l5t.W; a.b5t = l5t.b;
      a.w2 = l2.W; a.b2 = l2.b; a.w5 = l5.W; a.b5 = l5.b;
      a.reward = reward(); a.done = done(); a.ld_rd = R_;
      a.logp2 = logp2_; a.gamma = cfg.discount; a.c = ctl;
      a.nq1 = nq1_; a.nq2 = nq2_; a.q1 = q1_; a.q2 = q2_; a.dq1 = dq1_; a.dq2 = dq2_;
      a.dhid = dhid_; a.ld_dh = 2 * H_;
      a.metrics = metrics_dev_ + 3;
      a.counter = head_ctr_ + 1;
      launch_critic_td_head(a, s0);
    }
    {
      ColJob jobs[5] = {ColJob{hid_, dq1_, l2.dW, 2 * H_, B_, H_}, ColJob{dq1_, nullptr, l2.db, 1, B_, 1},
                        ColJob{hid_ + H_, dq2_, l5.dW, 2 * H_, B_, H_}, ColJob{dq2_, nullptr, l5.db, 1, B_, 1},
                        bias_job(B_, Mat{dhid_, 2 * H_}, l14)};
      launch_colreduce_multi(jobs, 5, s0);
    }
    linear_wgrad(gemm_, s0, B_, Mat{dhid_, 2 * H_}, Mat{zphi_, D_}, l14, Mat(), 0, false);
    launch_adam_polyak(crit_g_.p, crit_g_.g, crit_g_.m, crit_g_.v, crit_g_.n, &ctl->critic, crit_g_.target,
                       crit_g_.n_target, cfg.tau, &ctl->polyak_critic, s0);
  }

  void actor_step_chained() {  // ctrlsac_agent.py:295-325
    const float* eps = eps_dev_ + (size_t)B_ * A_;
    const Linear l14 = c14_.view(crit_g_);
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    {  // the UPDATED critic on frozen_phi(s, a_pi): hidden layer, then heads + actor / temperature loss + backward in one launch
      const Linear c2 = c2_.view(crit_g_), c5 = c5_.view(crit_g_);
      linear_fwd(gemm_, stream, B_, Mat{zpi_, D_}, l14, ACT_ELU, hid_, 2 * H_);
      ActorHeadArgs a;
      a.hid = hid_; a.ldh = 2 * H_; a.H = H_; a.B = B_;
      a.w2 = c2.W; a.b2 = c2.b; a.w5 = c5.W; a.b5 = c5.b;
      a.logp = logp_; a.target_entropy = (float)(-A_); a.learn_alpha = cfg.learn_alpha; a.c = ctl;
      a.q1 = q1_; a.q2 = q2_; a.dq1 = dq1_; a.dq2 = dq2_;
      a.dhid = dhid_; a.ld_dh = 2 * H_;
      a.dlogp_scalar = dlogp_;
      a.metrics = metrics_dev_ + 7;
      a.counter = head_ctr_ + 2;
      launch_actor_head(a, stream);
    }
    gemm_.begin_chain(stream);
    linear_dgrad(gemm_, stream, B_, Mat{dhid_, 2 * H_}, l14, DACT_NONE, Mat(), dzphi_, D_);
    linear_dgrad(gemm_, stream, B_, Mat{dzphi_, D_}, l3, DACT_ELU_OUT, Mat{hc2_, H_}, dh2_, H_);
    linear_dgrad(gemm_, stream, B_, Mat{dh2_, H_}, l2, DACT_ELU_OUT, Mat{hc1_, H_}, dh1_, H_);
    dgrad_to_action(Mat{dh1_, H_}, l1);
    gemm_.end_chain();
    actor_backward_chained(Mat{batch_, R_}, eps);
    actor_adam();
  }

  // twin heads on features z: hid = elu(z [l1|l4]^T + b), q1 = hid[:, :H] . l2, q2 = hid[:, H:] . l5
  void critic_forward(cudaStream_t s, const float* z, bool target, float* hid, float* q1, float* q2) {
    const Linear l14 = c14_.view(crit_g_, target), l2 = c2_.view(crit_g_, target), l5 = c5_.view(crit_g_, target);
    linear_fwd(gemm_, s, B_, Mat{z, D_}, l14, ACT_ELU, hid, 2 * H_);
    launch_rowdot_pair(RowDotJob{hid, l2.W, l2.b, q1, 2 * H_, H_}, RowDotJob{hid + H_, l5.W, l5.b, q2, 2 * H_, H_}, B_, s);
  }
  // d hid from (dq1, dq2) through the N = 1 heads and the ELU
  void critic_heads_backward_to_hidden() {
    const Linear l2 = c2_.view(crit_g_), l5 = c5_.view(crit_g_);
    launch_outer_dact(dq1_, l2.W, B_, H_, hid_, 2 * H_, DACT_ELU_OUT, dhid_, 2 * H_, stream);
    launch_outer_dact(dq2_, l5.W, B_, H_, hid_ + H_, 2 * H_, DACT_ELU_OUT, dhid_ + H_, 2 * H_, stream);
  }

  void critic_step() {  // ctrlsac_agent.py:257-293
    const float* eps = eps_dev_;
    cudaStream_t s0 = stream, s1 = side();
    fork();
    // Hoisted out of the actor step: a_pi ~ pi(s) and frozen_phi(s, a_pi) read only the actor, phi, the batch and the
    // noise -- nothing the critic step writes -- so they run beside it on an aux branch; the actor step joins it
    // before it evaluates the UPDATED critic on these features (reference order, ctrlsac_agent.py:299-305).
    cudaStream_t a0 = aux(0);
    wait_for(a0, mark(s0));
    const Mat spi = actor_forward_cat(Mat{batch_, R_}, eps_dev_ + (size_t)B_ * A_, cat_pi_, logp_, a0, /*set=*/0);
    phi_forward(a0, spi, Mat(), 0, zpi_, hc1_, hc2_);
    // main stream: a' ~ pi(s'), frozen_phi_target(s', a'), target critic
    const Mat s2a = actor_forward_cat(s2(), eps, cat_next_, logp2_, s0, /*set=*/1);
    phi_forward(s0, s2a, Mat(), 0, zmu_, h1_, h2_);  // zmu_ is free after the feature loop
    critic_forward(s0, zmu_, /*target=*/true, hid_t_, nq1_, nq2_);
    // side stream: frozen_phi_target(s, a) and the live critic on it
    phi_forward(s1, sa(), Mat(), 0, zphi_, hb1_, hb2_);
    critic_forward(s1, zphi_, /*target=*/false, hid_, q1_, q2_);
    join();
    launch_td_critic_loss(reward(), done(), R_, nq1_, nq2_, logp2_, q1_, q2_, B_, cfg.discount, ctl, dq1_, dq2_,
                          metrics_dev_ + 3, s0);
    // ---- backward (critic parameters only; the features are under no_grad)
    const Linear l14 = c14_.view(crit_g_), l2 = c2_.view(crit_g_), l5 = c5_.view(crit_g_);
    critic_heads_backward_to_hidden();
    {
      ColJob jobs[5] = {ColJob{hid_, dq1_, l2.dW, 2 * H_, B_, H_}, ColJob{dq1_, nullptr, l2.db, 1, B_, 1},
                        ColJob{hid_ + H_, dq2_, l5.dW, 2 * H_, B_, H_}, ColJob{dq2_, nullptr, l5.db, 1, B_, 1},
                        bias_job(B_, Mat{dhid_, 2 * H_}, l14)};
      launch_colreduce_multi(jobs, 5, s0);
    }
    linear_wgrad(gemm_, s0, B_, Mat{dhid_, 2 * H_}, Mat{zphi_, D_}, l14, Mat(), 0, false);
    // Adam on the critic; its Polyak (sac_agent.py:99-102, every `period` steps) only reads the updated critic and
    // nothing between here and the end of train() writes it, so it rides in the same launch.
    launch_adam_polyak(crit_g_.p, crit_g_.g, crit_g_.m, crit_g_.v, crit_g_.n, &ctl->critic, crit_g_.target,
                       crit_g_.n_target, cfg.tau, &ctl->polyak_critic, s0);
  }

  void actor_step() {  // ctrlsac_agent.py:295-325
    const float* eps = eps_dev_ + (size_t)B_ * A_;
    const Mat s{batch_, R_};
    join_aux(0, stream);  // a_pi, log pi and frozen_phi(s, a_pi) were computed beside the critic step
    critic_forward(stream, zpi_, false, hid_, q1_, q2_);
    launch_actor_alpha_loss(q1_, q2_, logp_, B_, (float)(-A_), cfg.learn_alpha, ctl, dq1_, dq2_, dlogp_,
                            metrics_dev_ + 7, stream);
    // ---- dgrad only, back to the action input of phi
    const Linear l14 = c14_.view(crit_g_);
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    critic_heads_backward_to_hidden();
    linear_dgrad(gemm_, stream, B_, Mat{dhid_, 2 * H_}, l14, DACT_NONE, Mat(), dzphi_, D_);
    linear_dgrad(gemm_, stream, B_, Mat{dzphi_, D_}, l3, DACT_ELU_OUT, Mat{hc2_, H_}, dh2_, H_);
    linear_dgrad(gemm_, stream, B_, Mat{dh2_, H_}, l2, DACT_ELU_OUT, Mat{hc1_, H_}, dh1_, H_);
    dgrad_to_action(Mat{dh1_, H_}, l1);
    actor_backward(s, eps);
    actor_adam();
  }

  int H_ = 0, D_ = 0, K_ = 0, off_r_ = 0, off_d_ = 0, off_s2_ = 0;
  ParamGroup feat_g_, crit_g_;
  LinearSlot p1_, p2_, p3_, m1_, m2_, m3_, th_, c14_, c2_, c5_;
  float *h1_ = nullptr, *h2_ = nullptr, *g1_ = nullptr, *g2_ = nullptr, *zphi_ = nullptr, *zmu_ = nullptr;
  float *dzphi_ = nullptr, *dzmu_ = nullptr, *dh2_ = nullptr, *dh1_ = nullptr, *logits_ = nullptr;
  float *dg2_ = nullptr, *dg1_ = nullptr, *hb1_ = nullptr, *hb2_ = nullptr, *hc1_ = nullptr, *hc2_ = nullptr, *zpi_ = nullptr;
  float *loss_rows_ = nullptr, *rpred_ = nullptr, *drp_ = nullptr, *hid_ = nullptr, *hid_t_ = nullptr,
        *dhid_ = nullptr;
  float *q1_ = nullptr, *q2_ = nullptr, *nq1_ = nullptr, *nq2_ = nullptr, *dq1_ = nullptr, *dq2_ = nullptr;
  float *logp2_ = nullptr;
  unsigned* head_ctr_ = nullptr;
  std::vector<std::string> names_;
};

}  // namespace

std::unique_ptr<Agent> make_ctrlsac_agent(const AgentConfig& cfg, cudaStream_t s) {
  return std::unique_ptr<Agent>(new CtrlSacAgent(cfg, s));
}

}  // namespace rlrep

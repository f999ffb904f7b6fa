// SPEDER-SAC update step (reference: agent/spedersac/spedersac_agent.py:181-322) as one stream of sm_100a kernels.
//
// Per train(): K x [gather 2B rows (update batch + independent batch) -> phi / mu trunks on all 2B rows -> spectral
// loss + reward head -> backward -> fused Adam(+Polyak of phi_target)] -> RFF-critic step on the live phi (no_grad) ->
// actor / temperature step -> critic Polyak.
//
// The second loss term mean((phi~ mu~^T)(phi~ mu~^T)^T) is evaluated as ||mu~ colsum(phi~)||^2 / B^2 (identical
// algebra, see kernels.cuh): two mat-vecs instead of two B x B GEMMs, and no TF32 rounding in the loss at all.
//
// Reference quirks kept: the critic and actor steps use the FIRST of the last iteration's two batches
// (spedersac_agent.py:299-300, 311-316); phi_target is Polyak-updated but never read; phi is live in the critic / actor
// steps and its gradients from the actor loss are discarded.
#include "agent_base.cuh"
#include "nets.cuh"

namespace rlrep {

namespace {

class SpederSacAgent final : public SacBase {
 public:
  SpederSacAgent(const AgentConfig& c, cudaStream_t s) : SacBase(c, s) {
    H_ = c.hidden_dim;  // critic_and_actor_hidden_dim
    D_ = c.feature_dim;
    K_ = c.k_feat;
    RLREP_CHECK(K_ >= 1 && K_ <= kMaxFeatureSteps, "extra_feature_steps out of range");
    RLREP_CHECK(D_ % 32 == 0, "feature_dim must be a multiple of 32");
    RLREP_CHECK(c.phi_hidden_depth >= 0 && c.mu_hidden_depth >= 0, "negative trunk depth");
    const RecordLayout lay = RecordLayout::of(S_, A_);
    off_r_ = lay.off_r;
    off_d_ = lay.off_d;
    off_s2_ = lay.off_s2;
    plan_common(K_ * 2 * B_, 2 * B_ * A_, lay.R, 2 * B_);

    // feature group: phi first so that phi_target is a prefix (spedersac_agent.py:147-166)
    feat_g_.name = "feature";
    phi_.plan(feat_g_, "phi.trunk", S_ + A_, c.phi_hidden_dim, D_, c.phi_hidden_depth);
    feat_g_.n_target = feat_g_.n;
    feat_g_.target_prefix_from = "phi.";
    feat_g_.target_prefix_to = "phi_target.";
    mu_.plan(feat_g_, "mu.trunk", S_, c.mu_hidden_dim, D_, c.mu_hidden_depth);
    th_ = add_linear(feat_g_, "theta.l", 1, D_, /*pad=*/false);
    feat_g_.want(arena_);

    crit_g_.name = "critic";
    critic_.plan(crit_g_, arena_, D_, H_, B_);
    crit_g_.n_target = crit_g_.n;
    crit_g_.target_prefix_from = "critic.";
    crit_g_.target_prefix_to = "critic_target.";
    crit_g_.want(arena_);

    const size_t BD2 = (size_t)2 * B_ * D_;
    phi_acts_.want(arena_, phi_, 2 * B_, true);
    mu_acts_.want(arena_, mu_, 2 * B_, true);
    phi_acts_b_.want(arena_, phi_, B_, false);
    phi_acts_c_.want(arena_, phi_, B_, true);
    arena_.want(&zpi_, (size_t)B_ * D_);
    arena_.want(&zphi_, BD2);
    arena_.want(&zmu_, BD2);
    arena_.want(&dzphi_, BD2);
    arena_.want(&dzmu_, BD2);
    arena_.want(&zb_, (size_t)B_ * D_);
    arena_.want(&u_, D_);
    arena_.want(&w_, D_);
    arena_.want(&diag_, B_);
    arena_.want(&c_, B_);
    arena_.want(&rpred_, B_);
    arena_.want(&drp_, B_);
    arena_.want(&dq_, 2 * B_);
    arena_.want(&logp2_, B_);
    finish_setup(0);

    names_ = {"total_loss", "model_loss", "r_loss", "q1_loss", "q2_loss", "q1", "q2", "actor_loss", "alpha_loss",
              "alpha"};
  }

  int idx_per_train() const override { return K_ * 2 * B_; }
  int eps_per_train() const override { return 2 * B_ * A_; }
  const std::vector<std::string>& metric_names() const override { return names_; }
  std::vector<ParamGroup*> groups() override { return {&feat_g_, &actor_g_, &crit_g_}; }
  void sync_targets_from_params() override {
    RLREP_CUDA(cudaMemcpyAsync(feat_g_.target, feat_g_.p, feat_g_.n_target * 4, cudaMemcpyDeviceToDevice, stream));
    RLREP_CUDA(cudaMemcpyAsync(crit_g_.target, crit_g_.p, crit_g_.n_target * 4, cudaMemcpyDeviceToDevice, stream));
    RLREP_CUDA(cudaStreamSynchronize(stream));
  }

 protected:
  void update(Ring& ring) override {  // spedersac_agent.py:291-322
    begin_update();
    launch_tick(ctl, base_tick(), stream);
    for (int k = 0; k < K_; ++k) {
      // rows [0, B): batch_1, rows [B, 2B): batch_2 -- drawn back to back by the host (:299-300)
      launch_gather(ring.data, R_ / 4, idx_dev_ + (size_t)k * 2 * B_, 2 * B_, batch_, stream);
      feature_step(k);
    }
    critic_step();
    actor_step();
  }

 private:
  Mat sa() const { return Mat{batch_, R_}; }
  Mat s2() const { return Mat{batch_ + off_s2_, R_}; }
  const float* reward() const { return batch_ + off_r_; }
  const float* done() const { return batch_ + off_d_; }

  void feature_step(int k) {  // spedersac_agent.py:181-219
    const Linear th = th_.view(feat_g_);
    cudaStream_t s0 = stream, s1 = side();
    const int B2 = 2 * B_;
    fork();
    trunk_forward(gemm_, s0, B2, phi_, feat_g_, false, sa(), Mat(), 0, phi_acts_, zphi_, D_);
    trunk_forward(gemm_, s1, B2, mu_, feat_g_, false, s2(), Mat(), 0, mu_acts_, zmu_, D_);
    {  // u = colsum(phi~)
      const ColJob job{zphi_ + (size_t)B_ * D_, nullptr, u_, D_, B_, D_};
      launch_colreduce_multi(&job, 1, s0);
    }
    join();
    launch_speder_rows(zphi_, zmu_, D_, B_, th.W, th.b, u_, diag_, rpred_, c_, s0);
    launch_speder_finalize(diag_, c_, rpred_, reward(), R_, B_, drp_, metrics_dev_ + 0, s0);
    {
      const ColJob jobs[3] = {ColJob{zmu_ + (size_t)B_ * D_, c_, w_, D_, B_, D_},  // w = mu~^T c
                              ColJob{zphi_, drp_, th.dW, D_, B_, D_},              // d theta.w
                              ColJob{drp_, nullptr, th.db, 1, B_, 1}};             // d theta.b
      launch_colreduce_multi(jobs, 3, s0);
    }
    launch_speder_grad(zphi_, zmu_, D_, B_, drp_, th.W, c_, u_, w_, dzphi_, dzmu_, s0);
    fork();
    {
      std::vector<ColJob> jobs;
      trunk_backward(gemm_, s0, B2, phi_, feat_g_, false, Mat{dzphi_, D_}, sa(), phi_acts_, true, &jobs, nullptr, 0, 0, 0);
      launch_bias_jobs(jobs, s0);
    }
    {
      std::vector<ColJob> jobs;
      trunk_backward(gemm_, s1, B2, mu_, feat_g_, false, Mat{dzmu_, D_}, s2(), mu_acts_, true, &jobs, nullptr, 0, 0, 0);
      launch_bias_jobs(jobs, s1);
    }
    join();
    launch_adam_polyak(feat_g_.p, feat_g_.g, feat_g_.m, feat_g_.v, feat_g_.n, &ctl->feat[k],
                       cfg.use_feature_target ? feat_g_.target : nullptr, feat_g_.n_target, cfg.feature_tau, nullptr,
                       s0);
  }

  void critic_step() {  // spedersac_agent.py:225-257
    const float* eps = eps_dev_;
    cudaStream_t s0 = stream, s1 = side();
    fork();
    // Hoisted out of the actor step (see agent_ctrlsac.cu): a_pi ~ pi(s) and phi(s, a_pi) read nothing the critic step
    // writes, so they run beside it on an aux branch; the actor step joins before it evaluates the updated critic.
    cudaStream_t a0 = aux(0);
    wait_for(a0, mark(s0));
    const Mat spi = actor_forward_cat(Mat{batch_, R_}, eps_dev_ + (size_t)B_ * A_, cat_pi_, logp_, a0, /*set=*/0);
    trunk_forward(gemm_, a0, B_, phi_, feat_g_, false, spi, Mat(), 0, phi_acts_c_, zpi_, D_);
    const Mat s2a = actor_forward_cat(s2(), eps, cat_next_, logp2_, s0, /*set=*/1);
    trunk_forward(gemm_, s0, B_, phi_, feat_g_, false, s2a, Mat(), 0, phi_acts_, zmu_, D_);
    critic_.forward(gemm_, s0, crit_g_, /*target=*/true, 0, zmu_);
    trunk_forward(gemm_, s1, B_, phi_, feat_g_, false, sa(), Mat(), 0, phi_acts_b_, zb_, D_);
    critic_.forward(gemm_, s1, crit_g_, /*target=*/false, 1, zb_);
    join();
    launch_td_critic_loss(reward(), done(), R_, critic_.q[0], critic_.q[0] + B_, logp2_, critic_.q[1], critic_.q[1] + B_,
                          B_, cfg.discount, ctl, dq_, dq_ + B_, metrics_dev_ + 3, s0);
    critic_.backward(gemm_, s0, crit_g_, 1, zb_, dq_, /*wgrad=*/true, nullptr);
    launch_adam_polyak(crit_g_.p, crit_g_.g, crit_g_.m, crit_g_.v, crit_g_.n, &ctl->critic, crit_g_.target,
                       crit_g_.n_target, cfg.tau, &ctl->polyak_critic, s0);
  }

  void actor_step() {  // spedersac_agent.py:259-289
    const float* eps = eps_dev_ + (size_t)B_ * A_;
    const Mat s{batch_, R_};
    join_aux(0, stream);
    critic_.forward(gemm_, stream, crit_g_, false, 0, zpi_);
    launch_actor_alpha_loss(critic_.q[0], critic_.q[0] + B_, logp_, B_, (float)(-A_), cfg.learn_alpha, ctl, dq_,
                            dq_ + B_, dlogp_, metrics_dev_ + 7, stream);
    critic_.backward(gemm_, stream, crit_g_, 0, zpi_, dq_, /*wgrad=*/false, dzphi_);
    const ActionGradDst ad = action_grad_dst(phi_.l[0].view(feat_g_));
    trunk_backward(gemm_, stream, B_, phi_, feat_g_, false, Mat{dzphi_, D_}, s, phi_acts_c_, false, nullptr, ad.dx, ad.ld,
                   ad.col0, ad.n_cols);
    actor_backward(s, eps);
    actor_adam();
  }

  int H_ = 0, D_ = 0, K_ = 0, off_r_ = 0, off_d_ = 0, off_s2_ = 0;
  ParamGroup feat_g_, crit_g_;
  Trunk phi_, mu_;
  TrunkActs phi_acts_, mu_acts_, phi_acts_b_, phi_acts_c_;
  float* zpi_ = nullptr;
  LinearSlot th_;
  RffCritic critic_;
  float *zphi_ = nullptr, *zmu_ = nullptr, *dzphi_ = nullptr, *dzmu_ = nullptr, *zb_ = nullptr;
  float *u_ = nullptr, *w_ = nullptr, *diag_ = nullptr, *c_ = nullptr, *rpred_ = nullptr, *drp_ = nullptr;
  float *dq_ = nullptr, *logp2_ = nullptr;
  std::vector<std::string> names_;
};

}  // namespace

std::unique_ptr<Agent> make_spedersac_agent(const AgentConfig& cfg, cudaStream_t s) {
  return std::unique_ptr<Agent>(new SpederSacAgent(cfg, s));
}

}  // namespace rlrep

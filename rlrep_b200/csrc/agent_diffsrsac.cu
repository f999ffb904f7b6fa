// Diff-SR-SAC update step (reference: agent/diffsrsac/diffsrsac_agent.py:205-343) as one stream of sm_100a kernels.
//
// Per train(): K x [gather -> DDPM perturbation of s' at host-drawn noise levels -> phi(s, a) and the
// grad-mu net on (s~', alpha-bar) -> score = phi^T grad-mu (the reference's bmm) -> noise-prediction loss ->
// backward -> fused Adam over phi | grad-mu] -> critic losses (metrics only) -> actor / temperature step -> Polyak.
//
// Reference quirks kept (SURVEY.md A.6 #1, #5): the RFF critic is NEVER optimised (its optimiser is bound to a
// discarded module) -- the critic step only reports losses, and critic_target drifts by Polyak rounding alone; phi is
// live (not frozen) in the critic / actor steps; the regulariser is multiplied by lambda = 0.
#include "agent_base.cuh"
#include "nets.cuh"

namespace rlrep {

namespace {

class DiffSrSacAgent final : public SacBase {
 public:
  DiffSrSacAgent(const AgentConfig& c, cudaStream_t s) : SacBase(c, s) {
    H_ = c.hidden_dim;
    D_ = c.feature_dim;
    K_ = c.k_feat;
    NL_ = c.num_noises;
    RLREP_CHECK(K_ >= 1 && K_ <= kMaxFeatureSteps, "extra_feature_steps out of range");
    RLREP_CHECK(D_ % 32 == 0, "feature_dim must be a multiple of 32");
    RLREP_CHECK(NL_ >= 1, "num_noises must be positive");
    const RecordLayout lay = RecordLayout::of(S_, A_);
    off_r_ = lay.off_r;
    off_d_ = lay.off_d;
    off_s2_ = lay.off_s2;
    // per feature iteration: B replay rows, then B noise levels; B*S Gaussian noise values
    plan_common(K_ * 2 * B_, K_ * B_ * S_ + 2 * B_ * A_, lay.R);

    // phi_optimizer and nablamu_optimizer (diffsrsac_agent.py:170-176) share lr / betas and always step together, so
    // their Adam updates are elementwise identical to one optimiser over phi | grad-mu: one launch.
    feat_g_.name = "feature";
    phi_.plan(feat_g_, "critic_feed_feature.z_vector", S_ + A_, c.phi_hidden_dim, D_, c.phi_hidden_depth);
    nabla_.plan(feat_g_, "nablamu_net.Mu_z_by_s_layer", S_ + 1, c.nabla_hidden_dim, D_ * S_, c.nabla_hidden_depth);
    feat_g_.want(arena_);

    crit_g_.name = "critic";
    critic_.plan(crit_g_, arena_, D_, H_, B_);
    crit_g_.n_target = crit_g_.n;
    crit_g_.target_prefix_from = "critic.";
    crit_g_.target_prefix_to = "critic_target.";
    crit_g_.want(arena_, /*with_opt=*/false);

    table_g_.name = "alphabars";
    table_off_ = table_g_.add("alphabars", 1, NL_);
    table_g_.want(arena_, /*with_opt=*/false);

    ld_x_ = round_up32(S_ + 1);
    ld_flat_ = round_up32(D_ * S_);
    phi_acts_.want(arena_, phi_, B_, true);
    phi_acts_b_.want(arena_, phi_, B_, false);
    phi_acts_c_.want(arena_, phi_, B_, true);
    arena_.want(&zpi_, (size_t)B_ * D_);
    nabla_acts_.want(arena_, nabla_, B_, true);
    arena_.want(&xin_, (size_t)B_ * ld_x_);
    arena_.want(&target_, (size_t)B_ * S_);
    arena_.want(&coef_, B_);
    arena_.want(&zphi_, (size_t)B_ * D_);
    arena_.want(&zb_, (size_t)B_ * D_);
    arena_.want(&dzphi_, (size_t)B_ * D_);
    arena_.want(&flat_, (size_t)B_ * D_ * S_);
    arena_.want(&dflat_, (size_t)B_ * D_ * S_ + 32);
    arena_.want(&dscore_, (size_t)B_ * S_);
    arena_.want(&loss_rows_, B_);
    arena_.want(&dq_, 2 * B_);
    arena_.want(&logp2_, B_);
    finish_setup(0);

    names_ = {"score_loss", "q1_loss", "q2_loss", "q1", "q2", "actor_loss", "alpha_loss", "alpha"};
  }

  int idx_per_train() const override { return K_ * 2 * B_; }
  int eps_per_train() const override { return K_ * B_ * S_ + 2 * B_ * A_; }
  const std::vector<std::string>& metric_names() const override { return names_; }
  std::vector<ParamGroup*> groups() override { return {&feat_g_, &actor_g_, &crit_g_, &table_g_}; }
  void sync_targets_from_params() override {
    RLREP_CUDA(cudaMemcpyAsync(crit_g_.target, crit_g_.p, crit_g_.n_target * 4, cudaMemcpyDeviceToDevice, stream));
    RLREP_CUDA(cudaStreamSynchronize(stream));
  }

 protected:
  bool is_replay_index(int i) const override { return (i / B_) % 2 == 0; }

  void update(Ring& ring) override {  // diffsrsac_agent.py:320-343
    begin_update();
    TickParams t = base_tick();
    t.critic_steps = 0;  // critic_optimizer never touches the RFF critic
    launch_tick(ctl, t, stream);
    for (int k = 0; k < K_; ++k) {
      launch_gather(ring.data, R_ / 4, idx_dev_ + (size_t)k * 2 * B_, B_, batch_, stream);
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

  void feature_step(int k) {  // critic_feeder_feature_step, diffsrsac_agent.py:271-318
    const long long* level = idx_dev_ + (size_t)k * 2 * B_ + B_;
    const float* noise = eps_dev_ + (size_t)k * B_ * S_;
    cudaStream_t s0 = stream, s1 = side();
    const int DS = D_ * S_;
    fork();
    trunk_forward(gemm_, s0, B_, phi_, feat_g_, false, sa(), Mat(), 0, phi_acts_, zphi_, D_);
    launch_diffsr_perturb(batch_ + off_s2_, R_, noise, level, table_g_.p + table_off_, NL_, cfg.sigma_scale, B_, S_, xin_,
                          ld_x_, target_, coef_, s1);
    trunk_forward(gemm_, s1, B_, nabla_, feat_g_, false, Mat{xin_, ld_x_}, Mat(), 0, nabla_acts_, flat_, DS);
    join();
    launch_diffsr_score(zphi_, flat_, D_, S_, target_, coef_, B_, dscore_, loss_rows_, s0);
    launch_sum_scaled(loss_rows_, B_, 1.f / (float)B_, metrics_dev_ + 0, s0);
    launch_diffsr_score_bwd(zphi_, flat_, D_, S_, B_, dscore_, dflat_, dzphi_, s0);
    fork();
    {
      std::vector<ColJob> jobs;
      trunk_backward(gemm_, s0, B_, phi_, feat_g_, false, Mat{dzphi_, D_}, sa(), phi_acts_, true, &jobs, nullptr, 0, 0, 0);
      launch_bias_jobs(jobs, s0);
    }
    {
      std::vector<ColJob> jobs;
      trunk_backward(gemm_, s1, B_, nabla_, feat_g_, false, Mat{dflat_, DS}, Mat{xin_, ld_x_}, nabla_acts_, true, &jobs,
                     nullptr, 0, 0, 0);
      launch_bias_jobs(jobs, s1);
    }
    join();
    launch_adam_polyak(feat_g_.p, feat_g_.g, feat_g_.m, feat_g_.v, feat_g_.n, &ctl->feat[k], nullptr, 0, 0.f, nullptr, s0);
  }

  void critic_step() {  // diffsrsac_agent.py:205-239: losses only
    const float* eps = eps_dev_ + (size_t)K_ * B_ * S_;
    cudaStream_t s0 = stream, s1 = side();
    fork();
    // Hoisted out of the actor step (see agent_ctrlsac.cu): a_pi ~ pi(s) and phi(s, a_pi) read nothing the critic step
    // writes, so they run beside it on an aux branch; the actor step joins before it evaluates the updated critic.
    cudaStream_t a0 = aux(0);
    wait_for(a0, mark(s0));
    const Mat spi = actor_forward_cat(Mat{batch_, R_}, eps_dev_ + (size_t)K_ * B_ * S_ + (size_t)B_ * A_, cat_pi_, logp_, a0, /*set=*/0);
    trunk_forward(gemm_, a0, B_, phi_, feat_g_, false, spi, Mat(), 0, phi_acts_c_, zpi_, D_);
    const Mat s2a = actor_forward_cat(s2(), eps, cat_next_, logp2_, s0, /*set=*/1);
    trunk_forward(gemm_, s0, B_, phi_, feat_g_, false, s2a, Mat(), 0, phi_acts_, zphi_, D_);
    critic_.forward(gemm_, s0, crit_g_, /*target=*/true, 0, zphi_);
    trunk_forward(gemm_, s1, B_, phi_, feat_g_, false, sa(), Mat(), 0, phi_acts_b_, zb_, D_);
    critic_.forward(gemm_, s1, crit_g_, /*target=*/false, 1, zb_);
    join();
    launch_td_critic_loss(reward(), done(), R_, critic_.q[0], critic_.q[0] + B_, logp2_, critic_.q[1], critic_.q[1] + B_,
                          B_, cfg.discount, ctl, dq_, dq_ + B_, metrics_dev_ + 1, s0);
  }

  void actor_step() {  // diffsrsac_agent.py:241-269
    const float* eps = eps_dev_ + (size_t)K_ * B_ * S_ + (size_t)B_ * A_;
    const Mat s{batch_, R_};
    join_aux(0, stream);
    critic_.forward(gemm_, stream, crit_g_, false, 0, zpi_);
    launch_actor_alpha_loss(critic_.q[0], critic_.q[0] + B_, logp_, B_, (float)(-A_), cfg.learn_alpha, ctl, dq_,
                            dq_ + B_, dlogp_, metrics_dev_ + 5, stream);
    critic_.backward(gemm_, stream, crit_g_, 0, zpi_, dq_, /*wgrad=*/false, dzphi_);
    const ActionGradDst ad = action_grad_dst(phi_.l[0].view(feat_g_));
    trunk_backward(gemm_, stream, B_, phi_, feat_g_, false, Mat{dzphi_, D_}, s, phi_acts_c_, false, nullptr, ad.dx, ad.ld,
                   ad.col0, ad.n_cols);
    actor_backward(s, eps);
    actor_adam();
    // update_target (sac_agent.py:99-102) still runs on the never-trained critic: tau*x + (1-tau)*x != x in fp32
    launch_polyak(crit_g_.p, crit_g_.target, crit_g_.n_target, cfg.tau, &ctl->polyak_critic, stream);
  }

  int H_ = 0, D_ = 0, K_ = 0, NL_ = 1000, off_r_ = 0, off_d_ = 0, off_s2_ = 0, ld_x_ = 0, ld_flat_ = 0;
  ParamGroup feat_g_, crit_g_, table_g_;
  size_t table_off_ = 0;
  Trunk phi_, nabla_;
  TrunkActs phi_acts_, phi_acts_b_, phi_acts_c_, nabla_acts_;
  float* zpi_ = nullptr;
  RffCritic critic_;
  float *xin_ = nullptr, *target_ = nullptr, *coef_ = nullptr, *zphi_ = nullptr, *zb_ = nullptr, *dzphi_ = nullptr;
  float *flat_ = nullptr, *dflat_ = nullptr, *dscore_ = nullptr, *loss_rows_ = nullptr;
  float *dq_ = nullptr, *logp2_ = nullptr;
  std::vector<std::string> names_;
};

}  // namespace

std::unique_ptr<Agent> make_diffsrsac_agent(const AgentConfig& cfg, cudaStream_t s) {
  return std::unique_ptr<Agent>(new DiffSrSacAgent(cfg, s));
}

}  // namespace rlrep

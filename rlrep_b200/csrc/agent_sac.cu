// Plain SAC update step (reference: agent/sac/sac_agent.py:105-188, agent/sac/critic.py:15-36) -- BASELINE config 1
// and the base every representation agent extends.  Twin Q MLPs on cat(s, a): the two first layers share their
// input, so they are stacked into one [2H, S+A] GEMM; the second layers and N = 1 heads run per head.
#include "agent_base.cuh"

namespace rlrep {

namespace {

class SacAgent final : public SacBase {
 public:
  SacAgent(const AgentConfig& c, cudaStream_t s, int members) : SacBase(c, s, members) {
    H_ = c.hidden_dim;
    RLREP_CHECK(H_ % 32 == 0, "hidden_dim must be a multiple of 32");
    const RecordLayout lay = RecordLayout::of(S_, A_);
    off_r_ = lay.off_r;
    off_d_ = lay.off_d;
    off_s2_ = lay.off_s2;
    plan_common(B_, 2 * B_ * A_, lay.R);

    crit_g_.name = "critic";
    const int in = S_ + A_;
    c0_.out = 2 * H_;
    c0_.in = in;
    c0_.ld = round_up32(in);
    c0_.out_alloc = 2 * H_;
    RLREP_CHECK(H_ % 32 == 0, "hidden_dim must be a multiple of 32");
    c0_.w_off = crit_g_.add("critic.Q1.0.weight", H_, in, c0_.ld);
    crit_g_.add("critic.Q2.0.weight", H_, in, c0_.ld);
    c0_.b_off = crit_g_.add("critic.Q1.0.bias", H_, 1);
    crit_g_.add("critic.Q2.0.bias", H_, 1);
    c1a_ = add_linear(crit_g_, "critic.Q1.2", H_, H_);
    c1b_ = add_linear(crit_g_, "critic.Q2.2", H_, H_);
    c2a_ = add_linear(crit_g_, "critic.Q1.4", 1, H_, false);
    c2b_ = add_linear(crit_g_, "critic.Q2.4", 1, H_, false);
    crit_g_.n_target = crit_g_.n;
    crit_g_.target_prefix_from = "critic.";
    crit_g_.target_prefix_to = "critic_target.";
    crit_g_.want(arena_);

    const size_t BH = (size_t)B_ * H_;
    arena_.want(&hid0_, 2 * BH);
    arena_.want(&hid1a_, BH);
    arena_.want(&hid1b_, BH);
    arena_.want(&dhid0_, 2 * BH);
    arena_.want(&dhid1a_, BH);
    arena_.want(&dhid1b_, BH);
    arena_.want(&q1_, B_);
    arena_.want(&q2_, B_);
    arena_.want(&nq1_, B_);
    arena_.want(&nq2_, B_);
    arena_.want(&dq1_, B_);
    arena_.want(&dq2_, B_);
    arena_.want(&logp2_, B_);
    finish_setup((size_t)4 << 20);
    names_ = {"q1_loss", "q2_loss", "q1", "q2", "actor_loss", "alpha_loss", "alpha"};
  }

  int idx_per_train() const override { return B_; }
  int eps_per_train() const override { return 2 * B_ * A_; }
  const std::vector<std::string>& metric_names() const override { return names_; }
  std::vector<ParamGroup*> groups() override { return {&crit_g_, &actor_g_}; }
  void sync_targets_from_params() override {
    copy_members(crit_g_.target, (size_t)mb.stride, crit_g_.p, (size_t)mb.stride, crit_g_.n_target * 4,
                 cudaMemcpyDeviceToDevice);
    RLREP_CUDA(cudaStreamSynchronize(stream));
  }

 protected:
  void update(Ring& ring) override {  // sac_agent.py:169-188
    begin_update();
    TickParams t = base_tick();
    t.k_feat = 0;
    launch_tick(ctl, t, stream, mb);
    launch_gather(ring.data, R_ / 4, idx_dev_, B_, batch_, stream, mb, ring_slot_);
    critic_step();
    actor_step();
  }

 private:
  // DoubleQCritic.forward on x = cat(x1, x2) (critic.py:26-36)
  void critic_forward(Mat x, Mat x2, int k1, bool target, float* q1, float* q2) {
    const Linear l0 = c0_.view(crit_g_, target), l1a = c1a_.view(crit_g_, target), l1b = c1b_.view(crit_g_, target);
    const Linear l2a = c2a_.view(crit_g_, target), l2b = c2b_.view(crit_g_, target);
    linear_fwd(gemm_, stream, B_, x, l0, ACT_ELU, hid0_, 2 * H_, x2, k1);
    linear_fwd(gemm_, stream, B_, Mat{hid0_, 2 * H_}, l1a, ACT_ELU, hid1a_, H_);
    linear_fwd(gemm_, stream, B_, Mat{hid0_ + H_, 2 * H_}, l1b, ACT_ELU, hid1b_, H_);
    launch_rowdot(hid1a_, H_, B_, H_, l2a.W, l2a.b, q1, stream, mb);
    launch_rowdot(hid1b_, H_, B_, H_, l2b.W, l2b.b, q2, stream, mb);
  }
  // (dq1, dq2) -> d hid1 -> d hid0 (activations of the matching critic_forward must be live)
  void critic_backward_to_hid0(bool with_wgrad) {
    const Linear l1a = c1a_.view(crit_g_), l1b = c1b_.view(crit_g_), l2a = c2a_.view(crit_g_), l2b = c2b_.view(crit_g_);
    launch_outer_dact(dq1_, l2a.W, B_, H_, hid1a_, H_, DACT_ELU_OUT, dhid1a_, H_, stream, mb);
    launch_outer_dact(dq2_, l2b.W, B_, H_, hid1b_, H_, DACT_ELU_OUT, dhid1b_, H_, stream, mb);
    if (with_wgrad) {
      launch_colreduce(hid1a_, H_, B_, H_, dq1_, l2a.dW, 0, stream, mb);
      launch_colreduce(dq1_, 1, B_, 1, nullptr, l2a.db, 0, stream, mb);
      launch_colreduce(hid1b_, H_, B_, H_, dq2_, l2b.dW, 0, stream, mb);
      launch_colreduce(dq2_, 1, B_, 1, nullptr, l2b.db, 0, stream, mb);
      linear_wgrad(gemm_, stream, B_, Mat{dhid1a_, H_}, Mat{hid0_, 2 * H_}, l1a);
      linear_wgrad(gemm_, stream, B_, Mat{dhid1b_, H_}, Mat{hid0_ + H_, 2 * H_}, l1b);
    }
    linear_dgrad(gemm_, stream, B_, Mat{dhid1a_, H_}, l1a, DACT_ELU_OUT, Mat{hid0_, 2 * H_}, dhid0_, 2 * H_);
    linear_dgrad(gemm_, stream, B_, Mat{dhid1b_, H_}, l1b, DACT_ELU_OUT, Mat{hid0_ + H_, 2 * H_}, dhid0_ + H_, 2 * H_);
  }

  void critic_step() {  // sac_agent.py:105-135
    const Mat sa{batch_, R_}, s2{batch_ + off_s2_, R_};
    const Mat s2a = actor_forward_cat(s2, eps_dev_, cat_next_, logp2_);
    critic_forward(s2a, Mat(), 0, /*target=*/true, nq1_, nq2_);
    critic_forward(sa, Mat(), 0, false, q1_, q2_);
    launch_td_critic_loss(batch_ + off_r_, batch_ + off_d_, R_, nq1_, nq2_, logp2_, q1_, q2_, B_, cfg.discount, ctl,
                          dq1_, dq2_, metrics_dev_ + 0, stream, 0, mb);
    critic_backward_to_hid0(true);
    linear_wgrad(gemm_, stream, B_, Mat{dhid0_, 2 * H_}, sa, c0_.view(crit_g_));
    launch_adam_polyak(crit_g_.p, crit_g_.g, crit_g_.m, crit_g_.v, crit_g_.n, &ctl->critic, crit_g_.target,
                       crit_g_.n_target, cfg.tau, &ctl->polyak_critic, stream, mb);
  }

  void actor_step() {  // sac_agent.py:138-166
    const float* eps = eps_dev_ + (size_t)B_ * A_;
    const Mat s{batch_, R_};
    const Mat spi = actor_forward_cat(s, eps, cat_pi_, logp_);
    critic_forward(spi, Mat(), 0, false, q1_, q2_);
    launch_actor_alpha_loss(q1_, q2_, logp_, B_, (float)(-A_), cfg.learn_alpha, ctl, dq1_, dq2_, dlogp_,
                            metrics_dev_ + 4, stream, mb);
    critic_backward_to_hid0(false);
    dgrad_to_action(Mat{dhid0_, 2 * H_}, c0_.view(crit_g_));
    actor_backward(s, eps);
    actor_adam();
  }

  int H_ = 0, off_r_ = 0, off_d_ = 0, off_s2_ = 0;
  ParamGroup crit_g_;
  LinearSlot c0_, c1a_, c1b_, c2a_, c2b_;
  float *hid0_ = nullptr, *hid1a_ = nullptr, *hid1b_ = nullptr, *dhid0_ = nullptr, *dhid1a_ = nullptr,
        *dhid1b_ = nullptr;
  float *q1_ = nullptr, *q2_ = nullptr, *nq1_ = nullptr, *nq2_ = nullptr, *dq1_ = nullptr, *dq2_ = nullptr;
  float *logp2_ = nullptr;
  std::vector<std::string> names_;
};

}  // namespace

std::unique_ptr<Agent> make_sac_agent(const AgentConfig& cfg, cudaStream_t s) {
  return std::unique_ptr<Agent>(new SacAgent(cfg, s, 1));
}
std::unique_ptr<Agent> make_sac_population(const AgentConfig& cfg, cudaStream_t s, int members) {
  return std::unique_ptr<Agent>(new SacAgent(cfg, s, members));
}

}  // namespace rlrep

// Batch-sharded CTRL-SAC update over N GPUs (BASELINE config 4; SURVEY.md 8e) -- one process per GPU, one handle per
// process, identical parameters on every rank, the GLOBAL batch of Bg = N * b rows split by rows.
//
// The reference has no distributed code; this is the data-parallel restatement of ctrlsac_agent.py:213-362 whose result
// is the single-process update on the global batch:
//   feature step   phi_local, mu_local on the rank's b rows
//                  all-gather mu              -> mu_all [Bg, D]                       (NCCL, NVLink / NVSwitch)
//                  logits_local = phi_local mu_all^T  [b, Bg]  (complete rows => the row log-sum-exp is local)
//                  G_local = (softmax - I) / Bg, diagonal at column rank * b + i
//                  d phi_local = G_local mu_all                      (local)
//                  d mu_all   = G_local^T phi_local  [Bg, D]   -> reduce-scatter -> rows of this rank, then * tanh'
//                  backward through phi / mu on the local rows, all-reduce of the parameter gradients, the SAME fused
//                  Adam(+Polyak) on every rank (all-reduce results are bit-identical across ranks, so parameters
//                  never diverge)
//   critic / actor plain data parallelism: means are over the global batch (every partial is divided by Bg), gradients
//                  and loss sums are all-reduced; the float64 temperature step runs on the all-reduced mean.
// Kernels are the single-GPU ones; b = 2048 rows per rank makes every GEMM throughput-bound, so the step runs eagerly
// (no graph).
//
// Overlap.  The all-gather of mu runs on a communication stream while phi's forward runs on the main stream, and the
// reduce-scatter of d mu_all while d z_phi and the phi backward are computed.  Pipelining the collectives in row slices
// of the rank's batch was measured on 8 x B200 (DESIGN.md section 6): 1 slice 7.45 ms / update, 2 slices 7.61, 4 slices
// 7.94 -- the smaller collectives lose more bandwidth, and take more SMs from the concurrent GEMMs, than the overlap wins.
#include "agent_base.cuh"
#include "comm.cuh"

namespace rlrep {

namespace {

class CtrlSacShardedAgent final : public SacBase {
 public:
  CtrlSacShardedAgent(const AgentConfig& c, cudaStream_t s, Comm* comm) : SacBase(c, s), comm_(comm) {
    RLREP_CHECK(comm_ != nullptr, "sharded agent needs a communicator");
    H_ = c.hidden_dim;
    D_ = c.feature_dim;
    K_ = c.k_feat;
    N_ = comm_->world;
    rank_ = comm_->rank;
    Bg_ = B_ * N_;
    cfg.use_graph = 0;
    dual_share_ = 1.0;  // throughput-bound GEMMs: plan each one for the whole GPU even when two branches overlap
    RLREP_CHECK(K_ >= 1 && K_ <= kMaxFeatureSteps, "extra_feature_steps out of range");
    RLREP_CHECK(H_ % 32 == 0 && D_ % 32 == 0 && B_ % 32 == 0, "hidden_dim, feature_dim and the per-rank batch must be multiples of 32");
    const RecordLayout lay = RecordLayout::of(S_, A_);
    off_r_ = lay.off_r;
    off_d_ = lay.off_d;
    off_s2_ = lay.off_s2;
    plan_common(K_ * B_, 2 * B_ * A_, lay.R);

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

    crit_g_.name = "critic";
    c14_.out = 2 * H_;
    c14_.in = D_;
    c14_.w_off = crit_g_.add("critic.l1.weight", H_, D_);
    crit_g_.add("critic.l4.weight", H_, D_);
    c14_.b_off = crit_g_.add("critic.l1.bias", H_, 1);
    crit_g_.add("critic.l4.bias", H_, 1);
    c2_ = add_linear(crit_g_, "critic.l2", 1, H_, false);
    c5_ = add_linear(crit_g_, "critic.l5", 1, H_, false);
    crit_g_.n_target = crit_g_.n;
    crit_g_.target_prefix_from = "critic.";
    crit_g_.target_prefix_to = "critic_target.";
    crit_g_.want(arena_);

    const size_t BH = (size_t)B_ * H_, BD = (size_t)B_ * D_;
    arena_.want(&h1_, BH); arena_.want(&h2_, BH); arena_.want(&g1_, BH); arena_.want(&g2_, BH);
    arena_.want(&zphi_, BD); arena_.want(&zmu_, BD); arena_.want(&dzphi_, BD); arena_.want(&dzmu_, BD);
    arena_.want(&dh2_, BH); arena_.want(&dh1_, BH); arena_.want(&dg2_, BH); arena_.want(&dg1_, BH);
    arena_.want(&zmu_all_, (size_t)Bg_ * D_);
    arena_.want(&dmu_all_, (size_t)Bg_ * D_);
    arena_.want(&logits_, (size_t)B_ * Bg_);
    arena_.want(&loss_rows_, B_);
    arena_.want(&rpred_, B_);
    arena_.want(&drp_, B_);
    arena_.want(&hid_, 2 * BH); arena_.want(&hid_t_, 2 * BH); arena_.want(&dhid_, 2 * BH);
    arena_.want(&q1_, B_); arena_.want(&q2_, B_); arena_.want(&nq1_, B_); arena_.want(&nq2_, B_);
    arena_.want(&dq1_, B_); arena_.want(&dq2_, B_);
    arena_.want(&logp2_, B_);
    arena_.want(&apart_, 4);
    finish_setup(0);

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
    for (int k = 0; k < K_; ++k) {
      launch_gather(ring.data, R_ / 4, idx_dev_ + (size_t)k * B_, B_, batch_, stream);
      feature_step(k);
    }
    critic_step();
    actor_step();
    comm_->all_reduce(metrics_dev_, 7, stream);  // additive partial means: feature, critic
    launch_alpha_step(apart_, cfg.learn_alpha, ctl, metrics_dev_ + 7, stream);
  }

 private:
  Mat sa() const { return Mat{batch_, R_}; }
  Mat s2() const { return Mat{batch_ + off_s2_, R_}; }
  const float* reward() const { return batch_ + off_r_; }
  const float* done() const { return batch_ + off_d_; }

  void phi_forward(Mat x, Mat x2, int k1, float* z) {
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    linear_fwd(gemm_, stream, B_, x, l1, ACT_ELU, h1_, H_, x2, k1);
    linear_fwd(gemm_, stream, B_, Mat{h1_, H_}, l2, ACT_ELU, h2_, H_);
    linear_fwd(gemm_, stream, B_, Mat{h2_, H_}, l3, ACT_NONE, z, D_);
  }

  void feature_step(int k) {
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    const Linear n1 = m1_.view(feat_g_), n2 = m2_.view(feat_g_), n3 = m3_.view(feat_g_);
    const Linear th = th_.view(feat_g_);
    const float inv_bg = 1.f / (float)Bg_;
    cudaStream_t s = stream, s1 = side();
    // mu on the side stream, phi on the main stream; the all-gather of mu runs on the communication stream.  Every rank
    // issues the collectives in the same host order, which is all NCCL asks for.
    cudaStream_t cs = aux(0);
    fork();
    linear_fwd(gemm_, s1, B_, s2(), n1, ACT_ELU, g1_, H_);
    linear_fwd(gemm_, s1, B_, Mat{g1_, H_}, n2, ACT_ELU, g2_, H_);
    linear_fwd(gemm_, s1, B_, Mat{g2_, H_}, n3, ACT_TANH, zmu_, D_);
    wait_for(cs, mark(s1));
    comm_->all_gather(zmu_, zmu_all_, (size_t)B_ * D_, cs);  // rank r's rows at row offset r * b of mu_all
    cudaEvent_t gathered = mark(cs);
    phi_forward(sa(), Mat(), 0, zphi_);
    wait_for(s, gathered);
    {  // logits_local[i, j] = <phi_i, mu_all_j>
      GemmArgs a;
      a.M = B_; a.N = Bg_; a.K = D_;
      a.A = zphi_; a.lda = D_;
      a.B = zmu_all_; a.ldb = D_;
      a.C = logits_; a.ldc = Bg_;
      gemm_.run(a, s);
    }
    join();
    // positives: local row i sits at column rank * b + i
    launch_ce_rows(logits_, Bg_, B_, Bg_, rank_ * B_, inv_bg, loss_rows_, s);
    launch_rowdot(zphi_, D_, B_, D_, th.W, th.b, rpred_, s);
    launch_feature_loss_finalize(loss_rows_, B_, rpred_, reward(), R_, inv_bg, drp_, metrics_dev_ + 0, s);
    // every rank's contribution to d mu of ALL rows: G_local^T phi_local -> reduce-scatter on the communication stream
    // while d z_phi and the phi backward are computed
    {
      GemmArgs a;
      a.M = Bg_; a.N = D_; a.K = B_;
      a.A = logits_; a.lda = Bg_; a.a_mn = true;
      a.B = zphi_; a.ldb = D_; a.b_mn = true;
      a.C = dmu_all_; a.ldc = D_;
      gemm_.run(a, s);
    }
    wait_for(cs, mark(s));
    comm_->reduce_scatter(dmu_all_, dzmu_, (size_t)B_ * D_, cs);
    cudaEvent_t scattered = mark(cs);
    {  // d z_phi = G_local mu_all + drp (x) theta.w
      GemmArgs a;
      a.M = B_; a.N = D_; a.K = Bg_;
      a.A = logits_; a.lda = Bg_;
      a.B = zmu_all_; a.ldb = D_; a.b_mn = true;
      a.C = dzphi_; a.ldc = D_;
      a.epi.r1_u = drp_; a.epi.r1_v = th.W;
      gemm_.run(a, s);
    }
    // side stream: the mu backward once its gradient has arrived; main stream: the phi backward
    fork();
    wait_for(s1, scattered);
    linear_wgrad(gemm_, s, B_, Mat{dzphi_, D_}, Mat{h2_, H_}, l3, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dzphi_, D_}, l3, DACT_ELU_OUT, Mat{h2_, H_}, dh2_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dh2_, H_}, Mat{h1_, H_}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, s, B_, Mat{dh2_, H_}, l2, DACT_ELU_OUT, Mat{h1_, H_}, dh1_, H_);
    linear_wgrad(gemm_, s, B_, Mat{dh1_, H_}, sa(), l1, Mat(), 0, false);
    {
      ColJob jobs[5] = {bias_job(B_, Mat{dzphi_, D_}, l3), bias_job(B_, Mat{dh2_, H_}, l2),
                        bias_job(B_, Mat{dh1_, H_}, l1), ColJob{zphi_, drp_, th.dW, D_, B_, D_},
                        ColJob{drp_, nullptr, th.db, 1, B_, 1}};
      launch_colreduce_multi(jobs, 5, s);
    }
    launch_mul_dact(dzmu_, zmu_, (size_t)B_ * D_, DACT_TANH_OUT, s1);
    linear_wgrad(gemm_, s1, B_, Mat{dzmu_, D_}, Mat{g2_, H_}, n3, Mat(), 0, false);
    linear_dgrad(gemm_, s1, B_, Mat{dzmu_, D_}, n3, DACT_ELU_OUT, Mat{g2_, H_}, dg2_, H_);
    linear_wgrad(gemm_, s1, B_, Mat{dg2_, H_}, Mat{g1_, H_}, n2, Mat(), 0, false);
    linear_dgrad(gemm_, s1, B_, Mat{dg2_, H_}, n2, DACT_ELU_OUT, Mat{g1_, H_}, dg1_, H_);
    linear_wgrad(gemm_, s1, B_, Mat{dg1_, H_}, s2(), n1, Mat(), 0, false);
    {
      ColJob jobs[3] = {bias_job(B_, Mat{dzmu_, D_}, n3), bias_job(B_, Mat{dg2_, H_}, n2),
                        bias_job(B_, Mat{dg1_, H_}, n1)};
      launch_colreduce_multi(jobs, 3, s1);
    }
    join_aux(0, s);
    join();
    comm_->all_reduce(feat_g_.g, feat_g_.n, s);
    launch_adam_polyak(feat_g_.p, feat_g_.g, feat_g_.m, feat_g_.v, feat_g_.n, &ctl->feat[k],
                       cfg.use_feature_target ? feat_g_.target : nullptr, feat_g_.n_target, cfg.feature_tau, nullptr, s);
  }

  void critic_forward(const float* z, bool target, float* hid, float* q1, float* q2) {
    const Linear l14 = c14_.view(crit_g_, target), l2 = c2_.view(crit_g_, target), l5 = c5_.view(crit_g_, target);
    linear_fwd(gemm_, stream, B_, Mat{z, D_}, l14, ACT_ELU, hid, 2 * H_);
    launch_rowdot_pair(RowDotJob{hid, l2.W, l2.b, q1, 2 * H_, H_}, RowDotJob{hid + H_, l5.W, l5.b, q2, 2 * H_, H_}, B_,
                       stream);
  }
  void critic_heads_backward_to_hidden() {
    const Linear l2 = c2_.view(crit_g_), l5 = c5_.view(crit_g_);
    launch_outer_dact(dq1_, l2.W, B_, H_, hid_, 2 * H_, DACT_ELU_OUT, dhid_, 2 * H_, stream);
    launch_outer_dact(dq2_, l5.W, B_, H_, hid_ + H_, 2 * H_, DACT_ELU_OUT, dhid_ + H_, 2 * H_, stream);
  }

  void critic_step() {
    const float* eps = eps_dev_;
    cudaStream_t s = stream;
    const Mat s2a = actor_forward_cat(s2(), eps, cat_next_, logp2_);
    phi_forward(s2a, Mat(), 0, zmu_);
    critic_forward(zmu_, /*target=*/true, hid_t_, nq1_, nq2_);
    phi_forward(sa(), Mat(), 0, zphi_);
    critic_forward(zphi_, /*target=*/false, hid_, q1_, q2_);
    launch_td_critic_loss(reward(), done(), R_, nq1_, nq2_, logp2_, q1_, q2_, B_, cfg.discount, ctl, dq1_, dq2_,
                          metrics_dev_ + 3, s, /*norm_B=*/Bg_);
    const Linear l14 = c14_.view(crit_g_), l2 = c2_.view(crit_g_), l5 = c5_.view(crit_g_);
    critic_heads_backward_to_hidden();
    {
      ColJob jobs[5] = {ColJob{hid_, dq1_, l2.dW, 2 * H_, B_, H_}, ColJob{dq1_, nullptr, l2.db, 1, B_, 1},
                        ColJob{hid_ + H_, dq2_, l5.dW, 2 * H_, B_, H_}, ColJob{dq2_, nullptr, l5.db, 1, B_, 1},
                        bias_job(B_, Mat{dhid_, 2 * H_}, l14)};
      launch_colreduce_multi(jobs, 5, s);
    }
    linear_wgrad(gemm_, s, B_, Mat{dhid_, 2 * H_}, Mat{zphi_, D_}, l14, Mat(), 0, false);
    comm_->all_reduce(crit_g_.g, crit_g_.n, s);
    launch_adam_polyak(crit_g_.p, crit_g_.g, crit_g_.m, crit_g_.v, crit_g_.n, &ctl->critic, crit_g_.target,
                       crit_g_.n_target, cfg.tau, &ctl->polyak_critic, s);
  }

  void actor_step() {
    const float* eps = eps_dev_ + (size_t)B_ * A_;
    const Mat s{batch_, R_};
    const Mat spi = actor_forward_cat(s, eps, cat_pi_, logp_);
    phi_forward(spi, Mat(), 0, zphi_);
    critic_forward(zphi_, false, hid_, q1_, q2_);
    launch_actor_loss_partial(q1_, q2_, logp_, B_, Bg_, (float)(-A_), ctl, dq1_, dq2_, dlogp_, apart_, stream);
    const Linear l14 = c14_.view(crit_g_);
    const Linear l1 = p1_.view(feat_g_), l2 = p2_.view(feat_g_), l3 = p3_.view(feat_g_);
    critic_heads_backward_to_hidden();
    linear_dgrad(gemm_, stream, B_, Mat{dhid_, 2 * H_}, l14, DACT_NONE, Mat(), dzphi_, D_);
    linear_dgrad(gemm_, stream, B_, Mat{dzphi_, D_}, l3, DACT_ELU_OUT, Mat{h2_, H_}, dh2_, H_);
    linear_dgrad(gemm_, stream, B_, Mat{dh2_, H_}, l2, DACT_ELU_OUT, Mat{h1_, H_}, dh1_, H_);
    dgrad_to_action(Mat{dh1_, H_}, l1);
    actor_backward(s, eps);
    comm_->all_reduce(actor_g_.g, actor_g_.n, stream);
    comm_->all_reduce(apart_, 2, stream);
    actor_adam();
  }

  Comm* comm_ = nullptr;
  int H_ = 0, D_ = 0, K_ = 0, N_ = 1, rank_ = 0, Bg_ = 0, off_r_ = 0, off_d_ = 0, off_s2_ = 0;
  ParamGroup feat_g_, crit_g_;
  LinearSlot p1_, p2_, p3_, m1_, m2_, m3_, th_, c14_, c2_, c5_;
  float *h1_ = nullptr, *h2_ = nullptr, *g1_ = nullptr, *g2_ = nullptr, *zphi_ = nullptr, *zmu_ = nullptr;
  float *dzphi_ = nullptr, *dzmu_ = nullptr, *dh2_ = nullptr, *dh1_ = nullptr, *dg2_ = nullptr, *dg1_ = nullptr;
  float *zmu_all_ = nullptr, *dmu_all_ = nullptr, *logits_ = nullptr;
  float *loss_rows_ = nullptr, *rpred_ = nullptr, *drp_ = nullptr, *hid_ = nullptr, *hid_t_ = nullptr, *dhid_ = nullptr;
  float *q1_ = nullptr, *q2_ = nullptr, *nq1_ = nullptr, *nq2_ = nullptr, *dq1_ = nullptr, *dq2_ = nullptr;
  float *logp2_ = nullptr, *apart_ = nullptr;
  std::vector<std::string> names_;
};

}  // namespace

std::unique_ptr<Agent> make_ctrlsac_sharded_agent(const AgentConfig& cfg, cudaStream_t s, Comm* comm) {
  return std::unique_ptr<Agent>(new CtrlSacShardedAgent(cfg, s, comm));
}

}  // namespace rlrep

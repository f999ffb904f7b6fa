// SacBase: what every SAC-family agent shares (reference: agent/sac/sac_agent.py) -- the tanh-Gaussian actor with
// its forward/backward, the control block with the float64 temperature, staging of the host-drawn indices and
// noise, metrics read-back, and the eager -> capture -> replay protocol of train().
// An agent built with members > 1 is a population (members.cuh): that many agents of this configuration, each with its
// own arena copy, trained by the one launch sequence every train() call runs.
#pragma once
#include "staging.cuh"

#include "agent.cuh"

namespace rlrep {

class SacBase : public Agent {
 public:
  SacBase(const AgentConfig& c, cudaStream_t s, int members = 1) {
    cfg = c;
    stream = s;
    S_ = c.state_dim;
    A_ = c.action_dim;
    B_ = c.batch;
    AH_ = c.actor_hidden_dim;
    members_ = members;
    RLREP_CHECK(S_ > 0 && A_ > 0 && B_ > 0, "bad agent dimensions");
    RLREP_CHECK(members_ >= 1 && members_ <= kActRows, "a population has 1 to 1024 members");
  }
  ~SacBase() override {
    for (cudaEvent_t e : events_) cudaEventDestroy(e);
    if (side_) cudaStreamDestroy(side_);
    for (cudaStream_t a : aux_)
      if (a) cudaStreamDestroy(a);
    if (metrics_host_) cudaFreeHost(metrics_host_);
    if (idx_host_) cudaFreeHost(idx_host_);
    if (eps_host_) cudaFreeHost(eps_host_);
    if (act_in_host_) cudaFreeHost(act_in_host_);
    if (act_out_host_) cudaFreeHost(act_out_host_);
  }

  void train(Ring& ring, const long long* idx_host, int n_idx, const float* eps_host, int n_eps, float* metrics_host,
             int n_metrics) override {
    Ring* rings[1] = {&ring};
    train_members(rings, idx_host, n_idx, eps_host, n_eps, metrics_host, n_metrics);
  }
  // rings[m], idx_host [members, idx_per_train()], eps_host [members, eps_per_train()] and metrics_host
  // [members, metric_names().size()] belong to member m.
  void train_members(Ring* const* rings, const long long* idx_host, int n_idx, const float* eps_host, int n_eps,
                     float* metrics_host, int n_metrics) override {
    const int ni = idx_per_train(), ne = eps_per_train(), nm = (int)metric_names().size();
    for (int m = 0; m < members_; ++m)
      RLREP_CHECK(rings[m]->S == S_ && rings[m]->A == A_, "ring shape does not match the agent" + member_note(m));
    RLREP_CHECK(n_idx == members_ * ni && n_eps == members_ * ne, "wrong number of indices / noise values");
    RLREP_CHECK(n_metrics >= members_ * nm, "metrics buffer too small");
    for (int m = 0; m < members_; ++m)
      for (int i = 0; i < ni; ++i) {
        const long long j = idx_host[(size_t)m * ni + i];
        RLREP_CHECK(!is_replay_index(i) || (j >= 0 && j < rings[m]->size), "replay index out of range" + member_note(m));
      }
    bind_rings(rings);
    RLREP_CUDA(cudaStreamSynchronize(stream));  // pinned staging is reused across calls
    std::memcpy(idx_host_, idx_host, (size_t)n_idx * sizeof(long long));
    to_members(idx_dev_, idx_host_, (size_t)ni * sizeof(long long), cudaMemcpyHostToDevice);
    if (is_device_pointer(eps_host)) {
      // noise drawn on the device by the caller (agents.py noise_device = "cuda"): it never touches the host
      to_members(eps_dev_, eps_host, (size_t)ne * sizeof(float), cudaMemcpyDeviceToDevice);
    } else {
      std::memcpy(eps_host_, eps_host, (size_t)n_eps * sizeof(float));
      to_members(eps_dev_, eps_host_, (size_t)ne * sizeof(float), cudaMemcpyHostToDevice);
    }
    const long long before = launch_count();
    const bool was_captured = graph_.captured();
    graph_.run(stream, cfg.use_graph != 0, [&] { update(*rings[0]); });
    if (!was_captured) launches_per_train_ = (int)(launch_count() - before);
    last_launches = launches_per_train_;
    // one device-to-host copy of every member's kNumMetrics-float block
    copy_members(metrics_host_, kNumMetrics * sizeof(float), metrics_dev_, (size_t)mb.stride, kNumMetrics * sizeof(float),
                 cudaMemcpyDeviceToHost);
    RLREP_CUDA(cudaStreamSynchronize(stream));
    for (int m = 0; m < members_; ++m)
      std::memcpy(metrics_host + (size_t)m * nm, metrics_host_ + (size_t)m * kNumMetrics, nm * sizeof(float));
  }

  float train_resident(Ring& ring, const long long* idx_host, const float* eps_host, int n_steps) override {
    Ring* rings[1] = {&ring};
    return train_resident_members(rings, idx_host, eps_host, n_steps);
  }
  // idx_host [n_steps, members, idx_per_train()], eps_host [n_steps, members, eps_per_train()]
  float train_resident_members(Ring* const* rings, const long long* idx_host, const float* eps_host, int n_steps) override {
    const int ni = idx_per_train(), ne = eps_per_train(), N = members_;
    RLREP_CHECK(n_steps > 0, "bad arguments");
    for (int m = 0; m < N; ++m) RLREP_CHECK(rings[m]->S == S_ && rings[m]->A == A_, "bad arguments");
    bind_rings(rings);
    long long* idx_all = nullptr;
    float* eps_all = nullptr;
    RLREP_CUDA(cudaMalloc(&idx_all, (size_t)n_steps * N * ni * sizeof(long long)));
    RLREP_CUDA(cudaMalloc(&eps_all, (size_t)n_steps * N * ne * sizeof(float)));
    RLREP_CUDA(cudaMemcpy(idx_all, idx_host, (size_t)n_steps * N * ni * sizeof(long long), cudaMemcpyHostToDevice));
    RLREP_CUDA(cudaMemcpy(eps_all, eps_host, (size_t)n_steps * N * ne * sizeof(float), cudaMemcpyHostToDevice));
    cudaEvent_t e0, e1;
    RLREP_CUDA(cudaEventCreate(&e0));
    RLREP_CUDA(cudaEventCreate(&e1));
    RLREP_CUDA(cudaStreamSynchronize(stream));
    RLREP_CUDA(cudaEventRecord(e0, stream));
    for (int i = 0; i < n_steps; ++i) {
      to_members(idx_dev_, idx_all + (size_t)i * N * ni, (size_t)ni * sizeof(long long), cudaMemcpyDeviceToDevice);
      to_members(eps_dev_, eps_all + (size_t)i * N * ne, (size_t)ne * sizeof(float), cudaMemcpyDeviceToDevice);
      graph_.run(stream, cfg.use_graph != 0, [&] { update(*rings[0]); });
    }
    RLREP_CUDA(cudaEventRecord(e1, stream));
    RLREP_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    RLREP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(idx_all);
    cudaFree(eps_all);
    return ms;
  }

  std::vector<ProfileEntry> profile_train(Ring& ring, const long long* idx_host, const float* eps_host) override {
    const int ni = idx_per_train(), ne = eps_per_train();
    RLREP_CUDA(cudaStreamSynchronize(stream));
    std::memcpy(idx_host_, idx_host, (size_t)ni * sizeof(long long));
    std::memcpy(eps_host_, eps_host, (size_t)ne * sizeof(float));
    RLREP_CUDA(cudaMemcpyAsync(idx_dev_, idx_host_, (size_t)ni * sizeof(long long), cudaMemcpyHostToDevice, stream));
    RLREP_CUDA(cudaMemcpyAsync(eps_dev_, eps_host_, (size_t)ne * sizeof(float), cudaMemcpyHostToDevice, stream));
    serial_ = true;  // one stream, so consecutive launch events bracket exactly one kernel
    profile_begin(stream);
    try {
      update(ring);
    } catch (...) {
      serial_ = false;
      throw;
    }
    serial_ = false;
    return profile_end(stream);
  }

  // select_action (sac_agent.py:89-96): eps == nullptr -> tanh(mu), else tanh(mu + std * eps).  Clamping to the
  // action range is done by the caller (the range belongs to the environment, not to this handle).  `rows` observations
  // are evaluated by ONE kernel launch per chunk of kActRows; the kernel reads them from, and writes the actions to, mapped
  // pinned host memory, so a call is: memcpy into the staging buffer, one launch, one stream synchronise.
  bool graph_stats(int* kernel_nodes, int* programmatic_edges) const override {
    return graph_.stats(kernel_nodes, programmatic_edges);
  }

  void act(const float* state_host, const float* eps_host, float* action_host) override {
    act_batch(state_host, eps_host, 1, action_host);
  }
  // One observation per member: states_host [members, S], eps_host [members, A] or nullptr -> actions_host [members, A],
  // one launch.
  void act_members(const float* states_host, const float* eps_host, float* actions_host) override {
    RLREP_CHECK(states_host && actions_host, "bad arguments");
    if (members_ == 1) return act_batch(states_host, eps_host, 1, actions_host);
    const Linear l0 = a0_.view(actor_g_), l1 = a1_.view(actor_g_), l2 = a2_.view(actor_g_);
    const int W = S_ + A_;
    RLREP_CUDA(cudaStreamSynchronize(stream));  // the staging buffers are reused
    for (int m = 0; m < members_; ++m) {
      float* dst = act_in_host_ + (size_t)m * W;
      std::memcpy(dst, states_host + (size_t)m * S_, S_ * sizeof(float));
      if (eps_host) std::memcpy(dst + S_, eps_host + (size_t)m * A_, A_ * sizeof(float));
    }
    launch_actor_act(act_in_dev_, 1, S_, A_, AH_, l0.W, l0.ld, l0.b, l1.W, l1.ld, l1.b, l2.W, l2.ld, l2.b,
                     eps_host != nullptr, act_out_dev_, stream, mb);
    RLREP_CUDA(cudaStreamSynchronize(stream));
    std::memcpy(actions_host, act_out_host_, (size_t)members_ * A_ * sizeof(float));
  }
  void act_batch(const float* states_host, const float* eps_host, int rows, float* actions_host) override {
    RLREP_CHECK(rows >= 0 && states_host && actions_host, "bad arguments");
    const Linear l0 = a0_.view(actor_g_), l1 = a1_.view(actor_g_), l2 = a2_.view(actor_g_);
    const int W = S_ + A_;
    for (int done = 0; done < rows; done += kActRows) {
      const int n = std::min(kActRows, rows - done);
      RLREP_CUDA(cudaStreamSynchronize(stream));  // the staging buffers are reused
      for (int r = 0; r < n; ++r) {
        float* dst = act_in_host_ + (size_t)r * W;
        std::memcpy(dst, states_host + (size_t)(done + r) * S_, S_ * sizeof(float));
        if (eps_host) std::memcpy(dst + S_, eps_host + (size_t)(done + r) * A_, A_ * sizeof(float));
      }
      launch_actor_act(act_in_dev_, n, S_, A_, AH_, l0.W, l0.ld, l0.b, l1.W, l1.ld, l1.b, l2.W, l2.ld, l2.b,
                       eps_host != nullptr, act_out_dev_, stream);
      RLREP_CUDA(cudaStreamSynchronize(stream));
      std::memcpy(actions_host + (size_t)done * A_, act_out_host_, (size_t)n * A_ * sizeof(float));
    }
  }

 protected:
  // Captured graphs bake ring.data into their gather nodes: a different ring (also one that happens to live at a freed
  // ring's address) invalidates the graph.  A population's members read their ring from a word in their arena
  // (ring_slot_), rewritten here whenever the set of rings changes.
  void bind_rings(Ring* const* rings) {
    bool same = true;
    for (int m = 0; m < members_; ++m) same = same && rings_bound_[m] == rings[m]->generation;
    if (same) return;
    graph_.reset();
    for (int m = 0; m < members_; ++m) rings_bound_[m] = rings[m]->generation;
    if (members_ > 1) {
      std::vector<const float*> data(members_);
      for (int m = 0; m < members_; ++m) data[m] = rings[m]->data;
      RLREP_CUDA(cudaStreamSynchronize(stream));
      to_members(ring_slot_, data.data(), sizeof(const float*), cudaMemcpyHostToDevice);
      RLREP_CUDA(cudaStreamSynchronize(stream));
    }
  }
  std::string member_note(int m) const { return members_ > 1 ? " (member " + std::to_string(m) + ")" : ""; }
  // dst_dev / src each hold `members_` blocks of `bytes`, one per member, at member pitch dpitch / spitch.
  void copy_members(void* dst, size_t dpitch, const void* src, size_t spitch, size_t bytes, cudaMemcpyKind kind) {
    if (members_ == 1) RLREP_CUDA(cudaMemcpyAsync(dst, src, bytes, kind, stream));
    else RLREP_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, bytes, members_, kind, stream));
  }
  // members_ dense blocks of `bytes` at src -> the same buffer of every member's arena
  void to_members(void* dst_dev, const void* src, size_t bytes, cudaMemcpyKind kind) {
    copy_members(dst_dev, (size_t)mb.stride, src, bytes, bytes, kind);
  }
  // One full train() worth of launches on `stream`, reading idx_dev_ / eps_dev_ and writing metrics_dev_.
  virtual void update(Ring& ring) = 0;

  // Independent kernel chains (phi | mu, target | live critic ...) run on a side stream between fork() and join().
  // Under graph capture these become parallel branches of the graph; each kernel here is latency- rather than
  // throughput-bound at B = 256, so overlapping two chains hides most of one of them.
  cudaStream_t side() {
    if (serial_) return stream;
    if (side_ == nullptr) RLREP_CUDA(cudaStreamCreateWithFlags(&side_, cudaStreamNonBlocking));
    return side_;
  }
  cudaEvent_t next_event() {
    if (ev_next_ == events_.size()) {
      cudaEvent_t e;
      RLREP_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      events_.push_back(e);
    }
    return events_[ev_next_++];
  }
  void fork() {
    gemm_.set_sm_share(dual_share_);
    if (serial_) return;
    cudaEvent_t e = next_event();
    RLREP_CUDA(cudaEventRecord(e, stream));
    RLREP_CUDA(cudaStreamWaitEvent(side(), e, 0));
  }
  void join() {
    gemm_.set_sm_share(1.0);
    if (serial_) return;
    cudaEvent_t e = next_event();
    RLREP_CUDA(cudaEventRecord(e, side()));
    RLREP_CUDA(cudaStreamWaitEvent(stream, e, 0));
  }
  void begin_update() { ev_next_ = 0; }

  // Finer-grained DAG edges for work that is off the critical path (weight / bias gradients run beside the dgrad
  // chain that the next layer is waiting for): aux(i) are extra streams, mark() / wait_for() build the edges, and
  // join_aux(i) folds an aux stream back into `to` (every forked stream must rejoin before the capture ends).
  cudaStream_t aux(int i) {
    if (serial_) return stream;
    if (aux_[i] == nullptr) RLREP_CUDA(cudaStreamCreateWithFlags(&aux_[i], cudaStreamNonBlocking));
    return aux_[i];
  }
  cudaEvent_t mark(cudaStream_t s) {
    if (serial_) return nullptr;
    cudaEvent_t e = next_event();
    RLREP_CUDA(cudaEventRecord(e, s));
    return e;
  }
  void wait_for(cudaStream_t s, cudaEvent_t e) {
    if (serial_ || e == nullptr) return;
    RLREP_CUDA(cudaStreamWaitEvent(s, e, 0));
  }
  void join_aux(int i, cudaStream_t to) {
    if (serial_) return;
    wait_for(to, mark(aux(i)));
  }

  // Position i of the index array is a replay-ring row (range-checked against the ring); agents that also receive
  // other host-drawn integers (Diff-SR's noise levels) override this.
  virtual bool is_replay_index(int /*i*/) const { return true; }

  void plan_common(int n_idx, int n_eps, int ring_R, int batch_rows = 0) {
    R_ = ring_R;
    LDH_ = round_up32(2 * A_);  // padded pitch of head_ / dhead_ (zero padding columns; weight rows are padded too)
    actor_g_.name = "actor";
    a0_ = add_linear(actor_g_, "actor.trunk.0", AH_, S_);  // agent/sac/actor.py:66-74
    a1_ = add_linear(actor_g_, "actor.trunk.2", AH_, AH_);
    a2_ = add_linear(actor_g_, "actor.trunk.4", 2 * A_, AH_);
    actor_g_.want(arena_);
    arena_.want(&ctl, 1);
    arena_.want(&metrics_dev_, kNumMetrics);
    arena_.want(&idx_dev_, n_idx);
    arena_.want(&eps_dev_, n_eps);
    arena_.want(&batch_, (size_t)(batch_rows > 0 ? batch_rows : B_) * R_);
    arena_.want(&ah1_, (size_t)B_ * AH_);
    arena_.want(&ah2_, (size_t)B_ * AH_);
    arena_.want(&head_, (size_t)B_ * round_up32(2 * A_));  // pitch LDH_: the head runs as an N = 32k tensor-core GEMM
    arena_.want(&bh1_, (size_t)B_ * AH_);
    arena_.want(&bh2_, (size_t)B_ * AH_);
    arena_.want(&bhead_, (size_t)B_ * round_up32(2 * A_));
    arena_.want(&logp_, B_);
    arena_.want(&dhead_, (size_t)B_ * LDH_);
    arena_.want(&dah2_, (size_t)B_ * AH_);
    arena_.want(&dah1_, (size_t)B_ * AH_);
    LDSA_ = round_up32(S_ + A_);
    arena_.want(&dsa_, (size_t)B_ * LDSA_);
    arena_.want(&cat_next_, (size_t)B_ * LDSA_);  // cat(s', a')   (critic step)
    arena_.want(&cat_pi_, (size_t)B_ * LDSA_);    // cat(s, a_pi)  (actor step)
    arena_.want(&dlogp_, 4);
    if (members_ > 1) arena_.want(&ring_slot_, 1);
    rings_bound_.assign(members_, 0);
    RLREP_CUDA(cudaMallocHost(&metrics_host_, (size_t)members_ * kNumMetrics * sizeof(float)));
    RLREP_CUDA(cudaMallocHost(&idx_host_, (size_t)members_ * (n_idx > 0 ? n_idx : 1) * sizeof(long long)));
    RLREP_CUDA(cudaMallocHost(&eps_host_, (size_t)members_ * (n_eps > 0 ? n_eps : 1) * sizeof(float)));
    // select_action staging: mapped pinned memory the policy kernel reads / writes directly
    RLREP_CUDA(cudaHostAlloc(&act_in_host_, (size_t)kActRows * (S_ + A_) * sizeof(float), cudaHostAllocMapped));
    RLREP_CUDA(cudaHostAlloc(&act_out_host_, (size_t)kActRows * A_ * sizeof(float), cudaHostAllocMapped));
    std::memset(act_in_host_, 0, (size_t)kActRows * (S_ + A_) * sizeof(float));
    RLREP_CUDA(cudaHostGetDevicePointer(&act_in_dev_, act_in_host_, 0));
    RLREP_CUDA(cudaHostGetDevicePointer(&act_out_dev_, act_out_host_, 0));
  }

  void finish_setup(size_t gemm_ws_floats) {
    arena_.commit(members_);
    if (members_ > 1) mb = Members{members_, (long long)arena_.bytes()};
    gemm_.init(static_cast<Precision>(cfg.precision), gemm_ws_floats);
    gemm_.set_members(mb);
    Control h;
    std::memset(&h, 0, sizeof(h));
    h.log_alpha = std::log(cfg.alpha0);  // torch.tensor(np.log(alpha)), float64
    h.alpha = (float)cfg.alpha0;
    for (int m = 0; m < members_; ++m)
      RLREP_CUDA(cudaMemcpyAsync(member_ptr(ctl, m * mb.stride), &h, sizeof(h), cudaMemcpyHostToDevice, stream));
    RLREP_CUDA(cudaStreamSynchronize(stream));
  }

  // actor(obs) -> head_, then rsample with eps -> action_out [B, A], logp_out [B]
  // action_out may point into a cat(obs, action) buffer (cat_next_ / cat_pi_, pitch LDSA_): pass cat = true to have
  // the sampling kernel copy obs in front of the action, so the next network reads ONE contiguous input.
  // `set` selects the activation buffers: 0 = the set actor_backward() reads (the actor step's forward), 1 = a scratch
  // set for forwards without a backward (a' = pi(s') of the critic step), so both can be in flight at once.
  Mat actor_forward_cat(Mat obs, const float* eps, float* cat_buf, float* logp_out, cudaStream_t s = nullptr, int set = 0) {
    if (s == nullptr) s = stream;
    const Linear l0 = a0_.view(actor_g_), l1 = a1_.view(actor_g_), l2 = a2_.view(actor_g_);
    float* h1 = set == 0 ? ah1_ : bh1_;
    float* h2 = set == 0 ? ah2_ : bh2_;
    float* hd = set == 0 ? head_ : bhead_;
    linear_fwd(gemm_, s, B_, obs, l0, ACT_ELU, h1, AH_);
    linear_fwd(gemm_, s, B_, Mat{h1, AH_}, l1, ACT_ELU, h2, AH_);
    linear_fwd(gemm_, s, B_, Mat{h2, AH_}, l2, ACT_NONE, hd, LDH_);
    launch_actor_sample(hd, LDH_, B_, A_, eps, cat_buf + S_, LDSA_, logp_out, s, obs.p, obs.ld, S_, mb);
    return Mat{cat_buf, LDSA_};
  }
  // The two halves of actor_forward_cat for callers that run the trunk GEMMs of several networks as one GEMM chain.
  void actor_trunk(Mat obs, int set, cudaStream_t s) {
    const Linear l0 = a0_.view(actor_g_), l1 = a1_.view(actor_g_), l2 = a2_.view(actor_g_);
    float* h1 = set == 0 ? ah1_ : bh1_;
    float* h2 = set == 0 ? ah2_ : bh2_;
    float* hd = set == 0 ? head_ : bhead_;
    linear_fwd(gemm_, s, B_, obs, l0, ACT_ELU, h1, AH_);
    linear_fwd(gemm_, s, B_, Mat{h1, AH_}, l1, ACT_ELU, h2, AH_);
    linear_fwd(gemm_, s, B_, Mat{h2, AH_}, l2, ACT_NONE, hd, LDH_);
  }
  // Both samples after actor_trunk(next_obs, 1) and actor_trunk(obs, 0), in one launch: cat(s', a') into cat_next_ with
  // log pi(a'|s') into logp_next, and cat(s, a_pi) into cat_pi_ with log pi(a_pi|s) into logp_.
  void actor_sample_cat_pair(Mat next_obs, const float* eps_next, float* logp_next, Mat obs, const float* eps_pi,
                             cudaStream_t s) {
    launch_actor_sample_pair(ActorSampleJob{bhead_, eps_next, cat_next_ + S_, logp_next, next_obs.p, next_obs.ld},
                             ActorSampleJob{head_, eps_pi, cat_pi_ + S_, logp_, obs.p, obs.ld}, LDH_, B_, A_, LDSA_, S_, s);
  }
  // actor_backward with the five GEMMs as one chain on the main stream (no aux branches)
  void actor_backward_chained(Mat obs, const float* eps) {
    const Linear l0 = a0_.view(actor_g_), l1 = a1_.view(actor_g_), l2 = a2_.view(actor_g_);
    launch_actor_sample_bwd(head_, LDH_, B_, A_, eps, dsa_ + S_, LDSA_, dlogp_, dhead_, LDH_, stream);
    gemm_.begin_chain(stream);
    linear_wgrad(gemm_, stream, B_, Mat{dhead_, LDH_}, Mat{ah2_, AH_}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, stream, B_, Mat{dhead_, LDH_}, l2, DACT_ELU_OUT, Mat{ah2_, AH_}, dah2_, AH_);
    linear_wgrad(gemm_, stream, B_, Mat{dah2_, AH_}, Mat{ah1_, AH_}, l1, Mat(), 0, false);
    linear_dgrad(gemm_, stream, B_, Mat{dah2_, AH_}, l1, DACT_ELU_OUT, Mat{ah1_, AH_}, dah1_, AH_);
    linear_wgrad(gemm_, stream, B_, Mat{dah1_, AH_}, obs, l0, Mat(), 0, false);
    gemm_.end_chain();
    const ColJob jobs[3] = {bias_job(B_, Mat{dhead_, LDH_}, l2), bias_job(B_, Mat{dah2_, AH_}, l1),
                            bias_job(B_, Mat{dah1_, AH_}, l0)};
    launch_colreduce_multi(jobs, 3, stream);
  }
  // Where the first layer of a network fed with cat(obs, action) writes its input gradient so that actor_backward finds
  // d(action) at dsa_[:, S:S+A].  On the tensor-core path the dgrad runs over ALL (padded) input columns -- N must be a
  // multiple of 32 there and the few extra columns are free -- otherwise only over the action columns.
  struct ActionGradDst {
    float* dx;
    int ld, col0, n_cols;
  };
  ActionGradDst action_grad_dst(const Linear& first) const {
    if (cfg.precision == PREC_TF32 && first.ld == LDSA_ && B_ >= 64) return {dsa_, LDSA_, 0, LDSA_};
    return {dsa_ + S_, LDSA_, S_, A_};
  }
  void dgrad_to_action(Mat dy, const Linear& first) {
    const ActionGradDst d = action_grad_dst(first);
    linear_dgrad(gemm_, stream, B_, dy, first, DACT_NONE, Mat(), d.dx, d.ld, d.col0, d.n_cols);
  }
  // Needs d(action) in dsa_[:, S:S+A] and *dlogp_; the activations of the matching actor_forward_cat(obs, eps, ..., set 0) must still be
  // in ah1_/ah2_/head_.  Leaves the actor gradients in actor_g_.g.
  void actor_backward(Mat obs, const float* eps) {
    const Linear l0 = a0_.view(actor_g_), l1 = a1_.view(actor_g_), l2 = a2_.view(actor_g_);
    // dgrad chain on the main stream; weight / bias gradients trail it on an aux branch
    cudaStream_t w = aux(1);
    launch_actor_sample_bwd(head_, LDH_, B_, A_, eps, dsa_ + S_, LDSA_, dlogp_, dhead_, LDH_, stream, mb);
    wait_for(w, mark(stream));
    linear_wgrad(gemm_, w, B_, Mat{dhead_, LDH_}, Mat{ah2_, AH_}, l2, Mat(), 0, false);
    linear_dgrad(gemm_, stream, B_, Mat{dhead_, LDH_}, l2, DACT_ELU_OUT, Mat{ah2_, AH_}, dah2_, AH_);
    wait_for(w, mark(stream));
    linear_wgrad(gemm_, w, B_, Mat{dah2_, AH_}, Mat{ah1_, AH_}, l1, Mat(), 0, false);
    linear_dgrad(gemm_, stream, B_, Mat{dah2_, AH_}, l1, DACT_ELU_OUT, Mat{ah1_, AH_}, dah1_, AH_);
    linear_wgrad(gemm_, stream, B_, Mat{dah1_, AH_}, obs, l0, Mat(), 0, false);
    wait_for(w, mark(stream));
    {
      const ColJob jobs[3] = {bias_job(B_, Mat{dhead_, LDH_}, l2), bias_job(B_, Mat{dah2_, AH_}, l1),
                              bias_job(B_, Mat{dah1_, AH_}, l0)};
      launch_colreduce_multi(jobs, 3, w, mb);
    }
    join_aux(1, stream);
  }
  void actor_adam() {
    launch_adam_polyak(actor_g_.p, actor_g_.g, actor_g_.m, actor_g_.v, actor_g_.n, &ctl->actor, nullptr, 0, 0.f,
                       nullptr, stream, mb);
  }
  TickParams base_tick() const {
    TickParams t;
    t.k_feat = cfg.k_feat;
    t.period = cfg.target_update_period;
    t.lr_feat = cfg.lr_feat;
    t.lr_critic = cfg.lr;
    t.lr_actor = cfg.lr_actor;
    t.lr_alpha = cfg.lr_alpha;
    t.critic_steps = 1;
    return t;
  }

  int S_ = 0, A_ = 0, B_ = 0, AH_ = 0, R_ = 0, LDH_ = 0, LDSA_ = 0;
  cudaStream_t side_ = nullptr;
  cudaStream_t aux_[2] = {nullptr, nullptr};
  static constexpr double kAuxShare = 0.25;  // SM share the GEMMs on an aux stream plan for
  // Batches up to this size run their GEMM groups as chains (gemm_chain.cuh); larger batches are throughput- rather than
  // latency-bound and keep one kernel per GEMM.
  static constexpr int kChainMaxBatch = 512;
  bool chained() const { return gemm_.chains_enabled() && B_ <= kChainMaxBatch; }
  std::vector<cudaEvent_t> events_;
  size_t ev_next_ = 0;
  bool serial_ = false;
  double dual_share_ = 0.5;  // SM share inside fork() / join()
  DeviceArena arena_;
  GemmRunner gemm_;
  GraphReplay graph_;
  std::vector<unsigned long long> rings_bound_;  // Ring::generation of each member's ring the captured graph was built against
  int members_ = 1;
  const float** ring_slot_ = nullptr;  // population: the member's ring (Ring::data), read by the gather
  int launches_per_train_ = 0;
  ParamGroup actor_g_;
  LinearSlot a0_, a1_, a2_;
  float *metrics_dev_ = nullptr, *metrics_host_ = nullptr;
  long long *idx_dev_ = nullptr, *idx_host_ = nullptr;
  float *eps_dev_ = nullptr, *eps_host_ = nullptr;
  float* batch_ = nullptr;
  float *ah1_ = nullptr, *ah2_ = nullptr, *head_ = nullptr, *logp_ = nullptr;
  float *dhead_ = nullptr, *dah2_ = nullptr, *dah1_ = nullptr, *dsa_ = nullptr, *dlogp_ = nullptr;
  float *cat_next_ = nullptr, *cat_pi_ = nullptr, *bh1_ = nullptr, *bh2_ = nullptr, *bhead_ = nullptr;
  static constexpr int kActRows = 1024;  // observations per select_action launch
  float *act_in_host_ = nullptr, *act_out_host_ = nullptr, *act_in_dev_ = nullptr, *act_out_dev_ = nullptr;
};

}  // namespace rlrep

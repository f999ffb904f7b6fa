// Bandwidth-/latency-bound kernels of the update step (everything that is not a GEMM):
// replay gather, contrastive log-sum-exp / cross-entropy, reward head, N=1 critic heads, TD target and
// critic loss, tanh-Gaussian actor sample / log-prob (forward + backward), actor / temperature loss,
// the fused multi-tensor Adam + Polyak kernel and the per-update control-block "tick".
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "epilogue.cuh"

namespace rlrep {

constexpr int kMaxFeatureSteps = 16;
constexpr int kNumMetrics = 32;

struct AdamHyper {
  float step_size;  // lr / (1 - beta1^t)
  float bc2_sqrt;   // sqrt(1 - beta2^t)
};

// Per-agent control block in device memory.  Everything that changes from one train() call to the next and
// would otherwise be a kernel argument lives here, so the whole update can be replayed as one CUDA graph.
struct Control {
  int steps;              // agent.steps (reference: sac_agent.py:173)
  int polyak_critic;      // steps % target_update_period == 0 (sac_agent.py:100)
  long long t_feat, t_critic, t_actor, t_alpha;  // Adam step counters
  AdamHyper feat[kMaxFeatureSteps];
  AdamHyper critic, actor;
  double alpha_step_size, alpha_bc2_sqrt;
  double log_alpha, la_m, la_v;  // temperature is float64 in the reference (sac_agent.py:66)
  float alpha;                   // float(exp(log_alpha)) as seen by fp32 kernels
};

struct TickParams {
  int k_feat;              // feature Adam steps per train() (0 = agent has no feature optimiser)
  int period;              // target_update_period
  double lr_feat, lr_critic, lr_actor, lr_alpha;
  int critic_steps;        // 1 if the critic optimiser steps this agent (0 for diffsrsac, SURVEY A.6 #1)
};

void launch_tick(Control* c, const TickParams& p, cudaStream_t s);

// Replay gather: out[b, :] = ring[idx[b], :], rows are rec4 float4 wide (128-bit loads/stores).
void launch_gather(const float* ring, int rec4, const long long* idx, int B, float* out, cudaStream_t s);
// Scatter of freshly added rows into the ring at slots (start + i) % capacity.
void launch_ring_write(float* ring, int rec4, long long capacity, long long start, const float* rows, int n,
                       cudaStream_t s);

// Contrastive soft-label CE with identity labels (ctrlsac_agent.py:226-231):
//   loss_i = logsumexp_j(l_ij) - l_{i, diag_off + i};  in place  l_ij <- (softmax_j(l_i)_j - [j == diag_off+i]) * inv_batch
void launch_ce_rows(float* logits, int ld, int rows, int cols, int diag_off, float inv_batch, float* loss_rows,
                    cudaStream_t s);

// y[i] = sum_j X[i,j] w[j] + b[0]  (N = 1 linear heads; one CTA per row)
void launch_rowdot(const float* X, int ld, int rows, int D, const float* w, const float* b, float* y, cudaStream_t s);
// Two such heads over the same rows in one launch (the twin Q heads).
struct RowDotJob {
  const float* X;
  const float* w;
  const float* b;
  float* y;
  int ld, D;
};
void launch_rowdot_pair(const RowDotJob& a, const RowDotJob& b, int rows, cudaStream_t s);
// out[j] (+)= sum_i u[i] * X[i,j]   (u == nullptr: plain column sum).  Deterministic.
void launch_colreduce(const float* X, int ld, int rows, int cols, const float* u, float* out, int accumulate,
                      cudaStream_t s);
// out[j] = sum_i X[i, j] for very tall X (rows ~ 1e5..1e6): `chunks` CTAs per 32 columns, partial is [chunks, cols].
// C[m, n] = epilogue(sum_g ws[g * group_stride + m * ldw + n]): the finish of a K-grouped GEMM (GemmArgs::k_groups), groups
// added in order.
void launch_kgroup_finish(const float* ws, int groups, int M, int N, int ldw, size_t group_stride, float* C, int ldc,
                          const Epilogue& epi, cudaStream_t s);
// Second stage alone: out[j] = sum_c partial[c * cols + j] in a fixed order (for kernels that produce per-CTA column
// partials as a by-product of another pass).
void launch_colsum_finish(const float* partial, int chunks, int cols, float* out, cudaStream_t s);
void launch_colsum_tall(const float* X, int ld, long long rows, int cols, float* partial, int chunks, float* out,
                        cudaStream_t s);
// Several column reductions in one launch (all the bias gradients of a network's backward pass).
struct ColJob {
  const float* X;
  const float* u;  // optional row weights
  float* out;
  int ld, rows, cols;
};
constexpr int kMaxColJobs = 8;
void launch_colreduce_multi(const ColJob* jobs, int n_jobs, cudaStream_t s);
// out[i,j] = u[i] * w[j] * dact(aux[i,j])   (backward of an N = 1 head into its hidden layer)
void launch_outer_dact(const float* u, const float* w, int rows, int cols, const float* aux, int ld_aux, int dact,
                       float* out, int ld_out, cudaStream_t s);

// Reward head loss (ctrlsac_agent.py:233): r_loss = 0.5 * mean((pred - r)^2); dpred = (pred - r) * inv_batch.
// Also finishes the feature metrics: model_loss = sum(loss_rows) * inv_batch, total = model + r.
void launch_feature_loss_finalize(const float* loss_rows, int rows, const float* pred, const float* reward, int ld_r,
                                  float inv_batch, float* dpred, float* metrics /*[total, model, r]*/, cudaStream_t s);

// Actor head -> action / log-prob (agent/sac/actor.py:76-91 + 40-43).
//   head [B, ld_head >= 2A] = (mu | raw log-std); eps [B, A];  out action [B, lda] (tanh(u)), logp [B]
// obs != nullptr: also copy obs[b, 0:S] to action[b, -S:0], i.e. build the contiguous cat(obs, action) row.
void launch_actor_sample(const float* head, int ld_head, int B, int A, const float* eps, float* action, int lda,
                         float* logp, cudaStream_t s, const float* obs = nullptr, int ld_obs = 0, int S = 0);
// Two independent launch_actor_sample calls with the same shapes (ld_head, B, A, lda, S) as one launch.
struct ActorSampleJob {
  const float* head;
  const float* eps;
  float* action;
  float* logp;
  const float* obs;
  int ld_obs;
};
void launch_actor_sample_pair(const ActorSampleJob& j0, const ActorSampleJob& j1, int ld_head, int B, int A, int lda, int S,
                              cudaStream_t s);
// Backward of the above: dhead [B, ld_dhead >= 2A] from d_action [B, ldd] and the per-row d_logp scalar.
// launch_ce_rows + launch_rowdot (reward head theta) + launch_feature_loss_finalize as one launch; `counter` is a
// zero-initialised device word owned by the caller (arrival counter of the row CTAs, re-armed by the kernel).
void launch_contrastive_head(float* logits, int ld, int rows, int cols, int diag_off, float inv_batch, const float* z, int ldz,
                             int D, const float* theta_w, const float* theta_b, const float* reward, int ld_r,
                             float* loss_rows, float* pred, float* dpred, float* metrics, unsigned* counter,
                             cudaStream_t s);
// select_action / batched policy evaluation in one launch: out[r, :] = tanh(mu(in[r, :S]) (+ std * in[r, S:S+A] if explore));
// `in` / `out` may be mapped pinned host memory (see actor_act_kernel).
void launch_actor_act(const float* in, int rows, int S, int A, int H, const float* W0, int ld0, const float* b0,
                      const float* W1, int ld1, const float* b1, const float* W2, int ld2, const float* b2, int explore,
                      float* out, cudaStream_t s);
void launch_actor_sample_bwd(const float* head, int ld_head, int B, int A, const float* eps, const float* d_action,
                             int ldd, const float* dlogp_scalar, float* dhead, int ld_dhead, cudaStream_t s);

// TD target + twin-critic MSE (ctrlsac_agent.py:263-286; sac_agent.py:112-123):
//   y = r + (1 - d) * gamma * (min(nq1, nq2) - alpha * logp2)
//   dq1 = 2 (q1 - y) / B, dq2 likewise;  metrics[0..3] = q1_loss, q2_loss, mean(q1), mean(q2)
void launch_td_critic_loss(const float* reward, const float* done, int ld_rd, const float* nq1, const float* nq2,
                           const float* logp2, const float* q1, const float* q2, int B, float gamma, const Control* c,
                           float* dq1, float* dq2, float* metrics, cudaStream_t s, int norm_B = 0);

// Fused heads of the chained CTRL critic / actor steps (kernels.cu "fused SAC heads"): hid_t / hid are [B, 2H] hidden
// activations of the twin critic (target / live), w2 / w5 the two N = 1 heads; outputs as the kernels they replace.
struct CriticHeadArgs {
  const float *hid_t, *hid;
  int ldh, H, B;
  const float *w2t, *b2t, *w5t, *b5t, *w2, *b2, *w5, *b5;
  const float *reward, *done;
  int ld_rd;
  const float* logp2;
  float gamma;
  const Control* c;
  float *nq1, *nq2, *q1, *q2, *dq1, *dq2, *dhid;
  int ld_dh;
  float* metrics;     // q1_loss, q2_loss, mean(q1), mean(q2)
  unsigned* counter;  // zero before the first launch; re-armed by the kernel
};
void launch_critic_td_head(const CriticHeadArgs& a, cudaStream_t s);
struct ActorHeadArgs {
  const float* hid;
  int ldh, H, B;
  const float *w2, *b2, *w5, *b5;
  const float* logp;
  float target_entropy;
  int learn_alpha;
  Control* c;
  float *q1, *q2, *dq1, *dq2, *dhid;
  int ld_dh;
  float* dlogp_scalar;
  float* metrics;  // actor_loss, alpha_loss, alpha
  unsigned* counter;
};
void launch_actor_head(const ActorHeadArgs& a, cudaStream_t s);

// Actor / temperature losses (ctrlsac_agent.py:308-320; sac_agent.py:146-161), single block:
//   actor_loss = mean(alpha * logp - min(q1, q2));  dq1/dq2 = -[argmin] / B;  *dlogp_scalar = alpha / B
//   alpha_loss = mean(alpha * (-logp - target_entropy)); fp64 Adam step on log_alpha inside the control block.
//   metrics[0..2] = actor_loss, alpha_loss, alpha (after the step, like `info['alpha'] = self.alpha`).
void launch_actor_alpha_loss(const float* q1, const float* q2, const float* logp, int B, float target_entropy,
                             int learn_alpha, Control* c, float* dq1, float* dq2, float* dlogp_scalar, float* metrics,
                             cudaStream_t s);

// Batch-sharded pieces (agent_ctrlsac_dp.cu).  norm_B = GLOBAL batch: every mean is a partial sum / norm_B that the
// caller all-reduces.  partial = {share of actor_loss, share of mean(-logp - target_entropy)}; alpha_step consumes the
// all-reduced pair: metrics = {actor_loss, alpha_loss, alpha} and the float64 Adam step on log_alpha.
void launch_actor_loss_partial(const float* q1, const float* q2, const float* logp, int B, int norm_B,
                               float target_entropy, const Control* c, float* dq1, float* dq2, float* dlogp_scalar,
                               float* partial, cudaStream_t s);
void launch_alpha_step(const float* reduced, int learn_alpha, Control* c, float* metrics, cudaStream_t s);
// x *= dact(aux), elementwise over n floats
void launch_mul_dact(float* x, const float* aux, size_t n, int dact, cudaStream_t s);

// ---- LV-Rep / VL-SAC (agent/vlsac/vlsac_agent.py, networks/vae.py) ----------------------------------------------
// out[b, dst + j] = in[b, src + j] for up to three column segments (builds cat(s, a, s') from a replay record).
struct ColSegment {
  int src, dst, len;
};
void launch_pack_columns(const float* in, int ld_in, float* out, int ld_out, int rows, const ColSegment* segs,
                         int n_segs, cudaStream_t s);
// Encoder.sample (vae.py:50-58): z = mean + eps * exp(clamp(raw_log_std, -20, 2)); head = [mean | raw_log_std].
void launch_vae_sample(const float* head, int ld_head, int B, int D, const float* eps, float* z, cudaStream_t s);
// Reconstruction losses (vlsac_agent.py:137-140): xr = [s'_hat (S) | r_hat]; dxr = d(0.5 mse_s + 0.5 mse_r);
// partial[block] = {sum (s'_hat - s')^2, sum (r_hat - r)^2}.  Padding columns of dxr [S+1, ld) are zeroed.
void launch_vae_recon_loss(const float* xr, int ld_xr, const float* next_state, const float* reward, int ld_rec, int B,
                           int S, float* dxr, float* partial, int n_blocks, cudaStream_t s);
// KL(q || p) of two diagonal Gaussians with clamped log-stds (vlsac_agent.py:143-150) and the backward of the whole
// ELBO into the encoder and prior heads: d_enc = [dz + dKL/dmean1 | (dz eps std1 + dKL/dls1) * clamp'],
// d_prior = [dKL/dmean2 | dKL/dls2 * clamp'];  partial[block] = sum KL.
void launch_vae_kl_bwd(const float* enc_head, const float* prior_head, int ld_head, int B, int D, const float* eps,
                       const float* dz, float* d_enc, float* d_prior, float* partial, int n_blocks, cudaStream_t s);
// metrics = {vae_loss, ml_loss, kl_loss, s_loss, r_loss}
void launch_vae_finalize(const float* recon_partial, int n_recon, const float* kl_partial, int n_kl, int B, int S, int D,
                         float* metrics, cudaStream_t s);
// Critic input (vlsac_agent.py:44-50): x[b*NN + j, :] = mean[b] + exp(clamp(raw_ls[b])) * noise[j].
void launch_noise_expand(const float* head, int ld_head, int B, int D, const float* noise, int NN, float* x,
                         cudaStream_t s);
// Its backward: d_head = [sum_j dx | (sum_j dx * noise_j) * std * clamp'].
void launch_noise_expand_bwd(const float* dx, const float* head, int ld_head, int B, int D, const float* noise, int NN,
                             float* d_head, cudaStream_t s);
// out[b, c] = mean_j hid[b*NN + j, c]   (vlsac_agent.py:53, :58)
void launch_group_mean(const float* hid, int ld, int B, int NN, int C, float* out, cudaStream_t s);
// dhid[b*NN + j, c] = dmean[b, c] / NN * elu'(hid[b*NN + j, c]);  colsum_partial[b, c] = sum_j dhid[b*NN + j, c]
void launch_group_mean_bwd(const float* dmean, const float* hid, int ld, int B, int NN, int C, float* dhid,
                           float* colsum_partial, cudaStream_t s);

// ---- SPEDER-SAC (agent/spedersac/spedersac_agent.py:181-219) ------------------------------------------------------
// Features of two batches are stacked: rows [0, B) belong to the update batch, rows [B, 2B) to the second, independent
// batch (phi~, mu~).  The spectral loss is
//   model = mean_i(-2 <phi_i, mu_i>) + mean_ij((phi~ mu~^T)(phi~ mu~^T)^T)
// and its second term equals ||mu~ u||^2 / B^2 with u = colsum(phi~) (sum_ij sum_k pa_ik pa_jk = sum_k (sum_i pa_ik)^2),
// so no B x B matrix is ever formed.
//   diag[i] = <phi_i, mu_i>, rpred[i] = <phi_i, theta_w> + theta_b, c[i] = <mu~_i, u>      (one warp per row)
void launch_speder_rows(const float* zphi, const float* zmu, int D, int B, const float* theta_w, const float* theta_b,
                        const float* u, float* diag, float* rpred, float* c, cudaStream_t s);
// drp = (rpred - r) / B;  metrics = {total_loss, model_loss, r_loss}
void launch_speder_finalize(const float* diag, const float* c, const float* rpred, const float* reward, int ld_r, int B,
                            float* drp, float* metrics, cudaStream_t s);
// dzphi[i] = -2/B mu_i + drp_i theta_w;  dzmu[i] = -2/B phi_i;  dzphi[B+i] = 2/B^2 w (w = mu~^T c);  dzmu[B+k] = 2/B^2 c_k u
void launch_speder_grad(const float* zphi, const float* zmu, int D, int B, const float* drp, const float* theta_w,
                        const float* c, const float* u, const float* w, float* dzphi, float* dzmu, cudaStream_t s);

// ---- Diff-SR-SAC (agent/diffsrsac/diffsrsac_agent.py:271-318) -----------------------------------------------------
// DDPM perturbation of s' at the host-drawn noise levels: ab = alphabars[level[b]];
//   xin[b] = [ sqrt(ab) s' + sqrt(1 - ab) noise | ab | 0 ... ]  (row pitch ld_x),  target = -(s~' - sqrt(ab) s'),
//   coef[b] = (1 - ab) * sigma.   `noise` is already scaled by sigma (torch.normal(0, sigma) drawn by the host).
void launch_diffsr_perturb(const float* next_state, int ld_rec, const float* noise, const long long* level,
                           const float* alphabars, int n_levels, float sigma, int B, int S, float* xin, int ld_x,
                           float* target, float* coef, cudaStream_t s);
// score[b, s] = sum_d phi[b, d] flat[b, d*S + s] (the reference's bmm);  diff = target - coef * score;
// loss_rows[b] = sum_s diff^2;  dscore = d(sum_b loss_rows / B) / dscore = -coef * 2/B * diff.
void launch_diffsr_score(const float* phi, const float* flat, int D, int S, const float* target, const float* coef, int B,
                         float* dscore, float* loss_rows, cudaStream_t s);
// dflat[b, d*S + s] = phi[b, d] dscore[b, s];  dphi[b, d] = sum_s dscore[b, s] flat[b, d*S + s]
void launch_diffsr_score_bwd(const float* phi, const float* flat, int D, int S, int B, const float* dscore, float* dflat,
                             float* dphi, cudaStream_t s);
// out[0] = scale * sum(x[0:n])   (single block, deterministic)
void launch_sum_scaled(const float* x, int n, float scale, float* out, cudaStream_t s);

// ---- DrQ-v2 pixel update (agent/diffsrdrq/network_arch/drqv2.py:60-135, drqv2.py:112-148) ----------------------------
// y[:, 0:n] = tanh(LayerNorm_n(x) * gamma + beta) (eps 1e-5); xhat / rstd are kept for the backward pass when non-null.
void launch_ln_tanh_fwd(const float* x, int ld_x, int B, int n, const float* gamma, const float* beta, float* y, int ld_y,
                        float* xhat, int ld_h, float* rstd, cudaStream_t s);
// Backward of the above: dx [B, ld_dx] (columns >= n zeroed), g_beta = dz and g_gamma = dz * xhat (their column sums are
// the LayerNorm parameter gradients).
void launch_ln_tanh_bwd(const float* dy, int ld_dy, const float* y, int ld_y, const float* xhat, int ld_h, const float* rstd,
                        int B, int n, const float* gamma, float* dx, int ld_dx, float* g_beta, float* g_gamma, int ld_g,
                        cudaStream_t s);
// Actor head + TruncatedNormal.sample(clip): mu = tanh(raw); action = clamp(mu + clamp(eps * std, +-clip), +-(1 - 1e-6)).
void launch_trunc_normal_sample(const float* raw, int ld_raw, int B, int A, const float* eps, float std, float clip,
                                float* mu, float* action, int ld_a, cudaStream_t s);
// Straight-through clamp: d raw = d action * (1 - mu^2); columns [A, ld_out) zeroed.
void launch_trunc_normal_bwd(const float* d_action, int ld_da, const float* mu, int B, int A, float* draw, int ld_out,
                             cudaStream_t s);
// y = r + discount * min(tq1, tq2); loss = mse over the stacked twin Q (mean over 2B); dq = 2 (q - y) / (2B);
// metrics = {critic_loss, mean(q_pred), mean(q_target), mean(reward)}
void launch_drq_critic_loss(const float* reward, const float* discount, const float* tq1, const float* tq2, const float* q1,
                            const float* q2, int B, float* dq1, float* dq2, float* metrics, cudaStream_t s);
// actor_loss = -mean(min(q1, q2)); dq = -1/B on the argmin; metrics = {actor_loss}
void launch_drq_actor_loss(const float* q1, const float* q2, int B, float* dq1, float* dq2, float* metrics, cudaStream_t s);

// ---- muLV-Rep DrQ-v2 pixel update (agent/mulvdrq/drqv2.py:313-461, vae.py:13-124; kernels_mulv.cu) ----------------------
// Gaussian heads are two [B, ld] matrices: mean (after tanh(LayerNorm)) and raw log-std (after LayerNorm; consumers clamp
// to [-20, 2]); padding columns [D, ld) are zero.
// y[:, 0:n] = act(LayerNorm_n(x) * gamma + beta), act = tanh or identity; columns [n, zero_to) of y zeroed.
void launch_ln_act_fwd(const float* x, int ld_x, int B, int n, const float* gamma, const float* beta, bool use_tanh,
                       float* y, int ld_y, int zero_to, float* xhat, int ld_h, float* rstd, cudaStream_t s);
// Backward: dx (columns [n, zero_to) zeroed); column sums of g_beta / g_gamma are the LayerNorm parameter gradients.
void launch_ln_act_bwd(const float* dy, int ld_dy, const float* y, int ld_y, const float* xhat, int ld_h, const float* rstd,
                       int B, int n, const float* gamma, bool use_tanh, float* dx, int ld_dx, int zero_to, float* g_beta,
                       float* g_gamma, int ld_g, cudaStream_t s);
// z[b, 0:D] = m + eps * exp(clamp(raw)) (Normal.rsample, vae.py:50-58); eps [B, D]; z [B, ld_z], padding zeroed.
void launch_gauss_sample(const float* m, const float* raw, int ld, int B, int D, const float* eps, float* z, int ld_z,
                         cudaStream_t s);
// w * KL(head 1 || head 2).mean() and the backward of the sample (dz) into head 1; head 2 also receives the critic's
// gradient (dcm, dcraw; nullable).  partial[block] = unweighted sum of KL elements.
void launch_gauss_kl_bwd(const float* m1, const float* raw1, const float* m2, const float* raw2, int ld, int B, int D,
                         const float* eps, const float* dz, float w, const float* dcm, const float* dcraw, float* dm1,
                         float* draw1, float* dm2, float* draw2, float* partial, int n_blocks, cudaStream_t s);
// Critic input (drqv2.py:177-183): x[b*NN + j] = m[b] + exp(clamp(raw[b])) * noise[j] * c_noise; x [B*NN, ld_x].
void launch_gauss_noise_expand(const float* m, const float* raw, int ld, int B, int D, const float* noise, int NN,
                               float c_noise, float* x, int ld_x, cudaStream_t s);
void launch_gauss_noise_expand_bwd(const float* dx, int ld_x, const float* raw, int ld, int B, int D, const float* noise,
                                   int NN, float c_noise, float* dm, float* draw, cudaStream_t s);
// launch_group_mean_bwd with the activation derivative as a parameter (the pixel critic uses ReLU).
void launch_group_mean_bwd_dact(const float* dmean, const float* hid, int ld, int B, int NN, int C, int dact, float* dhid,
                                float* colsum_partial, cudaStream_t s);
// y = r + discount * min(tq1, tq2); loss = smooth_l1(q1, y) + smooth_l1(q2, y); dq = clamp(q - y, +-1) / B;
// metrics = {critic_loss, mean(q1), mean(q2), mean(y)}
void launch_huber_critic_loss(const float* reward, const float* discount, const float* tq1, const float* tq2,
                              const float* q1, const float* q2, int B, float* dq1, float* dq2, float* metrics,
                              cudaStream_t s);
// out[0] = mse(r_hat, r); dr = w * 2 (r_hat - r) / B
void launch_reward_mse(const float* r_hat, const float* reward, int B, float w, float* dr, float* out, cudaStream_t s);

// ---- DRAFT: latent Diff-SR DrQ-v2 pixel update (agent/diffsrdrq/latent_diff_sr.py; kernels_ldiff.cu) -------------------
// LayerNorm + {0 none, 1 tanh, 2 swish}; same contract as launch_ln_act_fwd / _bwd (the backward also needs beta for swish).
void launch_ln_act2_fwd(const float* x, int ld_x, int B, int n, const float* gamma, const float* beta, int act, float* y,
                        int ld_y, int zero_to, float* xhat, int ld_h, float* rstd, cudaStream_t s);
void launch_ln_act2_bwd(const float* dy, int ld_dy, const float* y, int ld_y, const float* xhat, int ld_h, const float* rstd,
                        int B, int n, const float* gamma, const float* beta, int act, float* dx, int ld_dx, int zero_to,
                        float* g_beta, float* g_gamma, int ld_g, cudaStream_t s);
void launch_mish_fwd(const float* x, size_t n, float* y, cudaStream_t s);
void launch_mish_bwd(const float* dy, const float* x, size_t n, float* dx, cudaStream_t s);
// out = (accumulate ? out : 0) + x * (mask ? mask * inv_keep : 1): dropout with a host-drawn Bernoulli mask, and its backward
void launch_mask_scale(const float* x, const float* mask, float inv_keep, size_t n, int accumulate, float* out, cudaStream_t s);
// Diagonal-Gaussian posterior (vae_1d.py:24-48): h [N, 2L] = (mean | raw logvar, clamped to [-30, 20]); z = mean + std eps;
// partial[block] = sum of 0.5 (mean^2 + var - 1 - logvar)
void launch_posterior_fwd(const float* h, int N, int L, const float* eps, float* mean_out, float* z, float* partial,
                          int n_blocks, cudaStream_t s);
// dh from dz (gradient w.r.t. the sample), an optional gradient w.r.t. the mean of the first n_extra elements, and the
// KL term with weight w_kl (= kl weight / N rows)
void launch_posterior_bwd(const float* h, int N, int L, const float* eps, const float* dz, const float* dmean_extra,
                          int n_extra, float w_kl, float* dh, cudaStream_t s);
// zeta input [sqrt(ab) x + sqrt(1 - ab) noise | t_emb | 0] with row pitch ld; target = -noise; coef = sqrt(1 - ab) / feat
void launch_ldiff_perturb(const float* x, const float* noise, const float* ab, const float* temb, int B, int L, int T,
                          float inv_feat, float* zin, int ld, float* target, float* coef, cudaStream_t s);
void launch_ldiff_perturb_bwd(const float* dzin, int ld, const float* ab, int B, int L, float* dx, cudaStream_t s);
void launch_add_inplace(float* y, const float* x, size_t n, cudaStream_t s);
void launch_scale_inplace(float* p, size_t n, float scale, cudaStream_t s);  // n % 4 == 0

// Fused multi-tensor Adam (+ optional Polyak of a prefix of the arena into its target copy).
// One launch updates a whole optimiser group laid out as flat arrays p / g / m / v of n floats (n % 4 == 0).
//   torch.optim.Adam defaults: beta = (0.9, 0.999), eps = 1e-8, no weight decay / amsgrad.
//   target[0:n_polyak] = tau * p_new + (1 - tau) * target   when *polyak_flag != 0 (or flag == nullptr).
void launch_adam_polyak(float* p, const float* g, float* m, float* v, size_t n, const AdamHyper* hyper, float* target,
                        size_t n_polyak, float tau, const int* polyak_flag, cudaStream_t s);
// Polyak only (critic_target of agents whose critic optimiser never steps).
void launch_polyak(const float* p, float* target, size_t n, float tau, const int* polyak_flag, cudaStream_t s);

}  // namespace rlrep

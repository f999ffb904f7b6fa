/*
 * rlrep_b200 -- C ABI of the B200-native representation-learning update step.
 *
 * The reference (haotiansun14/rl-rep) has no FFI: its boundary is the duck-typed Python surface
 * `Agent(**kwargs)`, `agent.train(buffer, batch_size) -> dict`, `agent.select_action(state)`,
 * `ReplayBuffer.add/sample` (reference: main.py:71-144, utils/buffer.py:13-48, agent/sac/sac_agent.py:19-188).
 * This header is what a binding for that surface calls; `rlrep_b200/` (Python) is such a binding and
 * INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns int: 0 = ok, non-zero = error; rlrep_last_error() gives the message
 *     (thread-local);
 *   - `stream` arguments are a cudaStream_t passed as void* (NULL = the legacy default stream);
 *   - pointers named *_dev are device pointers, *_host are host pointers; the caller owns host buffers,
 *     the library owns every device allocation it makes and frees it in the matching *_destroy;
 *   - one handle = one agent (or one ring) = one stream; handles are independent (thread-compatible,
 *     not thread-safe per handle), so a population runs N handles per GPU;
 *   - there is no CPU fallback anywhere: without a CUDA device every compute call returns an error.
 */
#ifndef RLREP_B200_H_
#define RLREP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define RLREP_EXPORT __attribute__((visibility("default")))
#else
#define RLREP_EXPORT
#endif

#define RLREP_ABI_VERSION 3

RLREP_EXPORT int rlrep_abi_version(void);
RLREP_EXPORT const char* rlrep_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * Kernel-level entry points (used by the parity tests; the agent handles below call the same code).
 * ---------------------------------------------------------------------------------------------- */

/* Activation / activation-derivative selectors of the fused GEMM epilogue (see csrc/epilogue.cuh). */
enum { RLREP_ACT_NONE = 0, RLREP_ACT_ELU = 1, RLREP_ACT_RELU = 2, RLREP_ACT_TANH = 3, RLREP_ACT_SIN = 4 };
enum {
  RLREP_DACT_NONE = 0,
  RLREP_DACT_ELU_OUT = 1,
  RLREP_DACT_RELU_OUT = 2,
  RLREP_DACT_TANH_OUT = 3,
  RLREP_DACT_COS_PRE = 4
};

typedef struct rlrep_epilogue {
  const float* bias_dev;  /* [N] or NULL                                   */
  const float* r1_u_dev;  /* rank-1 term u[m] * v[n], both NULL to disable */
  const float* r1_v_dev;
  const float* aux_dev;   /* [M, ld_aux] operand of the activation derivative */
  float* pre_out_dev;     /* optional [M, ld_pre]: pre-activation values      */
  int ld_aux;
  int ld_pre;
  int act;
  int dact;
  int accumulate;         /* C += result */
  float scale;            /* accumulator scale, normally 1 */
} rlrep_epilogue;

/*
 * C[M,N] = epilogue(sum_k A(m,k) B(n,k)).  a_mn / b_mn = 0: operand is K-major (A[m*lda+k]); 1: MN-major
 * (A[k*lda+m]).  This single contraction covers nn.Linear forward (reference utils/util.py:85-96,
 * agent/ctrlsac/ctrlsac_agent.py:72-77), its dgrad and its wgrad, and the contrastive logits
 * phi(s,a) . mu(s')^T (ctrlsac_agent.py:229).
 *   path = 0: tcgen05 TF32 tensor-core kernel (TMA operands: 16-byte aligned bases, ld % 4 == 0)
 *   path = 1: CUDA-core exact-FP32 kernel (any alignment; optional second K segment A2 for cat() inputs)
 * bn / split_k = 0 lets the library choose; ws_dev (split-K partials, ws_floats floats) may be NULL.
 */
RLREP_EXPORT int rlrep_gemm(void* stream, int path, int M, int N, int K, const float* A_dev, int lda, int a_mn,
                            const float* A2_dev, int lda2, int K1, const float* B_dev, int ldb, int b_mn,
                            float* C_dev, int ldc, const rlrep_epilogue* epi, int bn, int split_k, float* ws_dev,
                            size_t ws_floats);

/* Tuning aid: plans the GEMM once (tensor maps encoded once, like the agent handles do), launches it `iters`
 * times back to back and reports the CUDA-event average in milliseconds plus the tile/split actually used. */
RLREP_EXPORT int rlrep_gemm_bench(void* stream, int path, int M, int N, int K, const float* A_dev, int lda, int a_mn,
                                  const float* B_dev, int ldb, int b_mn, float* C_dev, int ldc,
                                  const rlrep_epilogue* epi, int bn, int split_k, float* ws_dev, size_t ws_floats,
                                  int iters, float* ms_out, int* bn_out, int* split_out);

/* GEMM chain: a DAG of dependent GEMMs (the layers of a few small MLPs, forward or backward) executed by ONE persistent
 * tcgen05 kernel -- one CTA per SM walks a static item list, a dependent tile starts when the tiles it reads are complete
 * (csrc/gemm_chain.cuh).  The agent handles use this internally for every group of GEMMs between two elementwise kernels
 * when the batch is small; these three calls expose it for tests and tuning.  Usage (per thread): begin, add every GEMM in
 * program order (dependencies are inferred from the operands' address ranges), run.  `bn` / `split_k` = 0 lets the planner
 * choose per GEMM.  run launches the chain `iters` times (>= 1) and reports the CUDA-event average in milliseconds. */
RLREP_EXPORT int rlrep_gemm_chain_begin(void);
RLREP_EXPORT int rlrep_gemm_chain_add(int M, int N, int K, const float* A_dev, int lda, int a_mn, const float* B_dev,
                                      int ldb, int b_mn, float* C_dev, int ldc, const rlrep_epilogue* epi);
RLREP_EXPORT int rlrep_gemm_chain_run(void* stream, int bn, int split_k, int iters, float* ms_out, int* levels_out);
/* Debug aid: device buffer of 148 CTAs x 16 items x 10 slots uint64 %globaltimer stamps written by every chain launch
 * (NULL = off).  Events per item: 0 picked up, 1 dependencies satisfied, 2 TMA issued, 3 first operands landed,
 * 4 accumulator committed, 5 epilogue start, 6 split-K arrival, 7 tile published. */
RLREP_EXPORT int rlrep_gemm_chain_set_debug(unsigned long long* dev);

/* Debug aid (library built with -DRLREP_GEMM_TRACE): %globaltimer stamps (ns) taken by CTA (0,0,0) of the most
 * recent tcgen05 GEMM at: 0 entry, 1 setup done, 2 first operands landed, 3 last MMA issued, 4 accumulator complete,
 * 5 staged to shared, 6 cluster/CTA sync passed, 7 stores issued, 8 exit. */
RLREP_EXPORT int rlrep_gemm_trace(unsigned long long* out16_host);
/* Debug aid: device buffer of 80 uint64 into which CTA 0 of the persistent GEMM variant stamps %globaltimer for its first
 * 16 tiles (role * 16 + tile; roles: TMA issued, operands landed, accumulator committed, epilogue start, epilogue end). */
RLREP_EXPORT int rlrep_gemm_set_debug_buffer(unsigned long long* dev80);

/* ------------------------------------------------------------------------------------------------
 * Replay ring -- replaces utils/buffer.py:13-48 (ReplayBuffer.__init__ / add / sample).
 * Device-resident fp32 ring of packed records [s | a | r | d | pad | s' | pad]; see rlrep_ring_layout.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_ring rlrep_ring;

RLREP_EXPORT int rlrep_ring_create(int state_dim, int action_dim, long long capacity, rlrep_ring** out);
RLREP_EXPORT int rlrep_ring_destroy(rlrep_ring* ring);
/* Record layout in floats: total width and the offsets of action / reward / done / next_state (state is at 0). */
RLREP_EXPORT int rlrep_ring_layout(const rlrep_ring* ring, int* record_floats, int* off_action, int* off_reward,
                                   int* off_done, int* off_next_state);
RLREP_EXPORT int rlrep_ring_state(const rlrep_ring* ring, long long* size, long long* ptr, long long* capacity);
/* buffer.py:28-36 `add`, batched: n packed records [n, record_floats] are written at ptr, ptr+1, ... (mod capacity). */
RLREP_EXPORT int rlrep_ring_add_packed(rlrep_ring* ring, const float* rows_host, int n, void* stream);
/* Bulk fill from the reference's five column arrays (float64 if is_f64 else float32), n rows from slot 0. */
RLREP_EXPORT int rlrep_ring_load(rlrep_ring* ring, const void* state_host, const void* action_host,
                                 const void* next_state_host, const void* reward_host, const void* done_host,
                                 long long n, int is_f64, void* stream);
/* buffer.py:39-48 `sample` minus the index draw: out_dev[b, :] = record idx_host[b]; out_dev is [B, record_floats]. */
RLREP_EXPORT int rlrep_ring_gather(rlrep_ring* ring, const int64_t* idx_host, int B, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pixel replay ring -- replaces agent/diffsrdrq/helper_functions/efficient_buffer.py:35-136 (EfficientReplayBuffer:
 * storage + `gather_nstep_indices`; the mulvdrq loader's sample tuple, agent/mulvdrq/replay_buffer.py:149-168, has the
 * same six fields).  One uint8 frame per environment step lives in HBM; a batch is assembled by one kernel of 128-bit
 * copies into device tensors that rlrep_drq_update / rlrep_mulv_update / rlrep_ldiff_update accept in place of host
 * arrays.  Which slots may be sampled is host bookkeeping and stays with the caller (rlrep_b200.PixelReplayBuffer keeps it
 * exactly as the reference does).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_pixring rlrep_pixring;
RLREP_EXPORT int rlrep_pixring_create(long long capacity, int frame_bytes, int action_dim, int frame_stack, int nstep,
                                      rlrep_pixring** out);
RLREP_EXPORT int rlrep_pixring_destroy(rlrep_pixring* ring);
/* efficient_buffer.py:66-105 `add_data_point`, storage part: frame_host [frame_bytes] goes to slots [slot, slot + copies)
 * mod capacity (copies = frame_stack for the first observation of a trajectory, else 1); when has_step,
 * (action_host [action_dim], reward, discount) go to `slot`.  Writes are staged and shipped 64 at a time. */
RLREP_EXPORT int rlrep_pixring_write(rlrep_pixring* ring, long long slot, int copies, const unsigned char* frame_host,
                                     const float* action_host, float reward, float discount, int has_step);
RLREP_EXPORT int rlrep_pixring_flush(rlrep_pixring* ring);
/* efficient_buffer.py:108-136 `gather_nstep_indices` for n sampled slots idx_host: obs / nobs / sobs_dev
 * [n, frame_stack * frame_bytes] uint8 (sobs_dev may be NULL), act_dev [n, action_dim], rew_dev / dis_dev [n];
 * discount_vec_host [nstep] = discount^k as float32, next_dis = discount^nstep.  Outputs are complete on return. */
RLREP_EXPORT int rlrep_pixring_gather(rlrep_pixring* ring, const int64_t* idx_host, int n, const float* discount_vec_host,
                                      float next_dis, unsigned char* obs_dev, float* act_dev, float* rew_dev, float* dis_dev,
                                      unsigned char* nobs_dev, unsigned char* sobs_dev);

/* ------------------------------------------------------------------------------------------------
 * Agent handles -- replace `Agent(**kwargs)`, `agent.train(buffer, batch_size)`, `agent.select_action(state)`
 * (sac_agent.py:19-31,89-96,169-188; ctrlsac_agent.py:127-143,327-362; main.py:71-104,130,144).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_agent rlrep_agent;

enum { RLREP_ALG_SAC = 0, RLREP_ALG_CTRLSAC = 1, RLREP_ALG_VLSAC = 2, RLREP_ALG_SPEDERSAC = 3, RLREP_ALG_DIFFSRSAC = 4 };
enum { RLREP_PRECISION_TF32 = 0, RLREP_PRECISION_FP32 = 1 };

typedef struct rlrep_agent_config {
  int alg;
  int state_dim, action_dim, batch_size;
  int hidden_dim, feature_dim, actor_hidden_dim;
  int feature_steps;           /* extra_feature_steps + 1; 0 for sac */
  double lr_critic, lr_feature, lr_actor, lr_alpha;
  float discount, tau, feature_tau;
  double alpha;                /* initial temperature; log_alpha is kept in float64 like the reference */
  int target_update_period, auto_entropy_tuning, use_feature_target;
  int precision;               /* RLREP_PRECISION_*: tensor-core TF32 (default) or CUDA-core exact fp32 GEMMs */
  int use_cuda_graph;          /* replay train() as one CUDA graph after the first two calls */
  int phi_hidden_dim, phi_hidden_depth, mu_hidden_dim, mu_hidden_depth;     /* spedersac / diffsrsac */
  int nabla_mu_hidden_dim, nabla_mu_hidden_depth, num_noise, num_noises;
  float sigma_scale_factor;
} rlrep_agent_config;

RLREP_EXPORT int rlrep_agent_create(const rlrep_agent_config* cfg, void* stream, rlrep_agent** out);

/* Batch-sharded CTRL-SAC over N GPUs, one process per GPU (BASELINE config 4; the reference has no distributed code --
 * this is the data-parallel form of ctrlsac_agent.py:213-362 on a global batch of N * cfg->batch_size rows: all-gather of
 * mu(s'), reduce-scatter of its gradient, all-reduce of parameter gradients and loss sums over NCCL).  Rank 0 obtains a
 * 128-byte id, ships it to the other ranks out of band (torch.distributed, MPI, a file), every rank creates its
 * communicator and then its handle.  rlrep_agent_train takes the rank's OWN rows: idx [K * batch_size] and eps
 * [2 * batch_size * action_dim] are the rank's slices of the global draws; metrics are global and identical on all ranks. */
typedef struct rlrep_comm rlrep_comm;
RLREP_EXPORT int rlrep_comm_unique_id(unsigned char* out128);
RLREP_EXPORT int rlrep_comm_create(const unsigned char* id128, int rank, int world, rlrep_comm** out);
RLREP_EXPORT int rlrep_comm_destroy(rlrep_comm* comm);
RLREP_EXPORT int rlrep_comm_info(rlrep_comm* comm, int* rank, int* world, int* nccl_version, long long* collectives);
RLREP_EXPORT int rlrep_agent_create_sharded(const rlrep_agent_config* cfg, rlrep_comm* comm, void* stream,
                                            rlrep_agent** out);
RLREP_EXPORT int rlrep_agent_destroy(rlrep_agent* agent);

/* Parameters and Polyak targets under the reference's state_dict names ("phi.l1.weight", "critic_target.l2.bias",
 * ...), as device pointers (so PyTorch can view them, e.g. for NCCL) and through host copies. */
RLREP_EXPORT int rlrep_agent_num_tensors(rlrep_agent* agent, int* n);
RLREP_EXPORT int rlrep_agent_tensor_info(rlrep_agent* agent, int i, const char** name, float** ptr_dev, int* rows,
                                         int* cols);
RLREP_EXPORT int rlrep_agent_tensor_read(rlrep_agent* agent, int i, float* out_host);
RLREP_EXPORT int rlrep_agent_tensor_write(rlrep_agent* agent, int i, const float* in_host);
/* target <- parameter copies for every Polyak target (use after writing parameters). */
RLREP_EXPORT int rlrep_agent_sync_targets(rlrep_agent* agent);
RLREP_EXPORT int rlrep_agent_get_log_alpha(rlrep_agent* agent, double* log_alpha);
RLREP_EXPORT int rlrep_agent_set_log_alpha(rlrep_agent* agent, double log_alpha);
/* Optimiser / schedule state that is not a tensor: the agent's `steps` counter (gates the critic Polyak, sac_agent.py:100),
 * the Adam step counters of the four optimisers (bias correction) and the float64 temperature with its Adam moments.
 * Together with the "optim.m/<name>" / "optim.v/<name>" tensors it lets a checkpoint resume exactly where it stopped. */
typedef struct rlrep_optim_state {
  int steps;
  long long t_feature, t_critic, t_actor, t_alpha;
  double log_alpha, log_alpha_m, log_alpha_v;
} rlrep_optim_state;
RLREP_EXPORT int rlrep_agent_get_optim_state(rlrep_agent* agent, rlrep_optim_state* out);
RLREP_EXPORT int rlrep_agent_set_optim_state(rlrep_agent* agent, const rlrep_optim_state* in);
RLREP_EXPORT int rlrep_agent_get_steps(rlrep_agent* agent, int* steps);

/* One `agent.train(buffer, batch_size)`.  The caller draws the randomness exactly like the reference does
 * (np.random.randint for replay indices, torch.randn on the CPU generator for every epsilon; SURVEY.md A.5) and
 * passes it in; rlrep_agent_train_counts tells how many of each one call consumes.  metrics_host receives the
 * entries named by rlrep_agent_metric_name.  `eps_host` may also be a DEVICE pointer on the agent's GPU (noise drawn
 * there by the caller, e.g. torch.randn(device="cuda") like the reference run with device = cuda; the producing stream
 * must be complete): it is then copied device to device and never crosses PCIe. */
RLREP_EXPORT int rlrep_agent_train_counts(rlrep_agent* agent, int* n_idx, int* n_eps, int* n_metrics);
RLREP_EXPORT const char* rlrep_agent_metric_name(rlrep_agent* agent, int i);
RLREP_EXPORT int rlrep_agent_train(rlrep_agent* agent, rlrep_ring* ring, const int64_t* idx_host, int n_idx,
                                   const float* eps_host, int n_eps, float* metrics_host, int n_metrics);
/* select_action: eps_host == NULL -> tanh(mu) (explore=False), else tanh(mu + std * eps) with eps[action_dim]. */
RLREP_EXPORT int rlrep_agent_act(rlrep_agent* agent, const float* state_host, const float* eps_host,
                                 float* action_host);
/* Benchmark aids.  train_resident: n_steps updates back to back with all inputs already in HBM (indices / noise of
 * every step uploaded before the timed region), timed with CUDA events on the agent's stream; idx_host is
 * [n_steps * n_idx], eps_host [n_steps * n_eps].  profile_train: one eager train() with an event behind every kernel
 * launch; names[i] / ms[i] describe launch i, bytes[i] / flops[i] (either may be NULL) its ALGORITHMIC work -- operands
 * read once, results written once, 2 flop per MAC; 0 for latency-bound bookkeeping kernels (n_entries may exceed
 * max_entries; only max_entries are written). */
RLREP_EXPORT int rlrep_agent_train_resident(rlrep_agent* agent, rlrep_ring* ring, const int64_t* idx_host,
                                            const float* eps_host, int n_steps, float* total_ms);
RLREP_EXPORT int rlrep_agent_profile_train(rlrep_agent* agent, rlrep_ring* ring, const int64_t* idx_host,
                                           const float* eps_host, int max_entries, const char** names, float* ms,
                                           double* bytes, double* flops, int* n_entries);
/* ------------------------------------------------------------------------------------------------
 * DrQ-v2 pixel encoder -- replaces `Encoder.forward` / its autograd backward and `RandomShiftsAug`
 * (agent/diffsrdrq/network_arch/drqv2.py:21-57,138-167; agent/mulvdrq/drqv2.py:19-96).  First building block of the
 * pixel agents; the agents themselves are not assembled yet (DESIGN.md section 0).
 * Layer l = 0..3 is `convnet.{2l}`; weights are exchanged in the reference's layout [32, C_in, 3, 3] / [32].
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_conv_encoder rlrep_conv_encoder;
RLREP_EXPORT int rlrep_conv_encoder_create(int batch, int in_channels, int height, int precision, void* stream,
                                           rlrep_conv_encoder** out);
RLREP_EXPORT int rlrep_conv_encoder_destroy(rlrep_conv_encoder* enc);
/* what: 0 = weight, 1 = bias, 2 = weight gradient, 3 = bias gradient (host buffers, reference layout) */
RLREP_EXPORT int rlrep_conv_encoder_read(rlrep_conv_encoder* enc, int layer, int what, float* out_host);
RLREP_EXPORT int rlrep_conv_encoder_write(rlrep_conv_encoder* enc, int layer, int what, const float* in_host);
/* obs_dev uint8 [B, C, H, H]; shifts_dev int32 [B, 2] = (x, y) shift in [0, 8] or NULL; feat_dev fp32 [B, 32*h*h]
 * (h = 35 for 84-pixel frames) in the reference's flatten order.  backward consumes d(feat) of the same shape and
 * leaves dW / db readable. */
RLREP_EXPORT int rlrep_conv_encoder_forward(rlrep_conv_encoder* enc, const unsigned char* obs_dev, const int* shifts_dev,
                                            float* feat_dev);
RLREP_EXPORT int rlrep_conv_encoder_backward(rlrep_conv_encoder* enc, const float* dfeat_dev);
RLREP_EXPORT int rlrep_conv_encoder_feature_dim(rlrep_conv_encoder* enc, int* dim);
/* The same with a row pitch: ld_feat / ld_dfeat floats between rows (0 = dense; the columns past the feature dimension
 * are neither read nor written).  no_grad != 0 promises that no backward follows (layers 1-3 then run without column
 * matrices); backward after a no_grad forward fails.  forward / backward are the (0, 0) / 0 cases. */
RLREP_EXPORT int rlrep_conv_encoder_forward_pitched(rlrep_conv_encoder* enc, const unsigned char* obs_dev,
                                                    const int* shifts_dev, float* feat_dev, int ld_feat, int no_grad);
RLREP_EXPORT int rlrep_conv_encoder_backward_pitched(rlrep_conv_encoder* enc, const float* dfeat_dev, int ld_dfeat);
/* Copies an internal map to out_dev in NCHW, [B, 32, h_l, h_l] for layer l = 0..3 (h_l = 41, 39, 37, 35 for 84-pixel
 * frames): which 0 = the post-ReLU output of layer l (last forward), 1 = the gradient with respect to its
 * pre-activation, ReLU mask applied (last backward). */
RLREP_EXPORT int rlrep_conv_encoder_read_map(rlrep_conv_encoder* enc, int which, int layer, float* out_dev);

/* ------------------------------------------------------------------------------------------------
 * Pixel decoder on its own -- the 3 x ConvTranspose2d(s1) + ConvTranspose2d(s2) + Conv2d stack of muLV-Rep
 * (agent/mulvdrq/drqv2.py:98-117, out_kernel 2) and of the latent Diff-SR VAE (vae_1d.Decoder, out_kernel 3, stride-2
 * layer with output_padding 1), as the agents run it, for kernel-level tests.  Layer l = 0..3 is `deconvnet.{2l}`
 * (weights [ci, co, 3, 3] / [32]), layer 4 the output conv `deconvnet.8` ([3, 32, k, k] / [3]).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_conv_decoder rlrep_conv_decoder;
RLREP_EXPORT int rlrep_conv_decoder_create(int batch, int out_kernel, int precision, void* stream,
                                           rlrep_conv_decoder** out);
RLREP_EXPORT int rlrep_conv_decoder_destroy(rlrep_conv_decoder* dec);
/* what: 0 = weight, 1 = bias, 2 = weight gradient, 3 = bias gradient (host buffers, reference layout); write takes 0 / 1 */
RLREP_EXPORT int rlrep_conv_decoder_read(rlrep_conv_decoder* dec, int layer, int what, float* out_host);
RLREP_EXPORT int rlrep_conv_decoder_write(rlrep_conv_decoder* dec, int layer, int what, const float* in_host);
/* x_dev fp32 [B, 32*35*35] in the reference's (channel, row, column) order with row pitch ld_x (0 = dense); the
 * prediction [B, 3, 84, 84] stays in the handle. */
RLREP_EXPORT int rlrep_conv_decoder_forward(rlrep_conv_decoder* dec, const float* x_dev, int ld_x);
/* loss_dev[0] = 10 * mean |pred - (target / 255 - 0.5)|; target uint8 [B, 3, 84, 84]; keeps grad_scale * d loss / d pred */
RLREP_EXPORT int rlrep_conv_decoder_l1_loss(rlrep_conv_decoder* dec, const unsigned char* target_dev, float grad_scale,
                                            float* loss_dev);
/* loss_dev[0] = sum (pred - (shifted target / 255 - 0.5))^2 / B; shifts_dev int32 [B, 2] = (x, y) in [0, 8] or NULL */
RLREP_EXPORT int rlrep_conv_decoder_mse_sum_loss(rlrep_conv_decoder* dec, const unsigned char* target_dev,
                                                 const int* shifts_dev, float grad_scale, float* loss_dev);
/* parameter gradients of the five layers (readable with _read) and dx_dev [B, 32*35*35] with row pitch ld_dx (0 = dense;
 * the columns past 32*35*35 are not written) */
RLREP_EXPORT int rlrep_conv_decoder_backward(rlrep_conv_decoder* dec, float* dx_dev, int ld_dx);
/* Copies an internal map of the last forward / loss / backward to out_dev in NCHW: which 0 = the input of layer i
 * (i = 0..4, [B, 32, h_i, h_i]), 1 = the gradient with respect to it (ReLU mask applied for i > 0), 2 = pred,
 * 3 = grad_scale * d loss / d pred (both [B, 3, 84, 84]; i is ignored). */
RLREP_EXPORT int rlrep_conv_decoder_read_map(rlrep_conv_decoder* dec, int which, int i, float* out_dev);

/* ------------------------------------------------------------------------------------------------
 * Plain DrQ-v2 pixel agent -- replaces `DrQv2(obs_space, action_space, args)` and the updating half of
 * `DrQv2.train_step(replay_iter, step)` (agent/diffsrdrq/drqv2.py:12-148).  The caller keeps `_step` / `update_every`,
 * evaluates the std-dev schedule and draws the randomness in the reference's order on the CPU generator:
 * RandomShiftsAug's integer shifts for img then next_img ((x, y) per sample), then the standard-normal draws of the next
 * action and of the actor step.  Tensors are exposed under the reference's module names ("encoder.convnet.0.weight",
 * "critic.trunk.1.weight", "actor.policy.4.bias", "critic_target.Q2.2.weight", ...); conv weights of layers 2-4 are
 * stored as [32, (ky, kx, c_in)] (rlrep_b200/pixel.py permutes them to and from the reference's [32, c_in, 3, 3]).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_drq rlrep_drq;
typedef struct rlrep_drq_config {
  int batch_size, channels, height, action_dim, bn_dim, hidden_dim;
  double encoder_lr, actor_lr, critic_lr;
  float tau, stddev_clip;
  int precision;
} rlrep_drq_config;
RLREP_EXPORT int rlrep_drq_create(const rlrep_drq_config* cfg, void* stream, rlrep_drq** out);
RLREP_EXPORT int rlrep_drq_destroy(rlrep_drq* drq);
RLREP_EXPORT int rlrep_drq_num_tensors(rlrep_drq* drq, int* n);
RLREP_EXPORT int rlrep_drq_tensor_info(rlrep_drq* drq, int i, const char** name, float** ptr_dev, int* rows, int* cols);
RLREP_EXPORT int rlrep_drq_tensor_read(rlrep_drq* drq, int i, float* out_host);
RLREP_EXPORT int rlrep_drq_tensor_write(rlrep_drq* drq, int i, const float* in_host);
RLREP_EXPORT int rlrep_drq_sync_targets(rlrep_drq* drq);
/* img / next_img uint8 [B, C, H, H]; action [B, A]; reward, discount [B]; shifts int32 [2][B][2]; eps [2][B][A];
 * metrics_host[5] = {critic_loss, mean(q_pred), mean(q_target), mean(reward), actor_loss}.  All host pointers. */
RLREP_EXPORT int rlrep_drq_update(rlrep_drq* drq, const unsigned char* img, const float* action, const float* reward,
                                  const float* discount, const unsigned char* next_img, const int* shifts,
                                  const float* eps, float stddev, float* metrics_host);
/* select_action (drqv2.py:74-82) on n observations: obs uint8 [n, C, H, H] in host memory or device memory (a CUDA
 * tensor is copied device to device); eps_host == NULL -> dist.mean, else TruncatedNormal.sample(clip=None) with
 * eps_host [n, action_dim] ~ N(0, 1) and the schedule's stddev; actions_host [n, action_dim].  Runs the small-batch policy
 * (csrc/pixel_act.cu) in IEEE fp32 whatever the handle's precision, in chunks of 64 observations, on the handle's own
 * buffers: it reads the current weights, touches no update buffer, and may be called between updates.  Each action is
 * bit-identical to the n = 1 call on its observation.  n <= 0 or a null obs / actions pointer is an error.
 * rlrep_drq_act is the n = 1 case. */
RLREP_EXPORT int rlrep_drq_act_batch(rlrep_drq* drq, const unsigned char* obs, const float* eps_host, float stddev, int n,
                                     float* actions_host);
RLREP_EXPORT int rlrep_drq_act(rlrep_drq* drq, const unsigned char* obs_host, const float* eps_host, float stddev,
                               float* action_host);
/* Benchmark aids on the batch uploaded by the last rlrep_drq_update: n_steps updates back to back with CUDA-event timing;
 * one update with an event behind every launch (same contract as rlrep_agent_profile_train). */
RLREP_EXPORT int rlrep_drq_update_resident(rlrep_drq* drq, int n_steps, float stddev, float* total_ms);
RLREP_EXPORT int rlrep_drq_profile_update(rlrep_drq* drq, float stddev, int max_entries, const char** names, float* ms,
                                          double* bytes, double* flops, int* n_entries);
RLREP_EXPORT int rlrep_drq_last_launches(rlrep_drq* drq, int* launches);
/* Optimiser state that is not a tensor, for checkpoints.  The handle's tensor index also lists the Adam moments of every
 * parameter as "optim.m/<name>" / "optim.v/<name>" (same shape and layout as the parameter; torch.optim.Adam's exp_avg /
 * exp_avg_sq), and with these counters they let a resumed handle continue bit-identically.  The pixel agents' counters are
 * the Adam step counts: here t_feature counts the encoder's optimiser, t_critic the critic's, t_actor the actor's.  They
 * have no `steps` gate and no temperature: steps, t_alpha and log_alpha* read as 0, and set refuses non-zero values in
 * them.  Set takes effect at the next update (the Adam bias corrections are recomputed from the counters every update). */
RLREP_EXPORT int rlrep_drq_get_optim_state(rlrep_drq* drq, rlrep_optim_state* out);
RLREP_EXPORT int rlrep_drq_set_optim_state(rlrep_drq* drq, const rlrep_optim_state* in);

/* ------------------------------------------------------------------------------------------------
 * muLV-Rep DrQ-v2 pixel agent -- replaces `DrQV2Agent(obs_shape, action_shape, cfg)` and the updating half of
 * `DrQV2Agent.update(replay_iter, step)` + `update_actor` (agent/mulvdrq/drqv2.py:198-461) on `mulv_config.py`'s default
 * path (aug, no pre_aug, back_q2feat, tanh heads, ReLU critic, Huber loss, soft target updates).  The caller keeps
 * `up_every`, evaluates the std-dev schedule and draws the randomness in the reference's order on the CPU generator:
 * shift draws for img then next_img, randn[B, feat_dim] (feat_encoder.sample), the next action's standard normals,
 * randn[num_noise, feat_dim] for critic_target, for critic, the actor step's standard normals, randn for its critic.
 * Tensors carry the reference's module names ("encoder.convnet.0.weight", "feat_encoder.mean_linear.0.weight",
 * "feat_f_target.log_std_linear.1.bias", "decoder.deconvnet.6.weight", ...).  Conv weights of layers 2-4 are stored
 * [32, (ky, kx, c_in)], transposed-conv weights [(ky, kx, c_out), c_in]; rlrep_b200/pixel.py permutes them to and from
 * the reference's layouts.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_mulv rlrep_mulv;
typedef struct rlrep_mulv_config {
  int batch_size, channels, height, action_dim, feat_dim, hidden_dim, num_noise;
  double lr;
  float tau, stddev_clip, vae_w, mse_w, c_noise;
  int precision;
} rlrep_mulv_config;
RLREP_EXPORT int rlrep_mulv_create(const rlrep_mulv_config* cfg, void* stream, rlrep_mulv** out);
RLREP_EXPORT int rlrep_mulv_destroy(rlrep_mulv* h);
RLREP_EXPORT int rlrep_mulv_num_tensors(rlrep_mulv* h, int* n);
RLREP_EXPORT int rlrep_mulv_tensor_info(rlrep_mulv* h, int i, const char** name, float** ptr_dev, int* rows, int* cols);
RLREP_EXPORT int rlrep_mulv_tensor_read(rlrep_mulv* h, int i, float* out_host);
RLREP_EXPORT int rlrep_mulv_tensor_write(rlrep_mulv* h, int i, const float* in_host);
RLREP_EXPORT int rlrep_mulv_sync_targets(rlrep_mulv* h);
/* img / next_img uint8 [B, C, 84, 84]; img_step1 uint8 [B, 3, 84, 84] (last frame of the one-step-ahead observation);
 * action [B, A]; reward, discount [B]; shifts int32 [2][B][2]; eps_z [B, feat_dim]; eps_act [2][B][A];
 * noise [3][num_noise][feat_dim]; metrics_host[8] = {critic_loss, mean(q1), mean(q2), mean(target_q), s_loss, r_loss,
 * kl_loss, actor_loss}.  All host pointers. */
RLREP_EXPORT int rlrep_mulv_update(rlrep_mulv* h, const unsigned char* img, const float* action, const float* reward,
                                   const float* discount, const unsigned char* next_img, const unsigned char* img_step1,
                                   const int* shifts, const float* eps_z, const float* eps_act, const float* noise,
                                   float stddev, float* metrics_host);
/* act (drqv2.py:270-282) on n observations, with the contract of rlrep_drq_act_batch: obs uint8 [n, C, 84, 84] host or
 * device; eps_host == NULL -> dist.mean (eval_mode), else TruncatedNormal.sample(clip=None) with eps_host [n, action_dim]
 * ~ N(0, 1); actions_host [n, action_dim].  The exploration phase's uniform actions are the caller's (rlrep_b200/pixel.py).
 * rlrep_mulv_act is the n = 1 case. */
RLREP_EXPORT int rlrep_mulv_act_batch(rlrep_mulv* h, const unsigned char* obs, const float* eps_host, float stddev, int n,
                                      float* actions_host);
RLREP_EXPORT int rlrep_mulv_act(rlrep_mulv* h, const unsigned char* obs_host, const float* eps_host, float stddev,
                                float* action_host);
RLREP_EXPORT int rlrep_mulv_update_resident(rlrep_mulv* h, int n_steps, float stddev, float* total_ms);
RLREP_EXPORT int rlrep_mulv_profile_update(rlrep_mulv* h, float stddev, int max_entries, const char** names, float* ms,
                                           double* bytes, double* flops, int* n_entries);
RLREP_EXPORT int rlrep_mulv_last_launches(rlrep_mulv* h, int* launches);
/* Checkpoint counters with the contract of rlrep_drq_get_optim_state: t_critic is the Adam step count that every
 * representation and critic group shares (encoder, predict_encoder, decoder, feat_encoder, feat_decoder, feat_f, critic),
 * t_actor the actor's; t_feature advances with every update and drives no optimiser. */
RLREP_EXPORT int rlrep_mulv_get_optim_state(rlrep_mulv* h, rlrep_optim_state* out);
RLREP_EXPORT int rlrep_mulv_set_optim_state(rlrep_mulv* h, const rlrep_optim_state* in);

/* ------------------------------------------------------------------------------------------------
 * Latent Diff-SR DrQ-v2 pixel agent -- replaces
 * `LatentDiffSRDrQv2(obs_space, action_space, args)` and the updating half of `train_step(replay_iter, step)`
 * (agent/diffsrdrq/latent_diff_sr.py:13-139, :306-390) on configs/latent_diff_sr.yaml's path.  The caller keeps `_step` /
 * `update_every`, evaluates the std-dev schedule and draws ALL randomness in the reference's order on the CPU generator
 * (shift draws, posterior noise, diffusion levels and noise, the dropout masks of the online score network, the action
 * normals); see rlrep_b200/pixel.py:LatentDiffSRDrQv2._draw.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rlrep_ldiff rlrep_ldiff;
typedef struct rlrep_ldiff_config {
  int batch_size, action_dim, latent_dim, feature_dim, bn_dim, psi_hidden_dim, psi_hidden_depth, zeta_hidden_dim,
      zeta_hidden_depth, hidden_dim;
  double ae_lr, score_lr, actor_lr, critic_lr, weight_decay;
  float tau, kl_coef, ae_coef, stddev_clip;
  int precision;
} rlrep_ldiff_config;
typedef struct rlrep_ldiff_inputs { /* host pointers; N = 4 * batch frames, L = latent_dim */
  const unsigned char* frames;      /* [N, 3, 84, 84]: the 3B frames of img_stack, then the B newest next frames */
  const unsigned char* next_frames; /* [3B, 3, 84, 84] */
  const int* shifts;                /* [N, 2] per-frame shift; (4, 4) = no augmentation */
  const int* next_shifts;           /* [3B, 2] */
  const float *action, *reward, *discount;
  const float* eps_post;            /* [N, L] */
  const float *alphabar, *temb, *noise; /* [B], [B, L/2], [B, L] */
  const float* psi_masks;           /* [psi_depth][2B, psi_hidden]: rows [0, B) score step, [B, 2B) critic step */
  const float* zeta_masks;          /* [zeta_depth][B, zeta_hidden] */
  const float* eps_act;             /* [2][B][A] */
  float stddev;
} rlrep_ldiff_inputs;
RLREP_EXPORT int rlrep_ldiff_create(const rlrep_ldiff_config* cfg, void* stream, rlrep_ldiff** out);
RLREP_EXPORT int rlrep_ldiff_destroy(rlrep_ldiff* h);
RLREP_EXPORT int rlrep_ldiff_num_tensors(rlrep_ldiff* h, int* n);
RLREP_EXPORT int rlrep_ldiff_tensor_info(rlrep_ldiff* h, int i, const char** name, float** ptr_dev, int* rows, int* cols);
RLREP_EXPORT int rlrep_ldiff_tensor_read(rlrep_ldiff* h, int i, float* out_host);
RLREP_EXPORT int rlrep_ldiff_tensor_write(rlrep_ldiff* h, int i, const float* in_host);
RLREP_EXPORT int rlrep_ldiff_sync_targets(rlrep_ldiff* h);
/* metrics_host[8] = {recon_loss, kl_loss, score_loss, critic_loss, mean(q_pred), mean(q_target), mean(reward), actor_loss} */
RLREP_EXPORT int rlrep_ldiff_update(rlrep_ldiff* h, const rlrep_ldiff_inputs* in, float* metrics_host);
/* Measurement aids (bench.py), like rlrep_drq_update_resident / rlrep_drq_profile_update: n_steps updates on the inputs
 * the last rlrep_ldiff_update left in device memory, timed with CUDA events; one eager update with an event behind every
 * kernel launch. */
RLREP_EXPORT int rlrep_ldiff_update_resident(rlrep_ldiff* h, int n_steps, float stddev, float* total_ms);
RLREP_EXPORT int rlrep_ldiff_profile_update(rlrep_ldiff* h, float stddev, int max_entries, const char** names, float* ms,
                                            double* bytes, double* flops, int* n_entries);
RLREP_EXPORT int rlrep_ldiff_last_launches(rlrep_ldiff* h, int* launches);
/* Checkpoint counters with the contract of rlrep_drq_get_optim_state: t_feature counts the VAE's and the score network's
 * optimisers (one step count, like their one learning rate), t_critic the critic's, t_actor the actor's.  The score
 * blocks' unused `residual` layers have no optimiser state and no "optim.*" entries. */
RLREP_EXPORT int rlrep_ldiff_get_optim_state(rlrep_ldiff* h, rlrep_optim_state* out);
RLREP_EXPORT int rlrep_ldiff_set_optim_state(rlrep_ldiff* h, const rlrep_optim_state* in);

/* Kernels launched by the most recent train() (a graph replay counts the kernels it contains). */
/* Batched policy evaluation (utils/util.py:40-57 `eval_policy` over vectorised environments, or any caller that has many
 * observations at once): states_host [rows, state_dim], eps_host [rows, action_dim] or NULL (deterministic),
 * actions_host [rows, action_dim].  One kernel launch per 1024 rows; rlrep_agent_act is the rows = 1 case. */
RLREP_EXPORT int rlrep_agent_act_batch(rlrep_agent* agent, const float* states_host, const float* eps_host, int rows,
                                       float* actions_host);
RLREP_EXPORT int rlrep_agent_last_launches(rlrep_agent* agent, int* launches);
/* The captured train() graph: its kernel nodes, and how many of its edges are programmatic (a kernel that may start
 * while the kernel before it is still running, programmatic dependent launch).  Fails before the graph exists. */
RLREP_EXPORT int rlrep_agent_graph_stats(rlrep_agent* agent, int* kernel_nodes, int* programmatic_edges);

#ifdef __cplusplus
}
#endif
#endif /* RLREP_B200_H_ */

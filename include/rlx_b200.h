/*
 * rlx_b200.h — C-ABI of the B200-native (sm_100a) RL-X hot path.
 *
 * The reference (nico-bohlinger/RL-X) is pure Python and has no FFI of its own; its hot path is the body of
 * PPO.train() (rl_x/algorithms/ppo/pytorch/ppo.py:97-393) and SAC.train() (rl_x/algorithms/sac/pytorch/sac.py:89-348).
 * Each entry point below replaces a block of that Python; the block is cited as `ref:`.  The Python plugin
 * (rl_x_b200/algorithms/ppo/b200/ppo.py) binds these with ctypes — see INTEGRATION.md for the stub a maintainer
 * would add to the reference itself.
 *
 * Conventions
 *   - plain pointers + sizes only; no torch / C++ types.  All device pointers are raw CUDA device addresses
 *     (tensor.data_ptr()), row-major contiguous unless a leading dimension is given.
 *   - every device entry point is stream-ordered on `stream` (a cudaStream_t passed as void*; NULL = default stream),
 *     never allocates or frees memory, never synchronises the device.  Scratch is caller-provided
 *     (`*_workspace_bytes` queries).
 *   - return value: 0 = OK, negative = error (RLX_ERR_*); rlx_last_error_string() describes the last error of the
 *     calling thread.  Nothing throws across the boundary.
 *   - fp32 everywhere (the reference's parity path: bf16 autocast off, ppo.py:60-70); indices are int64 like
 *     np.arange(B) (ppo.py:273).
 */
#ifndef RLX_B200_H
#define RLX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLX_OK 0
#define RLX_ERR_INVALID_ARG (-1)
#define RLX_ERR_CUDA (-2)
#define RLX_ERR_WORKSPACE (-3)
#define RLX_ERR_UNSUPPORTED (-4)

/* ------------------------------------------------------------------------------------------------ library -- */
int rlx_version(void);                        /* ABI version, currently 1 */
const char* rlx_last_error_string(void);      /* thread-local, never NULL */
uint64_t rlx_launch_count(void);              /* kernels launched by this library since load / last reset */
void rlx_reset_launch_count(void);
void rlx_add_launch_count(uint64_t n);        /* account for kernels replayed through a captured CUDA graph */
/* Optional per-kernel-class device timing (CUDA events recorded around every launch on the launching stream).
 * rlx_timing_begin() enables it and clears the records; rlx_timing_end() synchronises the device, disables it and fills four
 * arrays of RLX_NKCLASS entries: summed duration (ms), launch count, summed ALGORITHMIC flops and bytes of each class. */
#define RLX_NKCLASS 14
int rlx_timing_begin(void);
int rlx_timing_end(double* ms, uint64_t* launches, double* flops, double* bytes);
const char* rlx_kernel_class_name(int cls);
/* GEMM engine used by the MLP entry points: 0 = fp32 SIMT (FFMA), 1 = tcgen05 3xTF32 (tensor cores, TMEM accumulators).
 * Returns the engine actually in effect (a request for 1 falls back to 0 with an error string if the shape is unsupported). */
int rlx_set_gemm_engine(int engine);
int rlx_get_gemm_engine(void);
/* The same choice for the dense layers of the FastSAC and PPO+LSTM entry points (their own switch: these paths were validated on the SIMT
 * engine).  1 routes every GEMM whose layout / epilogue / alignment the tcgen05 engine covers to it and leaves the rest on the SIMT
 * engine (e.g. the 101-column logits of the C51 critics, whose row pitch is not a multiple of 16 bytes).  Default 0.  Returns the value in effect. */
int rlx_set_aux_gemm_engine(int engine);
uint64_t rlx_aux_tc_gemm_count(void);     /* GEMMs of those two paths that ran on the tcgen05 engine since load */

/* Test hook: one plain fp32 GEMM through either engine.  layout 0: C[M,N] = A[M,K] B[N,K]^T; 1: C = A[M,K] B[K,N];
 * 2: C = A[K,M]^T B[K,N].  epilogue 0 none, 1 tanh(x + bias[n]) (layout 0), 2 x * (1 - aux[m,n]^2) (layout 1). */
int rlx_debug_gemm_f32(int engine, int layout, int epilogue, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                       const float* B, int64_t ldb, float* C, int64_t ldc, const float* bias, const float* aux, int64_t ldaux,
                       void* stream);

/* ------------------------------------------------------------------------------- numpy-compatible host RNG -- */
/* ref: self.rng = np.random.default_rng(self.seed)  (ppo.py:72; sac.py replay_buffer.py:8) — Generator(PCG64(SeedSequence(seed))).
 * state[0..1] = 128-bit LCG state (hi, lo); state[2..3] = increment (hi, lo); state[4] = has_uint32; state[5] = buffered uinteger. */
typedef struct rlx_pcg64 { uint64_t s[6]; } rlx_pcg64;
int rlx_pcg64_seed(uint64_t seed, rlx_pcg64* st);
uint64_t rlx_pcg64_next64(rlx_pcg64* st);
uint32_t rlx_pcg64_next32(rlx_pcg64* st);
/* ref: self.rng.shuffle(batch_indices)  (ppo.py:276) — in place, bit-exact with numpy.random.Generator.shuffle on a 1-D int64 array. HOST memory. */
int rlx_pcg64_shuffle_i64(rlx_pcg64* st, int64_t* a, int64_t n);
/* ref: self.rng.integers(high, size=n)  (sac/pytorch/replay_buffer.py:33-34) — int64 output, low = 0. HOST memory. */
int rlx_pcg64_integers_i64(rlx_pcg64* st, int64_t high, int64_t* out, int64_t n);
/* ref: self.rng.choice(self.batch_size, size=self.minibatch_size, replace=False)  (espo/pytorch/espo.py:256): bit-exact with
 * numpy.random.Generator.choice for an integer population, replace=False, shuffle=True, p=None.  Host function. */
int rlx_pcg64_choice_i64(rlx_pcg64* st, int64_t pop_size, int64_t size, int64_t* out);

/* ------------------------------------------------------------------------------------- PPO network layout -- */
/* Policy: obs -> hidden -> hidden -> act (tanh, tanh, linear) + logstd(act)   ref: policy.py:34-52
 * Critic: obs -> hidden -> hidden -> 1   (tanh, tanh, linear)                 ref: critic.py:23-41
 * All parameters live in ONE flat fp32 buffer; gradients and both Adam moments use the same layout.
 * Segment order (nn.Linear weights are [out, in] row-major exactly as in the reference state_dict):
 *   0 W1p[H,obs] 1 W1c[H,obs] 2 b1p[H] 3 b1c[H] 4 W2p[H,H] 5 W2c[H,H] 6 b2p[H] 7 b2c[H]
 *   8 W3p[A,H]   9 W3c[1,H]  10 b3p[A] 11 b3c[1] 12 logstd[A]
 * (policy and critic first layers are adjacent so that layer 1 runs as one [2H, obs] GEMM on the shared input.) */
#define RLX_PPO_NSEG 13
typedef struct rlx_ppo_dims { int32_t obs_dim, act_dim, hidden; } rlx_ppo_dims;
int64_t rlx_ppo_param_count(const rlx_ppo_dims* d);
/* offsets[RLX_PPO_NSEG+1]: start of each segment, last entry = total count.  is_critic[RLX_PPO_NSEG]: 0 policy / 1 critic. */
int rlx_ppo_param_layout(const rlx_ppo_dims* d, int64_t* offsets, int32_t* is_critic);

/* ------------------------------------------------------------------------------------------ rollout (acting) -- */
/* ref: policy.get_action_logprob(state) + critic.get_value(state)  (ppo.py:207-209; policy.py:61-73; critic.py:44-46)
 *   mean = MLP_p(obs); a = mean + exp(logstd) * noise; logp = sum_a Normal(mean, std).log_prob(a); value = MLP_c(obs)
 *   env_action = low + 0.5 * (clip(a,-1,1) + 1) * (high - low)   if clip_rescale else a
 * obs [n, obs_dim]; noise [n, act] standard-normal draws supplied by the caller, or NULL: a counter-based Philox4x32-10
 * stream keyed by (rng_seed, rng_offset, row) is used (rng_offset must advance by 1 per call).
 * deterministic != 0 reproduces get_deterministic_action (policy.py:85-93): a = mean, no noise, logp not written.
 * Outputs (any may be NULL): action [n, act] (unclipped sample, what ppo.py:233 stores), env_action [n, act],
 * logp [n], value [n].  workspace: rlx_ppo_forward_workspace_bytes(d, n). */
typedef struct rlx_ppo_forward_args {
  rlx_ppo_dims dims;
  int64_t n;
  const float* params;
  const float* obs;
  const float* noise;
  uint64_t rng_seed, rng_offset;
  const float* act_low;   /* [act] device */
  const float* act_high;  /* [act] device */
  int32_t clip_rescale;
  int32_t deterministic;
  float* action;
  float* env_action;
  float* logp;
  float* value;
  void* workspace;
  size_t workspace_bytes;
} rlx_ppo_forward_args;
size_t rlx_ppo_forward_workspace_bytes(const rlx_ppo_dims* d, int64_t n);
int rlx_ppo_forward_f32(const rlx_ppo_forward_args* a, void* stream);

/* ref: critic.get_value(x) alone  (ppo.py:253-254 next_values; critic.py:44-46).  obs [n, obs_dim] -> value [n]. */
int rlx_critic_forward_f32(const rlx_ppo_dims* d, const float* params, const float* obs, int64_t n, float* value,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ref: the per-step buffer writes  batch.rewards[step] = reward; batch.terminations[step] = terminated;
 * state = next_state  (ppo.py:231-245) plus the running `dones_this_rollout += done.sum()` (ppo.py:227) kept on device.
 * reward [n] f32; terminated/truncated [n] uint8 (torch.bool); next_obs [n, obs] may be NULL.
 * Writes rewards_row [n], terminations_row [n] (0/1 float), next_obs_dst [n, obs] (copy), done_count[0] += #done. */
int rlx_rollout_store_f32(const float* reward, const uint8_t* terminated, const uint8_t* truncated, const float* next_obs,
                          int64_t n, int64_t obs_dim, float* rewards_row, float* terminations_row, float* next_obs_dst,
                          int64_t* done_count, void* stream);
/* Same, plus device-side episode statistics with the semantics of the reference's torch-interface envs
 * (rl_x/environments/custom_mujoco/ant/warp_torch/environment.py:159-178, wrappers.py:15-33): episode_return[n] / episode_length[n]
 * (in/out running accumulators, zero-initialised by the caller) take this step's reward / +1; for an env whose episode ended
 * (terminated | truncated) done_return_row[i] / done_length_row[i] receive the finished episode's return / length and the accumulators
 * restart from zero; elsewhere the rows receive 0 (length 0 = "no episode ended here").  All four may be NULL (= rlx_rollout_store_f32). */
int rlx_rollout_store_stats_f32(const float* reward, const uint8_t* terminated, const uint8_t* truncated, const float* next_obs,
                                int64_t n, int64_t obs_dim, float* rewards_row, float* terminations_row, float* next_obs_dst,
                                int64_t* done_count, float* episode_return, float* episode_length, float* done_return_row,
                                float* done_length_row, void* stream);

/* ------------------------------------------------------------------------------------------------------ GAE -- */
/* ref: calculate_gae_advantages_and_returns  (ppo.py:110-118)
 *   delta = r + gamma * nv * (1 - term) - v;  A[t] = delta[t] + gamma*lambda*(1-term[t]) * A[t+1];  R = A + v
 * All arrays time-major [T, N].  Two ways to supply next values:
 *   next_values != NULL : full [T, N] tensor as in the reference (ppo.py:253-254)
 *   next_values == NULL : TORCH-interface shortcut, nv[t] = values[t+1] for t < T-1 and nv[T-1] = last_value[N]
 *                         (valid because next_states[t] is states[t+1], ppo.py:224-232,244; SURVEY §8 a5).
 * gamma / gae_lambda are the Python floats (doubles) of the config: TorchScript multiplies them in double before the
 * cast to fp32.  Bit-exact with the reference's fp32 arithmetic (same operation order, no FMA contraction). */
int rlx_gae_f32(const float* rewards, const float* terminations, const float* values, const float* next_values,
                const float* last_value, int64_t T, int64_t N, double gamma, double gae_lambda, float* advantages,
                float* returns, void* stream);
/* 1 (default): the GAE kernel stages its [steps x 32 envs] tiles into shared memory with TMA (cp.async.bulk.tensor.2d) whenever the arrays
 * are 16-byte aligned and N % 4 == 0; 0: always ordinary coalesced loads (the fallback for other shapes).  Results are bit-identical. */
int rlx_set_gae_tma(int on);

/* -------------------------------------------------------------------------------- minibatch gather + stats -- */
/* ref: batch_states[minibatch_indices], batch_actions[...], batch_log_probs[...], batch_advantages[...], batch_returns[...]
 * (ppo.py:277-284).  idx [count] int64 indices into the flattened (T*N) batch.  Gathers rows into contiguous
 * minibatch-ordered buffers; with count = B and idx = the epoch permutation, minibatch k is the slice [k*mb, (k+1)*mb).
 * out_states_ld: row pitch of out_states in floats (0 = obs_dim).  When it is larger than obs_dim the pad columns are written too:
 * out_states[:, obs_dim] = 1.0 (a constant-one feature used by the dW1 GEMM to emit the bias gradient), the rest 0. */
int rlx_gather_minibatch_f32(const int64_t* idx, int64_t count, int64_t obs_dim, int64_t act_dim, const float* states,
                             const float* actions, const float* log_probs, const float* advantages, const float* returns,
                             float* out_states, float* out_actions, float* out_log_probs, float* out_advantages,
                             float* out_returns, int64_t out_states_ld, void* stream);

/* ref: minibatch_advantages.mean(), .std() (unbiased)  (ppo.py:133-134), for `num_mb` consecutive minibatches of size mb
 * (last one may be short) over gathered advantages adv [count].  stats [num_mb, 2] = (mean, unbiased std). */
int rlx_advantage_stats_f32(const float* adv, int64_t count, int64_t mb, float* stats, void* stream);
/* sharded form (SURVEY.md §8 e): segment k = rows [offsets[k], offsets[k+1]) of x (offsets: [nseg+1] int64 ON THE DEVICE).
 * gsum == NULL: out[k] = sum of the segment.  Otherwise out[k] = sum (x - gsum[k]/gcount[k])^2.  The caller all-reduces `out` across
 * ranks between the two calls; mean = gsum/gcount, std = sqrt(q/(gcount-1)) reproduce ppo.py:133-134 on the global minibatch. */
int rlx_segment_moments_f32(const float* x, const int64_t* offsets, int64_t nseg, const float* gsum, const float* gcount, float* out,
                            void* stream);

/* ------------------------------------------------------------------------------- PPO minibatch update step -- */
/* Device-resident optimiser state: one struct per (policy, critic) pair.  ref: optim.Adam(lr, betas=(0.9,0.999), eps=1e-8)
 * x2 (ppo.py:82-84), clip_grad_norm_ x2 (ppo.py:146,162). */
typedef struct rlx_ppo_hparams {
  float clip_range;      /* ppo.py:46 */
  float entropy_coef;    /* ppo.py:47 */
  float critic_coef;     /* ppo.py:48 */
  float max_grad_norm;   /* ppo.py:49 */
  float adam_beta1, adam_beta2, adam_eps;
  float ratio_delta_metric; /* 0: metrics[4] = clip fraction (ppo.py:131).  1 (ESPO): metrics[4] = mean |ratio - 1| (espo.py:133, operator
                               "mean"); 2 (ESPO, operator "median", espo.py:59-60): torch.median(|ratio - 1|) = the lower median, by a
                               radix-select kernel (single-GPU minibatches).  ESPO's unclipped surrogate (espo.py:138) is clip_range = +inf */
} rlx_ppo_hparams;

/* Per-minibatch metric record written by the update (ref: ppo.py:285-294 .item() calls, kept on device instead). */
#define RLX_PPO_NMETRIC 8
/* 0 pg_loss 1 critic_loss 2 entropy_loss 3 approx_kl 4 clip_fraction (or ratio_delta) 5 policy_grad_norm 6 critic_grad_norm 7 count */

typedef struct rlx_ppo_minibatch_args {
  rlx_ppo_dims dims;
  int64_t m;                 /* rows in this minibatch (this rank's share) */
  int64_t m_global;          /* divisor of the mean reductions (= m on one GPU; global minibatch size when sharded) */
  const float* states;       /* [m, obs]  gathered */
  const float* actions;      /* [m, act] */
  const float* log_probs;    /* [m]  old log-probs */
  const float* advantages;   /* [m]  raw advantages */
  const float* returns;      /* [m] */
  const float* adv_stats;    /* [2] device: mean, unbiased std of the (global) minibatch advantages */
  float* params;             /* flat parameters (updated in place by the optimiser step) */
  float* grads;              /* flat gradient out [P] */
  float* exp_avg;            /* Adam m [P] */
  float* exp_avg_sq;         /* Adam v [P] */
  const float* lr;           /* [1] device: current learning rate (LinearLR runs on the host, ppo.py:302-304) */
  int64_t* step_count;       /* [1] device: Adam step counter, incremented by the optimiser kernel */
  rlx_ppo_hparams hp;
  float* metrics;            /* [RLX_PPO_NMETRIC] device, overwritten */
  void* workspace;
  size_t workspace_bytes;
  int64_t states_ld;         /* row pitch of `states` in floats; 0 = obs_dim (contiguous) */
  int32_t states_ones_col;   /* != 0: states[:, obs_dim] == 1.0 in every row (written by rlx_gather_minibatch_f32 when out_states_ld > obs):
                                lets the tensor-core dW1 GEMM produce the layer-1 bias gradient as one extra output column */
  int32_t reserved2;
} rlx_ppo_minibatch_args;
size_t rlx_ppo_minibatch_workspace_bytes(const rlx_ppo_dims* d, int64_t m);

/* ref: policy_loss_fn forward+backward (ppo.py:121-144) and critic_loss_fn forward+backward (ppo.py:153-160):
 * writes the flat gradient of (pg_loss - c_ent*entropy) wrt policy params and of c_v*mean(0.5 (v-R)^2) wrt critic
 * params (sums over the m local rows divided by m_global), and metrics[0..4].  Does NOT touch params. */
int rlx_ppo_minibatch_fwdbwd_f32(const rlx_ppo_minibatch_args* a, void* stream);

/* ref: clip_grad_norm_(policy) + Adam.step(); clip_grad_norm_(critic) + Adam.step()  (ppo.py:146-148,162-164;
 * torch/nn/utils/clip_grad.py; torch/optim/adam.py single-tensor path).  Reads grads (already all-reduced when
 * sharded), writes params/exp_avg/exp_avg_sq, increments step_count, writes metrics[5..6] (pre-clip norms). */
int rlx_gradnorm_clip_adam_f32(const rlx_ppo_minibatch_args* a, void* stream);

/* fwdbwd + clip/Adam for `num_mb` consecutive minibatches of gathered data (one epoch or part of it), all launched
 * from C with no host round trip.  states etc. point at the first row; minibatch k covers rows [k*mb, min((k+1)*mb, count)).
 * adv_stats [num_mb,2]; metrics [num_mb, RLX_PPO_NMETRIC].  Single-GPU only (no collective between the two halves). */
int rlx_ppo_update_epoch_f32(const rlx_ppo_minibatch_args* first, int64_t count, int64_t mb, void* stream);

/* --------------------------------------------------------------- multi-GPU gradient exchange (SURVEY.md §8 e) -- */
/* The reference is single-process (one optimiser.step per minibatch, ppo.py:146-148,162-164); data-parallel ranks have to
 * agree on the minibatch gradient in between loss.backward() and clip_grad_norm_.  rlx_comm is that exchange, done by the
 * library's own kernel over NVLink peer memory instead of a host-launched NCCL call: every rank writes its partial gradient
 * into a send slot that lives in ITS memory, and one kernel per rank waits on peer flags and sums all ranks' slots, in rank
 * order, straight from peer memory (one-shot all-reduce; the result is bit-identical on every rank).  The slots are double
 * buffered so no second barrier is needed.  One process per GPU; handles travel through any host channel the caller owns
 * (torch.distributed all_gather in the PPO class). */
#define RLX_COMM_MAX_WORLD 16
#define RLX_COMM_HANDLE_BYTES 64
typedef struct rlx_comm rlx_comm;
/* allocates this rank's flags + two send slots of `nfloats` floats on the current device */
int rlx_comm_create(int rank, int world, int64_t nfloats, rlx_comm** out);
/* writes the CUDA IPC handle of this rank's allocation (RLX_COMM_HANDLE_BYTES bytes) */
int rlx_comm_export_handle(rlx_comm* c, uint8_t* handle);
/* handles: [world, RLX_COMM_HANDLE_BYTES] in rank order (own entry ignored); maps every peer's allocation */
int rlx_comm_connect(rlx_comm* c, const uint8_t* handles);
/* device pointer of the slot the NEXT rlx_comm_allreduce_sum_f32 call reads (write the partial sums there) */
float* rlx_comm_send_buffer(rlx_comm* c);
/* convenience: device-to-device copy of src[0..n) into the send buffer (for callers whose producer cannot write there directly) */
int rlx_comm_stage_f32(rlx_comm* c, const float* src, int64_t n, void* stream);
/* out[i] = sum over ranks r = 0..world-1 (in that order) of rank r's send buffer [i], i < n <= nfloats.  Every rank must call
 * it the same number of times; the kernel spins on peer flags (and traps after ~20 s if a peer never arrives). */
int rlx_comm_allreduce_sum_f32(rlx_comm* c, float* out, int64_t n, void* stream);
int rlx_comm_destroy(rlx_comm* c);

/* Sharded form of rlx_ppo_update_epoch_f32: minibatch k covers this rank's counts[k] consecutive gathered rows and is divided by
 * global_counts[k]; per minibatch: fwdbwd into the send slot, peer all-reduce (gradient + metric sums) into first->grads
 * [P + RLX_PPO_NMETRIC], clip + Adam, metrics row k.  No host round trip and no NCCL call inside the epoch. */
int rlx_ppo_update_epoch_sharded_f32(const rlx_ppo_minibatch_args* first, int64_t num_mb, const int64_t* counts,
                                     const int64_t* global_counts, rlx_comm* comm, void* stream);


/* Loss head of rlx_ppo_minibatch_fwdbwd_f32: 0 (default) = the fused SIMT kernel, 2 = the fused kernel on the warp-level tensor path
 * (csrc/ppo_head_mma.cuh: both skinny products as 3xTF32 mma.sync tiles; fp32 mode, hidden 128/256/512, act <= 31 - other shapes and the
 * bf16 mode run engine 0).  Any other value is an error and leaves the setting unchanged.  Returns the engine in effect. */
int rlx_set_head_engine(int engine);
/* bf16-autocast mode of the PPO entry points (the reference's `bf16_mixed_precision_training`, ppo.py:98-107,123,155,208,253; its default).
 * on != 0: rlx_ppo_forward_f32 / rlx_critic_forward_f32 / rlx_ppo_minibatch_fwdbwd_f32 / rlx_gae_f32 round every value that torch's autocast
 * holds in a bf16 tensor to bf16 where torch rounds it - Linear inputs, weights and biases, Linear outputs, tanh outputs, the sampled action
 * and the bf16 subtraction / square inside its log-prob, gamma * next_values, and on the way back the gradients of those bf16 tensors and the
 * weight / bias gradients (one rounding of the complete fp32-accumulated sum) - while storage, losses, clipping and Adam stay fp32 as in
 * the reference.  bf16 values are exact TF32 operands, so the tensor-core GEMMs run ONE kind::tf32 MMA per product in this mode (fp32
 * accumulation in TMEM, as a bf16 tensor-core GEMM accumulates) instead of the three of the fp32-equivalent split.  Returns the setting. */
int rlx_set_autocast_bf16(int on);
/* tcgen05 engine on CTA pairs (cta_group::2, csrc/gemm_tc2.cu).  mode 0: single-CTA kernels only; 1: the weight-gradient GEMMs of the PPO
 * update run on pairs (256 x 256 / 256 x 192 tiles); 2 (default, with fwd_bn = 128): the forward / dX GEMMs too, with fwd_bn-wide pair tiles
 * (128: double-buffered accumulators, 256: single; other values keep the current setting).  Returns the mode. */
int rlx_set_tc_pair(int mode, int fwd_bn);

/* ------------------------------------------------------------------------------------------ PPO + LSTM path -- */
/* SURVEY.md §8 a18: rl_x/algorithms/ppo_lstm/flax (policy.py:36-146, critic.py:18-30, ppo_lstm.py:107-231), including the two policy
 * options lstm_obs_combine_method = "concat" | "film" (policy.py:57-59, 99-105) and share_lstm_obs_encoder (policy.py:51-53, 120-123).
 * The sources also compile for the host (g++ -DRLX_EMU) and are checked there against oracle/ppo_lstm_oracle.py
 * (tests/test_lstm_emulation.py); the default options have run on B200 since round 1, FiLM / shared encoder and the one-launch-per-step
 * recurrence were added after the round-2 GPU budget was spent (emulation-validated; GPU tests in tests/test_gpu_zzz_ppo_lstm.py).
 * Exact-fp32 SIMT GEMMs; ONE launch per time step for the recurrent part in both directions (carry reset + h.Wh + cell fused).
 *
 * Flat parameter layouts (fp32).  All kernels are stored [in, out] like Flax.  Policy segments, in order:
 *   0 We1 [obs,E] 1 be1 [E] 2 g1 [E] 3 n1 [E]      lstm_obs_encoder dense kernel/bias, LayerNorm scale/bias
 *   4 We2 [obs,E] 5 be2 [E] 6 g2 [E] 7 n2 [E]      obs_encoder (all four EMPTY with a shared encoder)
 *   8 Wi [E,4L] 9 Wh [L,4L] 10 bh [4L]             LSTM, gate blocks ordered i|f|g|o (Flax ii,if,ig,io / hi,hf,hg,ho)
 *   11 gl [L] 12 nl [L]                            lstm_ln
 *   13 Wt1 [E+L,H] (FiLM: [E,H]) 14 bt1 [H] 15 Wt2 [H,H] 16 bt2 [H] 17 Wm [H,A] 18 bm [A] 19 logstd [A]
 *   20 Wf [L,2E] 21 bf [2E]                        FiLM only (EMPTY otherwise): blocks gamma|beta (Flax lstm_film_gamma / lstm_film_beta)
 * Critic segments: 0 Wc1 [obs,H] 1 bc1 [H] 2 Wc2 [H,H] 3 bc2 [H] 4 Wc3 [H,1] 5 bc3 [1]. */
#define RLX_LSTM_POLICY_NSEG 22
#define RLX_LSTM_CRITIC_NSEG 6
#define RLX_LSTM_OPT_FILM 1            /* lstm_obs_combine_method = "film" */
#define RLX_LSTM_OPT_SHARED_ENCODER 2  /* share_lstm_obs_encoder = True */
typedef struct rlx_lstm_dims { int32_t obs_dim, act_dim, hidden, enc_dim, lstm_dim, options /* RLX_LSTM_OPT_* bits; 0 = reference defaults */; } rlx_lstm_dims;
int rlx_lstm_param_layout(const rlx_lstm_dims* d, int64_t* policy_offsets /*[NSEG+1]*/, int64_t* critic_offsets /*[NSEG+1]*/);
size_t rlx_lstm_minibatch_workspace_bytes(const rlx_lstm_dims* d, int64_t T, int64_t n_env);

/* Recurrence of rlx_lstm_ppo_minibatch_fwdbwd_f32: 0 (default) one launch per time step and direction; 1 ONE launch per direction - a block
 * owns a few envs for all T steps, recurrent kernel (Wh / Wh^T) resident in shared memory, hidden state / gate gradients exchanged through
 * shared memory with one barrier per step, cell state in a register.  Used when the kernel fits (lstm_dim <= 100 or so: 64 KB at 64), else
 * the per-step path runs.  Bit-identical results.  Returns the value in effect; the counter says how many such launches have run. */
int rlx_set_lstm_persistent(int on);
uint64_t rlx_lstm_persistent_launch_count(void);

typedef struct rlx_lstm_minibatch_args {
  rlx_lstm_dims dims;
  int64_t T, n_env;             /* sequence length, envs in this minibatch (ppo_lstm.py:58: minibatch_size // nr_steps) */
  const float* states;          /* [T, n_env, obs]   time-major like the reference's states[:, minibatch_env_indices] */
  const float* actions;         /* [T, n_env, act] */
  const float* log_probs;       /* [T, n_env] */
  const float* advantages;      /* [T, n_env] raw */
  const float* returns;         /* [T, n_env] */
  const float* dones;           /* [T, n_env] 0/1: done AFTER step t (policy.py:127-135) */
  const float* init_c;          /* [n_env, L] carry valid for states[0] */
  const float* init_h;          /* [n_env, L] */
  const float* adv_stats;       /* [2] device: mean and POPULATION std (jnp.std, ddof 0) of this minibatch's advantages (ppo_lstm.py:196-197) */
  const float* policy_params;
  const float* critic_params;
  float* policy_grads;          /* out, same layout as policy_params */
  float* critic_grads;
  float clip_range, entropy_coef, critic_coef, reserved;
  float* metrics;               /* [8] device: pg_loss, critic_loss, entropy_loss, approx_kl, clip_fraction, -, -, rows */
  void* workspace;
  size_t workspace_bytes;
} rlx_lstm_minibatch_args;
/* ref: loss_fn + grad (ppo_lstm.py:143-208): forward_sequence with carry reset, combined loss, gradients of its mean wrt both trees */
int rlx_lstm_ppo_minibatch_fwdbwd_f32(const rlx_lstm_minibatch_args* a, void* stream);

typedef struct rlx_lstm_step_args {
  rlx_lstm_dims dims;
  int64_t n;                    /* envs */
  const float* obs;             /* [n, obs] */
  float* c;                     /* [n, L] in: carry valid for obs (already reset where the previous step ended an episode); out: next carry */
  float* h;                     /* [n, L] */
  const float* noise;           /* [n, act] standard normal draws, or NULL: deterministic (action = mean, get_deterministic_action ppo_lstm.py:234-237) */
  const float* policy_params;
  const float* critic_params;   /* may be NULL together with `value` (evaluation) */
  const float* act_low;         /* [act] */
  const float* act_high;        /* [act] */
  int32_t clip_rescale;         /* action_clipping_and_rescaling (policy.py:149-157) */
  int32_t reserved;
  float* action;                /* [n, act] unclipped sample */
  float* env_action;            /* [n, act] what the env receives */
  float* logp;                  /* [n] or NULL */
  float* value;                 /* [n] or NULL */
  void* workspace;              /* rlx_lstm_minibatch_workspace_bytes(d, 1, n) */
  size_t workspace_bytes;
} rlx_lstm_step_args;
/* ref: get_action_and_value (ppo_lstm.py:107-118): Policy.apply_one_step + Gaussian sample + log-prob + critic value */
int rlx_lstm_step_f32(const rlx_lstm_step_args* a, void* stream);
/* ref: next_policy_lstm_carry * (1 - done) (ppo_lstm.py:283): done is [n] float 0/1 */
int rlx_lstm_mask_carry_f32(float* c, float* h, const float* done, int64_t n, int64_t lstm_dim, void* stream);
/* ref: critic.apply(params, x) (ppo_lstm.py:131): x [rows, obs] -> out [rows]; workspace: rlx_lstm_minibatch_workspace_bytes(d, 1, rows) */
int rlx_lstm_critic_forward_f32(const rlx_lstm_dims* d, const float* critic_params, const float* x, int64_t rows, float* out, void* workspace,
                                size_t workspace_bytes, void* stream);
/* out[0] = mean(x), out[1] = population std (jnp.std) of x[0..n); workspace: >= n + 2 * ceil(n / 256) + 8 floats */
int rlx_mean_popstd_f32(const float* x, int64_t n, float* out, float* workspace, void* stream);

/* ref: optax.chain(clip_by_global_norm(max_norm), adam(lr))  (ppo_lstm.py:88-103) on one flat tree: g *= max_norm/||g|| iff ||g|| >= max_norm
 * (no epsilon), then Adam with bias correction; step_count (device int64) is incremented; norm_out[0] = pre-clip ||g||.
 * workspace: >= ceil(n / 1024) floats. */
int rlx_optax_clip_adam_f32(float* params, const float* grads, float* mu, float* nu, int64_t n, const float* lr, int64_t* step_count,
                            float max_norm, float beta1, float beta2, float eps, float* norm_out, float* workspace, void* stream);

/* out[t, j, :] = src[t, env_idx[j], :]  for t < T, j < n  (the reference's x[:, minibatch_env_indices]); width = trailing dim (1 for [T, N]) */
int rlx_gather_env_columns_f32(const float* src, const int64_t* env_idx, int64_t T, int64_t N, int64_t n, int64_t width, float* out, void* stream);

/* -------------------------------------------------------------------------------------------- FastSAC update -- */
/* SURVEY.md §8 f4 (second half): rl_x/algorithms/fastsac/pytorch, fp32 path.  STATUS: written
 * without GPU access; numerics checked by running these sources in a host emulation build against oracle/fastsac_oracle.py, which
 * is pinned to the executed reference (tests/test_fastsac_emulation.py); on hardware since the round-1 driver run (tests/test_gpu_zzzz_fastsac.py).
 * Networks (fixed widths like the reference): policy Linear-LayerNorm-SiLU x3 (512, 256, 128) + mean / log_std heads (policy.py:36-48);
 * Q network Linear-LayerNorm-SiLU x3 (768, 384, 192) + nr_atoms logits on [state | action] (q_network.py:24-35).
 * Flat parameter layouts, torch [out, in] weights in state_dict order:
 *   policy: (W, b, ln_w, ln_b) x 3, mean.W [act,128], mean.b, log_std.W [act,128], log_std.b            -> 16 segments
 *   Q:      (W, b, ln_w, ln_b) x 3, head.W [atoms,192], head.b                                          -> 14 segments; q buffers hold q1 | q2 */
#define RLX_FASTSAC_POLICY_NSEG 16
#define RLX_FASTSAC_Q_NSEG 14
typedef struct rlx_fastsac_dims { int32_t obs_dim, act_dim, nr_atoms; } rlx_fastsac_dims;
int rlx_fastsac_param_layout(const rlx_fastsac_dims* d, int64_t* policy_offsets /*[17]*/, int64_t* q_offsets /*[15], one network*/);
size_t rlx_fastsac_workspace_bytes(const rlx_fastsac_dims* d, int64_t n);

typedef struct rlx_fastsac_hparams {
  float gamma, tau, v_min, v_max, target_entropy, log_std_min, log_std_max;
  float weight_decay, adam_beta1, adam_beta2, adam_eps, max_grad_norm;  /* max_grad_norm < 0: no clipping (fastsac.py:126-133) */
  float clipped_double_q;           /* != 0: both critics learn the target distribution of the smaller next value, the actor maximises
                                       min(q1, q2) (fastsac.py:117-120,179-182) */
} rlx_fastsac_hparams;

typedef struct rlx_fastsac_update_args {
  rlx_fastsac_dims dims;
  int64_t n;                        /* batch rows */
  const float* states;              /* [n, obs] normalised */
  const float* next_states;         /* [n, obs] normalised (critic update only) */
  const float* actions;             /* [n, act] (critic update only) */
  const float* rewards;             /* [n] n-step rewards */
  const float* dones;               /* [n] */
  const float* truncations;         /* [n] */
  const float* effective_n_steps;   /* [n] */
  const float* noise;               /* [n, act] standard normal draws of Normal.rsample() */
  const float* action_scale;        /* [act] policy.py:29-33 */
  float* policy_params;  float* policy_grads;  float* policy_m;  float* policy_v;
  float* q_params;       float* q_grads;       float* q_m;       float* q_v;        /* q1 | q2 */
  float* q_target_params;                                                           /* q1_target | q2_target */
  float* log_alpha;      float* alpha_state;   /* alpha_state [3]: grad, m, v */
  const float* lr;                  /* [1] device */
  int64_t* steps;                   /* [3] device: q, entropy, policy optimiser step counters */
  rlx_fastsac_hparams hp;
  float* metrics;                   /* critic update: q_loss, entropy_loss, q_min, q_max, entropy, critic_grad_norm, entropy_grad_norm (sq);
                                       policy update: policy_loss, alpha, policy_grad_norm */
  void* workspace;
  size_t workspace_bytes;
} rlx_fastsac_update_args;
/* ref: critic_and_entropy_loss_fn + both optimiser steps (fastsac.py:141-238) + the polyak update that follows it (:316-320) */
int rlx_fastsac_critic_update_f32(const rlx_fastsac_update_args* a, void* stream);
/* ref: policy_loss_fn + optimiser step (fastsac.py:106-138) */
int rlx_fastsac_policy_update_f32(const rlx_fastsac_update_args* a, void* stream);
/* ref: policy.get_action (policy.py:78-92); noise NULL: deterministic.  workspace as above */
int rlx_fastsac_act_f32(const rlx_fastsac_dims* d, const float* policy_params, const float* obs, const float* noise, const float* action_scale,
                        float log_std_min, float log_std_max, int64_t n, float* action, void* workspace, size_t workspace_bytes, void* stream);
/* ref: ObservationNormalizer (observation_normalizer.py:20-47): out = (x - mean) / (std + eps); update folds the batch statistics of x
 * into mean / var / std / count (Chan's formula) first when `update` != 0.  count: device int64[1]; workspace: >= 4 * obs * (n / 256 + 2) floats */
int rlx_fastsac_normalize_f32(const float* x, int64_t n, int64_t obs_dim, float* mean, float* var, float* std, int64_t* count, int32_t update,
                              float eps, float* out, float* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------- SAC path -- */
/* ref: ReplayBuffer.sample gathers  (sac/pytorch/replay_buffer.py:32-40):  rows states[idx1, idx2] etc. from the device ring.
 * ring arrays are [capacity_per_env, nr_envs, dim]; idx_t/idx_e [n] int64. */
int rlx_replay_sample_gather_f32(const int64_t* idx_t, const int64_t* idx_e, int64_t n, int64_t nr_envs, int64_t obs_dim,
                                 int64_t act_dim, const float* states, const float* next_states, const float* actions,
                                 const float* rewards, const float* terminations, float* out_states, float* out_next_states,
                                 float* out_actions, float* out_rewards, float* out_terminations, void* stream);

/* ref: Polyak update loop  (sac/pytorch/sac.py:238-242):  target = (1-tau)*target + tau*online over a flat buffer. */
/* ref: FastSAC's device-resident n-step replay, ReplayBuffer.sample  (fastsac/pytorch/replay_buffer.py:34-96), with the two index
 * draws (torch.randint, :37-38 / :63-64) passed in.  Ring arrays are [capacity, nr_envs, dim] (rewards / dones / truncations
 * [capacity, nr_envs]); `size` rows are filled, `pos` is the next write slot.  For sample i starting at (t, e) = (idx_t[i], idx_e[i]):
 *   states, actions: row (t, e);
 *   n_steps == 1:  next_states / rewards / dones / truncations of row (t, e), effective_n_steps = 1   (:36-47);
 *   n_steps  > 1:  rows t+j (mod capacity), j < n_steps; mask_j = prod_{l<j} (1 - dones[t+l]); reward = sum_j r_j * mask_j * discounts[j]
 *                  (summed in j order); effective_n_steps = sum_j mask_j; final row = first done or first truncation among the n
 *                  (the last one if none); next_states / dones / truncations are taken there.  When the ring is full the truncation
 *                  flag of the newest row (pos - 1) reads as 1 unless that row is a done (:50-57).
 * discounts: [n_steps] device array holding gamma ** arange(n_steps) as the caller's framework computes it (bit-exactness of the
 * power function is the caller's).  n_steps <= 32.  workspace: n int64 (the bootstrap row of every sample). */
int rlx_replay_sample_nstep_f32(const int64_t* idx_t, const int64_t* idx_e, int64_t n, int64_t capacity, int64_t nr_envs, int64_t obs_dim,
                                int64_t act_dim, int32_t n_steps, const float* discounts, int64_t size, int64_t pos, const float* states,
                                const float* next_states, const float* actions, const float* rewards, const float* dones,
                                const float* truncations, float* out_states, float* out_next_states, float* out_actions,
                                float* out_rewards, float* out_dones, float* out_truncations, float* out_effective_n_steps, int64_t* workspace,
                                void* stream);
int rlx_polyak_f32(float* target, const float* online, int64_t n, float tau, void* stream);

/* SAC networks (ref: sac/pytorch/policy.py:34-43, q_network.py:27-33), flat fp32 parameter layouts:
 *   policy [Pp]   : W1[H,O] b1[H] W2[H,H] b2[H] Wm[A,H] Ws[A,H] bm[A] bs[A]     (torso ReLU-ReLU, heads mean / log_std)
 *   q      [4][Pq]: W1[H,O+A] b1[H] W2[H,H] b2[H] W3[1,H] b3[1]   in the order q1, q2, q1_target, q2_target */
typedef struct rlx_sac_dims { int32_t obs_dim, act_dim, hidden; float log_std_min, log_std_max; } rlx_sac_dims;
int64_t rlx_sac_policy_param_count(int32_t obs_dim, int32_t act_dim, int32_t hidden);
int64_t rlx_sac_q_param_count(int32_t obs_dim, int32_t act_dim, int32_t hidden);
size_t rlx_sac_workspace_bytes(int32_t obs_dim, int32_t act_dim, int32_t hidden, int64_t batch);

/* ref: Policy.get_action / get_deterministic_action  (sac/pytorch/policy.py:45-73).  eps [n, act] = the standard-normal draws of
 * normal.rsample().  Outputs (nullable): action_tanh [n, act], env_action [n, act] (rescaled to [low, high]), logp [n]. */
int rlx_sac_act_f32(const rlx_sac_dims* d, const float* policy_params, const float* obs, const float* eps, int64_t n, const float* act_low,
                    const float* act_high, int32_t deterministic, float* action_tanh, float* env_action, float* logp, void* workspace,
                    size_t workspace_bytes, void* stream);

/* ref: one full SAC update  (sac.py:219-259): critic_loss_fn (target, twin-Q MSE, Adam over q1 U q2), Polyak, then
 * policy_and_entropy_loss_fn (actor loss through the updated critics, Adam; temperature loss, Adam).
 * metrics [RLX_SAC_NMETRIC]: 0 entropy/alpha 1 entropy/entropy 2 gradients/policy_grad_norm 3 gradients/critic_grad_norm
 *                            4 gradients/entropy_grad_norm 5 loss/q_loss 6 loss/policy_loss 7 loss/entropy_loss 8 q_value/q_value */
#define RLX_SAC_NMETRIC 12
typedef struct rlx_sac_update_args {
  rlx_sac_dims dims;
  int64_t batch;
  float* policy;            /* [Pp] */
  float* q;                 /* [4][Pq] */
  float* log_alpha;         /* [1] */
  const float* states;      /* [batch, obs]   sampled batch (rlx_replay_sample_gather_f32) */
  const float* next_states; /* [batch, obs] */
  const float* actions;     /* [batch, act] */
  const float* rewards;     /* [batch] */
  const float* terminations;/* [batch] */
  const float* eps_next;    /* [batch, act] rsample noise of pi(next_states)  (critic_loss_fn, sac.py:132) */
  const float* eps_cur;     /* [batch, act] rsample noise of pi(states)       (policy_and_entropy_loss_fn, sac.py:93) */
  const float* act_low;     /* [act] */
  const float* act_high;    /* [act] */
  float gamma, tau, target_entropy;
  float adam_beta1, adam_beta2, adam_eps;
  float* g_policy; float* m_policy; float* v_policy;            /* [Pp] each */
  float* g_q; float* m_q; float* v_q;                           /* [2*Pq] each (online nets) */
  float* g_log_alpha; float* m_log_alpha; float* v_log_alpha;   /* [1] each */
  const float* lr;          /* [1] device */
  int64_t* steps;           /* [3] device: Adam step counters of policy, q, log_alpha */
  float* metrics;           /* [RLX_SAC_NMETRIC] device */
  void* workspace;
  size_t workspace_bytes;
} rlx_sac_update_args;
int rlx_sac_update_f32(const rlx_sac_update_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RLX_B200_H */

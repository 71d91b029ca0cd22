// PPO MLP pair: forward (rollout / eval / bootstrap values) and the minibatch forward+backward+optimiser step.
//
// Network (ref: policy.py:45-52, critic.py:29-35): two independent 3-layer tanh MLPs on the same input.  They are
// evaluated as ONE pipeline over a fused activation layout [rows, 2H] = [policy half | critic half]:
//   layer 1   one GEMM  [rows, obs] x [2H, obs]^T          (shared A operand, SURVEY §8 a11)
//   layer 2   one batched GEMM (batch = 2 nets) [rows, H] x [H, H]^T on the two halves
//   layer 3   skinny head kernels (ppo_head.cuh) fused with sampling / loss
// Backward mirrors it: head -> (dW3 | dZ2) -> batched dW2 (split over rows) -> batched dH1*tanh' -> dW1 (split over rows),
// no dX for layer 1.  Bias gradients fall out of the dW GEMMs as row sums of the dZ operand.
#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_dispatch.cuh"
#include "ppo_head.cuh"
#include "ppo_head_mma.cuh"
#include "ppo_optim.cuh"

namespace rlx {

static bool use_tc(const rlx_ppo_dims& d) { return g_gemm_engine == 1 && tc_supported(d); }
extern bool g_tc_pair_force;  // gemm_tc.cu
}  // namespace rlx
// comm.cu: all-reduce of [gradient | metrics]; *nblk_out > 0 when the kernel also wrote that many (policy, critic) sum-of-squares partial pairs
int comm_allreduce_ppo(rlx_comm* c, float* out, int64_t n, const rlx_ppo_dims& d, float* norm_partials, long long* step_count, void* stream, int* nblk_out);
namespace rlx {

struct Splits {
  int splits, kchunk;
};
// choose a split-K factor for a [M' x N'] output reduced over `rows`: ~2 CTAs per SM for the SIMT engine, one persistent
// CTA per SM for the tcgen05 engine (k-chunks are multiples of 32 there: one 128-byte swizzle row of fp32)
// pair_bn > 0: the GEMM runs on CTA pairs (256 x pair_bn tiles, sm_count / 2 pairs)
static Splits choose_splits(long long rows, int out_m, int out_n, int batch, bool tc, int pair_bn = 0) {
  if (tc) {
    // persistent kernel, one CTA per SM: pick the split count whose tile total fills whole waves of SMs.  The tensor core accumulates
    // with round-toward-zero, so each TMEM accumulation chain is also kept <= 1024 rows (128 MMAs); the long part of the
    // reduction happens in the fp32 grad_reduce kernel (profiles/tc_accuracy_probe.py).
    const int bn = pair_bn > 0 ? pair_bn : ((out_n % 256 == 0) ? 256 : 128);
    const long long tiles = ceil_div(out_m, pair_bn > 0 ? 256 : 128) * ceil_div(out_n, bn) * batch;
    const long long smin = std::max<long long>(1, ceil_div(rows, 1024)), smax = std::max<long long>(smin, std::min<long long>(smin + 64, rows / 64));
    const long long sms = pair_bn > 0 ? sm_count() / 2 : sm_count();
    long long best = smin;
    double best_fill = -1.0;
    for (long long s = smin; s <= smax; ++s) {
      const long long t = tiles * s;
      const double fill = (double)t / (double)(ceil_div(t, sms) * sms);
      if (fill > best_fill + 0.02) { best_fill = fill; best = s; }
    }
    long long kchunk = std::max<long long>(32, ceil_div(ceil_div(rows, best), 32) * 32);
    return Splits{(int)ceil_div(rows, kchunk), (int)kchunk};
  }
  const long long tiles = ceil_div(out_m, GBM) * ceil_div(out_n, GBN) * batch;
  const long long target = (long long)sm_count() * 2;
  long long s = std::max<long long>(1, target / std::max<long long>(tiles, 1));
  s = std::min<long long>(s, std::max<long long>(1, rows / 256));  // at least 256 rows per split
  long long kchunk = std::max<long long>(8, ceil_div(ceil_div(rows, s), 8) * 8);
  return Splits{(int)ceil_div(rows, kchunk), (int)kchunk};
}

// bf16-autocast mode: dst = bf16-rounded copy of src (what `.to(torch.bfloat16)` of autocast's Linear does to the input and to the
// weights), except the [keep_lo, keep_hi) range, which is copied as is (logstd: an fp32 parameter no autocast op touches)
__global__ void __launch_bounds__(256) round_bf16_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n, long long keep_lo,
                                                         long long keep_hi) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float x = src[i];
    dst[i] = (i >= keep_lo && i < keep_hi) ? x : bf16r(x);
  }
}
static int launch_round_bf16(const float* src, float* dst, long long n, long long keep_lo, long long keep_hi, cudaStream_t st) {
  if (n <= 0) return RLX_OK;
  const unsigned grid = (unsigned)std::min<long long>(ceil_div(n, 256), (long long)sm_count() * 8);
  RLX_LAUNCH_C(KC_OTHER, 0, 8.0 * n, round_bf16_kernel, grid, 256, 0, st, src, dst, n, keep_lo, keep_hi);
  return RLX_OK;
}

struct FwdPlan {
  size_t off_H1, off_H2, off_P, off_X, total;
};
static FwdPlan plan_forward(const rlx_ppo_dims& d, long long n) {
  FwdPlan P;
  size_t o = 0;
  const size_t act_bytes = align_up((size_t)n * 2 * d.hidden * sizeof(float), 256);
  P.off_H1 = o; o += act_bytes;
  P.off_H2 = o; o += act_bytes;
  // bf16-autocast mode: rounded copies of the parameters and of the observations (always planned: the mode is a run-time switch)
  P.off_P = o; o += align_up((size_t)make_layout(d).total() * sizeof(float), 256);
  P.off_X = o; o += align_up((size_t)n * d.obs_dim * sizeof(float), 256);
  P.total = o;
  return P;
}

constexpr int kHeadWgradRows = 64;

struct TrainPlan {
  size_t off_H1, off_H2, off_dZ2, off_dZ1, off_dhead, off_headpart, off_part1, off_rs1, off_part2, off_part3, off_norm, off_barrier, off_P, off_X, off_ratio, total;
  int max_s1, max_s2, max_s3;
  int head_blocks, wgrad_chunks, norm_blocks, head_npart;
};
static int head_grid(long long m) { return (int)std::min<long long>(ceil_div(m, 16), (long long)sm_count() * 2); }

static TrainPlan plan_train(const rlx_ppo_dims& d, long long m) {
  TrainPlan P;
  const long long H = d.hidden, O = d.obs_dim, A = d.act_dim;
  P.max_s1 = std::max(choose_splits(m, (int)(2 * H), (int)O, 1, false).splits, choose_splits(m, (int)O + 1, (int)(2 * H), 1, true).splits);
  P.max_s1 = std::max(P.max_s1, choose_splits(m, (int)(2 * H), (int)O + 1, 1, true, 192).splits);  // CTA-pair orientation of dW1
  P.max_s2 = std::max(choose_splits(m, (int)H, (int)H, 2, false).splits, choose_splits(m, (int)H, (int)H, 2, true).splits);
  P.max_s2 = std::max(P.max_s2, choose_splits(m, (int)H, (int)H, 2, true, 256).splits);
  P.head_blocks = head_grid(m);
  P.head_npart = (int)(2 * A + 5 + 2 * H);
  P.wgrad_chunks = (int)ceil_div(m, kHeadWgradRows);
  // one (policy, critic) partial pair per CTA of whichever kernel leaves the squared norms behind: the <= SM-count grid of the exchange
  // kernel, the 64 CTAs of ppo_grad_sumsq_kernel, or the gradient-assembly grid (one CTA per 256 flat elements + one per 8 "tall" elements)
  P.norm_blocks = (int)std::max<long long>(std::max(64, sm_count()), ceil_div(make_layout(d).total(), 256) + ceil_div(2 * H + 2 * A + 1 + (A + 1) * H, 8) + 8);
  size_t o = 0;
  auto take = [&](size_t& off, size_t nfloats) {
    off = o;
    o += align_up(nfloats * sizeof(float), 256);
  };
  take(P.off_H1, (size_t)m * 2 * H);
  take(P.off_H2, (size_t)m * 2 * H);
  take(P.off_dZ2, (size_t)m * 2 * H);
  take(P.off_dZ1, (size_t)m * 2 * H);
  take(P.off_dhead, (size_t)m * (ceil_div(A + 1, 4) * 4));
  take(P.off_headpart, (size_t)P.head_blocks * P.head_npart);
  take(P.off_part1, (size_t)P.max_s1 * 2 * H * O);
  take(P.off_rs1, (size_t)P.max_s1 * 2 * H);
  take(P.off_part2, (size_t)P.max_s2 * 2 * H * H);
  const size_t dh_ld_plan = (size_t)(ceil_div(A + 1, 4) * 4);
  P.max_s3 = choose_splits(m, (int)dh_ld_plan, (int)H, 2, true).splits;
  take(P.off_part3, std::max<size_t>((size_t)P.wgrad_chunks * (A + 1) * H, (size_t)P.max_s3 * 2 * dh_ld_plan * H));
  take(P.off_norm, (size_t)P.norm_blocks * 2);
  take(P.off_barrier, 64);
  take(P.off_P, (size_t)make_layout(d).total());                          // bf16-autocast mode: rounded parameter copy
  take(P.off_X, (size_t)m * (size_t)(ceil_div(O + 1, 4) * 4));             // ... and rounded copy of the minibatch states (pitch <= obs + 4)
  take(P.off_ratio, (size_t)m);                                           // ESPO median: |ratio - 1| per row
  P.total = o;
  return P;
}

template <typename T>
static T* ws_ptr(void* ws, size_t off) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(ws) + off);
}

static size_t head_smem_bytes(const rlx_ppo_dims& d, bool train) {
  size_t s = ((size_t)d.act_dim * d.hidden + d.hidden) * sizeof(float);
  if (train) s += (size_t)8 * (2 * d.act_dim + 5 + 2 * d.hidden) * sizeof(float);
  return s;
}

// hidden layers: H1 = tanh(X W1cat^T + b1cat), H2 = tanh(H1 (blockdiag W2)^T + b2cat).  ldx = row pitch of X.
static int mlp_hidden_forward(const rlx_ppo_dims& d, const PpoLayout& L, const float* params, const float* X, long long ldx, long long rows,
                              float* H1, float* H2, cudaStream_t stream, int bf16 = 0) {
  const int H = L.H;
  const bool tc = use_tc(d);
  GemmP g{};
  g.A = X; g.B = params + L.off[W1P]; g.C = H1; g.bias = params + L.off[B1P];
  g.M = (int)rows; g.N = 2 * H; g.K = L.obs;
  g.lda = (int)ldx; g.ldb = L.obs; g.ldc = 2 * H;
  g.splits = 1; g.kchunk = (int)(ceil_div(L.obs, 8) * 8);
  g.bf16 = bf16;
  const int pair_fwd = tc ? tc_pair_fwd_bn() : 0;
  int rc = run_gemm<true, true, EPI_BIAS_TANH>(tc, g, 1, stream, KC_GEMM_FWD, rows, 2 * H, pair_fwd);
  if (rc) return rc;
  GemmP g2{};
  g2.A = H1; g2.B = params + L.off[W2P]; g2.C = H2; g2.bias = params + L.off[B2P];
  g2.M = (int)rows; g2.N = H; g2.K = H;
  g2.lda = 2 * H; g2.ldb = H; g2.ldc = 2 * H;
  g2.sA = H; g2.sB = (long long)H * H; g2.sC = H; g2.sBias = H;
  g2.splits = 1; g2.kchunk = (int)(ceil_div(H, 8) * 8);
  g2.bf16 = bf16;
  return run_gemm<true, true, EPI_BIAS_TANH>(tc, g2, 2, stream, KC_GEMM_FWD, rows, H, pair_fwd);
}

#define RLX_DISPATCH_NCH_1(CLS, FLOPS, BYTES, KERNEL, NCH_, BF_, grid, block, smem, stream, arg)                                    \
  do {                                                                                                                              \
    RLX_CHECK_CUDA(cudaFuncSetAttribute(KERNEL<NCH_, BF_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)));              \
    RLX_LAUNCH_C(CLS, FLOPS, BYTES, (KERNEL<NCH_, BF_>), grid, block, smem, stream, arg);                                           \
  } while (0)
#define RLX_DISPATCH_NCH_B(CLS, FLOPS, BYTES, H, KERNEL, BF_, grid, block, smem, stream, arg)                                       \
  do {                                                                                                                              \
    const int _nch = (int)ceil_div((H), 32);                                                                                        \
    if (_nch <= 2) RLX_DISPATCH_NCH_1(CLS, FLOPS, BYTES, KERNEL, 2, BF_, grid, block, smem, stream, arg);                           \
    else if (_nch <= 4) RLX_DISPATCH_NCH_1(CLS, FLOPS, BYTES, KERNEL, 4, BF_, grid, block, smem, stream, arg);                      \
    else if (_nch <= 8) RLX_DISPATCH_NCH_1(CLS, FLOPS, BYTES, KERNEL, 8, BF_, grid, block, smem, stream, arg);                      \
    else if (_nch <= 16) RLX_DISPATCH_NCH_1(CLS, FLOPS, BYTES, KERNEL, 16, BF_, grid, block, smem, stream, arg);                    \
    else RLX_DISPATCH_NCH_1(CLS, FLOPS, BYTES, KERNEL, 32, BF_, grid, block, smem, stream, arg);                                    \
  } while (0)
// bf16-autocast mode selects the kernels compiled with the bf16 roundings (h.bf16 is set by the callers)
#define RLX_DISPATCH_NCH(CLS, FLOPS, BYTES, H, KERNEL, grid, block, smem, stream, arg)                                              \
  do {                                                                                                                              \
    if ((arg).bf16) RLX_DISPATCH_NCH_B(CLS, FLOPS, BYTES, H, KERNEL, true, grid, block, smem, stream, arg);                         \
    else RLX_DISPATCH_NCH_B(CLS, FLOPS, BYTES, H, KERNEL, false, grid, block, smem, stream, arg);                                   \
  } while (0)

static bool head_dims_ok(const rlx_ppo_dims& d) {
  return dims_ok(d) && d.hidden <= 1024 && head_smem_bytes(d, true) <= 200 * 1024;
}

static int g_head_engine = 0;  // 0 fused SIMT kernel, 2 fused mma.sync kernel (rlx_set_head_engine)

static void fill_head_common(HeadP& h, const PpoLayout& L, const float* params, const float* H2, long long rows) {
  h.M = (int)rows; h.H = L.H; h.act = L.act;
  h.H2 = H2;
  h.W3p = params + L.off[W3P]; h.W3c = params + L.off[W3C];
  h.b3p = params + L.off[B3P]; h.b3c = params + L.off[B3C];
  h.logstd = params + L.off[LOGSTD];
}

}  // namespace rlx

using namespace rlx;

// ------------------------------------------------------------------------------------------------ forward API
extern "C" size_t rlx_ppo_forward_workspace_bytes(const rlx_ppo_dims* d, int64_t n) {
  if (d == nullptr || !head_dims_ok(*d) || n < 0) return 0;
  return plan_forward(*d, n).total;
}

extern "C" int rlx_ppo_forward_f32(const rlx_ppo_forward_args* a, void* stream) {
  RLX_CHECK_ARG(a != nullptr, "args is null");
  RLX_CHECK_ARG(head_dims_ok(a->dims), "unsupported dims (act <= 64, hidden <= 1024)");
  RLX_CHECK_ARG(a->n >= 0 && a->n < (1LL << 31), "bad row count");
  if (a->n == 0) return RLX_OK;
  RLX_CHECK_ARG(a->params && a->obs, "params / obs is null");
  RLX_CHECK_ARG(!a->env_action || !a->clip_rescale || (a->act_low && a->act_high), "action bounds required for clip_rescale");
  const FwdPlan P = plan_forward(a->dims, a->n);
  if (a->workspace == nullptr || a->workspace_bytes < P.total) {
    set_error("rlx_ppo_forward_f32: workspace too small (%zu < %zu)", a->workspace_bytes, P.total);
    return RLX_ERR_WORKSPACE;
  }
  const PpoLayout L = make_layout(a->dims);
  float* H1 = ws_ptr<float>(a->workspace, P.off_H1);
  float* H2 = ws_ptr<float>(a->workspace, P.off_H2);
  cudaStream_t st = (cudaStream_t)stream;
  const int bf16 = g_autocast_bf16;
  const float* params = a->params;
  const float* obs = a->obs;
  int rc;
  if (bf16) {
    float* pr = ws_ptr<float>(a->workspace, P.off_P);
    float* xr = ws_ptr<float>(a->workspace, P.off_X);
    rc = launch_round_bf16(a->params, pr, L.total(), L.off[LOGSTD], L.off[LOGSTD + 1], st);
    if (rc) return rc;
    rc = launch_round_bf16(a->obs, xr, a->n * (long long)L.obs, 0, 0, st);
    if (rc) return rc;
    params = pr;
    obs = xr;
  }
  rc = mlp_hidden_forward(a->dims, L, params, obs, a->dims.obs_dim, a->n, H1, H2, st, bf16);
  if (rc) return rc;
  HeadP h{};
  fill_head_common(h, L, params, H2, a->n);
  h.bf16 = bf16;
  h.noise = a->noise; h.seed = a->rng_seed; h.offset = a->rng_offset;
  h.act_low = a->act_low; h.act_high = a->act_high;
  h.clip_rescale = a->clip_rescale; h.deterministic = a->deterministic;
  h.action = a->action; h.env_action = a->env_action; h.logp_out = a->logp; h.value_out = a->value;
  const size_t smem = head_smem_bytes(a->dims, false);
  const int grid = head_grid(a->n);
  RLX_DISPATCH_NCH(KC_HEAD_ROLLOUT, 2.0 * a->n * L.H * (L.act + 1), 4.0 * a->n * (2.0 * L.H + 3.0 * L.act + 2), L.H, ppo_head_rollout_kernel, grid, 256, smem, st, h);
  return RLX_OK;
}

extern "C" int rlx_critic_forward_f32(const rlx_ppo_dims* d, const float* params, const float* obs, int64_t n, float* value,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  RLX_CHECK_ARG(d != nullptr, "dims is null");
  rlx_ppo_forward_args a{};
  a.dims = *d; a.n = n; a.params = params; a.obs = obs; a.deterministic = 1; a.value = value;
  a.workspace = workspace; a.workspace_bytes = workspace_bytes;
  return rlx_ppo_forward_f32(&a, stream);
}

// ---------------------------------------------------------------------------------------- minibatch update API
extern "C" size_t rlx_ppo_minibatch_workspace_bytes(const rlx_ppo_dims* d, int64_t m) {
  if (d == nullptr || !head_dims_ok(*d) || m < 0) return 0;
  return plan_train(*d, std::max<int64_t>(m, 1)).total;
}

static int check_mb_args(const rlx_ppo_minibatch_args* a, bool need_data) {
  RLX_CHECK_ARG(a != nullptr, "args is null");
  RLX_CHECK_ARG(head_dims_ok(a->dims), "unsupported dims (act <= 64, hidden <= 1024)");
  RLX_CHECK_ARG(a->m >= 0 && a->m < (1LL << 31) && a->m_global >= 1, "bad minibatch size");
  RLX_CHECK_ARG(a->params && a->grads, "params / grads is null");
  if (need_data && a->m > 0) {
    RLX_CHECK_ARG(a->states && a->actions && a->log_probs && a->advantages && a->returns && a->adv_stats, "null minibatch tensor");
  }
  const TrainPlan P = plan_train(a->dims, std::max<int64_t>(a->m, 1));
  if (a->workspace == nullptr || a->workspace_bytes < P.total) {
    set_error("rlx_ppo_minibatch: workspace too small (%zu < %zu)", a->workspace_bytes, P.total);
    return RLX_ERR_WORKSPACE;
  }
  return RLX_OK;
}

static long long tall_elements(const GradReduceP& r) {
  long long tall = 0;
  for (int gi = 0; gi < kNumGroups; ++gi)
    if (r.g[gi].nsplit > kTallSplit) tall += r.g[gi].len;
  return tall;
}
static double partial_bytes(const GradReduceP& r) {
  double b = 0;
  for (int gi = 0; gi < kNumGroups; ++gi) b += 4.0 * r.g[gi].nsplit * r.g[gi].len;
  return b;
}
static int launch_grad_reduce(const GradReduceP& r, cudaStream_t st) {
  const int flat_blocks = (int)ceil_div(r.total, 256);
  const int tall_blocks = (int)ceil_div(tall_elements(r), 8);  // 8 warps per CTA, one element per warp
  RLX_LAUNCH_C(KC_GRAD_REDUCE, 0, partial_bytes(r) + 4.0 * r.total, ppo_grad_reduce_kernel, (unsigned)(flat_blocks + tall_blocks), 256, 0, st, r, flat_blocks);
  return RLX_OK;
}

// `fuse_norms`: the assembly kernel also leaves the two squared clip norms in the workspace (off_barrier + 16 bytes) and bumps Adam's
// step counter, so that clip + Adam can follow without the separate sum-of-squares launch.
static int minibatch_fwdbwd(const rlx_ppo_minibatch_args* a, void* stream, bool fuse_norms = false);

extern "C" int rlx_ppo_minibatch_fwdbwd_f32(const rlx_ppo_minibatch_args* a, void* stream) { return minibatch_fwdbwd(a, stream); }

static int minibatch_fwdbwd(const rlx_ppo_minibatch_args* a, void* stream, bool fuse_norms) {
  int rc = check_mb_args(a, true);
  if (rc) return rc;
  const rlx_ppo_dims& d = a->dims;
  const PpoLayout L = make_layout(d);
  const long long m = a->m;
  const int H = L.H, O = L.obs, A = L.act;
  const long long ldx = a->states_ld > 0 ? a->states_ld : O;
  RLX_CHECK_ARG(ldx >= O, "states_ld smaller than obs_dim");
  RLX_CHECK_ARG(!a->states_ones_col || ldx > O, "states_ones_col needs states_ld > obs_dim");
  const bool tc = use_tc(d);
  const TrainPlan P = plan_train(d, std::max<long long>(m, 1));
  cudaStream_t st = (cudaStream_t)stream;
  void* ws = a->workspace;
  float* H1 = ws_ptr<float>(ws, P.off_H1);
  float* H2 = ws_ptr<float>(ws, P.off_H2);
  float* dZ2 = ws_ptr<float>(ws, P.off_dZ2);
  float* dZ1 = ws_ptr<float>(ws, P.off_dZ1);
  float* dhead = ws_ptr<float>(ws, P.off_dhead);
  float* headpart = ws_ptr<float>(ws, P.off_headpart);
  float* part1 = ws_ptr<float>(ws, P.off_part1);
  float* rs1 = ws_ptr<float>(ws, P.off_rs1);
  float* part2 = ws_ptr<float>(ws, P.off_part2);
  float* part3 = ws_ptr<float>(ws, P.off_part3);
  const float inv_mg = 1.f / (float)a->m_global;
  const int npart = P.head_npart;

  int head_blocks = 0, wgrad_chunks = 0, s1 = 0, s2 = 0, w3_nsplit = 0;
  long long w3_stride = (long long)(A + 1) * H, w3c_off = (long long)A * H;
  const int bf16 = g_autocast_bf16;
  const float* params = a->params;   // bf16 mode: the rounded copies below (what autocast's casts hand to every Linear)
  const float* states = a->states;
  if (m > 0) {
    if (bf16) {
      RLX_CHECK_ARG(ldx <= (long long)(ceil_div(O + 1, 4) * 4), "bf16 mode: states_ld larger than the planned rounded copy");
      float* pr = ws_ptr<float>(ws, P.off_P);
      float* xr = ws_ptr<float>(ws, P.off_X);
      rc = launch_round_bf16(a->params, pr, L.total(), L.off[LOGSTD], L.off[LOGSTD + 1], st);
      if (rc) return rc;
      rc = launch_round_bf16(a->states, xr, m * ldx, 0, 0, st);
      if (rc) return rc;
      params = pr;
      states = xr;
    }
    // ---- forward hidden layers
    rc = mlp_hidden_forward(d, L, params, states, ldx, m, H1, H2, st, bf16);
    if (rc) return rc;
    // ---- head: loss + dZ2 + dhead + block partials (incl. db2 = column sums of dZ2)
    HeadP h{};
    fill_head_common(h, L, params, H2, m);
    h.bf16 = bf16;
    h.actions = a->actions; h.logp_old = a->log_probs; h.adv = a->advantages; h.ret = a->returns; h.adv_stats = a->adv_stats;
    h.inv_mg = inv_mg; h.clip_range = a->hp.clip_range; h.critic_coef = a->hp.critic_coef;
    h.ratio_delta_metric = a->hp.ratio_delta_metric != 0.f ? 1 : 0;
    const bool want_median = a->hp.ratio_delta_metric == 2.f;  // ESPO delta_calc_operator = median (espo.py:59-60)
    h.ratio_abs = want_median ? ws_ptr<float>(ws, P.off_ratio) : nullptr;
    h.dZ2 = dZ2; h.dhead = dhead; h.block_partials = headpart;
    head_blocks = P.head_blocks;
    const size_t smem = head_smem_bytes(d, true);
    const int dh_ld = (int)(ceil_div(A + 1, 4) * 4);
    const bool fast_head = (A <= 31) && (H % 2 == 0) && (H <= 1024);
    const double head_flops = 4.0 * m * H * (A + 1), head_bytes = 4.0 * m * (4.0 * H + 2.0 * A + 5);
    if (fast_head) {
      HeadTrain2Extra ex{dh_ld};
      const bool vec_head = (H == 128 || H == 256 || H == 512);
      // fused head on the warp-level tensor path (ppo_head_mma.cuh): fp32 mode, <= 4 n-tiles of 8 head columns
      const int nt4 = (int)ceil_div(dh_ld, 8);
      const size_t smem4 = head4_smem_floats(H, A, nt4) * sizeof(float);
      const bool mma_head = vec_head && g_head_engine == 2 && !bf16 && nt4 <= 4 && smem4 <= 220 * 1024;
      if (mma_head) {
        head_blocks = (int)std::min<long long>(ceil_div(m, 16 * kHead4RowTiles), (long long)P.head_blocks);
#define RLX_HEAD4(H_, NT_)                                                                                                          \
  do {                                                                                                                              \
    RLX_CHECK_CUDA(cudaFuncSetAttribute(ppo_head_train4_kernel<H_, NT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4)); \
    RLX_LAUNCH_C(KC_HEAD_TRAIN, head_flops, head_bytes, (ppo_head_train4_kernel<H_, NT_>), head_blocks, 256, smem4, st, h, ex);     \
  } while (0)
#define RLX_HEAD4_NT(H_)              \
  do {                                \
    if (nt4 == 1) RLX_HEAD4(H_, 1);   \
    else if (nt4 == 2) RLX_HEAD4(H_, 2); \
    else if (nt4 == 3) RLX_HEAD4(H_, 3); \
    else RLX_HEAD4(H_, 4);            \
  } while (0)
        if (H == 128) RLX_HEAD4_NT(128);
        else if (H == 256) RLX_HEAD4_NT(256);
        else RLX_HEAD4_NT(512);
#undef RLX_HEAD4_NT
#undef RLX_HEAD4
      } else if (vec_head) {
#define RLX_HEAD3_B(H_, AM_, BF_)                                                                                                     \
  do {                                                                                                                                \
    RLX_CHECK_CUDA(cudaFuncSetAttribute(ppo_head_train3_kernel<H_, AM_, BF_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    RLX_LAUNCH_C(KC_HEAD_TRAIN, head_flops, head_bytes, (ppo_head_train3_kernel<H_, AM_, BF_>), head_blocks, 256, smem, st, h, ex);    \
  } while (0)
#define RLX_HEAD3(H_, AM_)                          \
  do {                                              \
    if (bf16) RLX_HEAD3_B(H_, AM_, true);           \
    else RLX_HEAD3_B(H_, AM_, false);               \
  } while (0)
#define RLX_HEAD3_ACT(H_)                      \
  do {                                         \
    if (A <= 8) RLX_HEAD3(H_, 8);              \
    else if (A <= 16) RLX_HEAD3(H_, 16);       \
    else if (A <= 24) RLX_HEAD3(H_, 24);       \
    else RLX_HEAD3(H_, 31);                    \
  } while (0)
        if (H == 128) RLX_HEAD3_ACT(128);
        else if (H == 256) RLX_HEAD3_ACT(256);
        else RLX_HEAD3_ACT(512);
#undef RLX_HEAD3_ACT
#undef RLX_HEAD3
#undef RLX_HEAD3_B
      } else {
        const int nch = (int)ceil_div(H, 32);
#define RLX_HEAD2_B(NCH_, AM_, BF_)                                                                                                   \
  do {                                                                                                                                \
    RLX_CHECK_CUDA(cudaFuncSetAttribute(ppo_head_train2_kernel<NCH_, AM_, BF_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    RLX_LAUNCH_C(KC_HEAD_TRAIN, head_flops, head_bytes, (ppo_head_train2_kernel<NCH_, AM_, BF_>), head_blocks, 256, smem, st, h, ex);  \
  } while (0)
#define RLX_HEAD2(NCH_, AM_)                        \
  do {                                              \
    if (bf16) RLX_HEAD2_B(NCH_, AM_, true);         \
    else RLX_HEAD2_B(NCH_, AM_, false);             \
  } while (0)
#define RLX_HEAD2_ACT(NCH_)                         \
  do {                                              \
    if (A <= 8) RLX_HEAD2(NCH_, 8);                 \
    else if (A <= 16) RLX_HEAD2(NCH_, 16);          \
    else if (A <= 24) RLX_HEAD2(NCH_, 24);          \
    else RLX_HEAD2(NCH_, 31);                       \
  } while (0)
        if (nch <= 2) RLX_HEAD2_ACT(2);
        else if (nch <= 4) RLX_HEAD2_ACT(4);
        else if (nch <= 8) RLX_HEAD2_ACT(8);
        else if (nch <= 16) RLX_HEAD2_ACT(16);
        else RLX_HEAD2_ACT(32);
#undef RLX_HEAD2_ACT
#undef RLX_HEAD2
#undef RLX_HEAD2_B
      }
      // ---- dW3 = dhead^T [act+1, m] . H2 [m, 2H]
      bool w3_done = false;
      if (tc) {
        // tensor cores: one MN-major GEMM per net half (batch 2); the act+1 (padded to dh_ld) gradient columns are the M side
        const Splits S3 = choose_splits(m, dh_ld, H, 2, true);
        GemmP g3{};
        g3.A = dhead; g3.B = H2; g3.C = part3;
        g3.M = dh_ld; g3.N = H; g3.K = (int)m;
        g3.lda = dh_ld; g3.ldb = 2 * H; g3.ldc = H;
        g3.sA = 0; g3.sB = H; g3.sC = (long long)dh_ld * H;
        g3.splits = S3.splits; g3.kchunk = S3.kchunk; g3.sSplitC = 2LL * dh_ld * H;
        g3.bf16 = bf16;
        rc = tc_gemm(g3, false, false, TC_NONE, 2, KC_HEAD_WGRAD, m, m, 0, nullptr, 0, 0, st);
        if (rc == RLX_OK) {
          w3_done = true;
          w3_nsplit = S3.splits;
          w3_stride = 2LL * dh_ld * H;
          w3c_off = (long long)dh_ld * H + (long long)A * H;  // net 1 (critic half of H2), row `act` of its [dh_ld, H] block
        } else if (rc != RLX_ERR_UNSUPPORTED) {
          return rc;
        }
      }
      if (!w3_done) {
        // SIMT: one thread per (policy, critic) column pair, 64 rows per CTA
        HeadWgrad2P w{(int)m, H, A, dh_ld, kHeadWgradRows, H2, dhead, part3};
        wgrad_chunks = (int)ceil_div(m, kHeadWgradRows);
        const unsigned wthreads = (unsigned)(ceil_div(H, 32) * 32);
        const size_t wsmem = (size_t)kHeadWgradRows * dh_ld * sizeof(float);
        const double wflops = 2.0 * m * H * (A + 1), wbytes = 4.0 * m * (2.0 * H + A + 1);
        if (A + 1 <= 4) RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<4>, wgrad_chunks, wthreads, wsmem, st, w);
        else if (A + 1 <= 8) RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<8>, wgrad_chunks, wthreads, wsmem, st, w);
        else if (A + 1 <= 12) RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<12>, wgrad_chunks, wthreads, wsmem, st, w);
        else if (A + 1 <= 16) RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<16>, wgrad_chunks, wthreads, wsmem, st, w);
        else if (A + 1 <= 20) RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<20>, wgrad_chunks, wthreads, wsmem, st, w);
        else if (A + 1 <= 24) RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<24>, wgrad_chunks, wthreads, wsmem, st, w);
        else RLX_LAUNCH_C(KC_HEAD_WGRAD, wflops, wbytes, ppo_head_wgrad3_kernel<32>, wgrad_chunks, wthreads, wsmem, st, w);
        w3_nsplit = wgrad_chunks;
      }
    } else {
      RLX_DISPATCH_NCH(KC_HEAD_TRAIN, head_flops, head_bytes, H, ppo_head_train_kernel, head_blocks, 256, smem, st, h);
      // ---- dW3 (thread per column, chunked over rows)
      HeadWgradP w{(int)m, H, A, kHeadWgradRows, H2, dhead, part3};
      wgrad_chunks = (int)ceil_div(m, kHeadWgradRows);
      dim3 wg((unsigned)wgrad_chunks, (unsigned)ceil_div(2 * H, 256));
      const size_t wsmem = (size_t)kHeadWgradRows * (A + 1) * sizeof(float);
      if (A <= 8) {
        RLX_LAUNCH_C(KC_HEAD_WGRAD, 2.0 * m * H * (A + 1), 4.0 * m * (2.0 * H + A + 1), ppo_head_wgrad_kernel<8>, wg, 256, wsmem, st, w);
      } else if (A <= 32) {
        RLX_LAUNCH_C(KC_HEAD_WGRAD, 2.0 * m * H * (A + 1), 4.0 * m * (2.0 * H + A + 1), ppo_head_wgrad_kernel<32>, wg, 256, wsmem, st, w);
      } else {
        RLX_CHECK_CUDA(cudaFuncSetAttribute(ppo_head_wgrad_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        RLX_LAUNCH_C(KC_HEAD_WGRAD, 2.0 * m * H * (A + 1), 4.0 * m * (2.0 * H + A + 1), ppo_head_wgrad_kernel<64>, wg, 256, wsmem, st, w);
      }
      w3_nsplit = wgrad_chunks;
    }
    // ---- dW2 : part2[split][net][o][i] = sum_rows dZ2[r, net*H+o] * H1[r, net*H+i]   (db2 comes from the head kernel)
    const int pair_dw = (tc && tc_pair_mode() >= 1 && H % 256 == 0) ? 256 : 0;
    const Splits S2 = choose_splits(m, H, H, 2, tc, pair_dw);
    s2 = S2.splits;
    GemmP g{};
    g.A = dZ2; g.B = H1; g.C = part2;
    g.M = H; g.N = H; g.K = (int)m;
    g.lda = 2 * H; g.ldb = 2 * H; g.ldc = H;
    g.sA = H; g.sB = H; g.sC = (long long)H * H;
    g.splits = S2.splits; g.kchunk = S2.kchunk; g.sSplitC = 2LL * H * H;
    g.bf16 = bf16;
    rc = run_gemm<false, false, EPI_NONE>(tc, g, 2, st, KC_GEMM_DW, m, m, pair_dw);
    if (rc) return rc;
    // ---- dZ1 = (dZ2 @ W2) * (1 - H1^2)   per net
    GemmP gd{};
    gd.A = dZ2; gd.B = params + L.off[W2P]; gd.C = dZ1; gd.aux = H1;
    gd.bf16 = bf16;
    gd.M = (int)m; gd.N = H; gd.K = H;
    gd.lda = 2 * H; gd.ldb = H; gd.ldc = 2 * H; gd.ldaux = 2 * H;
    gd.sA = H; gd.sB = (long long)H * H; gd.sC = H; gd.sAux = H;
    gd.splits = 1; gd.kchunk = (int)(ceil_div(H, 8) * 8);
    rc = run_gemm<true, false, EPI_DTANH>(tc, gd, 2, st, KC_GEMM_DX, m, H, tc ? tc_pair_fwd_bn() : 0);
    if (rc) return rc;
    // ---- dW1cat | db1cat : part1[split][o][i] = sum_rows dZ1[r, o] * X[r, i];  db1[o] = sum_rows dZ1[r, o]
    GemmP g1{};
    g1.A = dZ1; g1.B = states; g1.C = part1;
    g1.bf16 = bf16;
    g1.M = 2 * H; g1.N = O; g1.K = (int)m;
    g1.lda = 2 * H; g1.ldb = (int)ldx; g1.ldc = O;
    bool done = false;
    if (tc && a->states_ones_col && tc_pair_mode() >= 1 && (2 * H) % 256 == 0) {
      // CTA pairs, NOT transposed: M = 2H (whole 256-row pair tiles), N = O + 1 in 192-wide tiles (377 -> 2 x 192); the constant-one
      // column of X lands in output column O, which the epilogue diverts into rs1 (= db1)
      const Splits S1 = choose_splits(m, 2 * H, O + 1, 1, true, 192);
      GemmP gp = g1;
      gp.N = O + 1;
      gp.splits = S1.splits; gp.kchunk = S1.kchunk; gp.sSplitC = 2LL * H * O;
      rc = tc_gemm(gp, false, false, TC_NONE, 1, KC_GEMM_DW, m, m, O, rs1, 0, 2LL * H, st, 192);
      if (rc == RLX_OK) {
        done = true;
        s1 = S1.splits;
      } else if (rc != RLX_ERR_UNSUPPORTED) {
        return rc;
      }
    }
    if (!done && tc && a->states_ones_col) {
      // tensor-core path, computed TRANSPOSED: C^T[i, o] = sum_r X_aug[r, i] dZ1[r, o] with M = O+1 (the constant-one column of X
      // makes db1 the last output row) and N = 2H = full 256-wide tiles; the epilogue stores C^T transposed back into [o][i].
      const Splits S1 = choose_splits(m, O + 1, 2 * H, 1, true);
      GemmP gt{};
      gt.A = states; gt.B = dZ1; gt.C = part1;
      gt.bf16 = bf16;
      gt.M = O + 1; gt.N = 2 * H; gt.K = (int)m;
      gt.lda = (int)ldx; gt.ldb = 2 * H; gt.ldc = O;
      gt.splits = S1.splits; gt.kchunk = S1.kchunk; gt.sSplitC = 2LL * H * O;
      rc = tc_gemm_t(gt, false, false, TC_NONE, 1, KC_GEMM_DW, m, m, 0, rs1, 0, 2LL * H, st, 1, O);
      if (rc == RLX_OK) {
        done = true;
        s1 = S1.splits;
      } else if (rc != RLX_ERR_UNSUPPORTED) {
        return rc;
      }
    }
    if (!done) {
      const Splits S1 = choose_splits(m, 2 * H, O, 1, false);
      s1 = S1.splits;
      g1.rowsum = rs1;
      g1.splits = S1.splits; g1.kchunk = S1.kchunk; g1.sSplitC = 2LL * H * O; g1.sSplitRowsum = 2LL * H;
      rc = launch_sgemm<false, false, EPI_NONE>(g1, 1, st, KC_GEMM_DW);
      if (rc) return rc;
    }
  }
  // ---- assemble the flat gradient (m == 0: a rank that owns no row of this minibatch contributes zeros)
  GradReduceP r{};
  r.g[0] = GradGroup{L.off[W1P], 2LL * H * O, part1, s1, 2LL * H * O};
  r.g[1] = GradGroup{L.off[B1P], 2LL * H, rs1, s1, 2LL * H};
  r.g[2] = GradGroup{L.off[W2P], 2LL * H * H, part2, s2, 2LL * H * H};
  r.g[3] = GradGroup{L.off[B2P], 2LL * H, headpart + (2 * A + 5), head_blocks, (long long)npart};
  r.g[4] = GradGroup{L.off[W3P], (long long)A * H, part3, w3_nsplit, w3_stride};
  r.g[5] = GradGroup{L.off[B3P], 2LL * A + 1, headpart, head_blocks, (long long)npart};
  r.g[6] = GradGroup{L.off[W3C], (long long)H, part3 + w3c_off, w3_nsplit, w3_stride};
  r.total = L.total();
  r.logstd_off = L.off[LOGSTD];
  r.act = A;
  r.entropy_grad = -a->hp.entropy_coef * (float)m * inv_mg;
  r.grads = a->grads;
  r.head_partials = headpart; r.nblk = head_blocks; r.npart = npart; r.inv_mg = inv_mg; r.critic_coef = a->hp.critic_coef;
  r.logstd = a->params + L.off[LOGSTD];
  r.metrics = a->metrics; r.m_local = (float)m;
  r.bf16 = bf16;
  if (fuse_norms) {
    r.norm_partials = ws_ptr<float>(ws, P.off_norm);
    r.done = ws_ptr<unsigned int>(ws, P.off_barrier);
    r.norm_out = ws_ptr<float>(ws, P.off_barrier) + 4;
    r.step_count = (long long*)a->step_count;
    for (int i = 0; i <= RLX_PPO_NSEG; ++i) r.seg_off[i] = L.off[i];
    for (int i = 0; i < RLX_PPO_NSEG; ++i)
      if (seg_is_critic(i)) r.critic_mask |= (1u << i);
  }
  rc = launch_grad_reduce(r, st);
  if (rc) return rc;
  if (a->hp.ratio_delta_metric == 2.f && m > 0 && a->metrics != nullptr) {
    // metrics[4] <- torch.median(|ratio - 1|) of this minibatch, overwriting the mean the assembly kernel has just put there
    RLX_LAUNCH_C(KC_OTHER, 0, 16.0 * m, median_lower_kernel, 1, 1024, 0, st, ws_ptr<float>(ws, P.off_ratio), (long long)m, a->metrics + 4);
  }
  return RLX_OK;
}

static AdamP make_adam_params(const rlx_ppo_minibatch_args* a, const PpoLayout& L, const TrainPlan& P) {
  AdamP p{};
  p.total = L.total();
  for (int i = 0; i <= RLX_PPO_NSEG; ++i) p.seg_off[i] = L.off[i];
  p.critic_mask = 0;
  for (int i = 0; i < RLX_PPO_NSEG; ++i)
    if (seg_is_critic(i)) p.critic_mask |= (1u << i);
  p.params = a->params; p.grads = a->grads; p.m = a->exp_avg; p.v = a->exp_avg_sq;
  p.lr = a->lr; p.step_count = (long long*)a->step_count;
  p.max_norm = a->hp.max_grad_norm; p.beta1 = a->hp.adam_beta1; p.beta2 = a->hp.adam_beta2; p.eps = a->hp.adam_eps;
  p.norm_partials = ws_ptr<float>(a->workspace, P.off_norm);
  p.nblk_norm = P.norm_blocks;
  p.metrics = a->metrics;
  return p;
}

extern "C" int rlx_gradnorm_clip_adam_f32(const rlx_ppo_minibatch_args* a, void* stream) {
  int rc = check_mb_args(a, false);
  if (rc) return rc;
  RLX_CHECK_ARG(a->exp_avg && a->exp_avg_sq && a->lr && a->step_count, "optimizer state is null");
  const PpoLayout L = make_layout(a->dims);
  const TrainPlan P = plan_train(a->dims, std::max<int64_t>(a->m, 1));
  cudaStream_t st = (cudaStream_t)stream;
  AdamP p = make_adam_params(a, L, P);
  p.nblk_norm = 64;
  RLX_LAUNCH_C(KC_CLIP_ADAM, 0, 4.0 * L.total(), ppo_grad_sumsq_kernel, (unsigned)p.nblk_norm, 256, 0, st, p);
  RLX_LAUNCH_C(KC_CLIP_ADAM, 0, 28.0 * L.total(), ppo_clip_adam_kernel, (unsigned)ceil_div(L.total(), 256), 256, 0, st, p);
  return RLX_OK;
}

extern "C" int rlx_ppo_update_epoch_f32(const rlx_ppo_minibatch_args* first, int64_t count, int64_t mb, void* stream) {
  RLX_CHECK_ARG(first != nullptr && count >= 0 && mb > 0, "bad arguments");
  const int64_t nmb = ceil_div(count, mb);
  const int A = first->dims.act_dim;
  const int64_t O = first->states_ld > 0 ? first->states_ld : first->dims.obs_dim;  // row pitch of the gathered states
  cudaStream_t st = (cudaStream_t)stream;
  // clip norms fused into the gradient-assembly kernel (needs the optimiser state and the ticket word in the workspace zeroed once)
  bool norms_in_reduce = dims_ok(first->dims) && first->exp_avg && first->exp_avg_sq && first->lr && first->step_count && first->workspace;
  if (norms_in_reduce) {
    const TrainPlan P0 = plan_train(first->dims, std::max<int64_t>(std::min<int64_t>(mb, count), 1));
    if (first->workspace_bytes < P0.total) norms_in_reduce = false;
    else RLX_CHECK_CUDA(cudaMemsetAsync(ws_ptr<unsigned int>(first->workspace, P0.off_barrier), 0, 64, st));
  }
  for (int64_t k = 0; k < nmb; ++k) {
    rlx_ppo_minibatch_args a = *first;
    const int64_t r0 = k * mb;
    a.m = std::min<int64_t>(mb, count - r0);
    a.m_global = a.m;
    a.states = first->states + r0 * O;
    a.actions = first->actions + r0 * A;
    a.log_probs = first->log_probs + r0;
    a.advantages = first->advantages + r0;
    a.returns = first->returns + r0;
    a.adv_stats = first->adv_stats + 2 * k;
    a.metrics = first->metrics ? first->metrics + RLX_PPO_NMETRIC * k : nullptr;
    if (norms_in_reduce && a.m == std::min<int64_t>(mb, count)) {
      // the assembly kernel leaves the clip norms behind; clip + Adam read them (no separate sum-of-squares launch)
      int rc = minibatch_fwdbwd(&a, stream, true);
      if (rc) return rc;
      const PpoLayout La = make_layout(a.dims);
      const TrainPlan Pa = plan_train(a.dims, std::max<int64_t>(a.m, 1));
      AdamP ap = make_adam_params(&a, La, Pa);
      ap.norm_partials = ws_ptr<float>(a.workspace, Pa.off_barrier) + 4;
      ap.nblk_norm = 1;
      RLX_LAUNCH_C(KC_CLIP_ADAM, 0, 28.0 * La.total(), ppo_clip_adam_kernel, (unsigned)ceil_div(La.total(), 256), 256, 0, st, ap);
      continue;
    }
    // a short last minibatch (it has its own workspace plan) or no optimiser state: separate kernels
    int rc = rlx_ppo_minibatch_fwdbwd_f32(&a, stream);
    if (rc) return rc;
    rc = rlx_gradnorm_clip_adam_f32(&a, stream);
    if (rc) return rc;
  }
  return RLX_OK;
}

extern "C" int rlx_ppo_update_epoch_sharded_f32(const rlx_ppo_minibatch_args* first, int64_t num_mb, const int64_t* counts,
                                                const int64_t* global_counts, rlx_comm* comm, void* stream) {
  RLX_CHECK_ARG(first != nullptr && num_mb >= 0 && counts && global_counts && comm, "bad arguments");
  RLX_CHECK_ARG(first->metrics != nullptr, "metrics rows are required");
  const int A = first->dims.act_dim;
  const int64_t O = first->states_ld > 0 ? first->states_ld : first->dims.obs_dim;
  const int64_t P = make_layout(first->dims).total();
  cudaStream_t st = (cudaStream_t)stream;
  int64_t r0 = 0;
  for (int64_t k = 0; k < num_mb; ++k) {
    RLX_CHECK_ARG(counts[k] >= 0 && global_counts[k] >= 1, "bad minibatch sizes");
    rlx_ppo_minibatch_args a = *first;
    a.m = counts[k];
    a.m_global = global_counts[k];
    a.states = first->states + r0 * O;
    a.actions = first->actions + r0 * A;
    a.log_probs = first->log_probs + r0;
    a.advantages = first->advantages + r0;
    a.returns = first->returns + r0;
    a.adv_stats = first->adv_stats + 2 * k;
    float* send = rlx_comm_send_buffer(comm);  // partial gradient [P] followed by the partial metric sums
    a.grads = send;
    a.metrics = send + P;
    int rc = rlx_ppo_minibatch_fwdbwd_f32(&a, stream);
    if (rc) return rc;
    // the exchange kernel leaves the per-net squared norms of the reduced gradient behind (and bumps Adam's step counter):
    // clip + Adam follow directly, without a separate pass over the gradient
    const TrainPlan TP = plan_train(a.dims, std::max<int64_t>(a.m, 1));
    int nblk = 0;
    rc = comm_allreduce_ppo(comm, first->grads, P + RLX_PPO_NMETRIC, a.dims, ws_ptr<float>(a.workspace, TP.off_norm), (long long*)a.step_count, stream, &nblk);
    if (rc) return rc;
    a.grads = first->grads;
    a.metrics = first->grads + P;
    if (nblk > 0) {
      RLX_CHECK_ARG(a.exp_avg && a.exp_avg_sq && a.lr && a.step_count, "optimizer state is null");
      AdamP ap = make_adam_params(&a, make_layout(a.dims), TP);
      ap.nblk_norm = nblk;
      RLX_LAUNCH_C(KC_CLIP_ADAM, 0, 28.0 * P, ppo_clip_adam_kernel, (unsigned)ceil_div(P, 256), 256, 0, st, ap);
    } else {
      rc = rlx_gradnorm_clip_adam_f32(&a, stream);  // writes the two pre-clip norms next to the summed metrics
      if (rc) return rc;
    }
    RLX_CHECK_CUDA(cudaMemcpyAsync(first->metrics + RLX_PPO_NMETRIC * k, first->grads + P, RLX_PPO_NMETRIC * sizeof(float),
                                   cudaMemcpyDeviceToDevice, st));
    r0 += counts[k];
  }
  return RLX_OK;
}

// Test hook: one plain GEMM through either engine (single batch, no split): layout 0 = A k-major, B k-major (C = A B^T);
// 1 = A k-major, B n-major (C = A B); 2 = A m-major, B n-major (C = A^T B, A is [K, M]).  epilogue 0 none, 1 bias+tanh, 2 tanh'.
extern "C" int rlx_debug_gemm_f32(int engine, int layout, int epilogue, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                                  const float* B, int64_t ldb, float* C, int64_t ldc, const float* bias, const float* aux, int64_t ldaux,
                                  void* stream) {
  RLX_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0, "bad arguments");
  RLX_CHECK_ARG((epilogue == 0) || (epilogue == 1 && layout == 0 && bias) || (epilogue == 2 && layout == 1 && aux), "unsupported epilogue/layout");
  GemmP g{};
  g.A = A; g.B = B; g.C = C; g.bias = bias; g.aux = aux;
  g.M = (int)M; g.N = (int)N; g.K = (int)K;
  g.lda = (int)lda; g.ldb = (int)ldb; g.ldc = (int)ldc; g.ldaux = (int)ldaux;
  g.splits = 1; g.kchunk = (int)(ceil_div(K, 8) * 8);
  cudaStream_t st = (cudaStream_t)stream;
  const bool a_k = layout != 2, b_k = layout == 0;
  const long long a_rows = a_k ? M : K, b_rows = b_k ? N : K;
  if (engine >= 1 && engine <= 4) {
    // 1: single-CTA tcgen05 kernels; 2 / 3 / 4: CTA-pair kernels (cta_group::2) with 128 / 256 / 192-wide tiles
    const int pair_bn = engine == 2 ? 128 : engine == 3 ? 256 : engine == 4 ? 192 : 0;
    g_tc_pair_force = pair_bn != 0;
    const int rc = tc_gemm(g, a_k, b_k, epilogue, 1, KC_OTHER, a_rows, b_rows, 0, nullptr, 0, 0, st, pair_bn);
    g_tc_pair_force = false;
    if (rc == RLX_ERR_UNSUPPORTED) set_error("rlx_debug_gemm_f32: shape/alignment not supported by the tcgen05 engine");
    return rc;
  }
  if (layout == 0 && epilogue == 1) return launch_sgemm<true, true, EPI_BIAS_TANH>(g, 1, st);
  if (layout == 0) return launch_sgemm<true, true, EPI_NONE>(g, 1, st);
  if (layout == 1 && epilogue == 2) return launch_sgemm<true, false, EPI_DTANH>(g, 1, st);
  if (layout == 1) return launch_sgemm<true, false, EPI_NONE>(g, 1, st);
  return launch_sgemm<false, false, EPI_NONE>(g, 1, st);
}

extern "C" int rlx_set_head_engine(int engine) {
  if (engine == 0 || engine == 2) g_head_engine = engine;
  else set_error("rlx_set_head_engine: unknown engine %d", engine);
  return g_head_engine;
}

extern "C" int rlx_set_gemm_engine(int engine) {
  if (engine != 0 && engine != 1) {
    set_error("rlx_set_gemm_engine: unknown engine %d", engine);
    return g_gemm_engine;
  }
  g_gemm_engine = engine;
  return g_gemm_engine;
}

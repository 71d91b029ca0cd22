// Gradient assembly, gradient-norm clipping and Adam for the flat PPO parameter buffer.
//   grad_reduce : sums the split-K / per-block partial gradients into the flat gradient (fixed order => deterministic)
//   grad_sumsq  : per-net sum of squares partials (two nets: policy, critic) + Adam step counter increment
//   clip_adam   : clip coefficient per net + Adam update                      (ref: ppo.py:146-148,162-164)
#pragma once
#include "common.cuh"

namespace rlx {

struct GradGroup {
  long long off, len;      // range of the flat buffer
  const float* src;        // partials: element i of split s at src[s*stride + i]
  int nsplit;
  long long stride;
};
constexpr int kNumGroups = 7;

struct GradReduceP {
  GradGroup g[kNumGroups];
  long long total;
  long long logstd_off;
  int act;
  float entropy_grad;          // -entropy_coef * m / m_global, added to every logstd gradient
  float* grads;
  // metrics
  const float* head_partials;  // [nblk, npart]
  int nblk, npart;
  float inv_mg;
  float critic_coef;
  const float* logstd;
  float* metrics;              // [RLX_PPO_NMETRIC]
  float m_local;
  int bf16;                    // bf16-autocast mode: weight / bias gradients come out of bf16 GEMMs / reductions (fp32 accumulation, one rounding
                               // of the complete sum); logstd is an fp32 parameter outside every autocast op and is not rounded
  // Optional fused clip norms (rlx_ppo_update_epoch_f32): every CTA leaves the per-net sums of squares of the elements it assembled, the
  // LAST CTA to finish (atomic ticket) adds them up in a fixed order into norm_out[0..1] and bumps Adam's step counter - the separate
  // ppo_grad_sumsq_kernel launch (9 us of launch + latency for 1.3 MB) disappears.
  float* norm_partials;        // [gridDim.x, 2] or null (= feature off)
  float* norm_out;             // [2]: policy, critic sum of squares
  unsigned int* done;          // ticket counter, zero before the first launch; reset by the last CTA
  long long* step_count;
  long long seg_off[RLX_PPO_NSEG + 1];
  unsigned critic_mask;
};
__device__ __forceinline__ int grad_net_of(const GradReduceP& p, long long i) {
  int seg = 0;
#pragma unroll
  for (int s = 1; s < RLX_PPO_NSEG; ++s) seg += (i >= p.seg_off[s]) ? 1 : 0;
  return (p.critic_mask >> seg) & 1u;
}

// Groups with few partials per element (split-K GEMM outputs) are summed by one thread per element with 8 loads in flight;
// groups with many partials (per-CTA partials of the head kernels: hundreds per element) get one WARP per element, lanes
// striding over the partials, then a fixed-order shuffle tree.  Both orders are fixed => bitwise reproducible.
__device__ __forceinline__ float grad_sum_serial(const float* __restrict__ q, int nsplit, long long stride) {
  float s = 0.f;
  int sp = 0;
  for (; sp + 8 <= nsplit; sp += 8) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = q[(long long)(sp + u) * stride];
#pragma unroll
    for (int u = 0; u < 8; ++u) s += v[u];
  }
  for (; sp < nsplit; ++sp) s += q[(long long)sp * stride];
  return s;
}
__device__ __forceinline__ float grad_sum_warp(const float* __restrict__ q, int nsplit, long long stride, int lane) {
  float s = 0.f;
  for (int sp = lane; sp < nsplit; sp += 32) s += q[(long long)sp * stride];
  return warp_sum(s);
}
constexpr int kTallSplit = 160;  // groups with more partials than this (per-CTA partials of the head kernel) use a warp per element

__global__ void __launch_bounds__(256) ppo_grad_reduce_kernel(const GradReduceP p, const int flat_blocks) {
  float sq_p = 0.f, sq_c = 0.f;  // this thread's contribution to the two squared norms (fused-norm mode)
  if ((int)blockIdx.x < flat_blocks) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.total) {
      bool mine = true;
      float s = 0.f;
#pragma unroll
      for (int gi = 0; gi < kNumGroups; ++gi) {
        const GradGroup& g = p.g[gi];
        if (i >= g.off && i < g.off + g.len) {
          if (g.nsplit > kTallSplit) mine = false;
          else s = grad_sum_serial(g.src + (i - g.off), g.nsplit, g.stride);
        }
      }
      if (mine) {
        if (i >= p.logstd_off && i < p.logstd_off + p.act) s += p.entropy_grad;
        else s = bf16r_if(s, p.bf16);
        p.grads[i] = s;
        if (p.norm_partials != nullptr) { if (grad_net_of(p, i)) sq_c = s * s; else sq_p = s * s; }
      }
    }
  } else {
    // warp per element over the concatenation of the tall groups
    const int lane = threadIdx.x & 31;
    long long w = (long long)(blockIdx.x - flat_blocks) * (blockDim.x >> 5) + (threadIdx.x >> 5);
#pragma unroll
    for (int gi = 0; gi < kNumGroups; ++gi) {
      const GradGroup& g = p.g[gi];
      if (g.nsplit <= kTallSplit) continue;
      if (w >= 0 && w < g.len) {
        float s = grad_sum_warp(g.src + w, g.nsplit, g.stride, lane);
        const long long i = g.off + w;
        if (i >= p.logstd_off && i < p.logstd_off + p.act) s += p.entropy_grad;
        else s = bf16r_if(s, p.bf16);
        if (lane == 0) {
          p.grads[i] = s;
          if (p.norm_partials != nullptr) { if (grad_net_of(p, i)) sq_c = s * s; else sq_p = s * s; }
        }
        w = -1;
      } else if (w >= g.len) {
        w -= g.len;
      }
    }
  }
  if (blockIdx.x == 0 && p.metrics != nullptr) {
    // metric sums of this minibatch (ref: ppo.py:126-141,157): one warp per metric over the head block partials
    const int npart = p.npart, lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    if (wi < 4) {
      float s = 0.f;
      for (int b = lane; b < p.nblk; b += 32) s += p.head_partials[(long long)b * npart + 2 * p.act + 1 + wi];
      s = warp_sum(s) * p.inv_mg;
      if (lane == 0) {
        if (wi == 0) p.metrics[0] = s;                  // pg_loss
        if (wi == 1) p.metrics[1] = p.critic_coef * s;  // critic_loss
        if (wi == 2) p.metrics[3] = s;                  // approx_kl
        if (wi == 3) p.metrics[4] = s;                  // clip_fraction
      }
    }
    if (threadIdx.x == 128) {
      // entropy.mean(): sum_a (0.5 + 0.5*log(2*pi) + log(std_a)), identical for every row (torch Normal.entropy)
      float e = 0.f;
      for (int a = 0; a < p.act; ++a) e += 0.5f + 0.5f * 1.8378770664093453f + logf(expf(p.logstd[a]));
      p.metrics[2] = e * (p.m_local * p.inv_mg);
      p.metrics[7] = p.m_local;
    }
  }
  if (p.norm_partials != nullptr) {
    __shared__ float sh_n[34];
    __shared__ int s_last;
    sq_p = block_sum(sq_p, sh_n);
    sq_c = block_sum(sq_c, sh_n);
    if (threadIdx.x == 0) {
      p.norm_partials[2 * blockIdx.x] = sq_p;
      p.norm_partials[2 * blockIdx.x + 1] = sq_c;
      __threadfence();
      s_last = (atomicAdd(p.done, 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (s_last) {
      __threadfence();
      // fixed order: thread t adds partials t, t + 256, ...; then the block tree (same shape every launch => reproducible bits)
      float a = 0.f, b = 0.f;
      for (unsigned int q = threadIdx.x; q < gridDim.x; q += blockDim.x) {
        a += __ldcg(p.norm_partials + 2 * q);
        b += __ldcg(p.norm_partials + 2 * q + 1);
      }
      a = block_sum(a, sh_n);
      b = block_sum(b, sh_n);
      if (threadIdx.x == 0) {
        p.norm_out[0] = a;
        p.norm_out[1] = b;
        *p.done = 0u;
        if (p.step_count != nullptr) p.step_count[0] += 1;  // read by the clip_adam kernel launched after this one
      }
    }
  }
}

struct AdamP {
  long long total;
  long long seg_off[RLX_PPO_NSEG + 1];
  unsigned critic_mask;  // bit s set => segment s belongs to the critic
  float* params;
  const float* grads;
  float* m;
  float* v;
  const float* lr;
  long long* step_count;
  float max_norm, beta1, beta2, eps;
  float* norm_partials;  // [nblk_norm, 2]
  int nblk_norm;
  float* metrics;
};

__device__ __forceinline__ int adam_net_of(const AdamP& p, long long i) {
  int seg = 0;
#pragma unroll
  for (int s = 1; s < RLX_PPO_NSEG; ++s) seg += (i >= p.seg_off[s]) ? 1 : 0;
  return (p.critic_mask >> seg) & 1u;
}

__global__ void __launch_bounds__(256) ppo_grad_sumsq_kernel(const AdamP p) {
  __shared__ float sh[34];
  float sp = 0.f, sc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.total; i += (long long)gridDim.x * blockDim.x) {
    const float g = p.grads[i];
    if (adam_net_of(p, i)) sc = fmaf(g, g, sc); else sp = fmaf(g, g, sp);
  }
  sp = block_sum(sp, sh);
  sc = block_sum(sc, sh);
  if (threadIdx.x == 0) {
    p.norm_partials[2 * blockIdx.x] = sp;
    p.norm_partials[2 * blockIdx.x + 1] = sc;
    if (blockIdx.x == 0) p.step_count[0] += 1;  // read by the clip_adam kernel launched after this one
  }
}

__global__ void __launch_bounds__(256) ppo_clip_adam_kernel(const AdamP p) {
  __shared__ float s_coef[2];
  __shared__ float s_sc[3];
  if (threadIdx.x < 2) {
    float s = 0.f;
    for (int b = 0; b < p.nblk_norm; ++b) s += p.norm_partials[2 * b + threadIdx.x];
    const float norm = sqrtf(s);
    // clip_grad_norm_: clip_coef = max_norm / (total_norm + 1e-6), clamped to 1  (torch/nn/utils/clip_grad.py)
    s_coef[threadIdx.x] = fminf(p.max_norm / (norm + 1e-6f), 1.f);
    if (blockIdx.x == 0 && p.metrics != nullptr) p.metrics[5 + threadIdx.x] = norm;
  }
  if (threadIdx.x == 32) {
    // torch/optim/adam.py (_single_tensor_adam): step_size = lr / (1 - beta1^t); denom = sqrt(v)/sqrt(1 - beta2^t) + eps
    const double t = (double)p.step_count[0];
    const double bc1 = 1.0 - pow((double)p.beta1, t);
    const double bc2 = 1.0 - pow((double)p.beta2, t);
    s_sc[0] = (float)((double)p.lr[0] / bc1);
    s_sc[1] = (float)sqrt(bc2);
  }
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.total) return;
  const float g = p.grads[i] * s_coef[adam_net_of(p, i)];
  float m = p.m[i], v = p.v[i];
  m = m + (g - m) * (1.f - p.beta1);                 // exp_avg.lerp_(grad, 1 - beta1)
  v = v * p.beta2 + (1.f - p.beta2) * g * g;         // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
  const float denom = sqrtf(v) / s_sc[1] + p.eps;
  p.params[i] = p.params[i] - s_sc[0] * (m / denom); // param.addcdiv_(exp_avg, denom, value=-step_size)
  p.m[i] = m;
  p.v[i] = v;
}

// ------------------------------------------------------------------------------------------------ lower median (ESPO)
// torch.median of a 1-D tensor returns the LOWER of the two middle values: sorted(x)[(n - 1) / 2] (espo.py:57-63,133 applies it to
// |ratio - 1| of the minibatch).  Radix select on the bit patterns of the non-negative floats (their unsigned order is their numeric
// order): four passes of 8 bits, each a shared-memory histogram over the candidates that share the prefix found so far.  One CTA; n is a
// minibatch (<= a few 10^5 values).  A NaN anywhere makes torch.median NaN; so does this (NaN patterns sort above +inf and are counted).
__global__ void __launch_bounds__(1024) median_lower_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  __shared__ unsigned int hist[256];
  __shared__ unsigned int s_prefix, s_rank;
  __shared__ int s_nan;
  if (threadIdx.x == 0) { s_prefix = 0u; s_rank = (unsigned int)((n - 1) / 2); s_nan = 0; }
  __syncthreads();
  for (long long i = threadIdx.x; i < n; i += blockDim.x)
    if (x[i] != x[i]) s_nan = 1;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0u;
    __syncthreads();
    const unsigned int prefix = s_prefix;
    const unsigned int mask = pass == 0 ? 0u : (0xFFFFFFFFu << (shift + 8));
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
      const unsigned int u = __float_as_uint(fabsf(x[i]));
      if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned int r = s_rank, b = 0;
      while (b < 255 && r >= hist[b]) { r -= hist[b]; ++b; }
      s_rank = r;
      s_prefix = prefix | (b << shift);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = s_nan ? __int_as_float(0x7FC00000) : __uint_as_float(s_prefix);
}

}  // namespace rlx

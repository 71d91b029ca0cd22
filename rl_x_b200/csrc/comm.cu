// Gradient exchange between data-parallel ranks over NVLink peer memory (SURVEY.md §8 e): a one-shot all-reduce kernel that
// reads every rank's send slot through CUDA-IPC mapped pointers.  See rlx_b200.h for the protocol.
#include "common.cuh"
#include <string.h>

struct rlx_comm {
  int rank = 0, world = 1;
  int64_t nfloats = 0;
  size_t slot_bytes = 0;
  uint8_t* base = nullptr;                       // own allocation: [flags 1 KiB][slot 0][slot 1]
  uint8_t* peer[RLX_COMM_MAX_WORLD] = {};        // mapped peer allocations (peer[rank] == base)
  uint64_t seq = 0;                              // all-reduces issued so far
  bool connected = false;
};

namespace rlx {
namespace {

constexpr size_t kFlagBytes = 1024;
constexpr int kThreads = 512;

struct CommView {
  const float* slot[RLX_COMM_MAX_WORLD];          // every rank's send slot for this sequence number
  unsigned long long* flags[RLX_COMM_MAX_WORLD];  // every rank's flag array (flags[r][q]: rank q has published sequence number ...)
};
// Optional side product of the all-reduce: per-net sums of squares of the REDUCED vector (the two clip_grad_norm_ norms of the PPO update),
// one partial pair per CTA, so that no separate pass over the gradient is needed before clip + Adam.
struct CommSumsq {
  float* partials;          // [gridDim.x, 2] or null
  long long seg_off[RLX_PPO_NSEG + 1];
  unsigned critic_mask;
  long long total;          // elements beyond `total` (the metric tail riding along) are not part of any norm
  long long* step_count;    // optional: incremented once (Adam's step counter, as ppo_grad_sumsq_kernel does)
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// One launch per rank.  Block 0 publishes "my slot for `seq` is complete" (stream order put the gradient kernels before this
// one) into every rank's flag array; every block then waits until all ranks have published, and sums the slots in rank order.
// Peer data is read with ld.cv: peer lines must not be served from this SM's L1.
// WORLD > 0: compile-time rank count, so that the peer loads of one element are all in flight before the first add (one NVLink round
// trip per element instead of one per rank); WORLD == 0: any rank count.
__device__ __forceinline__ int comm_net_of(const CommSumsq& q, long long i);

template <int WORLD>
__global__ void __launch_bounds__(kThreads) comm_allreduce_kernel(CommView v, int rank, int world_rt, unsigned long long seq,
                                                                   float* __restrict__ out, long long n, CommSumsq q) {
  __shared__ float sh[34];
  float sp = 0.f, sc = 0.f;  // optional side product: per-net sums of squares of the reduced vector (see CommSumsq)
  const int world = WORLD > 0 ? WORLD : world_rt;
  if (blockIdx.x == 0 && threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(v.flags[threadIdx.x] + rank, seq);
  }
  if (threadIdx.x < world) {
    const unsigned long long* mine = v.flags[rank] + threadIdx.x;
    const unsigned long long t0 = global_ns();
    while (ld_acquire_sys(mine) < seq) {
      if (global_ns() - t0 > 20000000000ull) {
        printf("rlx_comm: rank %d waited 20 s for rank %d at sequence %llu\n", rank, (int)threadIdx.x, seq);
        __trap();
      }
    }
  }
  __syncthreads();
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    if (WORLD > 0) {
      float4 x[WORLD > 0 ? WORLD : 1];
#pragma unroll
      for (int r = 0; r < WORLD; ++r) x[r] = __ldcv(reinterpret_cast<const float4*>(v.slot[r]) + i);
      float4 acc = x[0];
#pragma unroll
      for (int r = 1; r < WORLD; ++r) { acc.x += x[r].x; acc.y += x[r].y; acc.z += x[r].z; acc.w += x[r].w; }  // rank order, as below
      reinterpret_cast<float4*>(out)[i] = acc;
      if (q.partials != nullptr) {
        const float e[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const long long idx = 4 * i + j;
          if (idx < q.total) { if (comm_net_of(q, idx)) sc = fmaf(e[j], e[j], sc); else sp = fmaf(e[j], e[j], sp); }
        }
      }
    } else {
      float4 acc = __ldcv(reinterpret_cast<const float4*>(v.slot[0]) + i);
      for (int r = 1; r < world; ++r) {
        const float4 x = __ldcv(reinterpret_cast<const float4*>(v.slot[r]) + i);
        acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
      }
      reinterpret_cast<float4*>(out)[i] = acc;
    }
  }
  if (blockIdx.x == 0) {
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) {
      float acc = __ldcv(v.slot[0] + i);
      for (int r = 1; r < world; ++r) acc += __ldcv(v.slot[r] + i);
      out[i] = acc;
      if (q.partials != nullptr && WORLD > 0 && i < q.total) { if (comm_net_of(q, i)) sc = fmaf(acc, acc, sc); else sp = fmaf(acc, acc, sp); }
    }
  }
  if (q.partials != nullptr && WORLD > 0) {
    sp = block_sum(sp, sh);
    sc = block_sum(sc, sh);
    if (threadIdx.x == 0) {
      q.partials[2 * blockIdx.x] = sp;
      q.partials[2 * blockIdx.x + 1] = sc;
      if (blockIdx.x == 0 && q.step_count != nullptr) q.step_count[0] += 1;
    }
  }
}

__device__ __forceinline__ int comm_net_of(const CommSumsq& q, long long i) {
  int seg = 0;
#pragma unroll
  for (int s = 1; s < RLX_PPO_NSEG; ++s) seg += (i >= q.seg_off[s]) ? 1 : 0;
  return (q.critic_mask >> seg) & 1u;
}

}  // namespace
}  // namespace rlx

using namespace rlx;

static_assert(sizeof(cudaIpcMemHandle_t) == RLX_COMM_HANDLE_BYTES, "CUDA IPC handle size changed");

extern "C" int rlx_comm_create(int rank, int world, int64_t nfloats, rlx_comm** out) {
  RLX_CHECK_ARG(out != nullptr && world >= 1 && world <= RLX_COMM_MAX_WORLD && rank >= 0 && rank < world && nfloats > 0, "bad arguments");
  rlx_comm* c = new rlx_comm();
  c->rank = rank; c->world = world; c->nfloats = nfloats;
  c->slot_bytes = align_up((size_t)nfloats * sizeof(float), 1024);
  const size_t total = kFlagBytes + 2 * c->slot_bytes;  // flags | send slot 0 | send slot 1
  static_assert(kFlagBytes >= RLX_COMM_MAX_WORLD * sizeof(unsigned long long), "flag area too small");
  cudaError_t e = cudaMalloc((void**)&c->base, total);  // plain cudaMalloc: exportable through cudaIpcGetMemHandle
  if (e == cudaSuccess) e = cudaMemset(c->base, 0, total);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    set_error("rlx_comm_create: CUDA error %s", cudaGetErrorString(e));
    if (c->base) cudaFree(c->base);
    delete c;
    return RLX_ERR_CUDA;
  }
  c->peer[rank] = c->base;
  c->connected = (world == 1);
  *out = c;
  return RLX_OK;
}

extern "C" int rlx_comm_export_handle(rlx_comm* c, uint8_t* handle) {
  RLX_CHECK_ARG(c != nullptr && handle != nullptr, "bad arguments");
  cudaIpcMemHandle_t h;
  RLX_CHECK_CUDA(cudaIpcGetMemHandle(&h, c->base));
  memcpy(handle, &h, sizeof(h));
  return RLX_OK;
}

extern "C" int rlx_comm_connect(rlx_comm* c, const uint8_t* handles) {
  RLX_CHECK_ARG(c != nullptr && handles != nullptr, "bad arguments");
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank || c->peer[r] != nullptr) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * RLX_COMM_HANDLE_BYTES, sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      set_error("rlx_comm_connect: cannot map rank %d's buffer (%s): no peer access between these GPUs?", r, cudaGetErrorString(e));
      cudaGetLastError();
      return RLX_ERR_CUDA;
    }
    c->peer[r] = (uint8_t*)p;
  }
  c->connected = true;
  return RLX_OK;
}

extern "C" float* rlx_comm_send_buffer(rlx_comm* c) {
  if (c == nullptr) return nullptr;
  return (float*)(c->base + kFlagBytes + ((c->seq + 1) & 1) * c->slot_bytes);
}

extern "C" int rlx_comm_stage_f32(rlx_comm* c, const float* src, int64_t n, void* stream) {
  RLX_CHECK_ARG(c != nullptr && src != nullptr && n > 0 && n <= c->nfloats, "bad arguments");
  RLX_CHECK_CUDA(cudaMemcpyAsync(rlx_comm_send_buffer(c), src, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return RLX_OK;
}

static int comm_allreduce(rlx_comm* c, float* out, int64_t n, void* stream, const CommSumsq* sumsq, int* nblk_out);

extern "C" int rlx_comm_allreduce_sum_f32(rlx_comm* c, float* out, int64_t n, void* stream) { return comm_allreduce(c, out, n, stream, nullptr, nullptr); }

// PPO update: all-reduce of [gradient | metric sums] with the two squared gradient norms of the reduced gradient as a side product at 2, 4
// and 8 ranks (returns the number of partial pairs written, 0 = none: the caller runs its own pass).
int comm_allreduce_ppo(rlx_comm* c, float* out, int64_t n, const rlx_ppo_dims& d, float* norm_partials, long long* step_count, void* stream,
                       int* nblk_out) {
  CommSumsq q{};
  const PpoLayout L = make_layout(d);
  for (int i = 0; i <= RLX_PPO_NSEG; ++i) q.seg_off[i] = L.off[i];
  for (int i = 0; i < RLX_PPO_NSEG; ++i)
    if (seg_is_critic(i)) q.critic_mask |= (1u << i);
  q.total = L.total();
  q.partials = norm_partials;
  q.step_count = step_count;
  return comm_allreduce(c, out, n, stream, &q, nblk_out);
}

static int comm_allreduce(rlx_comm* c, float* out, int64_t n, void* stream, const CommSumsq* sumsq, int* nblk_out) {
  if (nblk_out) *nblk_out = 0;
  RLX_CHECK_ARG(c != nullptr && out != nullptr && n > 0 && n <= c->nfloats, "bad arguments");
  RLX_CHECK_ARG(c->connected, "rlx_comm_connect has not been called");
  RLX_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 15) == 0, "out must be 16-byte aligned");
  c->seq += 1;
  CommView v{};
  for (int r = 0; r < c->world; ++r) {
    v.slot[r] = (const float*)(c->peer[r] + kFlagBytes + (c->seq & 1) * c->slot_bytes);
    v.flags[r] = (unsigned long long*)c->peer[r];
  }
  const int64_t n4 = std::max<int64_t>(n >> 2, 1);
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n4, kThreads), sm_count());
  // algorithmic bytes: every rank's slot read once + the result written once
  CommSumsq q1{};
  if (sumsq && (c->world == 2 || c->world == 4 || c->world == 8)) q1 = *sumsq;  // the generic-world instantiation does not compute them
#define RLX_COMM_LAUNCH(W)                                                                                                     \
  RLX_LAUNCH_C(KC_ALLREDUCE, 0, 4.0 * n * (c->world + 1), comm_allreduce_kernel<W>, grid, kThreads, 0, stream, v, c->rank, c->world, \
               (unsigned long long)c->seq, out, (long long)n, q1)
  switch (c->world) {
    case 2: RLX_COMM_LAUNCH(2); break;
    case 4: RLX_COMM_LAUNCH(4); break;
    case 8: RLX_COMM_LAUNCH(8); break;
    default: RLX_COMM_LAUNCH(0); break;
  }
#undef RLX_COMM_LAUNCH
  if (nblk_out && q1.partials) *nblk_out = (int)grid;
  return RLX_OK;
}

extern "C" int rlx_comm_destroy(rlx_comm* c) {
  if (c == nullptr) return RLX_OK;
  cudaDeviceSynchronize();
  for (int r = 0; r < c->world; ++r)
    if (r != c->rank && c->peer[r]) cudaIpcCloseMemHandle(c->peer[r]);
  if (c->base) cudaFree(c->base);
  delete c;
  return RLX_OK;
}

// Data-parallel exchange over NVLink peer memory (one process per GPU, CUDA IPC) — the step that follows the
// backward in a data-parallel run of training.py:47-51 (`loss.backward(); optimizer.step()`): the reference is
// single-device, SURVEY.md §8(e) adds one sum of the flat gradient per step.
//
// ONE kernel does reduce-scatter -> Adam -> all-gather:
//   phase 1  every rank stores slice r of its gradient into rank r's landing zone (peer stores), then raises
//            flag[r].grad[me] = epoch;
//   phase 2  rank r waits for all `world` flags, sums the `world` copies of ITS slice in rank order (fixed order:
//            bit-reproducible, and every rank ends up with bit-identical parameters), applies torch.optim.Adam
//            arithmetic to that slice only (optimizer work is sharded too), and stores the new parameters into
//            EVERY rank's parameter segment (peer stores); raises flag[r].param[me] = epoch;
//   phase 3  the last CTA waits for all parameter flags, so kernel completion == parameters of this step landed.
// Element n of the flat vector carries the loss (summed like a gradient, broadcast like a parameter).
// Flags only ever grow (epoch counter), nothing is reset, and the landing zone needs no double buffering: a peer
// can only start pushing step e+1 after it has seen MY parameter flag of step e, which I raise after my last read
// of the landing zone (see DESIGN.md §6).
#include <stdlib.h>
#include <string.h>

#include "tt_common.cuh"

namespace tt {
namespace {

constexpr int kMaxWorld = 8;
constexpr int kDpThreads = 256;
constexpr unsigned long long kSpinTimeoutNs = 4000000000ull;  // 4 s: a lost peer becomes an error, not a hung GPU

// TT_DP_TIMEOUT_MS overrides the spin timeout of the exchange / barrier kernels (rank-local work such as an
// evaluation on rank 0 must finish inside it, or be fenced by a host barrier first)
unsigned long long spin_timeout_ns() {
  static unsigned long long v = 0;
  if (!v) {
    const char* e = getenv("TT_DP_TIMEOUT_MS");
    const long long ms = e ? atoll(e) : 0;
    v = ms > 0 ? (unsigned long long)ms * 1000000ull : kSpinTimeoutNs;
  }
  return v;
}

struct DpLayout {
  size_t S;          // slice length in floats (multiple of 4)
  size_t recv_off;   // floats, from segment base
  size_t flag_off;   // bytes, from segment base
  size_t bytes;
};

__host__ __device__ inline DpLayout dp_layout(size_t n, int world) {
  DpLayout L;
  const size_t per = (n + 1 + (size_t)world - 1) / (size_t)world;
  L.S = (per + 63) & ~size_t(63);                    // 256-byte aligned slices
  L.recv_off = L.S * (size_t)world;                  // [0, world*S): parameters (+ loss at [n])
  L.flag_off = (L.recv_off + L.S * (size_t)world) * 4;  // [world*S, 2*world*S): landing zone [src rank][S]
  L.bytes = L.flag_off + 256;                        // flags: grad[world] | param[world] | error
  return L;
}

struct DpParams {
  float* seg[kMaxWorld];
  int world, rank;
  size_t n;
  const float* grad;  // [n+1] local
  float* m;
  float* v;
  float lr, beta1, beta2, eps;
  double* state;      // {t, beta1^t, beta2^t, -}
  unsigned* ctl;      // {epoch, ticket1, ticket2, error, then 4 x u64 diagnostics: ns until all gradient flags,
                      //  ns from there to the end of the kernel, calls, ns of the own push}
  unsigned long long timeout_ns;
};

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// waits until *flag >= epoch (wrap-safe); false on timeout
__device__ __forceinline__ bool wait_flag(const unsigned* flag, unsigned epoch, unsigned long long timeout_ns) {
  if ((int)(ld_acquire_sys(flag) - epoch) >= 0) return true;
  const unsigned long long t0 = globaltimer();
  for (;;) {
    for (int i = 0; i < 64; ++i)
      if ((int)(ld_acquire_sys(flag) - epoch) >= 0) return true;
    if (globaltimer() - t0 > timeout_ns) return false;
  }
}

__global__ void __launch_bounds__(kDpThreads) dp_rs_adam_ag_kernel(const __grid_constant__ DpParams p) {
  // Sticky error: once a peer has timed out (ctl[3] != 0) the protocol state (tickets, epoch, the peers' flags) is
  // no longer consistent, so every later launch is a no-op until the host has seen the error (DpExchange.check()
  // raises) — no update is ever applied on half-exchanged gradients.  The value is stable for the whole kernel only
  // when it is already set at launch; a timeout inside THIS launch makes the failing CTA return below.
  if (*reinterpret_cast<volatile unsigned*>(&p.ctl[3]) != 0u) return;
  const DpLayout L = dp_layout(p.n, p.world);
  const int tid = threadIdx.x, W = p.world, me = p.rank;
  const unsigned epoch = *reinterpret_cast<volatile unsigned*>(&p.ctl[0]) + 1u;
  // bias corrections of step t+1 (torch.optim.Adam: step_size = lr / (1 - beta1^t), denom = sqrt(v)/sqrt(1 - beta2^t) + eps)
  const double t = *reinterpret_cast<volatile double*>(&p.state[0]);
  const double b1p = (t == 0.0 ? 1.0 : *reinterpret_cast<volatile double*>(&p.state[1])) * (double)p.beta1;
  const double b2p = (t == 0.0 ? 1.0 : *reinterpret_cast<volatile double*>(&p.state[2])) * (double)p.beta2;
  const float step_size = (float)((double)p.lr / (1.0 - b1p));
  const float bc2_sqrt = (float)sqrt(1.0 - b2p);
  unsigned* my_flags = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(p.seg[me]) + L.flag_off);
  __shared__ int s_last, s_fail;
  if (tid == 0) s_fail = 0;
  const unsigned long long t_start = (blockIdx.x == 0 && tid == 0) ? globaltimer() : 0ull;
  unsigned long long t_flags = 0ull;

  const size_t S4 = L.S / 4;
  const size_t gstride = (size_t)gridDim.x * kDpThreads;
  const size_t g0 = (size_t)blockIdx.x * kDpThreads + tid;
  const size_t n1 = p.n + 1;

  // ---- phase 1: scatter my gradient slices to their owners (self copy last) ---------------------------------------
  for (int rr = 1; rr <= W; ++rr) {
    const int r = (me + rr) % W;
    float* dst = p.seg[r] + L.recv_off + (size_t)me * L.S;
    const size_t base = (size_t)r * L.S;
    for (size_t k4 = g0; k4 < S4; k4 += gstride) {
      const size_t j = base + k4 * 4;
      float4 g;
      if (j + 3 < n1) {
        g = *reinterpret_cast<const float4*>(p.grad + j);
      } else {
        g.x = j < n1 ? p.grad[j] : 0.f;
        g.y = j + 1 < n1 ? p.grad[j + 1] : 0.f;
        g.z = j + 2 < n1 ? p.grad[j + 2] : 0.f;
        g.w = 0.f;
      }
      *reinterpret_cast<float4*>(dst + k4 * 4) = g;
    }
  }
  __threadfence_system();
  __syncthreads();
  const unsigned long long t_pushed = (blockIdx.x == 0 && tid == 0) ? globaltimer() : 0ull;
  if (tid == 0) {
    const unsigned prev = atomicAdd(&p.ctl[1], 1u);
    if (prev == gridDim.x - 1) {  // every CTA of this rank has pushed: tell the owners
      __threadfence_system();
      for (int r = 0; r < W; ++r)
        st_release_sys(reinterpret_cast<unsigned*>(reinterpret_cast<char*>(p.seg[r]) + L.flag_off) + me, epoch);
      p.ctl[1] = 0;
    }
  }
  // ---- phase 2: reduce my slice in rank order, Adam, broadcast the new parameters ----------------------------------
  if (tid < W && !wait_flag(my_flags + tid, epoch, p.timeout_ns)) s_fail = 1;
  __syncthreads();
  if (blockIdx.x == 0 && tid == 0) t_flags = globaltimer();
  if (s_fail) {
    if (tid == 0) p.ctl[3] = 1;
    return;
  }
  {
    const float* recv = p.seg[me] + L.recv_off;
    float* mine = p.seg[me];
    const size_t base = (size_t)me * L.S;
    for (size_t k4 = g0; k4 < S4; k4 += gstride) {
      float4 a = __ldcg(reinterpret_cast<const float4*>(recv + k4 * 4));
      for (int r = 1; r < W; ++r) {
        const float4 b = __ldcg(reinterpret_cast<const float4*>(recv + (size_t)r * L.S + k4 * 4));
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      const size_t j = base + k4 * 4;
      float gi[4] = {a.x, a.y, a.z, a.w}, out[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const size_t jj = j + c;
        if (jj < p.n) {
          const float mi = p.m[jj] + (gi[c] - p.m[jj]) * (1.f - p.beta1);
          const float vi = p.v[jj] * p.beta2 + (1.f - p.beta2) * gi[c] * gi[c];
          p.m[jj] = mi;
          p.v[jj] = vi;
          const float denom = sqrtf(vi) / bc2_sqrt + p.eps;
          out[c] = __ldcg(mine + jj) - step_size * (mi / denom);
        } else {
          out[c] = jj == p.n ? gi[c] : 0.f;  // the loss rides in slot n
        }
      }
      const float4 o = make_float4(out[0], out[1], out[2], out[3]);
      for (int rr = 1; rr <= W; ++rr) {
        const int r = (me + rr) % W;
        *reinterpret_cast<float4*>(p.seg[r] + j) = o;
      }
    }
  }
  __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    const unsigned prev = atomicAdd(&p.ctl[2], 1u);
    s_last = (prev == gridDim.x - 1);
    if (s_last) {
      __threadfence_system();
      for (int r = 0; r < W; ++r)
        st_release_sys(reinterpret_cast<unsigned*>(reinterpret_cast<char*>(p.seg[r]) + L.flag_off) + W + me, epoch);
      p.state[0] = t + 1.0;
      p.state[1] = b1p;
      p.state[2] = b2p;
      p.ctl[2] = 0;
      p.ctl[0] = epoch;
    }
  }
  __syncthreads();
  // ---- phase 3: the last CTA holds the kernel open until every rank's parameter slice has landed here ----------------
  if (s_last && tid < W && !wait_flag(my_flags + W + tid, epoch, p.timeout_ns)) p.ctl[3] = 1;
  if (blockIdx.x == 0 && tid == 0) {  // diagnostics (CTA 0's view; it is not necessarily the last CTA)
    unsigned long long* d = reinterpret_cast<unsigned long long*>(p.ctl + 4);
    d[0] += t_flags - t_start;
    d[1] += globaltimer() - t_flags;
    d[2] += 1ull;
    d[3] += t_pushed - t_start;
  }
}

// one-CTA barrier across the ranks: flags[r] points at rank r's flag array ([world] slots, slot = source rank)
struct BarrierParams {
  unsigned* flags[kMaxWorld];
  int world, rank;
  unsigned* ctl;  // {epoch, -, -, error}
  unsigned long long timeout_ns;
};

__global__ void __launch_bounds__(32) peer_barrier_kernel(const __grid_constant__ BarrierParams p) {
  const int tid = threadIdx.x;
  const unsigned epoch = p.ctl[0] + 1u;
  __threadfence_system();
  if (tid < p.world) {
    st_release_sys(p.flags[tid] + p.rank, epoch);
    if (!wait_flag(p.flags[p.rank] + tid, epoch, p.timeout_ns)) p.ctl[3] = 1;
  }
  __syncwarp();
  if (tid == 0) p.ctl[0] = epoch;
}

// merge of per-rank top-k lists pulled straight from the peers' memory (corpus scan, §8e): same order as
// topk_merge_kernel — score descending, id ascending, ids < 0 ignored
struct MergeParams {
  const float* score[kMaxWorld];
  const long long* id[kMaxWorld];
  int world, Q, k;
  float* top_score;
  long long* top_id;
};

__global__ void __launch_bounds__(128) peer_topk_merge_kernel(const __grid_constant__ MergeParams p) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= p.Q) return;
  int head[kMaxWorld];
  for (int r = 0; r < p.world; ++r) head[r] = 0;
  for (int o = 0; o < p.k; ++o) {
    int best = -1;
    float bs = 0.f;
    long long bi = 0;
    for (int r = 0; r < p.world; ++r) {
      while (head[r] < p.k && p.id[r][(size_t)q * p.k + head[r]] < 0) ++head[r];
      if (head[r] >= p.k) continue;
      const float s = p.score[r][(size_t)q * p.k + head[r]];
      const long long i = p.id[r][(size_t)q * p.k + head[r]];
      if (best < 0 || s > bs || (s == bs && i < bi)) {
        best = r; bs = s; bi = i;
      }
    }
    if (best < 0) {
      p.top_score[(size_t)q * p.k + o] = __int_as_float(0xffffffff);
      p.top_id[(size_t)q * p.k + o] = -1;
    } else {
      p.top_score[(size_t)q * p.k + o] = bs;
      p.top_id[(size_t)q * p.k + o] = bi;
      ++head[best];
    }
  }
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" int tt_peer_alloc(size_t bytes, void** dev_ptr, void* handle_out) {
  TT_REQUIRE(dev_ptr && handle_out && bytes > 0, "tt_peer_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == TT_PEER_HANDLE_BYTES, "IPC handle size");
  void* p = nullptr;
  TT_CUDA(cudaMalloc(&p, bytes));
  TT_CUDA(cudaMemset(p, 0, bytes));
  TT_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  TT_CUDA(cudaIpcGetMemHandle(&h, p));
  memcpy(handle_out, &h, sizeof(h));
  *dev_ptr = p;
  return 0;
}

extern "C" int tt_peer_open(const void* handle, void** dev_ptr) {
  TT_REQUIRE(handle && dev_ptr, "tt_peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  TT_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

extern "C" int tt_peer_close(void* dev_ptr) {
  TT_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return 0;
}

extern "C" int tt_peer_free(void* dev_ptr) {
  TT_CUDA(cudaFree(dev_ptr));
  return 0;
}

extern "C" size_t tt_dp_segment_bytes(size_t n_param, int world) {
  if (world < 1 || world > kMaxWorld) return 0;
  return dp_layout(n_param, world).bytes;
}

extern "C" int tt_dp_reduce_adam(void* const* segments, int world, int rank, size_t n_param, const float* grad,
                                 float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                 double* state, unsigned* ctl, int max_ctas, tt_stream_t stream) {
  TT_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "tt_dp_reduce_adam: bad world/rank %d/%d",
             world, rank);
  TT_REQUIRE(segments && grad && exp_avg && exp_avg_sq && state && ctl, "tt_dp_reduce_adam: null argument");
  DpParams p{};
  for (int r = 0; r < world; ++r) {
    TT_REQUIRE(segments[r] != nullptr, "tt_dp_reduce_adam: segment of rank %d is null", r);
    p.seg[r] = reinterpret_cast<float*>(segments[r]);
  }
  p.world = world; p.rank = rank; p.n = n_param; p.grad = grad; p.m = exp_avg; p.v = exp_avg_sq;
  p.lr = lr; p.beta1 = beta1; p.beta2 = beta2; p.eps = eps; p.state = state; p.ctl = ctl;
  p.timeout_ns = spin_timeout_ns();
  const DpLayout L = dp_layout(n_param, world);
  // every CTA spins on peer flags, so the grid must be co-resident: never more than one CTA per SM
  long long ctas = (long long)((L.S / 4 + kDpThreads - 1) / kDpThreads);
  const int cap = max_ctas > 0 ? (max_ctas < sm_count() ? max_ctas : sm_count()) : sm_count();
  if (ctas > cap) ctas = cap;
  if (ctas < 1) ctas = 1;
  dp_rs_adam_ag_kernel<<<(unsigned)ctas, kDpThreads, 0, as_stream(stream)>>>(p);
  TT_LAUNCH_CHECK();
  return 0;
}

extern "C" int tt_peer_barrier(void* const* flags, int world, int rank, unsigned* ctl, tt_stream_t stream) {
  TT_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world && flags && ctl, "tt_peer_barrier: bad arguments");
  BarrierParams p{};
  for (int r = 0; r < world; ++r) {
    TT_REQUIRE(flags[r] != nullptr, "tt_peer_barrier: flags of rank %d are null", r);
    p.flags[r] = reinterpret_cast<unsigned*>(flags[r]);
  }
  p.world = world; p.rank = rank; p.ctl = ctl;
  p.timeout_ns = spin_timeout_ns();
  peer_barrier_kernel<<<1, 32, 0, as_stream(stream)>>>(p);
  TT_LAUNCH_CHECK();
  return 0;
}

extern "C" int tt_peer_topk_merge(const float* const* parts_score, const int64_t* const* parts_id, int world, int Q,
                                  int k, float* top_score, int64_t* top_id, tt_stream_t stream) {
  TT_REQUIRE(world >= 1 && world <= kMaxWorld && Q >= 0 && k >= 1, "tt_peer_topk_merge: bad shape");
  if (Q == 0) return 0;
  MergeParams p{};
  for (int r = 0; r < world; ++r) {
    TT_REQUIRE(parts_score[r] && parts_id[r], "tt_peer_topk_merge: null list for rank %d", r);
    p.score[r] = parts_score[r];
    p.id[r] = reinterpret_cast<const long long*>(parts_id[r]);
  }
  p.world = world; p.Q = Q; p.k = k; p.top_score = top_score; p.top_id = reinterpret_cast<long long*>(top_id);
  peer_topk_merge_kernel<<<(Q + 127) / 128, 128, 0, as_stream(stream)>>>(p);
  TT_LAUNCH_CHECK();
  return 0;
}

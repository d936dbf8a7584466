// Cosine triplet loss, forward and closed-form backward (backend/model.py:132-145).
// One warp per triplet; the batch sum is reduced in a fixed order (deterministic).
#include "tt_simt.cuh"

namespace tt {

namespace {

constexpr float kCosEps = 1e-8f;  // torch.cosine_similarity eps (per-vector clamp)

__global__ void __launch_bounds__(128) triplet_fwd_kernel(const float* __restrict__ q, const float* __restrict__ p,
                                                          const float* __restrict__ n, int B, int P, float margin,
                                                          float* __restrict__ stats) {
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= B) return;
  const float* qi = q + (size_t)i * P;
  const float* pi = p + (size_t)i * P;
  const float* ni = n + (size_t)i * P;
  float qq = 0.f, pp = 0.f, nn = 0.f, qp = 0.f, qn = 0.f;
  for (int c = lane; c < P; c += 32) {
    const float a = qi[c], b = pi[c], d = ni[c];
    qq = fmaf(a, a, qq);
    pp = fmaf(b, b, pp);
    nn = fmaf(d, d, nn);
    qp = fmaf(a, b, qp);
    qn = fmaf(a, d, qn);
  }
  qq = warp_sum(qq); pp = warp_sum(pp); nn = warp_sum(nn); qp = warp_sum(qp); qn = warp_sum(qn);
  if (lane == 0) {
    const float nq = sqrtf(qq), np_ = sqrtf(pp), nn_ = sqrtf(nn);
    const float cq = fmaxf(nq, kCosEps), cp = fmaxf(np_, kCosEps), cn = fmaxf(nn_, kCosEps);
    const float cos_p = qp / (cq * cp), cos_n = qn / (cq * cn);
    // relu(pos_dist - neg_dist + margin), model.py:140-143
    const float hinge = fmaxf((1.f - cos_p) - (1.f - cos_n) + margin, 0.f);
    float* s = stats + (size_t)i * 8;
    s[0] = cos_p; s[1] = cos_n; s[2] = hinge; s[3] = nq; s[4] = np_; s[5] = nn_; s[6] = qp; s[7] = qn;
  }
}

// loss = inv_batch * sum_i hinge_i, single CTA, fixed tree order
__global__ void __launch_bounds__(1024) loss_reduce_kernel(const float* __restrict__ stats, int B, float inv_batch,
                                                           float* __restrict__ loss) {
  __shared__ float s[1024];
  float v = 0.f;
  for (int i = threadIdx.x; i < B; i += 1024) v += stats[(size_t)i * 8 + 2];
  s[threadIdx.x] = v;
  __syncthreads();
  for (int off = 512; off > 0; off >>= 1) {
    if (threadIdx.x < off) s[threadIdx.x] += s[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) *loss = s[0] * inv_batch;
}

__global__ void __launch_bounds__(128)
    triplet_bwd_kernel(const float* __restrict__ q, const float* __restrict__ p, const float* __restrict__ n,
                       const float* __restrict__ stats, const float* __restrict__ dloss, float grad_scale, int B, int P,
                       float inv_batch, float* __restrict__ dq, float* __restrict__ dp, float* __restrict__ dn,
                       LossSplitOut sp) {
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= B) return;
  const float* s = stats + (size_t)i * 8;
  const float cos_p = s[0], cos_n = s[1], hinge = s[2], nq = s[3], np_ = s[4], nn_ = s[5];
  const float up = (dloss ? *dloss : 1.f) * grad_scale;
  // d loss / d hinge_i = inv_batch (mean); relu subgradient 0 at 0; d hinge/d cos_p = -1, d cos_n = +1
  const float gh = (hinge > 0.f) ? up * inv_batch : 0.f;
  const float cq = fmaxf(nq, kCosEps), cp = fmaxf(np_, kCosEps), cn = fmaxf(nn_, kCosEps);
  // cos(x,y) = x.y/(cx cy), cx = max(|x|,eps):  d/dx = y/(cx cy) - [|x|>eps] cos x/(cx |x|)
  const float a_qp = -gh / (cq * cp), a_qn = gh / (cq * cn);
  const float kq = (nq > kCosEps) ? (-gh * cos_p + gh * cos_n) / (cq * nq) : 0.f;
  const float kp = (np_ > kCosEps) ? (-gh * cos_p) / (cp * np_) : 0.f;
  const float kn = (nn_ > kCosEps) ? (gh * cos_n) / (cn * nn_) : 0.f;
  const size_t o = (size_t)i * P;
  for (int c = lane; c < P; c += 32) {
    const float a = q[o + c], b = p[o + c], d = n[o + c];
    const float gq = a_qp * b + a_qn * d - kq * a;
    const float gp = a_qp * a - kp * b;
    const float gn = a_qn * a - kn * d;
    if (dq) { dq[o + c] = gq; dp[o + c] = gp; dn[o + c] = gn; }
    if (sp.dy_hi) {
      const float gv[3] = {gq, gp, gn};
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        __nv_bfloat16 hi, lo;
        split_bf16(gv[t], hi, lo);
        const size_t row = (size_t)t * B + i;
        sp.dy_hi[row * P + c] = hi;
        sp.dy_lo[row * P + c] = lo;
        if (sp.dyt_hi) {
          const size_t tcol = row + ((long long)row >= sp.t_split_row ? sp.t_shift : 0);
          sp.dyt_hi[(size_t)c * sp.ldt + tcol] = hi;
          sp.dyt_lo[(size_t)c * sp.ldt + tcol] = lo;
        }
      }
    }
  }
}

// fused forward + backward (one warp per triplet, rows re-read from L1 for the gradient)
__global__ void __launch_bounds__(128)
    triplet_fused_kernel(const float* __restrict__ q, const float* __restrict__ p, const float* __restrict__ n, int B,
                         int P, float margin, float inv_batch, float grad_scale, float* __restrict__ stats,
                         float* __restrict__ loss, float* __restrict__ dq, float* __restrict__ dp,
                         float* __restrict__ dn, LossSplitOut sp, float* __restrict__ scratch) {
  __shared__ float s_h[4];
  __shared__ int s_last;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 4 + w;
  float hinge = 0.f;
  if (i < B) {
    const size_t o = (size_t)i * P;
    float qq = 0.f, pp = 0.f, nn = 0.f, qp = 0.f, qn = 0.f;
    for (int c = lane; c < P; c += 32) {
      const float a = q[o + c], b = p[o + c], d = n[o + c];
      qq = fmaf(a, a, qq);
      pp = fmaf(b, b, pp);
      nn = fmaf(d, d, nn);
      qp = fmaf(a, b, qp);
      qn = fmaf(a, d, qn);
    }
    qq = warp_sum(qq); pp = warp_sum(pp); nn = warp_sum(nn); qp = warp_sum(qp); qn = warp_sum(qn);
    const float nq = sqrtf(qq), np_ = sqrtf(pp), nn_ = sqrtf(nn);
    const float cq = fmaxf(nq, kCosEps), cp = fmaxf(np_, kCosEps), cn = fmaxf(nn_, kCosEps);
    const float cos_p = qp / (cq * cp), cos_n = qn / (cq * cn);
    hinge = fmaxf((1.f - cos_p) - (1.f - cos_n) + margin, 0.f);
    if (lane == 0) {
      float* s = stats + (size_t)i * 8;
      s[0] = cos_p; s[1] = cos_n; s[2] = hinge; s[3] = nq; s[4] = np_; s[5] = nn_; s[6] = qp; s[7] = qn;
    }
    const float gh = (hinge > 0.f) ? grad_scale * inv_batch : 0.f;
    const float a_qp = -gh / (cq * cp), a_qn = gh / (cq * cn);
    const float kq = (nq > kCosEps) ? (-gh * cos_p + gh * cos_n) / (cq * nq) : 0.f;
    const float kp = (np_ > kCosEps) ? (-gh * cos_p) / (cp * np_) : 0.f;
    const float kn = (nn_ > kCosEps) ? (gh * cos_n) / (cn * nn_) : 0.f;
    for (int c = lane; c < P; c += 32) {
      const float a = q[o + c], b = p[o + c], d = n[o + c];
      const float gv[3] = {a_qp * b + a_qn * d - kq * a, a_qp * a - kp * b, a_qn * a - kn * d};
      dq[o + c] = gv[0];
      dp[o + c] = gv[1];
      dn[o + c] = gv[2];
      if (sp.dy_hi) {
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          __nv_bfloat16 hi, lo;
          split_bf16(gv[t], hi, lo);
          const size_t row = (size_t)t * B + i;
          sp.dy_hi[row * P + c] = hi;
          sp.dy_lo[row * P + c] = lo;
        }
      }
    }
  }
  if (lane == 0) s_h[w] = hinge;
  __syncthreads();
  const int nblk = gridDim.x;
  unsigned* counter = reinterpret_cast<unsigned*>(scratch + nblk + 1);
  if (threadIdx.x == 0) {
    scratch[blockIdx.x] = (s_h[0] + s_h[1]) + (s_h[2] + s_h[3]);
    __threadfence();
    s_last = (atomicAdd(counter, 1u) == (unsigned)nblk - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // last block: fixed-order sum of the per-block partials (independent of which block arrived last)
  __shared__ float s_red[128];
  float v = 0.f;
  for (int b = threadIdx.x; b < nblk; b += 128) v += __ldcg(scratch + b);
  s_red[threadIdx.x] = v;
  __syncthreads();
  for (int off = 64; off > 0; off >>= 1) {
    if (threadIdx.x < off) s_red[threadIdx.x] += s_red[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *loss = s_red[0] * inv_batch;
    *counter = 0u;  // ready for the next launch / graph replay
  }
}

}  // namespace

int triplet_loss_fused(const float* q, const float* p, const float* n, int B, int P, float margin, float inv_batch,
                       float grad_scale, float* stats, float* loss, float* dq, float* dp, float* dn,
                       const LossSplitOut* split, float* scratch, cudaStream_t st) {
  TT_REQUIRE(B >= 1, "triplet loss: empty batch");
  LossSplitOut sp{};
  if (split) sp = *split;
  triplet_fused_kernel<<<(B + 3) / 4, 128, 0, st>>>(q, p, n, B, P, margin, inv_batch, grad_scale, stats, loss, dq, dp,
                                                    dn, sp, scratch);
  TT_LAUNCH_CHECK();
  return 0;
}

int triplet_loss_fwd(const float* q, const float* p, const float* n, int B, int P, float margin, float inv_batch,
                     float* stats, float* loss, cudaStream_t st) {
  if (B > 0) {
    triplet_fwd_kernel<<<(B + 3) / 4, 128, 0, st>>>(q, p, n, B, P, margin, stats);
    TT_LAUNCH_CHECK();
  }
  loss_reduce_kernel<<<1, 1024, 0, st>>>(stats, B, inv_batch, loss);
  TT_LAUNCH_CHECK();
  return 0;
}

int triplet_loss_bwd(const float* q, const float* p, const float* n, const float* stats, const float* dloss,
                     float grad_scale, int B, int P, float inv_batch, float* dq, float* dp, float* dn,
                     const LossSplitOut* split, cudaStream_t st) {
  if (B <= 0) return 0;
  LossSplitOut sp{};
  if (split) sp = *split;
  triplet_bwd_kernel<<<(B + 3) / 4, 128, 0, st>>>(q, p, n, stats, dloss, grad_scale, B, P, inv_batch, dq, dp, dn, sp);
  TT_LAUNCH_CHECK();
  return 0;
}

}  // namespace tt

extern "C" int tt_triplet_loss_fwd(const float* q, const float* p, const float* n, int B, int P, float margin,
                                   float inv_batch, float* stats, float* loss, tt_stream_t stream) {
  TT_REQUIRE(B >= 0 && P >= 1, "tt_triplet_loss_fwd: bad shape B=%d P=%d", B, P);
  return tt::triplet_loss_fwd(q, p, n, B, P, margin, inv_batch, stats, loss, tt::as_stream(stream));
}

extern "C" int tt_triplet_loss_bwd(const float* q, const float* p, const float* n, const float* stats,
                                   const float* dloss, int B, int P, float inv_batch, float* dq, float* dp, float* dn,
                                   tt_stream_t stream) {
  TT_REQUIRE(B >= 0 && P >= 1, "tt_triplet_loss_bwd: bad shape B=%d P=%d", B, P);
  TT_REQUIRE(dq && dp && dn, "tt_triplet_loss_bwd: null output");
  return tt::triplet_loss_bwd(q, p, n, stats, dloss, 1.f, B, P, inv_batch, dq, dp, dn, nullptr, tt::as_stream(stream));
}

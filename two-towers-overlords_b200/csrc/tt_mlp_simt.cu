// fp32 strict-parity projection MLP on CUDA cores (TT_PREC_FP32): a strided 64x64x16 SGEMM with a
// fused epilogue, a fixed-order split over the batch rows for the weight gradients, plus deterministic column sums
// for the bias gradients.
// Replaces backend/model.py:33-38,59 (forward) and what autograd does for it in training.py:50.
#include "tt_simt.cuh"

namespace tt {

namespace {

constexpr int BM = 64, BN = 64, BK = 16;

template <bool A_KFAST, bool B_KFAST>
__global__ void __launch_bounds__(256) sgemm_kernel(const SgemmArgs g) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  // slice blockIdx.z of a split contraction sums k in [kbeg, kend) into its own [M, ldc] block of C
  const int kbeg = blockIdx.z * g.kslice, kend = g.kslice ? min(g.K, kbeg + g.kslice) : g.K;
  float* __restrict__ C = g.C + (size_t)blockIdx.z * g.M * g.ldc;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = kbeg; k0 < kend; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      int m, k;
      if (A_KFAST) { k = idx & 15; m = idx >> 4; } else { m = idx & 63; k = idx >> 6; }
      const int gm = m0 + m, gk = k0 + k;
      As[k][m] = (gm < g.M && gk < kend) ? __ldg(g.A + gm * g.a_sm + gk * g.a_sk) : 0.f;
      int n, kb;
      if (B_KFAST) { kb = idx & 15; n = idx >> 4; } else { n = idx & 63; kb = idx >> 6; }
      const int gn = n0 + n, gkb = k0 + kb;
      Bs[kb][n] = (gn < g.N && gkb < kend) ? __ldg(g.B + gn * g.b_sn + gkb * g.b_sk) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j];
      if (g.bias) v += g.bias[n];
      if (g.relu) v = fmaxf(v, 0.f);
      const size_t o = (size_t)m * g.ldc + n;
      if (g.gate) v = (g.gate[o] > 0.f) ? v : 0.f;
      C[o] = g.accumulate ? (C[o] + v) : v;
    }
  }
}

// two-stage column sums for up to two matrices per launch (query | document rows): slices of rows are summed
// by separate CTAs into scratch[job][slice][N], then added in ascending slice order (deterministic).  The sums
// accumulate in double: the bias gradient of the document tower adds positive and negative rows whose dY nearly cancel
// column by column (condition number ~5e4 at B = 8256), where fp32 running sums over ~65 rows per thread were 2e-3 off.
__global__ void __launch_bounds__(256) colsum_partial_kernel(const float* __restrict__ X0, int M0,
                                                             const float* __restrict__ X1, int M1, int N, long long ld,
                                                             int S, float* __restrict__ scratch) {
  __shared__ double s[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int job = blockIdx.z, slice = blockIdx.y;
  const float* X = job ? X1 : X0;
  const int M = job ? M1 : M0;
  const int per = (M + S - 1) / S;
  const int r0 = slice * per, r1 = min(M, r0 + per);
  const int n = blockIdx.x * 32 + tx;
  double sum = 0.0;
  if (n < N)
    for (int m = r0 + ty; m < r1; m += 8) sum += (double)X[(size_t)m * ld + n];
  s[ty][tx] = sum;
  __syncthreads();
  if (ty == 0 && n < N) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += s[i][tx];
    scratch[((size_t)job * S + slice) * N + n] = (float)t;
  }
}

__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ scratch, int S, int N,
                                                           float* __restrict__ out0, float* __restrict__ out1,
                                                           int accumulate) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  const int job = blockIdx.y;
  if (n >= N) return;
  double t = 0.0;
  for (int i = 0; i < S; ++i) t += (double)scratch[((size_t)job * S + i) * N + n];
  float* out = job ? out1 : out0;
  if (accumulate == kAccumAfterSum) out[n] = out[n] + (float)t;
  else out[n] = accumulate ? (float)((double)out[n] + t) : (float)t;
}

// out[i] = sum_z partial[z][i], z ascending, in double (the weight-gradient slices of sgemm_rows); accumulate as for
// colsum2
__global__ void __launch_bounds__(256) slice_sum_kernel(const float* __restrict__ partial, int S, size_t n,
                                                        float* __restrict__ out, int accumulate) {
  const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  double t = 0.0;
  for (int z = 0; z < S; ++z) t += (double)partial[(size_t)z * n + i];
  if (accumulate == kAccumAfterSum) out[i] = out[i] + (float)t;
  else out[i] = accumulate ? (float)((double)out[i] + t) : (float)t;
}

}  // namespace

int colsum2(const float* X0, int M0, float* out0, const float* X1, int M1, float* out1, int N, long long ld,
            int accumulate, float* scratch, cudaStream_t st) {
  if (N <= 0) return 0;
  const int njobs = X1 ? 2 : 1;
  dim3 grid((N + 31) / 32, kColsumSlices, njobs);
  colsum_partial_kernel<<<grid, 256, 0, st>>>(X0, M0, X1, M1, N, ld, (int)kColsumSlices, scratch);
  TT_LAUNCH_CHECK();
  colsum_final_kernel<<<dim3((N + 255) / 256, njobs), 256, 0, st>>>(scratch, (int)kColsumSlices, N, out0, out1,
                                                                     accumulate);
  TT_LAUNCH_CHECK();
  return 0;
}

// the kernel instance for the operands' layouts, over `slices` row slices (sgemm_rows) or the whole K
static int launch_sgemm(const SgemmArgs& a, int slices, cudaStream_t st) {
  dim3 grid((a.N + BN - 1) / BN, (a.M + BM - 1) / BM, slices);
  const bool ak = a.a_sk == 1, bk = a.b_sk == 1;
  if (ak && bk) sgemm_kernel<true, true><<<grid, 256, 0, st>>>(a);
  else if (ak) sgemm_kernel<true, false><<<grid, 256, 0, st>>>(a);
  else if (bk) sgemm_kernel<false, true><<<grid, 256, 0, st>>>(a);
  else sgemm_kernel<false, false><<<grid, 256, 0, st>>>(a);
  TT_LAUNCH_CHECK();
  return 0;
}

int sgemm(const SgemmArgs& a, cudaStream_t st) {
  if (a.M <= 0 || a.N <= 0) return 0;
  return launch_sgemm(a, 1, st);
}

int row_slices(int K) {
  const int kb = (K + BK - 1) / BK, per = (kb + kRowSlices - 1) / kRowSlices;
  return kb ? (kb + per - 1) / per : 1;  // no empty slice
}

int sgemm_rows(const SgemmArgs& a, float* partial, cudaStream_t st) {
  if (a.M <= 0 || a.N <= 0) return 0;
  TT_REQUIRE(!a.bias && !a.relu && !a.gate && a.ldc == a.N, "sgemm_rows: plain dense output only");
  const int kb = (a.K + BK - 1) / BK, per = (kb + kRowSlices - 1) / kRowSlices, S = row_slices(a.K);
  SgemmArgs p = a;
  p.C = partial;
  p.accumulate = 0;
  p.kslice = per * BK;  // slice S - 1 starts at (S - 1) * per < kb k-steps: none is empty
  int rc = launch_sgemm(p, S, st);
  if (rc) return rc;
  const size_t n = (size_t)a.M * a.N;
  slice_sum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, S, n, a.C, a.accumulate);
  TT_LAUNCH_CHECK();
  return 0;
}

int mlp_fwd_fp32(const float* x, int M, int H, int P, const float* W1, const float* b1, const float* W2,
                 const float* b2, float* h, float* y, cudaStream_t st) {
  SgemmArgs g1{x, H, 1, W1, H, 1, h, P, M, P, H, b1, 1, nullptr, 0, 0};
  int rc = sgemm(g1, st);
  if (rc) return rc;
  SgemmArgs g2{h, P, 1, W2, P, 1, y, P, M, P, P, b2, 0, nullptr, 0, 0};
  return sgemm(g2, st);
}

int mlp_bwd_fp32(const float* dy, const float* x, const float* h, const float* W1, const float* W2, int M, int H,
                 int P, float* dW1, float* db1, float* dW2, float* db2, float* dx, int accumulate, float* dz1,
                 float* scratch, cudaStream_t st) {
  int rc;
  // the sums over the M batch rows: the bias gradients in colsum2's double slices, the weight gradients in
  // row_slices(M) fixed slices.  Positive and negative rows of the document tower's dY nearly cancel column by column
  // (condition number ~5e4 at M = 2B = 16512), where one fp32 FMA chain over all M rows left dW2 1.0e-3 off.
  float* partial = scratch;
  float* cs = scratch + (size_t)row_slices(M) * P * (P > H ? P : H);
  // db2[n] = sum_m dy[m,n];  dW2[n,k] = sum_m dy[m,n] h[m,k]
  if ((rc = colsum2(dy, M, db2, nullptr, 0, nullptr, P, P, accumulate, cs, st))) return rc;
  SgemmArgs gw2{dy, 1, P, h, 1, P, dW2, P, P, P, M, nullptr, 0, nullptr, accumulate, 0};
  if ((rc = sgemm_rows(gw2, partial, st))) return rc;
  // dz1 = (dy W2) * (h > 0)
  SgemmArgs gh{dy, P, 1, W2, 1, P, dz1, P, M, P, P, nullptr, 0, h, 0, 0};
  if ((rc = sgemm(gh, st))) return rc;
  if ((rc = colsum2(dz1, M, db1, nullptr, 0, nullptr, P, P, accumulate, cs, st))) return rc;
  // dW1[p,k] = sum_m dz1[m,p] x[m,k]
  SgemmArgs gw1{dz1, 1, P, x, 1, H, dW1, H, P, H, M, nullptr, 0, nullptr, accumulate, 0};
  if ((rc = sgemm_rows(gw1, partial, st))) return rc;
  if (dx) {
    SgemmArgs gx{dz1, P, 1, W1, 1, H, dx, H, M, H, P, nullptr, 0, nullptr, 0, 0};
    if ((rc = sgemm(gx, st))) return rc;
  }
  return 0;
}

size_t mlp_bwd_fp32_scratch_floats(int M, int H, int P) {
  return (size_t)row_slices(M) * P * (P > H ? P : H) + (size_t)kColsumSlices * P;
}

}  // namespace tt

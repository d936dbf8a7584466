#pragma once
#include "tt_common.cuh"

namespace tt {

// C[m,n] = epi( sum_k A(m,k) * B(n,k) ), A(m,k) = A[m*a_sm + k*a_sk], B(n,k) = B[n*b_sn + k*b_sk].
// epi: (+bias[n]) -> (relu) -> (* (gate[m*ldc+n] > 0)) -> (C += | C =)
// kslice > 0 (set by sgemm_rows): CTA z sums k in [z*kslice, (z+1)*kslice) into C + z*M*ldc
struct SgemmArgs {
  const float* A;
  long long a_sm, a_sk;
  const float* B;
  long long b_sn, b_sk;
  float* C;
  long long ldc;
  int M, N, K;
  const float* bias;
  int relu;
  const float* gate;
  int accumulate;
  int kslice;
};
int sgemm(const SgemmArgs& a, cudaStream_t st);

// `accumulate` of colsum2 and of the split-K reduction (launch_gemm): 0 = out is overwritten; kAccumOldFirst = the
// running sum starts from out (tt_encode_bwd); kAccumAfterSum = out = fl(out + sum) in fp32, the sum being exactly what
// 0 writes (tt_step_args.grad_accumulate, autograd's `.grad += new`)
constexpr int kAccumOldFirst = 1, kAccumAfterSum = 2;

// same sums for one or two matrices (X1 nullable) in two launches; scratch: 2 * kColsumSlices * N floats
constexpr int kColsumSlices = 32;
int colsum2(const float* X0, int M0, float* out0, const float* X1, int M1, float* out1, int N, long long ld,
            int accumulate, float* scratch, cudaStream_t st);

// C [M, N] dense (+)= sum_k A(m,k) B(n,k) as row_slices(K) fixed, non-empty slices of K (at most kRowSlices), each an
// sgemm into partial [slice][M*N], then added in ascending slice order in double; accumulate as for colsum2.  For the
// weight gradients, whose K is the batch: short fp32 chains, and a grid of slices x tiles instead of tiles alone.
constexpr int kRowSlices = 32;
int row_slices(int K);
int sgemm_rows(const SgemmArgs& a, float* partial, cudaStream_t st);

// fp32 strict-mode projection (tt_mlp_simt.cu).  mlp_bwd_fp32: dz1 [M, P]; scratch of
// mlp_bwd_fp32_scratch_floats(M, H, P) floats (weight-gradient slices, column-sum slices); accumulate as for colsum2
int mlp_fwd_fp32(const float* x, int M, int H, int P, const float* W1, const float* b1, const float* W2,
                 const float* b2, float* h, float* y, cudaStream_t st);
int mlp_bwd_fp32(const float* dy, const float* x, const float* h, const float* W1, const float* W2, int M, int H,
                 int P, float* dW1, float* db1, float* dW2, float* db2, float* dx, int accumulate, float* dz1,
                 float* scratch, cudaStream_t st);
size_t mlp_bwd_fp32_scratch_floats(int M, int H, int P);

// loss (tt_loss.cu)
struct LossSplitOut {  // optional operands for the tensor-core backward: dY as bf16 hi/lo, row-major + transposed
  __nv_bfloat16 *dy_hi, *dy_lo;    // [3B, P]
  __nv_bfloat16 *dyt_hi, *dyt_lo;  // [P, ldt]
  int ldt;
  int t_split_row, t_shift;        // transposed column of row r: r + (r >= t_split_row ? t_shift : 0)
};
int triplet_loss_fwd(const float* q, const float* p, const float* n, int B, int P, float margin, float inv_batch,
                     float* stats, float* loss, cudaStream_t st);
// forward + backward in one launch (the fused step): per-block hinge sums go to scratch[0 .. ceil(B/4)), the last block
// to finish adds them in index order (deterministic) and writes the loss; scratch[ceil(B/4) + 1] is the arrival counter,
// which must be zero before the first call (it is reset by the kernel, so graph replays need no memset)
int triplet_loss_fused(const float* q, const float* p, const float* n, int B, int P, float margin, float inv_batch,
                       float grad_scale, float* stats, float* loss, float* dq, float* dp, float* dn,
                       const LossSplitOut* split, float* scratch, cudaStream_t st);
int triplet_loss_bwd(const float* q, const float* p, const float* n, const float* stats, const float* dloss,
                     float grad_scale, int B, int P, float inv_batch, float* dq, float* dp, float* dn,
                     const LossSplitOut* split, cudaStream_t st);

}  // namespace tt

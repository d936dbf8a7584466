// tcgen05 / TMA (sm_100a) paths: projection GEMMs with fused epilogues and the tensor-core corpus scan.
#pragma once
#include "tt_common.cuh"
#include "tt_pool.cuh"

namespace tt {

size_t mlp_sm100_ws_bytes(int M, int H, int P);
int mlp_fwd_sm100(const float* x, int M, int H, int P, const float* W1, const float* b1, const float* W2,
                  const float* b2, float* h, float* y, int precision, void* ws, size_t ws_bytes, cudaStream_t st);
int mlp_bwd_sm100(const float* dy, const float* x, const float* h, const float* W1, const float* W2, int M, int H,
                  int P, float* dW1, float* db1, float* dW2, float* db2, float* dx, int accumulate, int precision,
                  void* ws, size_t ws_bytes, cudaStream_t st);

struct FusedAdam {  // optional optimiser in the tail of the persistent chain kernel (param == nullptr: gradients only)
  double* state;
  float *param, *grad, *exp_avg, *exp_avg_sq;
  size_t n;
  float lr, beta1, beta2, eps;
};

struct StepSm100 {
  PoolParams pool;  // xhat/cnt/nrm/err filled by the caller; split outputs filled by step_sm100
  int table_dtype;
  int B, H, P;
  const float *Wq1, *bq1, *Wq2, *bq2, *Wd1, *bd1, *Wd2, *bd2;
  float margin, inv_batch, grad_scale;
  float* loss;
  float *dWq1, *dbq1, *dWq2, *dbq2, *dWd1, *dbd1, *dWd2, *dbd2;
  float *h, *y, *stats, *dy;  // fp32 activations [3B,P] / [B,8]
  float* dxhat;               // [3B,H] nullable
  int n_split;                // 3 = bf16x3, 1 = bf16
  void* ws;
  size_t ws_bytes;
  int phases;                 // 0 / TT_STEP_FRONT | TT_STEP_BACK
  FusedAdam adam;
  bool chain;                 // persistent chain kernel (else one kernel per contraction)
  int grad_accumulate;        // 1: every gradient output becomes fl(old + new) (tt_step_args.grad_accumulate)
};
size_t step_sm100_ws_bytes(int B, int H, int P, int train_table);
int step_sm100(const StepSm100& s, cudaStream_t st);
// persistent chain kernel (tt_chain_sm100.cu): everything of the step after the pooled gather in ONE launch
bool chain_enabled();  // TT_CHAIN=0 selects the per-kernel chain for tt_step_args.chain == 0
int chain_sm100(const StepSm100& s, bool after_gather, cudaStream_t st);

// generic tensor-core contraction on bf16 (hi, lo) terms: C = act(A B^T + bias); act: 0 none, 1 ReLU, 2 GELU (erf)
int gemm_terms_sm100(const __nv_bfloat16* A_hi, const __nv_bfloat16* A_lo, long long lda, const __nv_bfloat16* B_hi,
                     const __nv_bfloat16* B_lo, long long ldb, int M, int N, int K, const float* bias, int act, float* C,
                     int ldc, __nv_bfloat16* C_hi, __nv_bfloat16* C_lo, cudaStream_t st);
int split_terms_sm100(const float* X, int R, int C, __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t st);

size_t scan_sm100_ws_bytes(int Q, long long N, int P, int k);
int scan_topk_sm100(const float* Qn, const float* Dn, const void* Qb, const void* Db, int Q, long long N, int P, int k,
                    long long id_base, float* top_score, long long* top_id, void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace tt

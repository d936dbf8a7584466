#pragma once
#include "tt_common.cuh"

namespace tt {

struct PoolSegDev {
  const void* table;
  const void* ids;
  const void* mask;
  int B, L, row0;
};

struct PoolParams {
  PoolSegDev seg[4];
  int nseg;
  int ids_dtype, mask_dtype;
  int vocab;
  float* xhat;  // [rows, H]
  float* cnt;   // [rows] nullable
  float* nrm;   // [rows] nullable
  int* err;     // nullable
  // optional operands for the tensor-core projection (bf16 hi/lo split, row-major)
  __nv_bfloat16* x_hi;   // [rows, H]
  __nv_bfloat16* x_lo;
  __nv_bfloat16* x_lo2;  // nullable third term: xhat - hi - lo
  int share_sm;  // 1: this launch runs beside other kernels (pipelined step): fewer rows in flight per warp
  // optional row aliases: output row alias_dst_row0 + i is a copy of output row alias_src_row0 + alias[i], i < alias_n
  // (in-batch negatives: negative i is the positive document of item alias[i]); nullptr = none
  const int* alias;
  int alias_n, alias_src_row0, alias_dst_row0;
  // optional precomputed pooled rows (a frozen front end encoded once per text): when row_index != nullptr the launch
  // copies output row r = s * row_B + i (s = 0 query, 1 positive, 2 negative) from row row_index[r] of rows_q (s = 0)
  // or rows_d, instead of pooling tokens; seg[], cnt and nrm are not used then
  const float* rows_q;
  const float* rows_d;
  long long rows_q_n, rows_d_n;
  const int* row_index;  // [3 * row_B]
  int row_B;
};

int pool_fwd_launch(PoolParams p, int table_dtype, int H, cudaStream_t st);

// backward (tt_pool_bwd.cu)
struct PoolBwdSeg {
  const void* ids;
  const void* mask;
  int B, L, row0;
};
size_t pool_bwd_ws_bytes(long long n_tokens, int vocab);
// g [rows,H]: per-sequence gradient of the masked SUM's mean, i.e. d(loss)/d(pooled mean)/cnt;
// dtable[id] (+)= sum over tokens with that id of mask_t * g[seq(t)], reduced in position order.
int pool_bwd_scatter(const PoolBwdSeg* segs, int nseg, int ids_dtype, int mask_dtype, const float* g,
                     int vocab, int H, float* dtable, int accumulate, void* ws, size_t ws_bytes,
                     cudaStream_t st);
// dxhat -> g: through F.normalize and the mean (rows [0,rows))
int pool_bwd_prep(const float* dxhat, const float* xhat, const float* cnt, const float* nrm, int rows,
                  int H, float* g, cudaStream_t st);

}  // namespace tt

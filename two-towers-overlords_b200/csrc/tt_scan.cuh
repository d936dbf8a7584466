#pragma once
#include "tt_common.cuh"

namespace tt {

int scan_splits(int Q, long long N);
size_t scan_fp32_ws_bytes(int Q, long long N, int k);
int scan_topk_fp32(const float* Qn, const float* Dn, int Q, long long N, int P, int k, long long id_base,
                   float* top_score, long long* top_id, void* ws, size_t ws_bytes, cudaStream_t st);
constexpr int kListedSplits = 64;
size_t scan_listed_ws_bytes(int cap, int k);
int scan_topk_fp32_listed(const float* Qn, const float* Dn, int Q, long long N, int P, int k, long long id_base,
                          const int* qlist, const int* qcount, int cap, float* top_score, long long* top_id, void* ws,
                          cudaStream_t st);
int scan_empty(int Q, int k, float* top_score, long long* top_id, cudaStream_t st);
int topk_merge(const float* ps, const long long* pi, int G, int Q, int k, float* os, long long* oi, cudaStream_t st);
int score_candidates(const float* Qn, const float* Dn, const long long* cand, int Q, int C, int P, int k,
                     long long id_base, float* os, long long* oi, float* all_scores, cudaStream_t st);

}  // namespace tt

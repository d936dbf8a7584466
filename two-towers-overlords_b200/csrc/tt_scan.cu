// Retrieval / evaluation kernels (reference: backend/training.py:244-311 restated as a batched scan).
//   - row normalisation with the per-vector clamp of torch.cosine_similarity
//   - exhaustive corpus scan with fused top-k (fp32 strict mode here; tensor-core mode in tt_scan_sm100.cu)
//   - exact candidate re-scoring, partial top-k merge, NDCG@k
// Order everywhere: (score descending, id ascending).
#include "tt_scan.cuh"

namespace tt {

namespace {

__device__ __forceinline__ bool better(float s1, long long i1, float s2, long long i2) {
  return s1 > s2 || (s1 == s2 && i1 < i2);
}

// ---- normalise rows ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) l2norm_rows_kernel(const float* __restrict__ x, long long N, int P, float eps,
                                                          float* __restrict__ y, __nv_bfloat16* __restrict__ yb) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= N) return;
  const float* xr = x + row * P;
  float sq = 0.f;
  for (int c = lane; c < P; c += 32) sq = fmaf(xr[c], xr[c], sq);
  sq = warp_sum(sq);
  const float d = fmaxf(sqrtf(sq), eps);
  for (int c = lane; c < P; c += 32) {
    const float v = xr[c] / d;
    if (y) y[row * P + c] = v;
    if (yb) yb[row * P + c] = __float2bfloat16_rn(v);
  }
}

// ---- fp32 scan with fused top-k --------------------------------------------------------------------
constexpr int SQ = 64, SD = 64, SK = 16;

__global__ void __launch_bounds__(256)
    scan_topk_fp32_kernel(const float* __restrict__ Qn, const float* __restrict__ Dn, int Q, long long N, int P, int k,
                          long long docs_per_split, long long id_base, float* __restrict__ part_score,
                          long long* __restrict__ part_id, const int* __restrict__ qlist,
                          const int* __restrict__ qcount, int slot0) {
  // indirect mode (qlist != null): this launch owns slots [slot0, slot0 + Q) of a device-side list of query rows
  // (the re-scan of queries whose tensor-core candidates could not be proven complete); empty tiles exit at once
  int n_slots = Q;
  if (qlist) {
    n_slots = min(Q, *qcount - slot0);
    if ((int)blockIdx.y * SQ >= n_slots) return;
  }
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float (*As)[SQ + 4] = reinterpret_cast<float (*)[SQ + 4]>(smem_raw);
  float (*Bs)[SD + 4] = reinterpret_cast<float (*)[SD + 4]>(smem_raw + sizeof(float) * SK * (SQ + 4));
  float (*S)[SD + 1] = reinterpret_cast<float (*)[SD + 1]>(smem_raw + sizeof(float) * SK * (SQ + 4 + SD + 4));
  float* l_score = reinterpret_cast<float*>(smem_raw + sizeof(float) * (SK * (SQ + 4 + SD + 4) + SQ * (SD + 1)));
  long long* l_id = reinterpret_cast<long long*>(l_score + SQ * k + (((SQ * k) & 1) ? 1 : 0));

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int q0 = blockIdx.y * SQ;
  const long long d_beg = (long long)blockIdx.x * docs_per_split;
  const long long d_end = min(d_beg + docs_per_split, N);

  for (int i = tid; i < SQ * k; i += 256) {
    l_score[i] = -INFINITY;
    l_id[i] = -1;
  }
  __syncthreads();

  for (long long d0 = d_beg; d0 < d_end; d0 += SD) {
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < P; k0 += SK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int idx = tid + i * 256;
        const int kk = idx & 15, r = idx >> 4;
        const int gq = q0 + r;
        const long long gd = d0 + r;
        const int gk = k0 + kk;
        const int qrow = (qlist && gq < n_slots) ? qlist[slot0 + gq] : gq;
        As[kk][r] = (gq < n_slots && gk < P) ? __ldg(Qn + (size_t)qrow * P + gk) : 0.f;
        Bs[kk][r] = (gd < d_end && gk < P) ? __ldg(Dn + (size_t)gd * P + gk) : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < SK; ++kk) {
        const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
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
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) S[ty * 4 + i][tx * 4 + j] = acc[i][j];
    __syncthreads();
    if (tid < SQ && q0 + tid < n_slots) {  // one thread per query walks its 64 scores in ascending doc id
      float* ls = l_score + tid * k;
      long long* li = l_id + tid * k;
      const int nd = (int)min((long long)SD, d_end - d0);
      float thr = ls[k - 1];
      for (int j = 0; j < nd; ++j) {
        const float sc = S[tid][j];
        if (sc > thr) {  // equal score with a larger id never displaces
          int pos = k - 1;
          while (pos > 0 && ls[pos - 1] < sc) {
            ls[pos] = ls[pos - 1];
            li[pos] = li[pos - 1];
            --pos;
          }
          ls[pos] = sc;
          li[pos] = id_base + d0 + j;
          thr = ls[k - 1];
        }
      }
    }
    __syncthreads();
  }
  for (int i = tid; i < SQ * k; i += 256) {
    const int r = i / k, c = i % k;
    if (q0 + r < n_slots) {
      const size_t o = ((size_t)blockIdx.x * Q + q0 + r) * k + c;
      part_score[o] = l_score[i];
      part_id[o] = l_id[i];
    }
  }
}

// ---- merge G sorted partial lists per query ----------------------------------------------------------
__global__ void __launch_bounds__(256) topk_merge_kernel(const float* __restrict__ ps, const long long* __restrict__ pi,
                                                         int G, int Q, int k, float* __restrict__ os,
                                                         long long* __restrict__ oi, const int* __restrict__ qlist,
                                                         const int* __restrict__ qcount, int slot0) {
  const int q = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= Q) return;
  int qo = q;  // output row; indirect mode scatters slot (slot0 + q) back to its query row
  if (qlist) {
    if (slot0 + q >= *qcount) return;
    qo = qlist[slot0 + q];
  }
  float last_s = INFINITY;
  long long last_i = -1;
  const int total = G * k;
  for (int r = 0; r < k; ++r) {
    float bs = -INFINITY;
    long long bi = -1;
    for (int c = lane; c < total; c += 32) {
      const int g = c / k, j = c % k;
      const size_t o = ((size_t)g * Q + q) * k + j;
      const long long id = pi[o];
      if (id < 0) continue;
      const float s = ps[o];
      // candidates strictly after the previous pick in the (score desc, id asc) order
      const bool after = (r == 0) || better(last_s, last_i, s, id);
      if (after && (bi < 0 || better(s, id, bs, bi))) {
        bs = s;
        bi = id;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float s2 = __shfl_xor_sync(0xffffffffu, bs, off);
      const long long i2 = __shfl_xor_sync(0xffffffffu, bi, off);
      if (i2 >= 0 && (bi < 0 || better(s2, i2, bs, bi))) {
        bs = s2;
        bi = i2;
      }
    }
    if (lane == 0) {
      os[(size_t)qo * k + r] = (bi >= 0) ? bs : -INFINITY;
      oi[(size_t)qo * k + r] = bi;
    }
    if (bi < 0) {
      for (int rr = r + 1; rr < k; ++rr)
        if (lane == 0) {
          os[(size_t)qo * k + rr] = -INFINITY;
          oi[(size_t)qo * k + rr] = -1;
        }
      break;
    }
    last_s = bs;
    last_i = bi;
  }
}

// ---- exact candidate scoring ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
    score_candidates_kernel(const float* __restrict__ Qn, const float* __restrict__ Dn, const long long* __restrict__ cand,
                            int Q, int C, int P, int k, long long id_base, float* __restrict__ os,
                            long long* __restrict__ oi, float* __restrict__ all_scores) {
  extern __shared__ float s_sc[];  // [C]
  const int q = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* qr = Qn + (size_t)q * P;
  const long long* cq = cand + (size_t)q * C;
  for (int c = warp; c < C; c += 4) {
    const long long d = cq[c];
    float dot = 0.f;
    if (d >= 0) {
      const float* dr = Dn + (size_t)d * P;
      for (int j = lane; j < P; j += 32) dot = fmaf(qr[j], dr[j], dot);
      dot = warp_sum(dot);
    }
    if (lane == 0) {
      s_sc[c] = dot;
      if (all_scores) all_scores[(size_t)q * C + c] = dot;
    }
  }
  __syncthreads();
  if (warp != 0) return;
  float last_s = INFINITY;
  long long last_i = -1;
  for (int r = 0; r < k; ++r) {
    float bs = -INFINITY;
    long long bi = -1;
    for (int c = lane; c < C; c += 32) {
      const long long id = cq[c];
      if (id < 0) continue;
      const float s = s_sc[c];
      const bool after = (r == 0) || better(last_s, last_i, s, id);
      if (after && (bi < 0 || better(s, id, bs, bi))) {
        bs = s;
        bi = id;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float s2 = __shfl_xor_sync(0xffffffffu, bs, off);
      const long long i2 = __shfl_xor_sync(0xffffffffu, bi, off);
      if (i2 >= 0 && (bi < 0 || better(s2, i2, bs, bi))) {
        bs = s2;
        bi = i2;
      }
    }
    if (lane == 0) {
      os[(size_t)q * k + r] = (bi >= 0) ? bs : -INFINITY;
      oi[(size_t)q * k + r] = (bi >= 0) ? bi + id_base : -1;
    }
    if (bi >= 0) {
      last_s = bs;
      last_i = bi;
    } else {
      last_s = -INFINITY;  // nothing left: every later rank is empty too
      last_i = -1;
    }
  }
}

// ---- NDCG@k from top-k ids and CSR relevant sets ---------------------------------------------------------
__global__ void ndcg_kernel(const long long* __restrict__ top_id, int Q, int k, int kk, const long long* __restrict__ off,
                            const long long* __restrict__ rel, double* __restrict__ out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  const long long b = off[q], e = off[q + 1];
  double dcg = 0.0, idcg = 0.0;
  for (int r = 0; r < kk; ++r) {
    const double disc = 1.0 / log2((double)r + 2.0);
    if (r < e - b) idcg += disc;
    const long long id = top_id[(size_t)q * k + r];
    if (id < 0) continue;
    long long lo = b, hi = e;  // binary search in the sorted relevant list
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (rel[mid] < id) lo = mid + 1; else hi = mid;
    }
    if (lo < e && rel[lo] == id) dcg += disc;
  }
  out[q] = (idcg == 0.0) ? 0.0 : dcg / idcg;
}

}  // namespace

int scan_splits(int Q, long long N) {
  const int qtiles = (Q + SQ - 1) / SQ;
  long long want = (2ll * sm_count() + qtiles - 1) / qtiles;
  const long long max_splits = (N + SD - 1) / SD;
  if (want > max_splits) want = max_splits;
  if (want < 1) want = 1;
  return (int)want;
}

// Dynamic shared memory of scan_topk_fp32_kernel: two operand tiles, the score tile and a k-long list per query
// (25,352 + 768 k bytes).  Past 48 KB (k > 30) the kernel must opt in, once per process; the 227 KB of an SM100 block
// are what bounds k.
static int fp32_scan_smem(int k, size_t* smem) {
  constexpr size_t kMaxSmem = 227 * 1024;
  *smem = sizeof(float) * (SK * (SQ + 4 + SD + 4) + SQ * (SD + 1)) + (size_t)SQ * k * 4 + 8 + (size_t)SQ * k * 8;
  TT_REQUIRE(*smem <= kMaxSmem, "tt_scan_topk: k=%d too large for the fp32 scan", k);
  static bool attr_done = false;
  if (*smem > 48 * 1024 && !attr_done) {
    TT_CUDA(cudaFuncSetAttribute(scan_topk_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    attr_done = true;
  }
  return 0;
}

// k > N rows of an empty shard: the (-inf, -1) padding every other path writes
__global__ void fill_empty_kernel(long long n, float* __restrict__ os, long long* __restrict__ oi) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    os[i] = -INFINITY;
    oi[i] = -1;
  }
}

int scan_empty(int Q, int k, float* top_score, long long* top_id, cudaStream_t st) {
  const long long n = (long long)Q * k;
  if (n <= 0) return 0;
  fill_empty_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, top_score, top_id);
  TT_LAUNCH_CHECK();
  return 0;
}

int topk_merge(const float* ps, const long long* pi, int G, int Q, int k, float* os, long long* oi, cudaStream_t st) {
  if (Q <= 0) return 0;
  topk_merge_kernel<<<(Q + 7) / 8, 256, 0, st>>>(ps, pi, G, Q, k, os, oi, nullptr, nullptr, 0);
  TT_LAUNCH_CHECK();
  return 0;
}

// Exact fp32 re-scan of the query rows listed on the device (qlist[0 .. *qcount)), `cap` slots per round; results
// overwrite top_score / top_id of exactly those rows.  ws: scan_listed_ws_bytes(cap, k).
size_t scan_listed_ws_bytes(int cap, int k) {
  return ws_round((size_t)kListedSplits * cap * k * 4) + ws_round((size_t)kListedSplits * cap * k * 8) + 512;
}

int scan_topk_fp32_listed(const float* Qn, const float* Dn, int Q, long long N, int P, int k, long long id_base,
                          const int* qlist, const int* qcount, int cap, float* top_score, long long* top_id, void* ws,
                          cudaStream_t st) {
  if (Q <= 0 || N <= 0) return 0;
  char* p = reinterpret_cast<char*>(ws);
  float* ps = ws_take<float>(p, (size_t)kListedSplits * cap * k);
  long long* pi = ws_take<long long>(p, (size_t)kListedSplits * cap * k);
  int S = kListedSplits;
  const long long max_splits = (N + SD - 1) / SD;
  if (S > max_splits) S = (int)max_splits;
  const long long per = ((N + S - 1) / S + SD - 1) / SD * SD;
  size_t smem;
  if (int rc = fp32_scan_smem(k, &smem)) return rc;
  for (int slot0 = 0; slot0 < Q; slot0 += cap) {  // later rounds find nothing to do unless > cap rows are listed
    const int nq = min(cap, Q - slot0);
    dim3 grid(S, (nq + SQ - 1) / SQ);
    scan_topk_fp32_kernel<<<grid, 256, smem, st>>>(Qn, Dn, nq, N, P, k, per, id_base, ps, pi, qlist, qcount, slot0);
    TT_LAUNCH_CHECK();
    topk_merge_kernel<<<(nq + 7) / 8, 256, 0, st>>>(ps, pi, S, nq, k, top_score, top_id, qlist, qcount, slot0);
    TT_LAUNCH_CHECK();
  }
  return 0;
}

int scan_topk_fp32(const float* Qn, const float* Dn, int Q, long long N, int P, int k, long long id_base,
                   float* top_score, long long* top_id, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (Q <= 0) return 0;
  const int S = scan_splits(Q, N);
  char* p = reinterpret_cast<char*>(ws);
  float* ps = ws_take<float>(p, (size_t)S * Q * k);
  long long* pi = ws_take<long long>(p, (size_t)S * Q * k);
  TT_REQUIRE((size_t)(p - reinterpret_cast<char*>(ws)) <= ws_bytes, "tt_scan_topk: workspace too small");
  const long long per = ((N + S - 1) / S + SD - 1) / SD * SD;
  size_t smem;
  if (int rc = fp32_scan_smem(k, &smem)) return rc;
  dim3 grid(S, (Q + SQ - 1) / SQ);
  scan_topk_fp32_kernel<<<grid, 256, smem, st>>>(Qn, Dn, Q, N, P, k, per, id_base, ps, pi, nullptr, nullptr, 0);
  TT_LAUNCH_CHECK();
  return topk_merge(ps, pi, S, Q, k, top_score, top_id, st);
}

size_t scan_fp32_ws_bytes(int Q, long long N, int k) {
  const int S = scan_splits(Q, N);
  return ws_round((size_t)S * Q * k * 4) + ws_round((size_t)S * Q * k * 8) + 512;
}

int score_candidates(const float* Qn, const float* Dn, const long long* cand, int Q, int C, int P, int k,
                     long long id_base, float* os, long long* oi, float* all_scores, cudaStream_t st) {
  if (Q <= 0) return 0;
  TT_REQUIRE(C >= 1 && C <= 12000, "tt_score_candidates: C=%d outside [1,12000]", C);
  score_candidates_kernel<<<Q, 128, (size_t)C * 4, st>>>(Qn, Dn, cand, Q, C, P, k, id_base, os, oi, all_scores);
  TT_LAUNCH_CHECK();
  return 0;
}

}  // namespace tt

extern "C" int tt_l2_normalize_rows(const float* x, int64_t N, int P, float eps, float* y, void* y_bf16,
                                    tt_stream_t stream) {
  TT_REQUIRE(N >= 0 && P >= 1, "tt_l2_normalize_rows: bad shape");
  if (N == 0) return 0;
  tt::l2norm_rows_kernel<<<(unsigned)((N + 7) / 8), 256, 0, tt::as_stream(stream)>>>(
      x, N, P, eps, y, reinterpret_cast<__nv_bfloat16*>(y_bf16));
  TT_LAUNCH_CHECK();
  return 0;
}

extern "C" int tt_score_candidates(const float* Qn, const float* Dn, const int64_t* cand, int Q, int C, int P, int k,
                                   int64_t id_base, float* top_score, int64_t* top_id, float* all_scores,
                                   tt_stream_t stream) {
  TT_REQUIRE(k >= 1 && k <= C, "tt_score_candidates: k=%d must be in [1,C=%d]", k, C);
  return tt::score_candidates(Qn, Dn, reinterpret_cast<const long long*>(cand), Q, C, P, k, id_base, top_score,
                              reinterpret_cast<long long*>(top_id), all_scores, tt::as_stream(stream));
}

extern "C" int tt_topk_merge(const float* parts_score, const int64_t* parts_id, int G, int Q, int k, float* top_score,
                             int64_t* top_id, tt_stream_t stream) {
  TT_REQUIRE(G >= 1 && k >= 1, "tt_topk_merge: bad shape");
  return tt::topk_merge(parts_score, reinterpret_cast<const long long*>(parts_id), G, Q, k, top_score,
                        reinterpret_cast<long long*>(top_id), tt::as_stream(stream));
}

extern "C" int tt_ndcg_at_k(const int64_t* top_id, int Q, int k, int kk, const int64_t* rel_offsets,
                            const int64_t* rel_ids, double* ndcg, tt_stream_t stream) {
  TT_REQUIRE(kk >= 1 && kk <= k, "tt_ndcg_at_k: kk=%d must be in [1,k=%d]", kk, k);
  if (Q <= 0) return 0;
  tt::ndcg_kernel<<<(Q + 127) / 128, 128, 0, tt::as_stream(stream)>>>(
      reinterpret_cast<const long long*>(top_id), Q, k, kk, reinterpret_cast<const long long*>(rel_offsets),
      reinterpret_cast<const long long*>(rel_ids), ndcg);
  TT_LAUNCH_CHECK();
  return 0;
}

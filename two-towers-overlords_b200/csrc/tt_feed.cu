// Batch assembly on the device (SURVEY.md §8f rank 1): the reference builds every batch in Python
// (backend/data.py:113-152: shuffle, per-item rejection loop for an in-batch negative, then the HF tokenizer pads the
// three text lists, model.py:43-48).  With a 0.25 ms step that loop is three orders of magnitude too slow, so the
// tokenised corpus lives in HBM as a ragged token bank and ONE kernel per step turns a slice of the epoch permutation
// into the six padded token tensors of a trainer slot, drawing the negatives on the way.
// The _mined entry points let an item take a hard negative mined by the corpus scan instead (tt_mine_negatives
// builds that table; the draw is documented in tt_b200.h).
#include "tt_common.cuh"

namespace tt {
namespace {

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

struct AssembleParams {
  const void* q_flat; const long long* q_off; int q_dtype;
  const void* d_flat; const long long* d_off; int d_dtype;
  const int* pair_q; const int* pair_d; const int* pair_qid;
  const int* order;
  int Bg, row0, B, Lq, Ld;
  unsigned long long seed;
  void* ids[3]; void* mask[3];
  int ids_dtype, mask_dtype;
  int* neg_out; int* err;
  bool use_mined;             // false: every negative is drawn in the batch (the entry points without _mined)
  tt_mined_negatives mined;   // copied by value: the kernels read the table and counts it points at
};

__device__ __forceinline__ void store_index(void* p, int dtype, size_t i, long long v) {
  switch (dtype) {
    case TT_I64: reinterpret_cast<long long*>(p)[i] = v; break;
    case TT_I32: reinterpret_cast<int*>(p)[i] = (int)v; break;
    case TT_U16: reinterpret_cast<unsigned short*>(p)[i] = (unsigned short)v; break;
    default: reinterpret_cast<unsigned char*>(p)[i] = (unsigned char)v; break;
  }
}

// In-batch negative of item i: uniform j in [0, Bg) redrawn until j != i and query_id[j] != query_id[i]
// (the accepted distribution of data.py:124-137); a pure function of (seed, i), so every rank of a data-parallel
// job draws the same negatives for the global batch without talking to the others.
__device__ int draw_negative(const AssembleParams& p, int i) {
  const int qi = p.pair_qid[p.order[i]];
  unsigned long long st = splitmix64(p.seed ^ ((unsigned long long)i * 0xD1342543DE82EF95ull));
  for (int attempt = 0; attempt < 256; ++attempt) {
    st = splitmix64(st);
    const int j = (int)(((st >> 32) * (unsigned long long)p.Bg) >> 32);
    if (j != i && p.pair_qid[p.order[j]] != qi) return j;
  }
  if (p.err) atomicExch(p.err, 2);  // no eligible partner (the reference loops forever here)
  return (i + 1) % p.Bg;
}

// Mined negative of item i (the formula tt_b200.h documents at tt_mined_negatives), or -1 when item i takes its
// in-batch negative.  A stream of its own, salted apart from draw_negative's, so the in-batch draws do not move.
__device__ int draw_mined(const AssembleParams& p, int i) {
  const int qrow = p.pair_q[p.order[i]];
  if (qrow < 0 || qrow >= p.mined.n_rows) {
    if (p.err) atomicExch(p.err, 3);
    return -1;
  }
  const int cnt = p.mined.count[qrow];
  if (cnt <= 0) return -1;
  const unsigned long long h0 =
      splitmix64(p.seed ^ 0x6A09E667F3BCC909ull ^ ((unsigned long long)i * 0x9E6C63D0676A9A99ull));
  const unsigned long long h1 = splitmix64(h0);
  if (!((float)(h1 >> 40) < p.mined.ratio * 16777216.0f)) return -1;
  const unsigned long long h2 = splitmix64(h1);
  const int col = (int)((h2 >> 32) % (unsigned long long)cnt);
  const int d = cnt <= p.mined.depth ? p.mined.table[(size_t)qrow * p.mined.depth + col] : -1;
  if (d < 0 || d >= p.mined.n_docs) {
    if (p.err) atomicExch(p.err, 3);
    return -1;
  }
  return d;
}

// document bank row of item i's negative; neg_out[b] = the in-batch item it came from, -1 for a mined one
__device__ int negative_row(const AssembleParams& p, int i, int b) {
  if (p.use_mined) {
    const int d = draw_mined(p, i);
    if (d >= 0) {
      if (p.neg_out) p.neg_out[b] = -1;
      return d;
    }
  }
  const int j = draw_negative(p, i);
  if (p.neg_out) p.neg_out[b] = j;
  return p.pair_d[p.order[j]];
}

// one CTA per output row: role 0 = query, 1 = positive, 2 = negative
__global__ void __launch_bounds__(64) assemble_triplets_kernel(const AssembleParams p) {
  const int role = blockIdx.x / p.B, b = blockIdx.x - role * p.B;
  const int i = p.row0 + b;  // index inside the global batch
  __shared__ int s_src;
  if (threadIdx.x == 0) {
    int src;
    if (role == 0) {
      src = p.pair_q[p.order[i]];
    } else if (role == 1) {
      src = p.pair_d[p.order[i]];
    } else {
      src = negative_row(p, i, b);
    }
    s_src = src;
  }
  __syncthreads();
  const int src = s_src;
  const int L = role == 0 ? p.Lq : p.Ld;
  const void* flat = role == 0 ? p.q_flat : p.d_flat;
  const long long* off = role == 0 ? p.q_off : p.d_off;
  const int dt = role == 0 ? p.q_dtype : p.d_dtype;
  const long long o0 = off[src];
  const int len = (int)min((long long)L, off[src + 1] - o0);  // truncation=True, max_length = L
  for (int t = threadIdx.x; t < L; t += blockDim.x) {
    const bool valid = t < len;
    store_index(p.ids[role], p.ids_dtype, (size_t)b * L + t, valid ? load_index(flat, dt, (size_t)(o0 + t)) : 0);
    store_index(p.mask[role], p.mask_dtype, (size_t)b * L + t, valid ? 1 : 0);
  }
}

// one thread per item: the bank rows of its query, its positive and its negative (a step with a pooled front end
// gathers precomputed pooled rows by these indices instead of pooling tokens)
__global__ void __launch_bounds__(128) assemble_triplet_rows_kernel(const AssembleParams p, int* __restrict__ rows_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  const int i = p.row0 + b;
  rows_out[2 * p.B + b] = negative_row(p, i, b);
  rows_out[b] = p.pair_q[p.order[i]];
  rows_out[p.B + b] = p.pair_d[p.order[i]];
}

// One warp per query: lane l holds rank l of the scan's list; a ballot over "kept" (a real id outside the query's
// exclusion list) gives every survivor its rank among the survivors, so the compaction keeps the scan's order.
__global__ void __launch_bounds__(128) mine_negatives_kernel(const long long* __restrict__ top_id, int Q, int k,
                                                             const long long* __restrict__ excl_off,
                                                             const int* __restrict__ excl_ids, int skip, int depth,
                                                             int* __restrict__ table, int* __restrict__ count) {
  const int r = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (r >= Q) return;
  const long long id = lane < k ? top_id[(size_t)r * k + lane] : -1;
  bool keep = id >= 0;
  if (keep) {  // binary search of the query's sorted exclusion list
    long long lo = excl_off[r], hi = excl_off[r + 1];
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      const long long v = excl_ids[mid];
      if (v == id) { keep = false; break; }
      if (v < id) lo = mid + 1; else hi = mid;
    }
  }
  const unsigned kept = __ballot_sync(0xffffffffu, keep);
  const int pos = __popc(kept & ((1u << lane) - 1u)) - skip;  // rank among the survivors after the skipped ones
  const int n = min(max(__popc(kept) - skip, 0), depth);
  if (keep && pos >= 0 && pos < depth) table[(size_t)r * depth + pos] = (int)id;
  if (lane >= n && lane < depth) table[(size_t)r * depth + lane] = -1;
  if (lane == 0) count[r] = n;
}

int check_slice(const char* who, const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                const int32_t* order, int Bg, int row0, int B) {
  TT_REQUIRE(pair_q && pair_d && pair_qid && order, "%s: null input", who);
  TT_REQUIRE(Bg >= 2 && row0 >= 0 && B >= 0 && row0 + B <= Bg, "%s: bad slice [%d,%d) of %d", who, row0, row0 + B, Bg);
  return 0;
}

int check_mined(const char* who, const tt_mined_negatives* m) {
  TT_REQUIRE(m != nullptr, "%s: null mined-negative descriptor", who);
  TT_REQUIRE(m->n_rows >= 0 && m->n_docs >= 0 && m->depth >= 1 && m->depth <= 32, "%s: bad table shape [%d,%d]",
             who, m->n_rows, m->depth);
  TT_REQUIRE(m->n_rows == 0 || (m->table && m->count), "%s: null table or count", who);
  TT_REQUIRE(m->ratio >= 0.0f && m->ratio <= 1.0f, "%s: ratio %g outside [0, 1]", who, (double)m->ratio);
  return 0;
}

int assemble_rows(const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid, const int32_t* order, int Bg,
                  int row0, int B, uint64_t seed, int32_t* rows_out, int32_t* neg_out, int* err_flag,
                  const tt_mined_negatives* mined, const char* who, tt_stream_t stream) {
  if (int rc = check_slice(who, pair_q, pair_d, pair_qid, order, Bg, row0, B)) return rc;
  TT_REQUIRE(rows_out != nullptr, "%s: null rows_out", who);
  if (B == 0) return 0;
  AssembleParams p{};
  p.pair_q = pair_q; p.pair_d = pair_d; p.pair_qid = pair_qid; p.order = order;
  p.Bg = Bg; p.row0 = row0; p.B = B; p.seed = seed;
  p.neg_out = neg_out; p.err = err_flag;
  if (mined) { p.use_mined = true; p.mined = *mined; }
  assemble_triplet_rows_kernel<<<(B + 127) / 128, 128, 0, as_stream(stream)>>>(p, rows_out);
  TT_LAUNCH_CHECK();
  return 0;
}

int assemble_tokens(const tt_token_bank* qbank, const tt_token_bank* dbank, const int32_t* pair_q, const int32_t* pair_d,
                    const int32_t* pair_qid, const int32_t* order, int Bg, int row0, int B, uint64_t seed, int Lq, int Ld,
                    void* q_ids, void* q_mask, void* p_ids, void* p_mask, void* n_ids, void* n_mask, int ids_dtype,
                    int mask_dtype, int32_t* neg_out, int* err_flag, const tt_mined_negatives* mined,
                    const char* who, tt_stream_t stream) {
  TT_REQUIRE(qbank && dbank, "%s: null input", who);
  if (int rc = check_slice(who, pair_q, pair_d, pair_qid, order, Bg, row0, B)) return rc;
  TT_REQUIRE(Lq >= 1 && Ld >= 1, "%s: bad lengths", who);
  for (int dt : {qbank->dtype, dbank->dtype, ids_dtype})
    TT_REQUIRE(dt == TT_I64 || dt == TT_I32 || dt == TT_U16, "%s: unsupported id dtype %d", who, dt);
  TT_REQUIRE(mask_dtype == TT_I64 || mask_dtype == TT_I32 || mask_dtype == TT_U8, "%s: unsupported mask dtype %d",
             who, mask_dtype);
  if (B == 0) return 0;
  AssembleParams p{};
  p.q_flat = qbank->flat; p.q_off = reinterpret_cast<const long long*>(qbank->offsets); p.q_dtype = qbank->dtype;
  p.d_flat = dbank->flat; p.d_off = reinterpret_cast<const long long*>(dbank->offsets); p.d_dtype = dbank->dtype;
  p.pair_q = pair_q; p.pair_d = pair_d; p.pair_qid = pair_qid; p.order = order;
  p.Bg = Bg; p.row0 = row0; p.B = B; p.Lq = Lq; p.Ld = Ld; p.seed = seed;
  p.ids[0] = q_ids; p.ids[1] = p_ids; p.ids[2] = n_ids;
  p.mask[0] = q_mask; p.mask[1] = p_mask; p.mask[2] = n_mask;
  p.ids_dtype = ids_dtype; p.mask_dtype = mask_dtype; p.neg_out = neg_out; p.err = err_flag;
  if (mined) { p.use_mined = true; p.mined = *mined; }
  assemble_triplets_kernel<<<3 * B, 64, 0, as_stream(stream)>>>(p);
  TT_LAUNCH_CHECK();
  return 0;
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" int tt_assemble_triplet_rows(const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                                        const int32_t* order, int Bg, int row0, int B, uint64_t seed,
                                        int32_t* rows_out, int32_t* neg_out, int* err_flag, tt_stream_t stream) {
  return assemble_rows(pair_q, pair_d, pair_qid, order, Bg, row0, B, seed, rows_out, neg_out, err_flag, nullptr,
                       "tt_assemble_triplet_rows", stream);
}

extern "C" int tt_assemble_triplet_rows_mined(const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                                              const int32_t* order, int Bg, int row0, int B, uint64_t seed,
                                              int32_t* rows_out, int32_t* neg_out, int* err_flag,
                                              const tt_mined_negatives* mined, tt_stream_t stream) {
  if (int rc = check_mined("tt_assemble_triplet_rows_mined", mined)) return rc;
  return assemble_rows(pair_q, pair_d, pair_qid, order, Bg, row0, B, seed, rows_out, neg_out, err_flag, mined,
                       "tt_assemble_triplet_rows_mined", stream);
}

extern "C" int tt_assemble_triplets(const tt_token_bank* qbank, const tt_token_bank* dbank, const int32_t* pair_q,
                                    const int32_t* pair_d, const int32_t* pair_qid, const int32_t* order, int Bg,
                                    int row0, int B, uint64_t seed, int Lq, int Ld, void* q_ids, void* q_mask,
                                    void* p_ids, void* p_mask, void* n_ids, void* n_mask, int ids_dtype, int mask_dtype,
                                    int32_t* neg_out, int* err_flag, tt_stream_t stream) {
  return assemble_tokens(qbank, dbank, pair_q, pair_d, pair_qid, order, Bg, row0, B, seed, Lq, Ld, q_ids, q_mask, p_ids,
                         p_mask, n_ids, n_mask, ids_dtype, mask_dtype, neg_out, err_flag, nullptr,
                         "tt_assemble_triplets", stream);
}

extern "C" int tt_assemble_triplets_mined(const tt_token_bank* qbank, const tt_token_bank* dbank, const int32_t* pair_q,
                                          const int32_t* pair_d, const int32_t* pair_qid, const int32_t* order, int Bg,
                                          int row0, int B, uint64_t seed, int Lq, int Ld, void* q_ids, void* q_mask,
                                          void* p_ids, void* p_mask, void* n_ids, void* n_mask, int ids_dtype,
                                          int mask_dtype, int32_t* neg_out, int* err_flag,
                                          const tt_mined_negatives* mined, tt_stream_t stream) {
  if (int rc = check_mined("tt_assemble_triplets_mined", mined)) return rc;
  return assemble_tokens(qbank, dbank, pair_q, pair_d, pair_qid, order, Bg, row0, B, seed, Lq, Ld, q_ids, q_mask, p_ids,
                         p_mask, n_ids, n_mask, ids_dtype, mask_dtype, neg_out, err_flag, mined,
                         "tt_assemble_triplets_mined", stream);
}

extern "C" int tt_mine_negatives(const int64_t* top_id, int Q, int k, const int64_t* excl_offsets,
                                 const int32_t* excl_ids, int skip, int depth, int32_t* table_out, int32_t* count_out,
                                 tt_stream_t stream) {
  TT_REQUIRE(Q >= 0, "tt_mine_negatives: bad Q %d", Q);
  TT_REQUIRE(depth >= 1 && skip >= 0 && skip + depth <= k && k <= 32,
             "tt_mine_negatives: need 1 <= depth, 0 <= skip, skip + depth <= k <= 32 (skip %d, depth %d, k %d)", skip,
             depth, k);
  TT_REQUIRE(top_id && excl_offsets && excl_ids && table_out && count_out, "tt_mine_negatives: null input");
  if (Q == 0) return 0;
  mine_negatives_kernel<<<(Q + 3) / 4, 128, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(top_id), Q, k,
                                                                    reinterpret_cast<const long long*>(excl_offsets),
                                                                    excl_ids, skip, depth, table_out, count_out);
  TT_LAUNCH_CHECK();
  return 0;
}

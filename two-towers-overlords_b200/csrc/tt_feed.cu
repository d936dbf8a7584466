// Batch assembly on the device (SURVEY.md §8f rank 1): the reference builds every batch in Python
// (backend/data.py:113-152: shuffle, per-item rejection loop for an in-batch negative, then the HF tokenizer pads the
// three text lists, model.py:43-48).  With a 0.25 ms step that loop is three orders of magnitude too slow, so the
// tokenised corpus lives in HBM as a ragged token bank and ONE kernel per step turns a slice of the epoch permutation
// into the six padded token tensors of a trainer slot, drawing the negatives on the way.
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
      const int j = draw_negative(p, i);
      if (p.neg_out) p.neg_out[b] = j;
      src = p.pair_d[p.order[j]];
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
  const int j = draw_negative(p, i);
  if (p.neg_out) p.neg_out[b] = j;
  rows_out[b] = p.pair_q[p.order[i]];
  rows_out[p.B + b] = p.pair_d[p.order[i]];
  rows_out[2 * p.B + b] = p.pair_d[p.order[j]];
}

int check_slice(const char* who, const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                const int32_t* order, int Bg, int row0, int B) {
  TT_REQUIRE(pair_q && pair_d && pair_qid && order, "%s: null input", who);
  TT_REQUIRE(Bg >= 2 && row0 >= 0 && B >= 0 && row0 + B <= Bg, "%s: bad slice [%d,%d) of %d", who, row0, row0 + B, Bg);
  return 0;
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" int tt_assemble_triplet_rows(const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                                        const int32_t* order, int Bg, int row0, int B, uint64_t seed,
                                        int32_t* rows_out, int32_t* neg_out, int* err_flag, tt_stream_t stream) {
  if (int rc = check_slice("tt_assemble_triplet_rows", pair_q, pair_d, pair_qid, order, Bg, row0, B)) return rc;
  TT_REQUIRE(rows_out != nullptr, "tt_assemble_triplet_rows: null rows_out");
  if (B == 0) return 0;
  AssembleParams p{};
  p.pair_q = pair_q; p.pair_d = pair_d; p.pair_qid = pair_qid; p.order = order;
  p.Bg = Bg; p.row0 = row0; p.B = B; p.seed = seed;
  p.neg_out = neg_out; p.err = err_flag;
  assemble_triplet_rows_kernel<<<(B + 127) / 128, 128, 0, as_stream(stream)>>>(p, rows_out);
  TT_LAUNCH_CHECK();
  return 0;
}

extern "C" int tt_assemble_triplets(const tt_token_bank* qbank, const tt_token_bank* dbank, const int32_t* pair_q,
                                    const int32_t* pair_d, const int32_t* pair_qid, const int32_t* order, int Bg,
                                    int row0, int B, uint64_t seed, int Lq, int Ld, void* q_ids, void* q_mask,
                                    void* p_ids, void* p_mask, void* n_ids, void* n_mask, int ids_dtype, int mask_dtype,
                                    int32_t* neg_out, int* err_flag, tt_stream_t stream) {
  TT_REQUIRE(qbank && dbank, "tt_assemble_triplets: null input");
  if (int rc = check_slice("tt_assemble_triplets", pair_q, pair_d, pair_qid, order, Bg, row0, B)) return rc;
  TT_REQUIRE(Lq >= 1 && Ld >= 1, "tt_assemble_triplets: bad lengths");
  for (int dt : {qbank->dtype, dbank->dtype, ids_dtype})
    TT_REQUIRE(dt == TT_I64 || dt == TT_I32 || dt == TT_U16, "tt_assemble_triplets: unsupported id dtype %d", dt);
  TT_REQUIRE(mask_dtype == TT_I64 || mask_dtype == TT_I32 || mask_dtype == TT_U8,
             "tt_assemble_triplets: unsupported mask dtype %d", mask_dtype);
  if (B == 0) return 0;
  AssembleParams p{};
  p.q_flat = qbank->flat; p.q_off = reinterpret_cast<const long long*>(qbank->offsets); p.q_dtype = qbank->dtype;
  p.d_flat = dbank->flat; p.d_off = reinterpret_cast<const long long*>(dbank->offsets); p.d_dtype = dbank->dtype;
  p.pair_q = pair_q; p.pair_d = pair_d; p.pair_qid = pair_qid; p.order = order;
  p.Bg = Bg; p.row0 = row0; p.B = B; p.Lq = Lq; p.Ld = Ld; p.seed = seed;
  p.ids[0] = q_ids; p.ids[1] = p_ids; p.ids[2] = n_ids;
  p.mask[0] = q_mask; p.mask[1] = p_mask; p.mask[2] = n_mask;
  p.ids_dtype = ids_dtype; p.mask_dtype = mask_dtype; p.neg_out = neg_out; p.err = err_flag;
  assemble_triplets_kernel<<<3 * B, 64, 0, as_stream(stream)>>>(p);
  TT_LAUNCH_CHECK();
  return 0;
}

/*
 * tt_b200.h — C ABI of the B200-native two-tower hot path (libtt_b200.so).
 *
 * This is the drop-in boundary for the path BASELINE.json's north_star names.
 * The reference (freemvmt/two-towers-overlords) is pure Python and has no FFI;
 * the functions below are what a ctypes binding placed under the reference's
 * backend/model.py + backend/training.py surface would bind (INTEGRATION.md shows
 * the stub).  Each entry point cites the reference lines it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates);
 *     the library never allocates or frees persistent memory;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = ok, non-zero = error; tt_last_error() gives the text
 *     (thread-local); nothing throws across the boundary;
 *   - row-major everywhere; H = hidden size of the token table (384 for MiniLM),
 *     P = projection_dim; all float buffers are fp32 unless a dtype says else.
 *   - no torch types, no CPU fallback: a call on a machine without an sm_100
 *     device returns an error.
 */
#ifndef TT_B200_H
#define TT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TT_B200_VERSION 100 /* major*100 + minor */

typedef void* tt_stream_t; /* cudaStream_t */

/* element types of caller buffers */
enum tt_dtype {
  TT_F32 = 0,
  TT_BF16 = 1,
  TT_I64 = 2,
  TT_I32 = 3,
  TT_U16 = 4,
  TT_U8 = 5
};

/* arithmetic of the projection / scan contractions */
enum tt_precision {
  TT_PREC_FP32 = 0,   /* fp32 FFMA on CUDA cores: strict-parity mode                         */
  TT_PREC_BF16X3 = 1, /* tcgen05 bf16 MMA, 3-term hi/lo split, fp32 accumulate (~2^-16 rel.) */
  TT_PREC_BF16 = 2    /* tcgen05 bf16 MMA, single pass, fp32 accumulate (~2^-8 rel.)         */
};

int tt_version(void);
const char* tt_last_error(void);
/* Diagnostics: kernels this library has launched (or captured into a CUDA graph) in this process so far. */
unsigned long long tt_launch_count(void);
/* sm count / compute capability of the current device; error if it is not sm_100. */
int tt_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * Tower front end: token-row gather + attention-masked mean + L2 normalise.
 * Replaces backend/model.py:48-56 (tokens→device, `pretrained_model(**tokens)` restated as
 * E[input_ids] per north_star, `_mean_pooling` model.py:63-72, `F.normalize` model.py:56).
 *   table [vocab,H] f32|bf16; ids [B,L] i64|i32|u16; mask [B,L] i64|i32|u8 (0 = padding).
 *   xhat [B,H]: (sum_t m_t E[id_t] / max(sum m, 1e-9)) / max(||.||, 1e-12)
 *   cnt [B] = sum_t m_t (unclamped); nrm [B] = L2 norm of the mean (unclamped).  cnt/nrm may be NULL.
 *   err_flag (nullable, device int): set to 1 if any unmasked id is outside [0,vocab).
 * ---------------------------------------------------------------------------------------- */
int tt_pool_fwd(const void* table, int table_dtype, int vocab, int H,
                const void* ids, int ids_dtype, const void* mask, int mask_dtype,
                int B, int L, float* xhat, float* cnt, float* nrm, int* err_flag,
                tt_stream_t stream);

/* Up to 4 segments in one launch (query / positive / negative batches of a triplet step). Rows of
 * segment s land at xhat[row0[s] ..]; segments may use different tables (the reference keeps one
 * backbone copy per tower, model.py:84-85). */
typedef struct tt_pool_seg {
  const void* table;
  const void* ids;
  const void* mask;
  int B;
  int L;
  int row0;
  int _pad;
} tt_pool_seg;
int tt_pool_fwd_multi(const tt_pool_seg* segs, int nseg, int table_dtype, int vocab, int H,
                      int ids_dtype, int mask_dtype, float* xhat, float* cnt, float* nrm,
                      int* err_flag, tt_stream_t stream);

/* Backward of tt_pool_fwd into the token table (north_star config 3, "trainable table"; the
 * reference freezes the backbone, model.py:28-30,51 — see DESIGN.md D2).  Deterministic:
 * (token id, position) pairs are radix-sorted, each touched row is reduced in position order and
 * written once; no float atomics.
 *   dxhat, xhat [B,H]; cnt, nrm [B] from the forward; dtable [vocab,H] f32 is OVERWRITTEN
 *   (zero rows for untouched ids) unless accumulate != 0.
 *   ws: scratch of at least tt_pool_bwd_ws_bytes(B,L,vocab,H) bytes. */
size_t tt_pool_bwd_ws_bytes(int B, int L, int vocab, int H);
int tt_pool_bwd(const float* dxhat, const float* xhat, const float* cnt, const float* nrm,
                const void* ids, int ids_dtype, const void* mask, int mask_dtype, int B, int L,
                int vocab, int H, float* dtable, int accumulate, void* ws, size_t ws_bytes,
                tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Projection MLP of one tower: y = relu(x W1^T + b1) W2^T + b2      (model.py:33-38,59)
 *   x [M,H]; W1 [P,H]; b1 [P]; W2 [P,P]; b2 [P]; h [M,P] (post-ReLU, saved for backward); y [M,P].
 *   ws: scratch of tt_mlp_ws_bytes(M,H,P,precision) bytes.
 * ---------------------------------------------------------------------------------------- */
size_t tt_mlp_ws_bytes(int M, int H, int P, int precision);
int tt_encode_fwd(const float* x, int M, int H, int P, const float* W1, const float* b1,
                  const float* W2, const float* b2, float* h, float* y, int precision, void* ws,
                  size_t ws_bytes, tt_stream_t stream);
/* Backward of tt_encode_fwd (what autograd does for model.py:59 inside training.py:50).
 *   dy [M,P]; grads dW1 [P,H], db1 [P], dW2 [P,P], db2 [P] are overwritten, or added to when
 *   accumulate != 0 (the document tower is called twice per step, training.py:41-42);
 *   dx [M,H] nullable (only needed when the table trains). */
int tt_encode_bwd(const float* dy, const float* x, const float* h, const float* W1,
                  const float* W2, int M, int H, int P, float* dW1, float* db1, float* dW2,
                  float* db2, float* dx, int accumulate, int precision, void* ws, size_t ws_bytes,
                  tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Cosine triplet loss (model.py:132-145):
 *   cos(x,y) = sum_i (x_i/max(||x||,1e-8)) (y_i/max(||y||,1e-8))
 *   hinge_i = relu((1-cos(q_i,p_i)) - (1-cos(q_i,n_i)) + margin);  loss = inv_batch * sum_i hinge_i
 *   inv_batch = 1/B for one GPU, 1/B_global under data parallelism.
 *   stats [B,8] = {cos_p, cos_n, hinge, |q|, |p|, |n|, q.p, q.n} saved for backward.
 * ---------------------------------------------------------------------------------------- */
int tt_triplet_loss_fwd(const float* q, const float* p, const float* n, int B, int P, float margin,
                        float inv_batch, float* stats, float* loss, tt_stream_t stream);
/* dloss: device scalar (upstream gradient of the loss; NULL means 1).  dq/dp/dn [B,P]. */
int tt_triplet_loss_bwd(const float* q, const float* p, const float* n, const float* stats,
                        const float* dloss, int B, int P, float inv_batch, float* dq, float* dp,
                        float* dn, tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * One whole triplet training step, forward + backward (training.py:37-50 without the optimiser):
 * pool(q), pool(p), pool(n) -> both tower MLPs -> loss -> gradients of the 8 projection tensors
 * (and of the tables when dtable_q/dtable_d are non-NULL).  Gradients are OVERWRITTEN (see grad_accumulate).
 * ---------------------------------------------------------------------------------------- */
typedef struct tt_step_args {
  /* tokens */
  const void* q_ids;  const void* q_mask;  int Lq;
  const void* p_ids;  const void* p_mask;
  const void* n_ids;  const void* n_mask;  int Ld;
  int ids_dtype, mask_dtype;
  int B;             /* triplets on this GPU                         */
  /* frozen (or trainable) token tables */
  const void* table_q; const void* table_d; int table_dtype; int vocab; int H;
  /* projection parameters, fp32 */
  int P;
  const float *Wq1, *bq1, *Wq2, *bq2, *Wd1, *bd1, *Wd2, *bd2;
  /* loss */
  float margin; float inv_batch; float grad_scale; /* upstream d(loss) (1 normally)  */
  /* outputs */
  float* loss;       /* [1]                                          */
  float *dWq1, *dbq1, *dWq2, *dbq2, *dWd1, *dbd1, *dWd2, *dbd2;
  float *dtable_q, *dtable_d; /* nullable                            */
  int* err_flag;     /* nullable                                     */
  int precision;
  void* ws; size_t ws_bytes;  /* >= tt_step_ws_bytes(...); zero-fill it once before its first use (it holds an
                                 arrival counter that every call leaves at zero again)                        */
  int phases;        /* 0 = whole step; TT_STEP_FRONT = pooled gather only (reads tokens + tables, or the pooled
                        banks below, not the projection weights, so it may overlap the previous step's parameter
                        exchange);
                        TT_STEP_BACK = everything after it, on the same workspace                             */
  /* optional optimiser (training.py:51 `optimizer.step()`; adam_param NULL = gradients only): torch.optim.Adam
   * arithmetic on ONE flat fp32 parameter buffer of adam_n elements.  The 8 projection tensors above must be
   * slices of adam_param, and their gradients slices of adam_grad, at equal 16-byte aligned offsets; exp_avg /
   * exp_avg_sq are flat buffers of the same length.  adam_state: 4 doubles as for tt_adam_step_dev, advanced once
   * per call that has TT_STEP_BACK.  With the tensor-core precisions the update runs in the tail of the step's
   * persistent chain kernel (no extra launch); otherwise it is launched after the step.                        */
  double* adam_state;
  float *adam_param, *adam_grad, *adam_exp_avg, *adam_exp_avg_sq;
  size_t adam_n;
  float adam_lr, adam_beta1, adam_beta2, adam_eps;
  int chain;         /* tensor-core precisions: how everything after the pooled gather is launched.
                        1 = ONE persistent kernel (both layers, loss in the layer-2 epilogue, backward, bias sums,
                        gradient reduction, optimiser); 2 = one kernel per contraction (small kernels a concurrent
                        look-ahead gather can slip between); 0 = library default: TT_CHAIN env (1 / 0 = per-kernel),
                        else 1.  Keep the same choice for the TT_STEP_FRONT and TT_STEP_BACK calls of one step.   */
  /* optional in-batch negatives (NULL = the negatives are gathered from n_ids / n_mask like any document).
   * The reference's batcher draws every negative among the OTHER items' positive documents of the same batch
   * (backend/data.py:113-137), so negative row i is the same token sequence as positive row neg_index[i]
   * (0 <= neg_index[i] < B, int32 on the device).  Given the indices, the pooled gather visits every positive
   * once and writes its pooled row to the negative rows that name it — the same bits as gathering the same tokens
   * again, for half the document rows read; n_ids / n_mask are not read anywhere in the call then.  With table
   * gradients (dtable_q / dtable_d) each negative's gradient row g_n[i] (d loss / d masked token sum) is folded
   * into the positive it copies: g'_p[j] = ((g_p[j] + g_n[i1]) + g_n[i2]) + ... over the negatives i1 < i2 < ...
   * naming j, in fp32 and ascending i, and the document table's gradient (or its Adam step) sums over the
   * positives' tokens only.  That is the same gradient as walking the negatives' tokens, up to the fp32 summation
   * order.  An index out of range raises err_flag and adds nothing to any positive.                          */
  const int32_t* neg_index;
  /* optional frozen front end (NULL = pool tokens as before): rows of F.normalize(masked_mean(backbone(text)))
   * computed once per text.  Output row i     = pooled_q[pooled_index[i]],
   *                           row B + i       = pooled_d[pooled_index[B + i]],
   *                           row 2B + i      = pooled_d[pooled_index[2B + i]]   (int32 [3B] on the device).
   * Rows are fp32 [rows, H], 16-byte aligned.  Tokens and tables are not read (may be NULL).  Needs frozen tables
   * and neg_index == NULL.  An index outside [0, rows) sets err_flag and reads row 0.  cnt / nrm of the pooled
   * rows are not known then: only the table gradient reads them, and it is refused.
   * These five fields were appended while TT_B200_VERSION stayed at 100, so the version does not tell the two
   * layouts apart.  A caller compiled against a header without them passes a shorter struct, and the library
   * reads whatever follows it as pooled_*: rebuild such a caller against this header (the ctypes mirror in
   * _native.py lists them), and zero-initialise the struct as before.                                          */
  const float* pooled_q; int64_t pooled_q_rows;
  const float* pooled_d; int64_t pooled_d_rows;
  const int32_t* pooled_index;
  /* gradient accumulation (the reference's `loss / accumulation_steps; backward()` over the micro-batches of a
   * window, backend/training.py:66-133): 0 = the gradient outputs are OVERWRITTEN as described above; 1 = every
   * gradient output (the 8 projection gradients, and dtable_q / dtable_d when given) becomes fl(old + new) in fp32,
   * where new is exactly what the same call writes with 0 — autograd's `.grad += new`.  The loss is still overwritten
   * with this call's loss.  With adam_param set the optimiser consumes the accumulated gradient, so a window of a
   * micro-batches is a - 1 calls with grad_accumulate = 1 and no optimiser, then one with both (the first call of a
   * window that carries nothing uses 0; set grad_scale = 1/a for the reference's scaling).  Appended, like the
   * pooled_* fields, while TT_B200_VERSION stayed at 100: rebuild callers against this header.                    */
  int grad_accumulate;
  /* optional optimiser of the token tables (NULL = the table gradients are only computed, as above): when
   * table_param_q / table_param_d are set and the call has TT_STEP_BACK, the table gradient of this call (plus the old
   * dtable_* when grad_accumulate = 1) is consumed by one dense torch.optim.Adam step on EVERY row of both tables, run
   * in the scatter-add's epilogue; dtable_q / dtable_d are then not written (still give them: they select the trainable
   * table and hold a window's partial sum).  An untouched row has gradient 0: its moments decay, and it still moves once
   * its exp_avg is non-zero.  The tables share the projections' step count and hyper-parameters (adam_state is
   * advanced by this call before the table update reads it, adam_lr / adam_beta1 / adam_beta2 / adam_eps), so these
   * fields need adam_param.  table_param_q / table_param_d must be table_q / table_d (distinct fp32 tables);
   * table_exp_avg* are fp32 [vocab, H].  Appended, like grad_accumulate, while TT_B200_VERSION stayed at 100: rebuild
   * callers against this header.                                                                                   */
  float *table_param_q, *table_param_d;
  float *table_exp_avg_q, *table_exp_avg_sq_q, *table_exp_avg_d, *table_exp_avg_sq_d;
} tt_step_args;
#define TT_STEP_FRONT 1
#define TT_STEP_BACK 2
size_t tt_step_ws_bytes(int B, int Lq, int Ld, int H, int P, int vocab, int precision,
                        int train_table);
int tt_triplet_step(const tt_step_args* args, tt_stream_t stream);

/* Adam update, same arithmetic as torch.optim.Adam defaults used at training.py:436
 * (betas 0.9/0.999, eps 1e-8, no weight decay, no amsgrad): n fp32 elements, `step` is the
 * 1-based step count AFTER this update.  grad_scale multiplies the gradient first (e.g. 1/world). */
int tt_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n,
                 float lr, float beta1, float beta2, float eps, int step, float grad_scale,
                 tt_stream_t stream);

/* Graph-capturable variant: the step count and beta powers live in device memory
 * (state: 4 doubles {t, beta1^t, beta2^t, unused}, zero-initialised = "no step taken yet" — a zeroed
 * state is advanced to t=1 by the first call), so replaying a captured graph advances the bias
 * correction without any host-side argument change. */
int tt_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n,
                     float lr, float beta1, float beta2, float eps, double* state, float grad_scale,
                     tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Retrieval / evaluation (training.py:244-311 restated as a batched exhaustive scan).
 * ---------------------------------------------------------------------------------------- */
/* y[i,:] = x[i,:] / max(||x[i,:]||, eps)  (the per-vector clamp of torch.cosine_similarity,
 * training.py:297-299, eps = 1e-8).  In place allowed (y == x).  y_bf16 nullable: bf16 copy. */
int tt_l2_normalize_rows(const float* x, int64_t N, int P, float eps, float* y, void* y_bf16,
                         tt_stream_t stream);

/* Exhaustive corpus scan: for every query the k best documents of this shard by dot product of
 * the (already normalised) rows, ties broken by ascending id.  The score matrix is never stored.
 *   Qn [Q,P] f32, Dn [N,P] f32 (TT_PREC_FP32) — or bf16 copies Qb/Db for the tensor-core scan, in
 *   which case the fp32 arrays are still used to re-score the k_cand best candidates exactly.
 *   id_base: global id of local document 0 (corpus sharding, one shard per GPU).
 *   top_score [Q,k] f32 descending; top_id [Q,k] i64 (-1 where fewer than k docs exist).
 *   ws: tt_scan_ws_bytes(Q,N,P,k,precision) bytes. */
size_t tt_scan_ws_bytes(int Q, int64_t N, int P, int k, int precision);
int tt_scan_topk(const float* Qn, const float* Dn, const void* Qb, const void* Db, int Q, int64_t N,
                 int P, int k, int64_t id_base, int precision, float* top_score, int64_t* top_id,
                 void* ws, size_t ws_bytes, tt_stream_t stream);

/* Exact fp32 scores of per-query candidate lists (validation mode of evaluate_model,
 * training.py:253-267,288-299): cand [Q,C] i64 local doc indices (-1 = padding).
 * Writes the k best per query (score desc, id asc). */
int tt_score_candidates(const float* Qn, const float* Dn, const int64_t* cand, int Q, int C, int P,
                        int k, int64_t id_base, float* top_score, int64_t* top_id,
                        float* all_scores /* [Q,C] nullable: every candidate's score */,
                        tt_stream_t stream);

/* Merge G partial top-k lists per query (corpus shards after the all-gather):
 * parts_score/parts_id [G,Q,k] -> [Q,k], order (score desc, id asc), ids < 0 ignored. */
int tt_topk_merge(const float* parts_score, const int64_t* parts_id, int G, int Q, int k,
                  float* top_score, int64_t* top_id, tt_stream_t stream);

/* NDCG@k of binary relevance from top-k ids (sklearn.metrics.ndcg_score semantics used at
 * training.py:304-309, tie-free case): rel_offsets [Q+1] / rel_ids (CSR, global ids, each list
 * sorted ascending), ndcg [Q] f64.  IDCG = sum_{r<min(R,k)} 1/log2(r+2); ndcg = 0 when R == 0.
 * kk <= k evaluates NDCG@kk from the first kk entries. */
int tt_ndcg_at_k(const int64_t* top_id, int Q, int k, int kk, const int64_t* rel_offsets,
                 const int64_t* rel_ids, double* ndcg, tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Data parallelism over NVLink peer memory (SURVEY.md §8e; the reference is single-device, this is the one
 * exchange a data-parallel training.py:47-51 needs).  One process per GPU; segments are exchanged as CUDA IPC
 * handles (the host side ships the 64 handle bytes through torch.distributed).  These four calls are the only
 * ones that allocate: IPC needs memory whose allocation base the library knows.
 * ---------------------------------------------------------------------------------------- */
#define TT_PEER_HANDLE_BYTES 64
int tt_peer_alloc(size_t bytes, void** dev_ptr, void* handle_out /* TT_PEER_HANDLE_BYTES */); /* zero-filled */
int tt_peer_open(const void* handle, void** dev_ptr); /* maps a peer's segment into this process */
int tt_peer_close(void* dev_ptr);
int tt_peer_free(void* dev_ptr);

/* Segment layout for n_param fp32 parameters on `world` ranks (S = slice = ceil((n_param+1)/world) rounded up to 64):
 *   floats [0, world*S)            the parameters, slot [n_param] = the step's global loss
 *   floats [world*S, 2*world*S)    gradient landing zone [source rank][S]
 *   then 256 bytes of flags        grad-arrived[world] | param-arrived[world]
 * The caller points its flat parameter tensor at offset 0 of its own segment. */
size_t tt_dp_segment_bytes(size_t n_param, int world);

/* ONE kernel: reduce-scatter of the flat gradient (+ loss in slot n_param) over peer stores, torch.optim.Adam
 * arithmetic (training.py:436 defaults) on this rank's slice, all-gather of the new parameters into every rank's
 * segment.  Sums run in rank order, so all ranks hold bit-identical parameters and a run is bit-reproducible.
 *   segments[world]: every rank's segment as mapped in THIS process (own entry = the local pointer);
 *   grad [n_param+1] local; exp_avg / exp_avg_sq [n_param] local (only this rank's slice is touched);
 *   state: 4 doubles {t, beta1^t, beta2^t, -}; ctl: 16 u32 {epoch, ticket, ticket, error, then four u64
 *   diagnostics: ns until all gradient flags, ns from there to kernel end, calls, ns of the own push}, both
 *   zero-initialised, local.  ctl[3] != 0 after a call means a peer did not answer within 4 s.
 *   max_ctas: upper bound on the CTAs used (<= SM count; 0 = one per SM, measured best at N = 8) — every CTA spins on peer flags, so
 *   the grid must be co-resident with whatever else runs concurrently. */
int tt_dp_reduce_adam(void* const* segments, int world, int rank, size_t n_param, const float* grad,
                      float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                      double* state, unsigned* ctl, int max_ctas, tt_stream_t stream);

/* Barrier across the ranks on `stream`: flags[r] = rank r's flag array (>= world u32, zero-initialised, peer
 * memory), ctl as above (its own 4 u32). */
int tt_peer_barrier(void* const* flags, int world, int rank, unsigned* ctl, tt_stream_t stream);

/* tt_topk_merge reading every shard's [Q,k] list in place from its owner's peer memory (corpus scan, §8e);
 * bracket it with tt_peer_barrier so the lists are complete before and not overwritten during the merge. */
int tt_peer_topk_merge(const float* const* parts_score, const int64_t* const* parts_id, int world, int Q, int k,
                       float* top_score, int64_t* top_id, tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Batch assembly on the device (backend/data.py:113-152 + the tokenizer padding of model.py:43-48, for a
 * tokenised corpus resident in HBM — SURVEY.md §8f rank 1).  A token bank is ragged: `flat` holds the ids of all
 * texts back to back (i64|i32|u16), text r occupies flat[offsets[r] .. offsets[r+1]).
 *   pair_q / pair_d / pair_qid [n_pairs]: bank row of the query, bank row of the positive passage and the query id
 *   of every (query, positive) pair of the dataset; order [Bg]: the dataset pairs that form this step's GLOBAL
 *   batch (a slice of the epoch permutation); this rank assembles items [row0, row0 + B) of it.
 *   Negative of item i = positive passage of item j, j uniform in [0, Bg) redrawn until j != i and
 *   query_id[j] != query_id[i]; j is a pure function of (seed, i), so all ranks agree on the global batch's
 *   negatives.  neg_out [B] (nullable) receives j.  err_flag (nullable) is set to 2 if an item has no partner.
 *   Outputs: ids [B,Lq] / [B,Ld] / [B,Ld] (i64|i32|u16, zero padded, truncated to L) and masks (i64|i32|u8).
 * ---------------------------------------------------------------------------------------- */
typedef struct tt_token_bank {
  const void* flat;
  const int64_t* offsets;
  int dtype;
  int _pad;
} tt_token_bank;
int tt_assemble_triplets(const tt_token_bank* qbank, const tt_token_bank* dbank, const int32_t* pair_q,
                         const int32_t* pair_d, const int32_t* pair_qid, const int32_t* order, int Bg, int row0,
                         int B, uint64_t seed, int Lq, int Ld, void* q_ids, void* q_mask, void* p_ids, void* p_mask,
                         void* n_ids, void* n_mask, int ids_dtype, int mask_dtype, int32_t* neg_out, int* err_flag,
                         tt_stream_t stream);
/* The same batch as bank ROWS instead of tokens (for a step with tt_step_args.pooled_index): rows_out [3B] int32 =
 * query rows | positive rows | negative rows, i.e. pair_q[order[row0 + i]], pair_d[order[row0 + i]] and
 * pair_d[order[neg_out[i]]].  The negatives are drawn by the same code as in tt_assemble_triplets, so for equal
 * arguments they are the same items.  neg_out (nullable) and err_flag as there. */
int tt_assemble_triplet_rows(const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                             const int32_t* order, int Bg, int row0, int B, uint64_t seed,
                             int32_t* rows_out, int32_t* neg_out, int* err_flag, tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Hard negatives mined with the corpus scan (DPR / ANCE style): the passages the current towers rank highest for a
 * query that are not its positives.
 *
 * tt_mine_negatives: top_id [Q,k] i64 = tt_scan_topk / tt_topk_merge lists of query-bank rows (score desc, id asc,
 * -1 padding); excl_offsets [Q+1] i64 / excl_ids i32 = CSR exclusion list of every query, sorted ascending within
 * each query.  Each list is walked in rank order, every id of the query's exclusion list is dropped, the first `skip`
 * survivors are dropped, and the next up to `depth` survivors are written in rank order to table_out [Q,depth] i32;
 * count_out [Q] i32 = how many were written, the rest of the row is -1.  Needs 1 <= depth, 0 <= skip,
 * skip + depth <= k <= 32.
 *
 * tt_assemble_triplets_mined / tt_assemble_triplet_rows_mined: tt_assemble_triplets / tt_assemble_triplet_rows whose
 * item i may take its negative from the table instead.  With qrow = pair_q[order[i]], x ^ y bitwise xor, u >> s a
 * logical shift, all arithmetic on uint64 mod 2^64 and splitmix64 as in the in-batch draw:
 *   h0 = splitmix64(seed ^ 0x6A09E667F3BCC909 ^ (i * 0x9E6C63D0676A9A99)),  h1 = splitmix64(h0),  h2 = splitmix64(h1)
 *   hard = count[qrow] > 0  and  float(h1 >> 40) < ratio * 2^24           (fp32 compare, both sides exact)
 *   hard item:  negative = document row table[qrow][(h2 >> 32) mod count[qrow]],  neg_out[i - row0] = -1
 *   otherwise:  the in-batch draw of tt_assemble_triplets, unchanged (neg_out = its item j)
 * so ratio = 0, or all counts 0, gives the batches of the entry points without _mined bit for bit, and every rank of
 * a data-parallel job draws the same negatives.  A qrow outside [0, n_rows), a count above depth or a table entry
 * outside [0, n_docs) sets err_flag to 3 and the item falls back to its in-batch draw.
 * ---------------------------------------------------------------------------------------- */
typedef struct tt_mined_negatives {
  const int32_t* table;   /* [n_rows, depth] document-bank rows, device */
  const int32_t* count;   /* [n_rows] valid entries per row, device     */
  int depth;
  int n_rows;             /* query-bank rows                            */
  int n_docs;             /* document-bank rows                         */
  float ratio;            /* probability of a hard negative, [0, 1]     */
} tt_mined_negatives;
int tt_mine_negatives(const int64_t* top_id, int Q, int k, const int64_t* excl_offsets, const int32_t* excl_ids,
                      int skip, int depth, int32_t* table_out, int32_t* count_out, tt_stream_t stream);
int tt_assemble_triplets_mined(const tt_token_bank* qbank, const tt_token_bank* dbank, const int32_t* pair_q,
                               const int32_t* pair_d, const int32_t* pair_qid, const int32_t* order, int Bg, int row0,
                               int B, uint64_t seed, int Lq, int Ld, void* q_ids, void* q_mask, void* p_ids,
                               void* p_mask, void* n_ids, void* n_mask, int ids_dtype, int mask_dtype, int32_t* neg_out,
                               int* err_flag, const tt_mined_negatives* mined, tt_stream_t stream);
int tt_assemble_triplet_rows_mined(const int32_t* pair_q, const int32_t* pair_d, const int32_t* pair_qid,
                                   const int32_t* order, int Bg, int row0, int B, uint64_t seed, int32_t* rows_out,
                                   int32_t* neg_out, int* err_flag, const tt_mined_negatives* mined,
                                   tt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Measurement probe (bench.py): L2 -> SM read bandwidth.  Every SM streams `buf` (`bytes` long, cache-resident
 * when it fits the 126 MB L2) `iters` times with coalesced 16-byte loads at full occupancy; the caller times the
 * launch with CUDA events: GB/s = bytes * iters / seconds.  This is the ceiling of the pooled gather, whose token
 * tables stay resident in L2 (the reference's counterpart is nn.Embedding inside backend/model.py:51-52).
 * ctas_per_sm <= 0 selects 8 (x 256 threads).  sink: 4 writable bytes. */
/* ------------------------------------------------------------------------------------------
 * The reference's full backbone (SURVEY.md D1): the frozen MiniLM-L6 BertModel of backend/model.py:24,
 * run forward-only under no_grad at backend/model.py:51-52; output[0] = last hidden state.
 * All pointers are device pointers.  Weight matrices are torch Linear weights [out, in] given as their
 * bf16 (hi, lo) terms (tt_split_bf16_terms, once: the backbone is frozen); wqkv = rows of query | key | value.
 * ---------------------------------------------------------------------------------------- */
typedef struct tt_encoder_layer {
  const void *wqkv_hi, *wqkv_lo; const float* bqkv;      /* [3H, H], [3H] */
  const void *wo_hi, *wo_lo;     const float* bo;        /* [H, H], [H]   */
  const float *ln1_g, *ln1_b;                            /* attention.output.LayerNorm */
  const void *w1_hi, *w1_lo;     const float* b1;        /* intermediate.dense [I, H]  */
  const void *w2_hi, *w2_lo;     const float* b2;        /* output.dense [H, I]        */
  const float *ln2_g, *ln2_b;                            /* output.LayerNorm           */
} tt_encoder_layer;
typedef struct tt_encoder_weights {
  const float *word_emb, *pos_emb, *type_emb;            /* [vocab,H], [max_pos,H], row 0 of [2,H] */
  const float *emb_ln_g, *emb_ln_b;
  int vocab, max_pos, hidden, heads, inter, n_layers;
  float ln_eps;
  const tt_encoder_layer* layers;                        /* HOST array of n_layers entries */
} tt_encoder_weights;
size_t tt_encoder_ws_bytes(int tokens, int hidden, int inter);
/* hidden_out [B*L, hidden] f32 = last hidden state; ids [B,L] (any index dtype), mask [B,L] (attention mask:
 * masked KEYS get softmax weight 0; masked query positions are still computed, as in the reference, and are
 * ignored by the masked mean that follows).  err_flag (nullable) is set on an out-of-range token id. */
int tt_encoder_fwd(const tt_encoder_weights* w, const void* ids, int ids_dtype, const void* mask, int mask_dtype,
                   int B, int L, float* hidden_out, int* err_flag, void* ws, size_t ws_bytes, tt_stream_t stream);
/* fp32 [rows, cols] dense -> bf16 terms hi = rn(x), lo = rn(x - hi). */
int tt_split_bf16_terms(const float* x, int rows, int cols, void* hi, void* lo, tt_stream_t stream);

/* Diagnostics / parity tests: device address of a named internal buffer of a tensor-core step workspace:
 * "trace" (task timeline of the persistent chain kernel after a TT_CHAIN_TRACE=1 step: [160][128] pairs of
 * {task << 4 | event, globaltimer ns}; the launch does not clear it, so the caller zeroes it before the launch it
 * wants to trace, or slots of earlier launches remain), "x_hi" / "x_lo" / "x_lo2" (bf16 terms [3B,H] of the pooled rows; x_lo2 in
 * bf16x3 steps only), "h_hi" / "h_lo" / "dy_hi" / "dy_lo" (bf16 terms [3B,P]); rows q | p | n. */
int tt_debug_step_buffer(void* ws, int B, int Lq, int Ld, int H, int P, int vocab, int precision, int train_table,
                         const char* name, void** ptr);
int tt_ubench_l2_read(const void* buf, size_t bytes, int iters, int ctas_per_sm, void* sink, tt_stream_t stream);
/* Self-test of the MN-major tcgen05 operand path (the persistent chain kernel's weight gradients contract over the
 * batch rows of row-major activations without transposed copies): D[128,128] fp32 = sum_k A[k][m] * B[k][n] for
 * A, B [K,128] bf16 row-major on the device, K a multiple of 64.  One CTA; for tests.                           */
int tt_selftest_mn_major(const void* A, const void* B, int K, float* D, tt_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TT_B200_H */

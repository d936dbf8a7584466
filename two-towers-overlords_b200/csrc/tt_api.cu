// C-ABI entry points of libtt_b200.so that orchestrate several kernels (see include/tt_b200.h).
#include <stdarg.h>
#include <string.h>

#include "tt_pool.cuh"
#include "tt_scan.cuh"
#include "tt_simt.cuh"
#include "tt_sm100.cuh"
#include "tt_step_ws.cuh"

namespace tt {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_cuda(cudaError_t e, const char* what, const char* file, int line) {
  if (e == cudaSuccess) return 0;
  set_error("CUDA error %s (%d) at %s:%d in `%s`", cudaGetErrorString(e), (int)e, file, line, what);
  return 1;
}

static unsigned long long g_launches = 0;
void note_launch() { __atomic_fetch_add(&g_launches, 1ull, __ATOMIC_RELAXED); }

int sm_count() {
  static int cached = 0;
  if (cached) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  cached = n;
  return n;
}

namespace {

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float beta1, float beta2, float eps, float step_size,
                            float bc2_sqrt, float grad_scale) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * grad_scale;
  // torch.optim.Adam (single/multi-tensor, non-fused): lerp, mul+addcmul, sqrt/bc2_sqrt + eps, addcdiv
  const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
  const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] = p[i] - step_size * (mi / denom);
}

__global__ void adam_advance_kernel(double* state, double beta1, double beta2) {
  const double t = state[0];
  state[0] = t + 1.0;
  state[1] = (t == 0.0 ? 1.0 : state[1]) * beta1;
  state[2] = (t == 0.0 ? 1.0 : state[2]) * beta2;
}

__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                float* __restrict__ v, size_t n, float lr, float beta1, float beta2, float eps,
                                const double* __restrict__ state, float grad_scale) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float step_size = adam_step_size(state, lr);
  const float bc2_sqrt = adam_bc2_sqrt(state);
  float pi = p[i], mi = m[i], vi = v[i];
  adam_element(pi, mi, vi, g[i] * grad_scale, beta1, beta2, eps, step_size, bc2_sqrt);
  m[i] = mi;
  v[i] = vi;
  p[i] = pi;
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" int tt_version(void) { return TT_B200_VERSION; }
extern "C" const char* tt_last_error(void) { return tt::g_err; }
extern "C" unsigned long long tt_launch_count(void) { return __atomic_load_n(&tt::g_launches, __ATOMIC_RELAXED); }

extern "C" int tt_device_info(int* sms, int* cc_major, int* cc_minor) {
  int dev = 0;
  TT_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  TT_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sms) *sms = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  TT_REQUIRE(prop.major == 10, "libtt_b200 is built for sm_100a only; device is sm_%d%d", prop.major, prop.minor);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// tower MLP
// ------------------------------------------------------------------------------------------------
// fp32: h (forward without h) or dz1 [M, P], then the backward's slice sums
extern "C" size_t tt_mlp_ws_bytes(int M, int H, int P, int precision) {
  if (precision == TT_PREC_FP32)
    return ws_round((size_t)M * P * 4) + ws_round(mlp_bwd_fp32_scratch_floats(M, H, P) * 4) + 256;
  return mlp_sm100_ws_bytes(M, H, P) + 256;
}

static int check_mlp_shape(const char* who, int M, int H, int P, int precision) {
  TT_REQUIRE(M >= 0 && H >= 1 && P >= 1, "%s: bad shape M=%d H=%d P=%d", who, M, H, P);
  TT_REQUIRE(precision == TT_PREC_FP32 || precision == TT_PREC_BF16X3 || precision == TT_PREC_BF16,
             "%s: unknown precision %d", who, precision);
  if (precision != TT_PREC_FP32)
    TT_REQUIRE(H % 64 == 0 && P % 64 == 0, "%s: tensor-core precision needs H and P multiples of 64 (H=%d P=%d)", who,
               H, P);
  return 0;
}

extern "C" int tt_encode_fwd(const float* x, int M, int H, int P, const float* W1, const float* b1, const float* W2,
                             const float* b2, float* h, float* y, int precision, void* ws, size_t ws_bytes,
                             tt_stream_t stream) {
  int rc = check_mlp_shape("tt_encode_fwd", M, H, P, precision);
  if (rc) return rc;
  if (M == 0) return 0;
  cudaStream_t st = as_stream(stream);
  TT_REQUIRE(ws_bytes >= tt_mlp_ws_bytes(M, H, P, precision), "tt_encode_fwd: workspace too small");
  if (precision == TT_PREC_FP32) {
    float* hbuf = h ? h : reinterpret_cast<float*>(ws);
    return mlp_fwd_fp32(x, M, H, P, W1, b1, W2, b2, hbuf, y, st);
  }
  return mlp_fwd_sm100(x, M, H, P, W1, b1, W2, b2, h, y, precision, ws, ws_bytes, st);
}

extern "C" int tt_encode_bwd(const float* dy, const float* x, const float* h, const float* W1, const float* W2, int M,
                             int H, int P, float* dW1, float* db1, float* dW2, float* db2, float* dx, int accumulate,
                             int precision, void* ws, size_t ws_bytes, tt_stream_t stream) {
  int rc = check_mlp_shape("tt_encode_bwd", M, H, P, precision);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  if (M == 0) {
    if (!accumulate) {
      TT_CUDA(cudaMemsetAsync(dW1, 0, (size_t)P * H * 4, st));
      TT_CUDA(cudaMemsetAsync(db1, 0, (size_t)P * 4, st));
      TT_CUDA(cudaMemsetAsync(dW2, 0, (size_t)P * P * 4, st));
      TT_CUDA(cudaMemsetAsync(db2, 0, (size_t)P * 4, st));
    }
    return 0;
  }
  TT_REQUIRE(ws_bytes >= tt_mlp_ws_bytes(M, H, P, precision), "tt_encode_bwd: workspace too small");
  if (precision == TT_PREC_FP32) {
    char* p = reinterpret_cast<char*>(ws);
    float* dz1 = ws_take<float>(p, (size_t)M * P);
    return mlp_bwd_fp32(dy, x, h, W1, W2, M, H, P, dW1, db1, dW2, db2, dx, accumulate, dz1, reinterpret_cast<float*>(p),
                        st);
  }
  return mlp_bwd_sm100(dy, x, h, W1, W2, M, H, P, dW1, db1, dW2, db2, dx, accumulate, precision, ws, ws_bytes, st);
}

// ------------------------------------------------------------------------------------------------
// whole triplet step
// ------------------------------------------------------------------------------------------------
struct ApiStepWs {
  float *xhat, *cnt, *nrm, *h, *y, *stats, *dy, *dz1, *dxhat, *g;
  float* fp32_scratch;  // mlp_bwd_fp32's slice sums, shared by both towers (fp32 only)
  void* pool_ws;
  size_t pool_ws_bytes;
  void* mma_ws;
  size_t mma_ws_bytes;
};

static size_t carve_step_ws(char* base, int B, int Lq, int Ld, int H, int P, int vocab, int precision, int train_table,
                            ApiStepWs* out) {
  char* p = base;
  const size_t R = (size_t)3 * B;
  ApiStepWs w{};
  w.xhat = ws_take<float>(p, R * H);
  w.cnt = ws_take<float>(p, R);
  w.nrm = ws_take<float>(p, R);
  w.h = ws_take<float>(p, R * P);
  w.y = ws_take<float>(p, R * P);
  w.stats = ws_take<float>(p, (size_t)B * 8);
  w.dy = ws_take<float>(p, R * P);
  w.dz1 = ws_take<float>(p, R * P);
  if (train_table) {
    w.dxhat = ws_take<float>(p, R * H);
    w.g = ws_take<float>(p, R * H);
    const long long ntok = (long long)B * Lq > 2ll * B * Ld ? (long long)B * Lq : 2ll * B * Ld;
    w.pool_ws_bytes = pool_bwd_ws_bytes(ntok, vocab);
    w.pool_ws = ws_take<char>(p, w.pool_ws_bytes);
  }
  if (precision != TT_PREC_FP32) {
    w.mma_ws_bytes = step_sm100_ws_bytes(B, H, P, train_table);
    w.mma_ws = ws_take<char>(p, w.mma_ws_bytes);
  } else {
    w.fp32_scratch = ws_take<float>(p, mlp_bwd_fp32_scratch_floats(2 * B, H, P));
  }
  if (out) *out = w;
  return (size_t)(p - base) + 256;
}

extern "C" int tt_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                float beta1, float beta2, float eps, double* state, float grad_scale,
                                tt_stream_t stream);

extern "C" size_t tt_step_ws_bytes(int B, int Lq, int Ld, int H, int P, int vocab, int precision, int train_table) {
  return carve_step_ws(nullptr, B, Lq, Ld, H, P, vocab, precision, train_table, nullptr);
}

// Diagnostics and parity tests: device address of a named internal buffer of a tensor-core step workspace.
//   "trace"  per-CTA task timeline of the last TT_CHAIN_TRACE=1 step: [160][128] x {task << 4 | event, globaltimer ns};
//            the launch does not clear it (a memset would sit between the pooled gather and the chain kernel, its
//            programmatic dependent): the caller zeroes it first, or slots of earlier launches remain
//   "x_hi" / "x_lo" / "x_lo2"            bf16 terms [3B, H] of the pooled rows xhat (rows q | p | n; x_lo2 is written by
//                                        bf16x3 steps only)
//   "h_hi" / "h_lo" / "dy_hi" / "dy_lo"  bf16 terms [3B, P] of the hidden activations / of dY (rows q | p | n)
extern "C" int tt_debug_step_buffer(void* ws, int B, int Lq, int Ld, int H, int P, int vocab, int precision,
                                    int train_table, const char* name, void** ptr) {
  TT_REQUIRE(ws && name && ptr && precision != TT_PREC_FP32, "tt_debug_step_buffer: bad arguments");
  ApiStepWs w;
  carve_step_ws(reinterpret_cast<char*>(ws), B, Lq, Ld, H, P, vocab, precision, train_table, &w);
  tt::StepWs m;
  tt::carve_step(reinterpret_cast<char*>(w.mma_ws), B, H, P, train_table, &m);
  void* out = nullptr;
  if (!strcmp(name, "trace")) out = m.trace;
  else if (!strcmp(name, "x_hi")) out = m.x_hi;
  else if (!strcmp(name, "x_lo")) out = m.x_lo;
  else if (!strcmp(name, "x_lo2")) out = m.x_lo2;
  else if (!strcmp(name, "h_hi")) out = m.h_hi;
  else if (!strcmp(name, "h_lo")) out = m.h_lo;
  else if (!strcmp(name, "dy_hi")) out = m.dy_hi;
  else if (!strcmp(name, "dy_lo")) out = m.dy_lo;
  TT_REQUIRE(out != nullptr, "tt_debug_step_buffer: unknown buffer '%s'", name);
  *ptr = out;
  return 0;
}

extern "C" int tt_triplet_step(const tt_step_args* a, tt_stream_t stream) {
  TT_REQUIRE(a != nullptr, "tt_triplet_step: null args");
  const int B = a->B, H = a->H, P = a->P;
  int rc = check_mlp_shape("tt_triplet_step", B, H, P, a->precision);
  if (rc) return rc;
  TT_REQUIRE(B >= 1, "tt_triplet_step: empty batch");
  const int train_table = (a->dtable_q != nullptr || a->dtable_d != nullptr) ? 1 : 0;
  TT_REQUIRE(!train_table || (a->dtable_q && a->dtable_d), "tt_triplet_step: give both table gradients or neither");
  TT_REQUIRE(a->grad_accumulate == 0 || a->grad_accumulate == 1, "tt_triplet_step: grad_accumulate must be 0 or 1, got %d",
             a->grad_accumulate);
  const int acc = a->grad_accumulate;
  const bool table_adam = a->table_param_q != nullptr || a->table_param_d != nullptr;
  if (table_adam) {
    TT_REQUIRE(a->table_param_q && a->table_param_d, "tt_triplet_step: give both table_param_q and table_param_d or "
               "neither");
    TT_REQUIRE(train_table, "tt_triplet_step: the table optimiser needs the table gradients (dtable_q / dtable_d)");
    TT_REQUIRE(a->table_dtype == TT_F32, "tt_triplet_step: the table optimiser needs fp32 tables");
    TT_REQUIRE(a->table_param_q == a->table_q && a->table_param_d == a->table_d && a->table_q != a->table_d,
               "tt_triplet_step: table_param_q / table_param_d must be the two distinct tables the step gathers from");
    TT_REQUIRE(a->adam_param != nullptr, "tt_triplet_step: the table optimiser shares the projections' step count: it "
               "needs adam_param");
    TT_REQUIRE(a->adam_state && a->table_exp_avg_q && a->table_exp_avg_sq_q && a->table_exp_avg_d &&
               a->table_exp_avg_sq_d, "tt_triplet_step: the table optimiser needs adam_state and all four table moments");
  }
  const size_t need = tt_step_ws_bytes(B, a->Lq, a->Ld, H, P, a->vocab, a->precision, train_table);
  TT_REQUIRE(a->ws && a->ws_bytes >= need, "tt_triplet_step: workspace too small (%zu < %zu)", a->ws_bytes, need);
  cudaStream_t st = as_stream(stream);
  ApiStepWs w;
  carve_step_ws(reinterpret_cast<char*>(a->ws), B, a->Lq, a->Ld, H, P, a->vocab, a->precision, train_table, &w);

  // 1. pooled gather for q | p | n rows
  PoolParams pp{};
  pp.nseg = 3;
  pp.seg[0] = PoolSegDev{a->table_q, a->q_ids, a->q_mask, B, a->Lq, 0};
  pp.seg[1] = PoolSegDev{a->table_d, a->p_ids, a->p_mask, B, a->Ld, B};
  pp.seg[2] = PoolSegDev{a->table_d, a->n_ids, a->n_mask, B, a->Ld, 2 * B};
  pp.ids_dtype = a->ids_dtype;
  pp.mask_dtype = a->mask_dtype;
  pp.vocab = a->vocab;
  pp.xhat = w.xhat;
  pp.cnt = w.cnt;
  pp.nrm = w.nrm;
  pp.err = a->err_flag;
  if (a->neg_index) {  // in-batch negatives: the n rows are copies of the p rows they name
    pp.nseg = 2;
    pp.alias = a->neg_index;
    pp.alias_n = B;
    pp.alias_src_row0 = B;
    pp.alias_dst_row0 = 2 * B;
  }
  if (a->pooled_index) {  // frozen front end computed once per text: rows are copied, not pooled
    TT_REQUIRE(!train_table, "tt_triplet_step: pooled_index needs frozen tables (dtable_q / dtable_d must be NULL)");
    TT_REQUIRE(!a->neg_index, "tt_triplet_step: pooled_index and neg_index are exclusive (name the negatives' rows in "
               "pooled_index instead)");
    pp.rows_q = a->pooled_q; pp.rows_q_n = a->pooled_q_rows;
    pp.rows_d = a->pooled_d; pp.rows_d_n = a->pooled_d_rows;
    pp.row_index = a->pooled_index;
    pp.row_B = B;
  }

  float* dxhat = train_table ? w.dxhat : nullptr;
  bool adam_done = false;
  TT_REQUIRE(a->phases >= 0 && a->phases <= (TT_STEP_FRONT | TT_STEP_BACK), "tt_triplet_step: bad phases %d", a->phases);
  const bool front = a->phases == 0 || (a->phases & TT_STEP_FRONT), back = a->phases == 0 || (a->phases & TT_STEP_BACK);
  if (a->precision == TT_PREC_FP32) {
    if (front && (rc = pool_fwd_launch(pp, a->table_dtype, H, st))) return rc;
    if (!back) return 0;
    // 2. both towers
    if ((rc = mlp_fwd_fp32(w.xhat, B, H, P, a->Wq1, a->bq1, a->Wq2, a->bq2, w.h, w.y, st))) return rc;
    if ((rc = mlp_fwd_fp32(w.xhat + (size_t)B * H, 2 * B, H, P, a->Wd1, a->bd1, a->Wd2, a->bd2, w.h + (size_t)B * P,
                           w.y + (size_t)B * P, st)))
      return rc;
    // 3. loss, 4. its gradient
    const float* yq = w.y;
    const float* yp = w.y + (size_t)B * P;
    const float* yn = w.y + (size_t)2 * B * P;
    if ((rc = triplet_loss_fwd(yq, yp, yn, B, P, a->margin, a->inv_batch, w.stats, a->loss, st))) return rc;
    if ((rc = triplet_loss_bwd(yq, yp, yn, w.stats, nullptr, a->grad_scale, B, P, a->inv_batch, w.dy,
                               w.dy + (size_t)B * P, w.dy + (size_t)2 * B * P, nullptr, st)))
      return rc;
    // 5. tower backward (document tower: positives and negatives in one M = 2B pass); grad_accumulate adds the old
    // gradient after the sum, as the tensor-core chains do
    const int facc = acc ? kAccumAfterSum : 0;
    if ((rc = mlp_bwd_fp32(w.dy, w.xhat, w.h, a->Wq1, a->Wq2, B, H, P, a->dWq1, a->dbq1, a->dWq2, a->dbq2, dxhat, facc,
                           w.dz1, w.fp32_scratch, st)))
      return rc;
    if ((rc = mlp_bwd_fp32(w.dy + (size_t)B * P, w.xhat + (size_t)B * H, w.h + (size_t)B * P, a->Wd1, a->Wd2, 2 * B, H,
                           P, a->dWd1, a->dbd1, a->dWd2, a->dbd2, dxhat ? dxhat + (size_t)B * H : nullptr, facc,
                           w.dz1 + (size_t)B * P, w.fp32_scratch, st)))
      return rc;
  } else {
    StepSm100 s{};
    s.pool = pp;
    s.table_dtype = a->table_dtype;
    s.B = B; s.H = H; s.P = P;
    s.Wq1 = a->Wq1; s.bq1 = a->bq1; s.Wq2 = a->Wq2; s.bq2 = a->bq2;
    s.Wd1 = a->Wd1; s.bd1 = a->bd1; s.Wd2 = a->Wd2; s.bd2 = a->bd2;
    s.margin = a->margin; s.inv_batch = a->inv_batch; s.grad_scale = a->grad_scale;
    s.loss = a->loss;
    s.dWq1 = a->dWq1; s.dbq1 = a->dbq1; s.dWq2 = a->dWq2; s.dbq2 = a->dbq2;
    s.dWd1 = a->dWd1; s.dbd1 = a->dbd1; s.dWd2 = a->dWd2; s.dbd2 = a->dbd2;
    s.h = w.h; s.y = w.y; s.stats = w.stats; s.dy = w.dy;
    s.dxhat = dxhat;
    s.n_split = (a->precision == TT_PREC_BF16X3) ? 3 : 1;
    s.grad_accumulate = acc;
    s.ws = w.mma_ws; s.ws_bytes = w.mma_ws_bytes;
    s.phases = a->phases;
    TT_REQUIRE(a->chain >= 0 && a->chain <= 2, "tt_triplet_step: bad chain selector %d", a->chain);
    s.chain = a->chain == 1 || (a->chain == 0 && chain_enabled());
    if (a->adam_param && s.chain) {  // the optimiser rides in the chain kernel's tail
      s.adam = FusedAdam{a->adam_state, a->adam_param, a->adam_grad, a->adam_exp_avg, a->adam_exp_avg_sq, a->adam_n,
                         a->adam_lr, a->adam_beta1, a->adam_beta2, a->adam_eps};
      adam_done = true;
    }
    if ((rc = step_sm100(s, st))) return rc;
    if (!back) return 0;
  }
  if (a->adam_param && !adam_done) {
    TT_REQUIRE(a->adam_state && a->adam_grad && a->adam_exp_avg && a->adam_exp_avg_sq,
               "tt_triplet_step: the optimiser needs state, grad and both moments");
    if ((rc = tt_adam_step_dev(a->adam_param, a->adam_grad, a->adam_exp_avg, a->adam_exp_avg_sq, a->adam_n, a->adam_lr,
                               a->adam_beta1, a->adam_beta2, a->adam_eps, a->adam_state, 1.f, stream)))
      return rc;
  }
  // 6. table gradients (D2 extension), or with table_param_* the tables' Adam step in the scatter-add's epilogue.  Every
  // path above has advanced adam_state for this step in stream order, so the tables use the projections' step count
  if (train_table) {
    if ((rc = pool_bwd_prep(w.dxhat, w.xhat, w.cnt, w.nrm, 3 * B, H, w.g, st))) return rc;
    const TableAdam tq{a->table_param_q, a->table_exp_avg_q, a->table_exp_avg_sq_q, a->adam_lr, a->adam_beta1,
                       a->adam_beta2, a->adam_eps, a->adam_state};
    const TableAdam td{a->table_param_d, a->table_exp_avg_d, a->table_exp_avg_sq_d, a->adam_lr, a->adam_beta1,
                       a->adam_beta2, a->adam_eps, a->adam_state};
    PoolBwdSeg sq{a->q_ids, a->q_mask, B, a->Lq, 0};
    if ((rc = pool_bwd_scatter(&sq, 1, a->ids_dtype, a->mask_dtype, w.g, a->vocab, H, a->dtable_q, acc, w.pool_ws,
                               w.pool_ws_bytes, st, table_adam ? &tq : nullptr)))
      return rc;
    PoolBwdSeg sd[2] = {{a->p_ids, a->p_mask, B, a->Ld, B}, {a->n_ids, a->n_mask, B, a->Ld, 2 * B}};
    int nsd = 2;
    if (a->neg_index) {  // negative i pooled positive neg_index[i]'s tokens: fold its g row into that positive's
      if ((rc = pool_bwd_fold_neg(a->neg_index, B, H, w.g + (size_t)2 * B * H, w.g + (size_t)B * H, st))) return rc;
      nsd = 1;
    }
    if ((rc = pool_bwd_scatter(sd, nsd, a->ids_dtype, a->mask_dtype, w.g, a->vocab, H, a->dtable_d, acc, w.pool_ws,
                               w.pool_ws_bytes, st, table_adam ? &td : nullptr)))
      return rc;
  }
  return 0;
}

extern "C" int tt_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                            float beta1, float beta2, float eps, int step, float grad_scale, tt_stream_t stream) {
  TT_REQUIRE(step >= 1, "tt_adam_step: step must be >= 1");
  if (n == 0) return 0;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const float step_size = (float)((double)lr / bc1);
  const float bc2_sqrt = (float)sqrt(bc2);
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, beta1,
                                                                         beta2, eps, step_size, bc2_sqrt, grad_scale);
  TT_LAUNCH_CHECK();
  return 0;
}

extern "C" int tt_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                float beta1, float beta2, float eps, double* state, float grad_scale,
                                tt_stream_t stream) {
  TT_REQUIRE(state != nullptr, "tt_adam_step_dev: null state");
  cudaStream_t st = as_stream(stream);
  adam_advance_kernel<<<1, 1, 0, st>>>(state, beta1, beta2);
  TT_LAUNCH_CHECK();
  if (n == 0) return 0;
  adam_dev_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                eps, state, grad_scale);
  TT_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// corpus scan
// ------------------------------------------------------------------------------------------------
extern "C" size_t tt_scan_ws_bytes(int Q, int64_t N, int P, int k, int precision) {
  if (N <= 0) return 0;  // an empty shard only writes padding (and has no document splits to plan)
  if (precision == TT_PREC_FP32) return scan_fp32_ws_bytes(Q, N, k);
  return scan_sm100_ws_bytes(Q, N, P, k);
}

extern "C" int tt_scan_topk(const float* Qn, const float* Dn, const void* Qb, const void* Db, int Q, int64_t N, int P,
                            int k, int64_t id_base, int precision, float* top_score, int64_t* top_id, void* ws,
                            size_t ws_bytes, tt_stream_t stream) {
  TT_REQUIRE(Q >= 0 && N >= 0 && P >= 1 && k >= 1, "tt_scan_topk: bad shape Q=%d N=%lld P=%d k=%d", Q, (long long)N, P,
             k);
  cudaStream_t st = as_stream(stream);
  if (Q == 0) return 0;
  TT_REQUIRE(ws_bytes >= tt_scan_ws_bytes(Q, N, P, k, precision), "tt_scan_topk: workspace too small");
  if (N == 0) return scan_empty(Q, k, top_score, reinterpret_cast<long long*>(top_id), st);
  if (precision == TT_PREC_FP32)
    return scan_topk_fp32(Qn, Dn, Q, N, P, k, id_base, top_score, reinterpret_cast<long long*>(top_id), ws, ws_bytes,
                          st);
  TT_REQUIRE(Qb && Db, "tt_scan_topk: the tensor-core scan needs bf16 copies of queries and documents");
  return scan_topk_sm100(Qn, Dn, Qb, Db, Q, N, P, k, id_base, top_score, reinterpret_cast<long long*>(top_id), ws,
                         ws_bytes, st);
}

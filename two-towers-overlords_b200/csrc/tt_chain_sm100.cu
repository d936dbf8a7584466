// The projection chain of one training step as ONE persistent kernel (north_star (2): the tower MLP on tcgen05 with
// cosine distance + margin loss fused into the second layer's epilogue, forward and backward).  Replaces
// backend/model.py:33-38,59,132-145 and what autograd does for them inside backend/training.py:40-51.
//
// One CTA per SM walks a static queue of tile tasks in dependency order; kernel boundaries of the per-kernel chain
// (tt_gemm_sm100.cu: split -> fwd1 -> fwd2 -> loss -> dY^T -> dz1 -> dW2 -> colsums -> dW1 -> reduce) become
// per-row-tile ready counters in global memory:
//
//   S    weights -> bf16 terms                                           SIMT, one task per CTA
//   F1   h  = relu(x W1^T + b1)        -> (hi,lo) terms                   tile (row tile, col tile)
//   F2L  y  = h W2^T + b2 for the q | p | n rows of 128 triplets (three accumulators), then in the SAME epilogue:
//        partial |q|^2,|p|^2,|n|^2,q.p,q.n over this tile's columns -> exchanged with the sibling column tiles through
//        global memory -> cosines, hinge, closed-form dY straight from TMEM -> dY (hi,lo), db2 partials
//   DZ   dz1 = (dY W2) * (h > 0)       -> (hi,lo), db1 partials
//   DX   dxhat = dz1 W1                (only when the token tables train)
//   DW2  dW2 partial = dY^T h  over a chunk of batch rows                 raw fp32 partial tile
//   DW1  dW1 partial = dz1^T x over a chunk of batch rows
//   G    gradients = fixed-order sums of the partials; loss; Adam step-count advance
//
// No transposed copy of anything exists: contractions whose reduction runs over the OUTER dimension of a row-major
// operand (the weight gradients dW = dY^T h, dz1^T x reduce over batch rows; dz1 = dY W2 and dxhat = dz1 W1 reduce
// over the weights' rows) read that operand as it lies in memory — TMA boxes of 64 k-rows x 64 elements, 128-byte
// swizzle — and describe it to tcgen05.mma as MN-MAJOR (instruction-descriptor bits 15 / 16; shared-memory descriptor:
// leading offset 8192 B between the two 64-element boxes of a 128-wide tile, stride offset 1024 B between groups of 8
// k-rows, 2048 B per K = 16 step; checked bit-exact against the host by tt_selftest_mn_major / tests/test_cuda_parity.py).
//
// Warp roles per CTA: warp 0 = TMA producer (also waits for a task's dependencies), warp 1 = TMEM owner + single-thread
// tcgen05.mma issuer, warps 2-9 = epilogue (two warps per TMEM lane quarter, 64 columns each).  The accumulators form
// a ring of four 128-column TMEM buffers, so an epilogue overlaps the following main loops.  All sums have a fixed
// order: results are bit-reproducible run to run.
#include <stdlib.h>

#include "tt_ptx.cuh"
#include "tt_step_ws.cuh"
#include "tt_tma.cuh"

namespace tt {

namespace {

using namespace ptx;

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int kMaxStages = 6;
constexpr int kAcc = 4;  // TMEM accumulator ring
constexpr int kEpiThreads = 256;
constexpr int kThreads = 64 + kEpiThreads;
constexpr uint32_t kABytes = BM * BK * 2, kBBytes = BN * BK * 2, kStageBytes = kABytes + kBBytes;
constexpr int kSplitPad = 66;  // bf16 elements per row of a transposed 64 x 64 staging tile
// Per-epilogue-warp row staging: a thread owns a tile row (TMEM lane), so direct stores would scatter 16-byte pieces
// over 32 rows per instruction; instead the warp parks a [32 rows x 16 | 32 columns] block in shared memory and writes
// it out with whole sectors / lines per row.  The split phase's transpose tiles overlay the same bytes.
constexpr int kRowStage = 3072;   // per warp: 2 x 1536 (two bf16 blocks of 16 columns) or 2560 (fp32, 16 columns)
constexpr int kTermPitch = 48;    // bytes per row of a 16-column bf16 block (32 B + pad: conflict-free 16 B accesses)
constexpr int kTermBlock = 32 * kTermPitch;
constexpr int kF32Pitch = 80;     // bytes per row of a 16-column fp32 block (64 B + pad)
constexpr int kCsBytes = 2 * 8 * 64 * 4;
constexpr int kStagingBytes = kCsBytes /*column sums*/ + 8 * kRowStage /*row staging | split tiles*/ + 64;
static_assert(2 * 64 * kSplitPad * 2 <= 8 * kRowStage, "split tiles overlay the row staging");
constexpr size_t chain_smem(int stages) { return (size_t)stages * kStageBytes + 1024 + 256 + kStagingBytes; }
constexpr float kCosEps = 1e-8f;  // torch.cosine_similarity eps (per-vector clamp), backend/model.py:134
constexpr long long kSpinLimit = 4000000000ll;

enum { T_S = 0, T_T, T_F1, T_F2L, T_DZ, T_DX, T_DW2, T_DW1, T_G, T_COUNT };

struct TowerMaps {  // K-major bf16 operand terms of one tower (box 128 rows x 64 k)
  CUtensorMap x[3], w1[3];   // F1:  [rows,H] x [P,H]                          boxes of 128 rows x 64 k
  CUtensorMap h[2], w2[2];   // F2:  [rows,P] x [P,P]   (w2: boxes of 64 rows — the loss tiles are 64 columns wide;
                             //      DZ reads the same boxes as its MN-major B operand: 64 k-rows x 64 columns)
  CUtensorMap dy[2];         // DZ:  A = dY [rows,P] K-major;  B = W2 [k][n] MN-major (w2 above)
  CUtensorMap dz[2], w1k[2];  // DX:  A = dz1 [rows,P] K-major; B = W1 [k][n] MN-major
  CUtensorMap dyk[2], hk[2];  // DW2: A = dY [k = batch row][m], B = h [k][n], both MN-major (boxes of 64 rows x 64)
  CUtensorMap dzk[2], xk[2];  // DW1: A = dz1 [k][m], B = x [k][n], both MN-major
};

struct SplitJobC {  // fp32 [R, C] dense -> bf16 terms hi/lo[/lo2] [R, C]
  const float* X;
  bf16 *hi, *lo, *lo2;
  int R, C;
  int f4_0;    // first float4 of this matrix in the flat pass over all jobs
};

struct alignas(64) ChainParams {
  TowerMaps tm[2];
  int B, H, P, RTB, NC, NCH, NCF;  // NCF: 64-column tiles of the fused layer-2 / loss phase
  int pairs, terms, pairs1, terms1;
  int kcb, nch[2], kbt[2];
  int off[T_COUNT + 1];
  int stages, n_sj, n_split_f4, n_split_f4_w1;
  int nS;        // tasks of the S, T and G phases: one per CTA
  int use_pdl;   // launched as a programmatic dependent of the pooled gather: wait for it before touching x
  SplitJobC sj[6];
  float margin, inv_batch, grad_scale;
  const float *b1[2], *b2[2];
  float *h, *y, *dy, *dz1, *dxhat, *stats, *loss;
  bf16 *h_hi, *h_lo, *dy_hi, *dy_lo, *dz_hi, *dz_lo;
  float *part2, *part1;
  float *dW1[2], *db1[2], *dW2[2], *db2[2];
  float *stat_part, *cs1, *cs2, *hinge_part, *ybuf;
  unsigned* ctr;
  int n_counters;
  // optional fused optimiser: torch.optim.Adam on the flat parameter buffer the 8 tensors are slices of
  double* adam_state;  // {t, beta1^t, beta2^t, -}: advanced once per launch (by the first task), read by the tail
  float *adam_p, *adam_g, *adam_m, *adam_v;
  float lr, beta1, beta2, eps;
  int grad_accumulate;  // 1: a gradient element becomes fl(old + its fixed-order sum), and Adam consumes that
  unsigned total_signals, dw2_signals;
  unsigned long long* trace;  // nullable (TT_CHAIN_TRACE=1)
};

// ---- cross-CTA hand-off ------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void signal(unsigned* p) {
  asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ unsigned ld_relaxed(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Polls with relaxed loads (an acquire load invalidates the SM's L1 on every poll, which evicts the epilogue warps'
// bias lines and register spills) and orders everything after the successful poll with one acquire fence.
__device__ __forceinline__ void wait_counter(const unsigned* p, unsigned target) {
  if (ld_relaxed(p) < target) {
    const long long t0 = clock64();
    while (ld_relaxed(p) < target) {
      __nanosleep(32);
      if (clock64() - t0 > kSpinLimit) __trap();  // a protocol bug fails the launch instead of hanging the GPU
    }
  }
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

struct Task {
  int type, i;
};
__device__ __forceinline__ Task decode(const ChainParams& p, int idx) {
  int t = 0;
#pragma unroll
  for (int k = 1; k < T_COUNT; ++k)
    if (idx >= p.off[k]) t = k;
  return Task{t, idx - p.off[t]};
}

struct RowTile {
  int r, seg, t, trow, grow, valid;
};
// row tile u = 3 r + seg: 128 rows of segment seg (q | p | n) starting at triplet 128 r
__device__ __forceinline__ RowTile row_tile(const ChainParams& p, int u) {
  RowTile rt;
  rt.r = u / 3;
  rt.seg = u - 3 * rt.r;
  rt.t = rt.seg != 0;
  rt.trow = (rt.seg == 2 ? p.B : 0) + rt.r * BM;  // row inside the tower's operand (document tower: p rows, n rows)
  rt.grow = rt.seg * p.B + rt.r * BM;             // row inside the [3B, .] activations
  rt.valid = min(BM, p.B - rt.r * BM);
  return rt;
}

struct Sub {
  const CUtensorMap *a, *b;
  int terms, pairs, m0, n0, kb0, nkb;
  int bn;  // MMA N = rows of the B box (128, or 64 for the loss tiles)
  int amn, bmn;  // operand is MN-major: two boxes of 64 k-rows x 64 elements at (m0 | m0 + 64, k) instead of one K-major box
};
__device__ __forceinline__ int n_subs(int type) {
  return (type == T_S || type == T_T || type == T_G) ? 0 : 1;
}

__device__ __forceinline__ void dw_chunk(const ChainParams& p, int ci, int& t, int& j) {
  t = ci >= p.nch[0];
  j = ci - (t ? p.nch[0] : 0);
}

__device__ __forceinline__ Sub get_sub(const ChainParams& p, Task tk, int k) {
  Sub s;
  s.terms = p.terms;
  s.pairs = p.pairs;
  s.kb0 = 0;
  s.bn = BN;
  s.amn = s.bmn = 0;
  switch (tk.type) {
    case T_F1: {
      const RowTile rt = row_tile(p, tk.i / p.NC);
      s.a = p.tm[rt.t].x; s.b = p.tm[rt.t].w1;
      s.terms = p.terms1; s.pairs = p.pairs1;
      s.m0 = rt.trow; s.n0 = (tk.i % p.NC) * BN; s.nkb = p.H / BK;
    } break;
    case T_F2L: {  // task = ((r, c), seg): layer 2 of 128 rows of one row group (q | p | n) x 64 columns
      const int seg = tk.i % 3, rc = tk.i / 3, r = rc / p.NCF, t = seg != 0;
      s.a = p.tm[t].h; s.b = p.tm[t].w2;
      s.m0 = (seg == 2 ? p.B : 0) + r * BM; s.n0 = (rc % p.NCF) * 64; s.nkb = p.P / BK;
      s.bn = 64;
    } break;
    case T_DZ: {
      const RowTile rt = row_tile(p, tk.i / p.NC);
      s.a = p.tm[rt.t].dy; s.b = p.tm[rt.t].w2; s.bmn = 1;
      s.m0 = rt.trow; s.n0 = (tk.i % p.NC) * BN; s.nkb = p.P / BK;
    } break;
    case T_DX: {
      const RowTile rt = row_tile(p, tk.i / p.NCH);
      s.a = p.tm[rt.t].dz; s.b = p.tm[rt.t].w1k; s.bmn = 1;
      s.m0 = rt.trow; s.n0 = (tk.i % p.NCH) * BN; s.nkb = p.P / BK;
    } break;
    case T_DW2: {
      const int nt_ = p.NC * p.NC, tile = tk.i % nt_;
      int t, j;
      dw_chunk(p, tk.i / nt_, t, j);
      s.a = p.tm[t].dyk; s.b = p.tm[t].hk; s.amn = s.bmn = 1;
      s.m0 = (tile / p.NC) * BM; s.n0 = (tile % p.NC) * BN;
      s.kb0 = j * p.kcb; s.nkb = min(p.kcb, p.kbt[t] - s.kb0);
    } break;
    default: {  // T_DW1
      const int nt_ = p.NC * p.NCH, tile = tk.i % nt_;
      int t, j;
      dw_chunk(p, tk.i / nt_, t, j);
      s.a = p.tm[t].dzk; s.b = p.tm[t].xk; s.amn = s.bmn = 1;
      s.m0 = (tile / p.NCH) * BM; s.n0 = (tile % p.NCH) * BN;
      s.kb0 = j * p.kcb; s.nkb = min(p.kcb, p.kbt[t] - s.kb0);
    } break;
  }
  return s;
}

__device__ __forceinline__ unsigned* h_ready(const ChainParams& p) { return p.ctr + 8; }
__device__ __forceinline__ unsigned* dy_ready(const ChainParams& p) { return p.ctr + 8 + 3 * p.RTB; }
__device__ __forceinline__ unsigned* dz_ready(const ChainParams& p) { return p.ctr + 8 + 6 * p.RTB; }
__device__ __forceinline__ unsigned* stat_ready(const ChainParams& p) { return p.ctr + 8 + 9 * p.RTB; }
__device__ __forceinline__ unsigned* y_ready(const ChainParams& p) { return p.ctr + 8 + 10 * p.RTB; }  // [RTB * NCF]

// every row tile [seg][r] that holds one of the batch rows [k0, k1) of tower t must have all NC column tiles done
__device__ __forceinline__ void wait_rows(const ChainParams& p, const unsigned* ready, unsigned need, int t, int k0,
                                          int k1) {
  if (t == 0) {
    for (int r = k0 / BM; r <= (k1 - 1) / BM; ++r) wait_counter(ready + r, need);
    return;
  }
  if (k0 < p.B)
    for (int r = k0 / BM; r <= (min(k1, p.B) - 1) / BM; ++r) wait_counter(ready + p.RTB + r, need);
  if (k1 > p.B)
    for (int r = (max(k0, p.B) - p.B) / BM; r <= (k1 - p.B - 1) / BM; ++r) wait_counter(ready + 2 * p.RTB + r, need);
}

__device__ __forceinline__ void wait_deps(const ChainParams& p, Task tk) {
  switch (tk.type) {
    case T_F1: wait_counter(p.ctr + 0, (unsigned)p.nS); break;
    case T_F2L: {
      const int seg = tk.i % 3, r = tk.i / 3 / p.NCF;
      wait_counter(p.ctr + 2, (unsigned)p.nS);  // second-layer weight terms (and transposes)
      wait_counter(h_ready(p) + seg * p.RTB + r, p.NC);
    } break;
    case T_DZ: {
      const RowTile rt = row_tile(p, tk.i / p.NC);
      wait_counter(dy_ready(p) + rt.seg * p.RTB + rt.r, p.NCF);
    } break;
    case T_DX: {
      const RowTile rt = row_tile(p, tk.i / p.NCH);
      wait_counter(dz_ready(p) + rt.seg * p.RTB + rt.r, p.NC);
    } break;
    case T_DW2:
    case T_DW1: {
      const int nt_ = tk.type == T_DW2 ? p.NC * p.NC : p.NC * p.NCH;
      int t, j;
      dw_chunk(p, tk.i / nt_, t, j);
      const int k0 = j * p.kcb * BK, k1 = min(k0 + p.kcb * BK, t ? 2 * p.B : p.B);
      if (tk.type == T_DW2) wait_rows(p, dy_ready(p), p.NCF, t, k0, k1);
      else wait_rows(p, dz_ready(p), p.NC, t, k0, k1);
    } break;
    default: break;
  }
}

// ---- epilogue helpers --------------------------------------------------------------------------------------
// sum over the 32 lanes of each of 16 per-lane values; every lane returns the total of column (lane >> 1) & 15
__device__ __forceinline__ float colsum16(const float (&v)[16], int lane) {
  float a[8], b[4], c[2];
  const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4, h2 = lane & 2;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float keep = h16 ? v[8 + j] : v[j], send = h16 ? v[j] : v[8 + j];
    a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float keep = h8 ? a[4 + j] : a[j], send = h8 ? a[j] : a[4 + j];
    b[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const float keep = h4 ? b[2 + j] : b[j], send = h4 ? b[j] : b[2 + j];
    c[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  const float keep = h2 ? c[1] : c[0], send = h2 ? c[0] : c[1];
  float d = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  d += __shfl_xor_sync(0xffffffffu, d, 1);
  return d;
}

__device__ __forceinline__ void store16(float* dst, const float (&v)[16]) {
  float4* d = reinterpret_cast<float4*>(dst);
#pragma unroll
  for (int j = 0; j < 4; ++j) d[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

__device__ __forceinline__ void split16(const float (&v)[16], bf16 (&hi)[16], bf16 (&lo)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) split_bf16(v[j], hi[j], lo[j]);
}
// this lane's 16 bf16 (32 B) -> row `lane` of a staged block
__device__ __forceinline__ void stage16(uint8_t* blk, int lane, const bf16 (&x)[16]) {
  uint4* d = reinterpret_cast<uint4*>(blk + lane * kTermPitch);
  d[0] = reinterpret_cast<const uint4*>(x)[0];
  d[1] = reinterpret_cast<const uint4*>(x)[1];
}
// staged block [32 rows][16 bf16] -> g[(row0 + r) * ld + n ..], rows r < vr: two lanes per row, 16 rows per instruction
__device__ __forceinline__ void flush16(const uint8_t* blk, int lane, bf16* g, size_t row0, int n, int ld, int vr) {
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int r = it * 16 + (lane >> 1), sg = lane & 1;
    if (r < vr)
      *reinterpret_cast<uint4*>(g + (row0 + r) * ld + n + sg * 8) =
          *reinterpret_cast<const uint4*>(blk + r * kTermPitch + sg * 16);
  }
}
// fp32: this lane's 16 values -> row `lane` of a staged [32][16] block
__device__ __forceinline__ void stage_f32(uint8_t* blk, int lane, const float (&v)[16]) {
  float4* d = reinterpret_cast<float4*>(blk + lane * kF32Pitch);
#pragma unroll
  for (int j = 0; j < 4; ++j) d[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
// staged [32 rows][16 fp32] -> g[(row0 + r) * ld + n ..]: four lanes per row (two whole sectors), eight rows per instruction
__device__ __forceinline__ void flush_f32(const uint8_t* blk, int lane, float* g, size_t row0, int n, size_t ld, int vr) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int r = it * 8 + (lane >> 2), sg = lane & 3;
    if (r < vr)
      *reinterpret_cast<float4*>(g + (row0 + r) * ld + n + sg * 4) =
          *reinterpret_cast<const float4*>(blk + r * kF32Pitch + sg * 16);
  }
}

struct EpiCtx {
  uint32_t tmem_base;
  uint64_t *acc_full, *acc_empty;
  float* cs_s;  // [2][8][64]
  bf16* sp_s;   // [2][64][kSplitPad]
  float* hs_s;  // [4]
  uint8_t* rs;  // this warp's row staging (kRowStage bytes)
  int we, q, hf, lane, tid;  // epilogue warp 0..7, TMEM lane quarter, column half, lane, epilogue thread 0..255
  int ab;
  uint32_t aph;
  unsigned long long* trace;  // this CTA's timeline slots (nullable)
  int tslot, tidx;
};

// timeline event of the current task: kind 0 = start, 1 = end, 2 = accumulators ready, 3 = sibling sums arrived
__device__ __forceinline__ void trace_ev(EpiCtx& e, int kind) {
  if (e.trace && e.tid == 0 && e.tslot < kTraceSlots) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    e.trace[e.tslot * 2] = ((unsigned long long)e.tidx << 2) | (unsigned long long)kind;
    e.trace[e.tslot * 2 + 1] = t;
    ++e.tslot;
  }
}

__device__ __forceinline__ uint32_t acc_addr(const EpiCtx& e, int buf, int chunk) {
  return e.tmem_base + ((uint32_t)(e.q * 32) << 16) + (uint32_t)(buf * BN + e.hf * 64 + chunk * 16);
}
__device__ __forceinline__ void acc_advance(EpiCtx& e, int n) {
  e.ab += n;
  if (e.ab >= kAcc) {
    e.ab -= kAcc;
    e.aph ^= 1u;
  }
}
// all writes of this CTA's epilogue visible device-wide (also to TMA reads of other CTAs), then one signal per counter
__device__ __forceinline__ void publish(const EpiCtx& e) {
  fence_proxy_async();
  __threadfence();
  epi_bar();
}

// per-warp column sums of one chunk -> staging; reduce_cs() then adds the four lane quarters in a fixed order
__device__ __forceinline__ void stage_cs(const EpiCtx& e, int slot, int chunk, float d) {
  if ((e.lane & 1) == 0) e.cs_s[(slot * 8 + e.we) * 64 + chunk * 16 + (e.lane >> 1)] = d;
}
// col: column of the tile; cw: columns per epilogue warp (64 for 128-wide tiles, 32 for the 64-wide loss tiles)
__device__ __forceinline__ float reduce_cs(const EpiCtx& e, int slot, int col, int cw = 64) {
  const int hf = col / cw, cc = col - hf * cw;
  float s = 0.f;
#pragma unroll
  for (int quarter = 0; quarter < 4; ++quarter) s += e.cs_s[(slot * 8 + hf * 4 + ((quarter - 2) & 3)) * 64 + cc];
  return s;
}

__device__ __forceinline__ uint32_t pack_bf16(bf16 a, bf16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// weights of both towers -> bf16 terms: one flat float4 pass over all matrices, every load of a thread in flight at once
__device__ void epi_split(const ChainParams& p, EpiCtx& e, int task_i) {
  const int nS = p.nS;
  if (task_i == 0 && e.tid == 0 && p.adam_state) {
    // torch.optim.Adam's step count and beta powers live on the device so that a graph replay advances them; the
    // tail (epi_grad) reads them through the S -> ... -> G dependency chain
    const double t = p.adam_state[0];
    p.adam_state[0] = t + 1.0;
    p.adam_state[1] = (t == 0.0 ? 1.0 : p.adam_state[1]) * (double)p.beta1;
    p.adam_state[2] = (t == 0.0 ? 1.0 : p.adam_state[2]) * (double)p.beta2;
  }
  // (a) flat pass, first-layer weights first
  constexpr int U = 4;
  const int gstride = nS * kEpiThreads;
  for (int part = 0; part < 2; ++part) {
    const int lo_i = part ? p.n_split_f4_w1 : 0, hi_i = part ? p.n_split_f4 : p.n_split_f4_w1;
    for (int base = lo_i + task_i * kEpiThreads + e.tid; base < hi_i; base += U * gstride) {
      float4 v[U];
      int ji[U], li[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = base + u * gstride;
        ji[u] = -1;
        if (i < hi_i) {
          int j = 0;
          for (int k = 1; k < p.n_sj; ++k)
            if (i >= p.sj[k].f4_0) j = k;
          ji[u] = j;
          li[u] = i - p.sj[j].f4_0;
          v[u] = __ldg(reinterpret_cast<const float4*>(p.sj[j].X) + li[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (ji[u] < 0) continue;
        const SplitJobC& J = p.sj[ji[u]];
        const float x[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
        bf16 h[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) split_bf16(x[k], h[k], l[k]);
        reinterpret_cast<uint2*>(J.hi)[li[u]] = make_uint2(pack_bf16(h[0], h[1]), pack_bf16(h[2], h[3]));
        reinterpret_cast<uint2*>(J.lo)[li[u]] = make_uint2(pack_bf16(l[0], l[1]), pack_bf16(l[2], l[3]));
        if (J.lo2) {
          bf16 m[4];
#pragma unroll
          for (int k = 0; k < 4; ++k)
            m[k] = __float2bfloat16_rn((x[k] - __bfloat162float(h[k])) - __bfloat162float(l[k]));
          reinterpret_cast<uint2*>(J.lo2)[li[u]] = make_uint2(pack_bf16(m[0], m[1]), pack_bf16(m[2], m[3]));
        }
      }
    }
    if (part == 0) {  // layer 1 can start
      publish(e);
      if (e.tid == 0) signal(p.ctr + 0);
    }
  }
  publish(e);
  if (e.tid == 0) signal(p.ctr + 2);
}

__device__ __forceinline__ int warp_valid_rows(const EpiCtx& e, int valid) { return max(0, min(32, valid - e.q * 32)); }

__device__ void epi_f1(const ChainParams& p, EpiCtx& e, int task_i) {
  const RowTile rt = row_tile(p, task_i / p.NC);
  const int n0 = (task_i % p.NC) * BN;
  mbar_wait(&e.acc_full[e.ab], e.aph);
  tc_fence_after();
  trace_ev(e, 2);
  const int row = e.q * 32 + e.lane;
  const bool ok = row < rt.valid;
  const int vr = warp_valid_rows(e, rt.valid);
  const size_t wrow0 = (size_t)rt.grow + e.q * 32;
  const float* bias = p.b1[rt.t];
  for (int ch = 0; ch < 4; ++ch) {
    const int n = n0 + e.hf * 64 + ch * 16;
    if (n >= p.P) break;  // warp-uniform
    float v[16];
    tmem_ld16(acc_addr(e, e.ab, ch), v);
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j] + __ldg(bias + n + j), 0.f);
    alignas(16) bf16 hi[16], lo[16];
    split16(v, hi, lo);
    stage16(e.rs, e.lane, hi);
    stage16(e.rs + kTermBlock, e.lane, lo);
    if (ok && p.h) store16(p.h + (wrow0 + e.lane) * p.P + n, v);
    __syncwarp();
    flush16(e.rs, e.lane, p.h_hi, wrow0, n, p.P, vr);
    flush16(e.rs + kTermBlock, e.lane, p.h_lo, wrow0, n, p.P, vr);
    __syncwarp();
  }
  tc_fence_before();
  mbar_arrive(&e.acc_empty[e.ab]);
  acc_advance(e, 1);
  publish(e);
  if (e.tid == 0) signal(h_ready(p) + rt.seg * p.RTB + rt.r);
}

// Layer 2 and the loss.  Task ((r, c), seg) owns the 128 x 64 tile of y for ONE row group (q | p | n) of 128 triplets:
//   1. y = acc + b2 goes to an exchange buffer (layout [column][row]: every access of a warp is one 128 B line) and
//      the accumulator is released; the three tasks of (r, c) run on three CTAs at the same time and wait for each other;
//   2. every task reads all three tiles and forms the partial |q|^2, |p|^2, |n|^2, q.p, q.n of its columns; the seg 0
//      task publishes them; all tasks of row tile r wait until the partials of every column tile have arrived;
//   3. cosines, hinge, and the closed-form dY of the task's OWN row group -> (hi, lo) terms row-major and transposed,
//      db2 partial sums.
__device__ void epi_f2l(const ChainParams& p, EpiCtx& e, int task_i) {
  const int seg = task_i % 3, rc = task_i / 3, r = rc / p.NCF, c = rc % p.NCF, n0 = c * 64;
  const int valid = min(BM, p.B - r * BM);
  const int row = e.q * 32 + e.lane;
  const bool ok = row < valid;
  const int vr = warp_valid_rows(e, valid);
  const int trip = r * BM + row;
  const size_t wrow0 = (size_t)seg * p.B + (size_t)r * BM + e.q * 32;  // this warp's first row in the [3B, P] arrays
  mbar_wait(&e.acc_full[e.ab], e.aph);
  tc_fence_after();
  trace_ev(e, 2);
  const uint32_t accb = e.tmem_base + ((uint32_t)(e.q * 32) << 16) + (uint32_t)(e.ab * BN + e.hf * 32);
  const float* bias = p.b2[seg != 0];
  float* X = p.ybuf + (size_t)rc * 3 * 64 * 128;  // [seg][64 columns][128 rows]
  float own[32];  // this task's y values of the thread's 32 columns stay in registers
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int col = e.hf * 32 + ch * 16;
    float v[16];
    tmem_ld16(accb + ch * 16, v);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      v[j] += __ldg(bias + n0 + col + j);
      own[ch * 16 + j] = v[j];
      X[((size_t)(seg * 64 + col + j)) * 128 + row] = v[j];
    }
    if (p.y && ok) store16(p.y + ((size_t)seg * p.B + trip) * p.P + n0 + col, v);
  }
  tc_fence_before();
  mbar_arrive(&e.acc_empty[e.ab]);  // the accumulator is free: the next main loop may overwrite it
  acc_advance(e, 1);
  __threadfence();
  epi_bar();
  if (e.tid == 0) {
    signal(y_ready(p) + rc);
    wait_counter(y_ready(p) + rc, 3u);
  }
  epi_bar();
  // ---- the other two row groups' values of the same (triplet, column)s: all 64 loads in flight at once -----------------
  const int s1 = seg == 0 ? 1 : 0, s2 = seg == 2 ? 1 : 2;  // the two foreign groups, ascending
  float f1[32], f2[32];
  {
    const float* x1 = X + (size_t)(s1 * 64 + e.hf * 32) * 128 + row;
    const float* x2 = X + (size_t)(s2 * 64 + e.hf * 32) * 128 + row;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      f1[j] = __ldcg(x1 + (size_t)j * 128);
      f2[j] = __ldcg(x2 + (size_t)j * 128);
    }
  }
  // q, p, n views of (own, f1, f2): seg 0 -> (own, f1, f2), seg 1 -> (f1, own, f2), seg 2 -> (f1, f2, own)
  float qq = 0.f, pp = 0.f, nn = 0.f, qp = 0.f, qn = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const float a = seg == 0 ? own[j] : f1[j];
    const float b = seg == 0 ? f1[j] : (seg == 1 ? own[j] : f2[j]);
    const float d = seg == 2 ? own[j] : f2[j];
    qq = fmaf(a, a, qq);
    pp = fmaf(b, b, pp);
    nn = fmaf(d, d, nn);
    qp = fmaf(a, b, qp);
    qn = fmaf(a, d, qn);
  }
  // one slot of partial sums per column tile: the two column halves of the tile meet in shared memory first
  const int nslots = p.NCF;
  float* xs = e.cs_s;  // [5][128] (the column-sum staging is idle until the stores below)
  if (seg == 0 && e.hf == 1) {
    xs[row] = qq; xs[128 + row] = pp; xs[256 + row] = nn; xs[384 + row] = qp; xs[512 + row] = qn;
  }
  epi_bar();
  if (seg == 0 && e.hf == 0) {
    float* sp = p.stat_part + ((size_t)(r * nslots + c) * 5) * 128 + row;
    sp[0] = qq + xs[row]; sp[128] = pp + xs[128 + row]; sp[256] = nn + xs[256 + row]; sp[384] = qp + xs[384 + row];
    sp[512] = qn + xs[512 + row];
    __threadfence();
  }
  epi_bar();
  if (e.tid == 0) {
    if (seg == 0) signal(stat_ready(p) + r);
    wait_counter(stat_ready(p) + r, (unsigned)p.NCF);
  }
  epi_bar();
  trace_ev(e, 3);
  // ---- the whole row's sums, slot order fixed (identical in every task of this row tile) ------------------------
  qq = pp = nn = qp = qn = 0.f;
  for (int s0 = 0; s0 < nslots; s0 += 4) {  // four slots (20 loads) in flight; the additions keep slot order
    float v[4][5];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float* sp = p.stat_part + ((size_t)(r * nslots + min(s0 + u, nslots - 1)) * 5) * 128 + row;
#pragma unroll
      for (int w = 0; w < 5; ++w) v[u][w] = __ldcg(sp + 128 * w);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (s0 + u < nslots) {
        qq += v[u][0]; pp += v[u][1]; nn += v[u][2]; qp += v[u][3]; qn += v[u][4];
      }
  }
  const float nq = sqrtf(qq), np_ = sqrtf(pp), nn_ = sqrtf(nn);
  const float cq = fmaxf(nq, kCosEps), cp = fmaxf(np_, kCosEps), cn = fmaxf(nn_, kCosEps);
  const float cos_p = qp / (cq * cp), cos_n = qn / (cq * cn);
  // relu(pos_dist - neg_dist + margin), model.py:140-143
  const float hinge = ok ? fmaxf((1.f - cos_p) - (1.f - cos_n) + p.margin, 0.f) : 0.f;
  const float gh = (hinge > 0.f) ? p.grad_scale * p.inv_batch : 0.f;  // 0 for rows past the batch: their dY is 0
  // dY of this task's row group = c_own * own + c1 * f1 + c2 * f2  (closed-form gradient of the two cosines)
  const float a_qp = -gh / (cq * cp), a_qn = gh / (cq * cn);
  float c_own, c1, c2;
  if (seg == 0) {  // dq = a_qp p + a_qn n - kq q
    c_own = -((nq > kCosEps) ? (-gh * cos_p + gh * cos_n) / (cq * nq) : 0.f); c1 = a_qp; c2 = a_qn;
  } else if (seg == 1) {  // dp = a_qp q - kp p
    c_own = -((np_ > kCosEps) ? (-gh * cos_p) / (cp * np_) : 0.f); c1 = a_qp; c2 = 0.f;
  } else {  // dn = a_qn q - kn n
    c_own = -((nn_ > kCosEps) ? (gh * cos_n) / (cn * nn_) : 0.f); c1 = a_qn; c2 = 0.f;
  }
  if (seg == 0 && c == 0 && e.hf == 0) {
    if (ok) {
      float* s = p.stats + (size_t)trip * 8;
      s[0] = cos_p; s[1] = cos_n; s[2] = hinge; s[3] = nq; s[4] = np_; s[5] = nn_; s[6] = qp; s[7] = qn;
    }
    const float hsum = warp_sum(hinge);
    if (e.lane == 0) e.hs_s[e.q] = hsum;
  }
  uint8_t* blk_hi = e.rs;
  uint8_t* blk_lo = e.rs + kTermBlock;
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int n = n0 + e.hf * 32 + ch * 16;
    float g[16];
#pragma unroll
    for (int j = 0; j < 16; ++j)
      g[j] = ok ? (c_own * own[ch * 16 + j] + c1 * f1[ch * 16 + j] + c2 * f2[ch * 16 + j]) : 0.f;
    alignas(16) bf16 hi[16], lo[16];
    split16(g, hi, lo);
    stage16(blk_hi, e.lane, hi);
    stage16(blk_lo, e.lane, lo);
    if (ok && p.dy) store16(p.dy + ((size_t)seg * p.B + trip) * p.P + n, g);
    __syncwarp();
    flush16(blk_hi, e.lane, p.dy_hi, wrow0, n, p.P, vr);
    flush16(blk_lo, e.lane, p.dy_lo, wrow0, n, p.P, vr);
    __syncwarp();
    stage_cs(e, 0, ch, colsum16(g, e.lane));
  }
  epi_bar();
  if (e.tid < 64) p.cs2[(size_t)(seg * p.RTB + r) * p.P + n0 + e.tid] = reduce_cs(e, 0, e.tid, 32);  // db2 partials
  if (seg == 0 && c == 0 && e.tid == 0) p.hinge_part[r] = (e.hs_s[0] + e.hs_s[1]) + (e.hs_s[2] + e.hs_s[3]);
  publish(e);
  if (e.tid == 0) {
    signal(dy_ready(p) + seg * p.RTB + r);
    signal(p.ctr + 1);
  }
}

__device__ void epi_dz(const ChainParams& p, EpiCtx& e, int task_i) {
  const RowTile rt = row_tile(p, task_i / p.NC);
  const int n0 = (task_i % p.NC) * BN;
  mbar_wait(&e.acc_full[e.ab], e.aph);
  tc_fence_after();
  trace_ev(e, 2);
  const int row = e.q * 32 + e.lane;
  const bool ok = row < rt.valid;
  const int vr = warp_valid_rows(e, rt.valid);
  const size_t wrow0 = (size_t)rt.grow + e.q * 32;
  for (int ch = 0; ch < 4; ++ch) {
    const int n = n0 + e.hf * 64 + ch * 16;
    if (n >= p.P) break;
    float v[16];
    tmem_ld16(acc_addr(e, e.ab, ch), v);
    const size_t o = (wrow0 + e.lane) * p.P + n;
    if (ok) {
      // ReLU gate from the hi term of h: bf16 rounding keeps the sign and never turns a normal positive value into 0
      alignas(16) bf16 g[16];
      reinterpret_cast<uint4*>(g)[0] = __ldcg(reinterpret_cast<const uint4*>(p.h_hi + o));
      reinterpret_cast<uint4*>(g)[1] = __ldcg(reinterpret_cast<const uint4*>(p.h_hi + o) + 1);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __bfloat162float(g[j]) > 0.f ? v[j] : 0.f;
      if (p.dz1) store16(p.dz1 + o, v);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = 0.f;
    }
    alignas(16) bf16 hi[16], lo[16];
    split16(v, hi, lo);
    stage16(e.rs, e.lane, hi);  // (rows past the batch are zero: the weight-gradient contraction reads whole k-blocks)
    stage16(e.rs + kTermBlock, e.lane, lo);
    __syncwarp();
    flush16(e.rs, e.lane, p.dz_hi, wrow0, n, p.P, vr);
    flush16(e.rs + kTermBlock, e.lane, p.dz_lo, wrow0, n, p.P, vr);
    __syncwarp();
    stage_cs(e, 0, ch, colsum16(v, e.lane));
  }
  tc_fence_before();
  mbar_arrive(&e.acc_empty[e.ab]);
  acc_advance(e, 1);
  epi_bar();
  if (e.tid < BN && n0 + e.tid < p.P)
    p.cs1[(size_t)(rt.seg * p.RTB + rt.r) * p.P + n0 + e.tid] = reduce_cs(e, 0, e.tid);
  publish(e);
  if (e.tid == 0) {
    signal(dz_ready(p) + rt.seg * p.RTB + rt.r);
    signal(p.ctr + 1);
  }
}

// fp32 tile of this warp (32 rows x 64 columns) -> g, through the staging block, 16 columns at a time
__device__ __forceinline__ void epi_store_f32(const ChainParams& p, EpiCtx& e, float* g, size_t wrow0, int n0, int N,
                                              size_t ld, int vr) {
  for (int ch = 0; ch < 4; ++ch) {
    const int n = n0 + e.hf * 64 + ch * 16;
    if (n >= N) break;
    float v[16];
    tmem_ld16(acc_addr(e, e.ab, ch), v);
    stage_f32(e.rs, e.lane, v);
    __syncwarp();
    flush_f32(e.rs, e.lane, g, wrow0, n, ld, vr);
    __syncwarp();
  }
}

__device__ void epi_dx(const ChainParams& p, EpiCtx& e, int task_i) {
  const RowTile rt = row_tile(p, task_i / p.NCH);
  const int n0 = (task_i % p.NCH) * BN;
  mbar_wait(&e.acc_full[e.ab], e.aph);
  tc_fence_after();
  trace_ev(e, 2);
  epi_store_f32(p, e, p.dxhat, (size_t)rt.grow + e.q * 32, n0, p.H, p.H, warp_valid_rows(e, rt.valid));
  tc_fence_before();
  mbar_arrive(&e.acc_empty[e.ab]);
  acc_advance(e, 1);
}

// raw partial sums of one (chunk, tile) of a weight gradient: part[chunk][M][N]
__device__ void epi_dw(const ChainParams& p, EpiCtx& e, Task tk) {
  const bool two = tk.type == T_DW2;
  const int N = two ? p.P : p.H, ntn = two ? p.NC : p.NCH, nt_ = p.NC * ntn;
  const int ci = tk.i / nt_, tile = tk.i % nt_;
  const int m0 = (tile / ntn) * BM, n0 = (tile % ntn) * BN;
  float* part = (two ? p.part2 : p.part1) + (size_t)ci * p.P * N;
  mbar_wait(&e.acc_full[e.ab], e.aph);
  tc_fence_after();
  trace_ev(e, 2);
  epi_store_f32(p, e, part, (size_t)m0 + e.q * 32, n0, N, N, warp_valid_rows(e, p.P - m0));
  tc_fence_before();
  mbar_arrive(&e.acc_empty[e.ab]);
  acc_advance(e, 1);
  __threadfence();
  epi_bar();
  if (e.tid == 0) {
    if (two) signal(p.ctr + 5);  // the second-layer gradient's partial tiles: the tail sums them without waiting for dW1
    signal(p.ctr + 1);
  }
}

__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

struct AdamCoef {
  float step_size, bc2_sqrt;
};
// torch.optim.Adam (non-fused, no weight decay / amsgrad): lerp, mul + addcmul, sqrt / bc2_sqrt + eps, addcdiv
__device__ __forceinline__ float adam1(const ChainParams& p, const AdamCoef& k, float g, float& m, float& v, float w) {
  m = m + (g - m) * (1.f - p.beta1);
  v = v * p.beta2 + (1.f - p.beta2) * g * g;
  const float denom = sqrtf(v) / k.bc2_sqrt + p.eps;
  return w - k.step_size * (m / denom);
}
// gradient element(s) at dst (a slice of the flat gradient buffer; added to what dst holds when accumulating) -> memory,
// and the Adam update of the parameter,
// exp_avg and exp_avg_sq elements at the same offset of their flat buffers
__device__ __forceinline__ void emit4(const ChainParams& p, const AdamCoef& k, float4* dst, float4 g) {
  if (p.grad_accumulate) g = add4(*dst, g);
  *dst = g;
  if (!p.adam_p) return;
  const size_t off = reinterpret_cast<float*>(dst) - p.adam_g;
  float4 m = *reinterpret_cast<float4*>(p.adam_m + off), v = *reinterpret_cast<float4*>(p.adam_v + off);
  float4 w = *reinterpret_cast<float4*>(p.adam_p + off);
  w.x = adam1(p, k, g.x, m.x, v.x, w.x);
  w.y = adam1(p, k, g.y, m.y, v.y, w.y);
  w.z = adam1(p, k, g.z, m.z, v.z, w.z);
  w.w = adam1(p, k, g.w, m.w, v.w, w.w);
  *reinterpret_cast<float4*>(p.adam_m + off) = m;
  *reinterpret_cast<float4*>(p.adam_v + off) = v;
  *reinterpret_cast<float4*>(p.adam_p + off) = w;
}
__device__ __forceinline__ void emit1(const ChainParams& p, const AdamCoef& k, float* dst, float g) {
  if (p.grad_accumulate) g = *dst + g;
  *dst = g;
  if (!p.adam_p) return;
  const size_t off = dst - p.adam_g;
  float m = p.adam_m[off], v = p.adam_v[off];
  p.adam_p[off] = adam1(p, k, g, m, v, p.adam_p[off]);
  p.adam_m[off] = m;
  p.adam_v[off] = v;
}

// gradients = fixed-order sums of the partials (chunk order / row-tile order) [-> Adam]; task 0 also finishes the loss.
// Nothing else reads the fp32 parameters any more at this point (the weights were split into bf16 terms by S, the
// biases were last read by the F1 / F2L epilogues, all of which have signalled), so they are updated in place.
__device__ void epi_grad(const ChainParams& p, EpiCtx& e, int task_i) {
  // phase A needs the dW2 partial tiles only: CTAs that run out of contraction tasks start here while others still work
  // on dW1 (W2's fp32 values were last read by S, so its Adam update is safe already)
  if (e.tid == 0) wait_counter(p.ctr + 5, p.dw2_signals);
  epi_bar();
  trace_ev(e, 2);
  AdamCoef k{0.f, 1.f};
  if (p.adam_p) {
    const volatile double* st = p.adam_state;
    k.step_size = (float)((double)p.lr / (1.0 - st[1]));
    k.bc2_sqrt = (float)sqrt(1.0 - st[2]);
  }
  const int nG = p.off[T_COUNT] - p.off[T_G];
  // A weight gradient pair (both towers) is a list of float4 items cut into chunks of 512 that the CTAs CLAIM (one
  // atomic per chunk): a CTA that arrives early takes more of them, the CTA that finishes the last contraction task
  // finds little left.  A thread keeps two items and, per item, four chunk loads in flight; the additions keep the
  // order of the batch-row chunks, so the sums do not depend on who computes them.
  volatile int* claim_s = reinterpret_cast<volatile int*>(e.cs_s);  // (the column-sum staging is idle in this phase)
  int round = 0;
  auto sum_pairs = [&](unsigned* claim, const float* part, float* const (&dW)[2], size_t n4) {
    auto locate = [&](size_t item, const float4*& src, float4*& dst, int& nch) {
      const int t = item >= n4;
      const size_t i = item - (t ? n4 : 0);
      nch = p.nch[t];
      src = reinterpret_cast<const float4*>(part) + (size_t)(t ? p.nch[0] : 0) * n4 + i;
      dst = reinterpret_cast<float4*>(dW[t]) + i;
    };
    const size_t ntot = 2 * n4;
    const int nchunks = (int)((ntot + 2 * kEpiThreads - 1) / (2 * kEpiThreads));
    for (;;) {
      if (e.tid == 0) claim_s[round & 1] = (int)atomicAdd(claim, 1u);
      epi_bar();
      const int c = claim_s[round & 1];
      ++round;
      if (c >= nchunks) break;
      const size_t it = (size_t)c * 2 * kEpiThreads + e.tid;
      if (it >= ntot) continue;
      const float4* src[2];
      float4* dst[2];
      int nch[2];
      const bool two = it + kEpiThreads < ntot;
      locate(it, src[0], dst[0], nch[0]);
      locate(two ? it + kEpiThreads : it, src[1], dst[1], nch[1]);
      float4 acc[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
      const int nmax = max(nch[0], nch[1]);
      for (int j = 0; j < nmax; j += 4) {
        float4 t[2][4];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4)
            t[u][c4] = (j + c4 < nch[u]) ? __ldcg(src[u] + (size_t)(j + c4) * n4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4)
            if (j + c4 < nch[u]) acc[u] = add4(acc[u], t[u][c4]);
      }
      emit4(p, k, dst[0], acc[0]);
      if (two) emit4(p, k, dst[1], acc[1]);
    }
  };
  sum_pairs(p.ctr + 6, p.part2, p.dW2, (size_t)p.P * p.P / 4);
  // phase B: everything else has signalled
  if (e.tid == 0) wait_counter(p.ctr + 1, p.total_signals);
  epi_bar();
  sum_pairs(p.ctr + 7, p.part1, p.dW1, (size_t)p.P * p.H / 4);
  // bias gradients: one output per warp at a time, the lanes take the row-tile partials (lane-strided, then a fixed
  // xor tree), so every CTA shares this tail instead of the first few
  {
    const int nout = 4 * p.P;  // db2[0] | db2[1] | db1[0] | db1[1]
    const int gw = task_i * 8 + e.we, nw = nG * 8;
    for (int o = gw; o < nout; o += nw) {
      const int which = o / p.P, n = o - which * p.P, t = which & 1;
      const float* src;
      int cnt;
      if (which < 2) {
        src = p.cs2 + (size_t)(t ? p.RTB : 0) * p.P + n;
        cnt = t ? 2 * p.RTB : p.RTB;
      } else {
        src = p.cs1 + (size_t)(t ? p.RTB : 0) * p.P + n;
        cnt = t ? 2 * p.RTB : p.RTB;
      }
      float s = 0.f;
      for (int r = e.lane; r < cnt; r += 32) s += __ldcg(src + (size_t)r * p.P);
      s = warp_sum(s);
      if (e.lane == 0) emit1(p, k, (which < 2 ? p.db2[t] : p.db1[t]) + n, s);
    }
  }
  if (task_i == 0 && e.tid == 0) {
    float s = 0.f;
    for (int r = 0; r < p.RTB; ++r) s += __ldcg(p.hinge_part + r);
    *p.loss = s * p.inv_batch;
  }
  // The last tail task to finish clears the dependency counters for the next launch (every other task of this
  // launch has completed by then: the tail waited for all of them), so a graph replay needs no memset node.
  epi_bar();
  if (e.tid == 0) {
    __threadfence();
    if (atomicAdd(p.ctr + 4, 1u) == (unsigned)nG - 1u) {
      for (int i = 0; i < p.n_counters; ++i) p.ctr[i] = 0u;
    }
  }
}

__global__ void __launch_bounds__(kThreads, 1) chain_kernel(const __grid_constant__ ChainParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const int NS = p.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NS * kStageBytes);
  uint64_t* empty = full + kMaxStages;
  uint64_t* acc_full = empty + kMaxStages;
  uint64_t* acc_empty = acc_full + kAcc;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + kAcc);
  uint8_t* staging = smem + NS * kStageBytes + 256;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < kAcc; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], kEpiThreads);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kAcc * BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_tasks = p.off[T_COUNT];

  if (warp == 0) {
    if (elect_one()) {  // ---- TMA producer: dependencies, then the operand tiles of every sub-tile ------------
      int s = 0;
      uint32_t ph = 0;
      if (p.use_pdl) pdl_wait();
      for (int idx = blockIdx.x; idx < n_tasks; idx += gridDim.x) {
        const Task tk = decode(p, idx);
        const int ns = n_subs(tk.type);
        if (ns == 0) continue;
        wait_deps(p, tk);
        fence_proxy_async();  // other CTAs' generic-proxy writes (acquired above) before this thread's TMA reads
        for (int k = 0; k < ns; ++k) {
          const Sub sb = get_sub(p, tk, k);
          for (int kb = sb.kb0; kb < sb.kb0 + sb.nkb; ++kb) {
            for (int j = 0; j < sb.terms; ++j) {
              mbar_wait(&empty[s], ph ^ 1u);
              mbar_arrive_expect_tx(&full[s], kABytes + (uint32_t)sb.bn * BK * 2);
              uint8_t* sa = smem + s * kStageBytes;
              uint8_t* sbm = sa + kABytes;
              if (sb.amn) {  // MN-major: [64 k-rows][64 m] boxes for m0 .. m0+63 and m0+64 .. m0+127
                tma_load_2d(sa, &sb.a[j], &full[s], sb.m0, kb * BK);
                tma_load_2d(sa + kABytes / 2, &sb.a[j], &full[s], sb.m0 + 64, kb * BK);
              } else {
                tma_load_2d(sa, &sb.a[j], &full[s], kb * BK, sb.m0);
              }
              if (sb.bmn) {
                tma_load_2d(sbm, &sb.b[j], &full[s], sb.n0, kb * BK);
                tma_load_2d(sbm + kBBytes / 2, &sb.b[j], &full[s], sb.n0 + 64, kb * BK);
              } else {
                tma_load_2d(sbm, &sb.b[j], &full[s], kb * BK, sb.n0);
              }
              if (++s == NS) {
                s = 0;
                ph ^= 1u;
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {  // ---- MMA issuer ----------------------------------------------------------------------
      constexpr uint32_t idesc128 = make_idesc_bf16(BM, BN), idesc64 = make_idesc_bf16(BM, 64);
      const uint32_t ring = smem_u32(smem);
      int s = 0, ab = 0;
      uint32_t ph = 0, aph = 0;
      for (int idx = blockIdx.x; idx < n_tasks; idx += gridDim.x) {
        const Task tk = decode(p, idx);
        const int ns = n_subs(tk.type);
        for (int k = 0; k < ns; ++k) {
          const Sub sb = get_sub(p, tk, k);
          // MN-major operands: instruction-descriptor bits 15 (A) / 16 (B)
          const uint32_t idesc = (sb.bn == BN ? idesc128 : idesc64) | ((uint32_t)sb.amn << 15) | ((uint32_t)sb.bmn << 16);
          // per K = 16 step a K-major operand advances 32 B inside its 128-byte rows, an MN-major one two groups of
          // 8 k-rows (2 x 1024 B); descriptor units are 16 B
          const uint64_t a_step = sb.amn ? 128 : 2, b_step = sb.bmn ? 128 : 2;
          mbar_wait(&acc_empty[ab], aph ^ 1u);
          tc_fence_after();
          const uint32_t acc = tmem_base + (uint32_t)(ab * BN);
          for (int kbi = 0; kbi < sb.nkb; ++kbi) {
            uint32_t slot_addr[3];
            int slot_id[3];
            for (int j = 0; j < sb.terms; ++j) {
              mbar_wait(&full[s], ph);
              slot_id[j] = s;
              slot_addr[j] = ring + (uint32_t)s * kStageBytes;
              if (++s == NS) {
                s = 0;
                ph ^= 1u;
              }
            }
            tc_fence_after();
            for (int pair = 0; pair < sb.pairs; ++pair) {
              const int ai = (0x201100 >> (4 * pair)) & 3, bi = (0x021010 >> (4 * pair)) & 3;
              const uint64_t da = sb.amn ? make_smem_desc_sw128_mn(slot_addr[ai], kABytes / 2) : make_smem_desc_sw128(slot_addr[ai]),
                             db = sb.bmn ? make_smem_desc_sw128_mn(slot_addr[bi] + kABytes, kBBytes / 2)
                                         : make_smem_desc_sw128(slot_addr[bi] + kABytes);
#pragma unroll
              for (int kk = 0; kk < BK / 16; ++kk)
                mma_bf16(acc, da + a_step * kk, db + b_step * kk, idesc, (kbi | pair | kk) != 0);
            }
            for (int j = 0; j < sb.terms; ++j) mma_commit(&empty[slot_id[j]]);
          }
          mma_commit(&acc_full[ab]);
          if (++ab == kAcc) {
            ab = 0;
            aph ^= 1u;
          }
        }
      }
    }
  } else {  // ---- epilogue warps ------------------------------------------------------------------------------
    EpiCtx e;
    e.tmem_base = tmem_base;
    e.acc_full = acc_full;
    e.acc_empty = acc_empty;
    e.cs_s = reinterpret_cast<float*>(staging);
    e.sp_s = reinterpret_cast<bf16*>(staging + kCsBytes);
    e.rs = staging + kCsBytes + (warp - 2) * kRowStage;
    e.hs_s = reinterpret_cast<float*>(staging + kCsBytes + 8 * kRowStage);
    e.we = warp - 2;
    e.q = warp & 3;
    e.hf = e.we >> 2;
    e.lane = lane;
    e.tid = threadIdx.x - 64;
    e.ab = 0;
    e.aph = 0;
    e.trace = p.trace ? p.trace + (size_t)blockIdx.x * kTraceSlots * 2 : nullptr;
    e.tslot = 0;
    for (int idx = blockIdx.x; idx < n_tasks; idx += gridDim.x) {
      const Task tk = decode(p, idx);
      e.tidx = idx;
      trace_ev(e, 0);
      switch (tk.type) {
        case T_S:
          epi_split(p, e, tk.i);
          if (p.use_pdl) pdl_wait();  // the pooled gather's xhat terms are read from here on
          break;
        case T_F1: epi_f1(p, e, tk.i); break;
        case T_F2L: epi_f2l(p, e, tk.i); break;
        case T_DZ: epi_dz(p, e, tk.i); break;
        case T_DX: epi_dx(p, e, tk.i); break;
        case T_DW2:
        case T_DW1: epi_dw(p, e, tk); break;
        default: epi_grad(p, e, tk.i); break;
      }
      trace_ev(e, 1);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kAcc * BN);
}

// operand ring depth (6 x 32 KB + 29 KB of epilogue staging still fit the 227 KB; 5 measured best)
constexpr int kChainStages = 5;
static_assert(kChainStages <= kMaxStages, "the barrier block holds kMaxStages slots");

int chain_debug_out() {  // TT_CHAIN_FP32_OUT=1: also write h, y, dY and dz1 in fp32 (diagnostics; read per call)
  const char* e = getenv("TT_CHAIN_FP32_OUT");
  return e ? atoi(e) : 0;
}

int map_terms(CUtensorMap* m, int n, const bf16* const* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
              uint32_t box_rows = BM) {
  for (int i = 0; i < n; ++i) {
    const bf16* base = ptr[i] ? ptr[i] : ptr[0];  // unused terms alias the first (never loaded)
    int rc = make_map_bf16_kmajor(&m[i], base, rows, cols, ld, box_rows);
    if (rc) return rc;
  }
  return 0;
}

}  // namespace

bool chain_enabled() {
  const char* e = getenv("TT_CHAIN");  // 0 = the per-kernel chain of tt_gemm_sm100.cu; read per call (tests toggle it)
  return e ? atoi(e) != 0 : true;
}

// Everything of the step after the pooled gather.  after_gather: the pooled gather is the previous launch of this
// stream (whole-step call): the kernel is then launched as its programmatic dependent, splits the weights while the
// gather's last CTAs drain and waits for it (griddepcontrol.wait) before it reads xhat.  s.adam (optional): torch.optim.Adam on the flat parameter buffer in
// the kernel's tail, step count and beta powers advanced on the device.
int chain_sm100(const StepSm100& s, bool after_gather, cudaStream_t st) {
  const int B = s.B, H = s.H, P = s.P;
  StepWs w;
  carve_step(reinterpret_cast<char*>(s.ws), B, H, P, s.dxhat != nullptr, &w);
  static bool attr_done = false;
  if (!attr_done) {
    TT_CUDA(cudaFuncSetAttribute(chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chain_smem(kChainStages)));
    attr_done = true;
  }
  static thread_local ChainParams p;  // ~8 KB: kept off the stack; copied into the launch before this returns
  p = ChainParams{};
  int rc;
  const float* W1[2] = {s.Wq1, s.Wd1};
  const float* W2[2] = {s.Wq2, s.Wd2};
  const int row0[2] = {0, B}, rows[2] = {B, 2 * B};
  const bool x3 = s.n_split == 3;
  for (int t = 0; t < 2; ++t) {
    TowerMaps& m = p.tm[t];
    const size_t oH = (size_t)row0[t] * H, oP = (size_t)row0[t] * P;
    const bf16* x[3] = {w.x_hi + oH, x3 ? w.x_lo + oH : nullptr, x3 ? w.x_lo2 + oH : nullptr};
    const bf16* w1[3] = {w.w1_hi[t], w.w1_lo[t], w.w1_lo2[t]};
    const bf16* hh[2] = {w.h_hi + oP, w.h_lo + oP};
    const bf16* w2[2] = {w.w2_hi[t], w.w2_lo[t]};
    const bf16* dy[2] = {w.dy_hi + oP, w.dy_lo + oP};
    const bf16* dz[2] = {w.dz_hi + oP, w.dz_lo + oP};
    if ((rc = map_terms(m.x, 3, x, rows[t], H, H))) return rc;
    if ((rc = map_terms(m.w1, 3, w1, P, H, H))) return rc;
    if ((rc = map_terms(m.h, 2, hh, rows[t], P, P))) return rc;
    if ((rc = map_terms(m.w2, 2, w2, P, P, P, 64))) return rc;
    if ((rc = map_terms(m.dy, 2, dy, rows[t], P, P))) return rc;
    if ((rc = map_terms(m.dz, 2, dz, rows[t], P, P))) return rc;
    // MN-major operands: the same row-major arrays, boxes of 64 k-rows x 64 elements
    if ((rc = map_terms(m.w1k, 2, w1, P, H, H, 64))) return rc;
    if ((rc = map_terms(m.dyk, 2, dy, rows[t], P, P, 64))) return rc;
    if ((rc = map_terms(m.hk, 2, hh, rows[t], P, P, 64))) return rc;
    if ((rc = map_terms(m.dzk, 2, dz, rows[t], P, P, 64))) return rc;
    if ((rc = map_terms(m.xk, 2, x, rows[t], H, H, 64))) return rc;
  }
  p.B = B; p.H = H; p.P = P;
  p.RTB = (B + BM - 1) / BM; p.NC = (P + BN - 1) / BN; p.NCH = (H + BN - 1) / BN; p.NCF = P / 64;
  p.pairs = x3 ? 3 : 1; p.terms = x3 ? 2 : 1;
  p.pairs1 = x3 ? 6 : 1; p.terms1 = x3 ? 3 : 1;  // layer 1 (its ReLU sign gates the backward): 6-product split
  for (int t = 0; t < 2; ++t) p.kbt[t] = (rows[t] + BK - 1) / BK;
  p.kcb = 8;
  {
    const char* e = getenv("TT_CHAIN_KCB");  // test hook: k-blocks (64 batch rows each) per weight-gradient chunk
    if (e && atoi(e) >= 4) p.kcb = atoi(e) / 4 * 4;
  }
  while ((p.kbt[0] + p.kcb - 1) / p.kcb + (p.kbt[1] + p.kcb - 1) / p.kcb > 48) p.kcb += 8;
  for (int t = 0; t < 2; ++t) p.nch[t] = (p.kbt[t] + p.kcb - 1) / p.kcb;
  const int grid = sm_count();
  // the 3 * NCF loss tasks of one row tile wait for each other inside their epilogues: they must sit on distinct CTAs
  TT_REQUIRE(grid >= 3 * (P / 64), "tt_triplet_step: projection dim %d needs %d co-resident CTAs, the device has %d SMs", P,
             3 * (P / 64), grid);
  const int n_rt = 3 * p.RTB, nchs = p.nch[0] + p.nch[1];
  const int count[T_COUNT] = {grid,
                              0,  // (T: the xhat transposition of earlier builds; no transposed copy exists any more)
                              n_rt * p.NC,
                              n_rt * p.NCF,
                              n_rt * p.NC,
                              s.dxhat ? n_rt * p.NCH : 0,
                              nchs * p.NC * p.NC,
                              nchs * p.NC * p.NCH,
                              grid};
  p.off[0] = 0;
  for (int k = 0; k < T_COUNT; ++k) p.off[k + 1] = p.off[k] + count[k];
  p.total_signals = (unsigned)(count[T_F2L] + count[T_DZ] + count[T_DW2] + count[T_DW1]);
  p.dw2_signals = (unsigned)count[T_DW2];
  p.stages = kChainStages;
  // weights of both towers -> bf16 terms (+ transposes for the backward contractions); the first-layer weights come
  // first in the flat pass: layer 1 starts as soon as THEY are split (counter 0), the rest signals counter 2
  int f4 = 0;
  p.n_sj = 0;
  for (int t = 0; t < 2; ++t) {
    p.sj[p.n_sj++] = SplitJobC{W1[t], w.w1_hi[t], w.w1_lo[t], x3 ? w.w1_lo2[t] : nullptr, P, H, f4};
    f4 += P * H / 4;
  }
  p.n_split_f4_w1 = f4;
  for (int t = 0; t < 2; ++t) {
    p.sj[p.n_sj++] = SplitJobC{W2[t], w.w2_hi[t], w.w2_lo[t], nullptr, P, P, f4};
    f4 += P * P / 4;
  }
  p.n_split_f4 = f4;
  p.margin = s.margin; p.inv_batch = s.inv_batch; p.grad_scale = s.grad_scale;
  p.b1[0] = s.bq1; p.b1[1] = s.bd1; p.b2[0] = s.bq2; p.b2[1] = s.bd2;
  const bool dbg = chain_debug_out() != 0;
  p.h = dbg ? s.h : nullptr; p.y = dbg ? s.y : nullptr; p.dy = dbg ? s.dy : nullptr; p.dz1 = dbg ? w.dz1 : nullptr;
  p.dxhat = s.dxhat; p.stats = s.stats; p.loss = s.loss;
  p.h_hi = w.h_hi; p.h_lo = w.h_lo;
  p.dy_hi = w.dy_hi; p.dy_lo = w.dy_lo;
  p.dz_hi = w.dz_hi; p.dz_lo = w.dz_lo;
  p.part2 = w.partial2; p.part1 = w.partial;
  p.dW1[0] = s.dWq1; p.dW1[1] = s.dWd1; p.db1[0] = s.dbq1; p.db1[1] = s.dbd1;
  p.dW2[0] = s.dWq2; p.dW2[1] = s.dWd2; p.db2[0] = s.dbq2; p.db2[1] = s.dbd2;
  p.stat_part = w.stat_part; p.cs1 = w.cs1; p.cs2 = w.cs2; p.hinge_part = w.hinge_part; p.ybuf = w.ybuf;
  p.ctr = w.counters;
  p.n_counters = w.n_counters;
  p.nS = grid;
  p.grad_accumulate = s.grad_accumulate;
  if (s.adam.param) {
    const FusedAdam& a = s.adam;
    TT_REQUIRE(a.state && a.grad && a.exp_avg && a.exp_avg_sq, "tt_triplet_step: fused Adam needs state, grad and both moments");
    const float* W[8] = {s.Wq1, s.bq1, s.Wq2, s.bq2, s.Wd1, s.bd1, s.Wd2, s.bd2};
    float* G[8] = {s.dWq1, s.dbq1, s.dWq2, s.dbq2, s.dWd1, s.dbd1, s.dWd2, s.dbd2};
    const size_t len[8] = {(size_t)P * H, (size_t)P, (size_t)P * P, (size_t)P, (size_t)P * H, (size_t)P, (size_t)P * P, (size_t)P};
    for (int i = 0; i < 8; ++i) {
      const ptrdiff_t off = G[i] - a.grad;
      TT_REQUIRE(off >= 0 && (size_t)off + len[i] <= a.n && W[i] == a.param + off && off % 4 == 0,
                 "tt_triplet_step: fused Adam wants the 8 projection tensors and their gradients to be slices of the "
                 "flat buffers at equal, 16-byte aligned offsets (tensor %d)", i);
    }
    p.adam_state = a.state; p.adam_p = a.param; p.adam_g = a.grad; p.adam_m = a.exp_avg; p.adam_v = a.exp_avg_sq;
    p.lr = a.lr; p.beta1 = a.beta1; p.beta2 = a.beta2; p.eps = a.eps;
  }
  {
    const char* e = getenv("TT_CHAIN_TRACE");
    p.trace = (e && atoi(e) != 0 && grid <= kTraceCtas) ? w.trace : nullptr;
    if (p.trace) TT_CUDA(cudaMemsetAsync(w.trace, 0, (size_t)kTraceCtas * kTraceSlots * 16, st));
  }
  // (no memset of the counters: the workspace is zero-filled once by its owner and every launch leaves them at zero)
  p.use_pdl = after_gather ? 1 : 0;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = chain_smem(p.stages);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = p.use_pdl ? 1 : 0;
  TT_CUDA(cudaLaunchKernelEx(&cfg, chain_kernel, p));
  TT_LAUNCH_CHECK();
  return 0;
}

}  // namespace tt

// Pooled gather: token-row gather + attention-masked mean + L2 normalise, one CTA per sequence.
// Replaces backend/model.py:48-56,63-72 of the reference (see include/tt_b200.h).
//
// HBM-bound byte work: each unmasked token costs one H-wide row read (H*4 B fp32 / H*2 B bf16).
// A warp reads one row per step as fully coalesced 16 B (fp32) / 8 B (bf16) per-lane vectors,
// UNROLL rows in flight per warp, 4 warps per sequence, fp32 accumulation in registers, cross-warp
// reduction staged in shared memory, warp-shuffle reduction for the norm.
#include "tt_pool.cuh"

namespace tt {

namespace {

constexpr int kPoolThreads = 128;
constexpr int kPoolWarps = kPoolThreads / 32;
constexpr int kMaxL = 512;  // tokenizer max_length at backend/model.py:44

template <typename TE>
struct RowVec;
template <>
struct RowVec<float> {
  using V = float4;
  static __device__ __forceinline__ V zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  static __device__ __forceinline__ V load(const float* row, int vec) {
    return __ldg(reinterpret_cast<const float4*>(row) + vec);
  }
  static __device__ __forceinline__ void fma(float w, const V& v, float* acc) {
    acc[0] = fmaf(w, v.x, acc[0]);
    acc[1] = fmaf(w, v.y, acc[1]);
    acc[2] = fmaf(w, v.z, acc[2]);
    acc[3] = fmaf(w, v.w, acc[3]);
  }
};
template <>
struct RowVec<__nv_bfloat16> {
  using V = uint2;  // 4 bf16
  static __device__ __forceinline__ V zero() { return make_uint2(0u, 0u); }
  static __device__ __forceinline__ V load(const __nv_bfloat16* row, int vec) {
    return __ldg(reinterpret_cast<const uint2*>(row) + vec);
  }
  static __device__ __forceinline__ void fma(float w, const V& v, float* acc) {
    acc[0] = fmaf(w, __uint_as_float(v.x << 16), acc[0]);
    acc[1] = fmaf(w, __uint_as_float(v.x & 0xffff0000u), acc[1]);
    acc[2] = fmaf(w, __uint_as_float(v.y << 16), acc[2]);
    acc[3] = fmaf(w, __uint_as_float(v.y & 0xffff0000u), acc[3]);
  }
};

// Four consecutive columns [col, col + 4) of output row `row`: xhat and, for the tensor-core projection, its bf16
// hi / lo (/ lo2) terms.  The one place that defines the split, shared by the pooling and the row-gather kernels.
__device__ __forceinline__ void store_pooled4(const PoolParams& p, int H, size_t row, int col, float4 x) {
  *reinterpret_cast<float4*>(p.xhat + row * H + col) = x;
  if (p.x_hi) {  // operands of the tensor-core projection: bf16 hi/lo(/lo2) split, row-major
    const float xv[4] = {x.x, x.y, x.z, x.w};
    __nv_bfloat16 hi[4], lo[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) split_bf16(xv[c], hi[c], lo[c]);
    *reinterpret_cast<uint2*>(p.x_hi + row * H + col) = *reinterpret_cast<uint2*>(hi);
    *reinterpret_cast<uint2*>(p.x_lo + row * H + col) = *reinterpret_cast<uint2*>(lo);
    if (p.x_lo2) {
      __nv_bfloat16 l2[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) l2[c] = __float2bfloat16_rn((xv[c] - __bfloat162float(hi[c])) - __bfloat162float(lo[c]));
      *reinterpret_cast<uint2*>(p.x_lo2 + row * H + col) = *reinterpret_cast<uint2*>(l2);
    }
  }
}

// Pooled-row front end: output row r is a copy of a precomputed pooled row (PoolParams::row_index), written with the
// same terms the pooling epilogue writes.  One warp per row, coalesced 16-byte loads; the whole launch moves
// 3B * H * 4 bytes (9.4 MB at B = 2048, H = 384).
constexpr int kRowThreads = 256;
__global__ void __launch_bounds__(kRowThreads) pooled_rows_kernel(const PoolParams p, int H) {
  pdl_launch();  // as pool_fwd_kernel: a programmatic dependent may start filling SMs
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (kRowThreads / 32) + (threadIdx.x >> 5);
  if (r >= 3 * p.row_B) return;
  const bool q = r < p.row_B;
  const long long n = q ? p.rows_q_n : p.rows_d_n;
  long long src = __ldg(p.row_index + r);
  if (src < 0 || src >= n) {
    if (lane == 0 && p.err) atomicExch(p.err, 1);
    src = 0;
  }
  const float4* in = reinterpret_cast<const float4*>((q ? p.rows_q : p.rows_d) + (size_t)src * H);
  for (int v = lane; v < H / 4; v += 32) store_pooled4(p, H, (size_t)r, v * 4, __ldg(in + v));
}

template <typename TE, int NV, int UNROLL>
__global__ void __launch_bounds__(kPoolThreads) pool_fwd_kernel(const PoolParams p) {
  constexpr int H = NV * 128;
  __shared__ unsigned s_row[kMaxL];
  __shared__ float s_w[kMaxL];
  __shared__ __align__(16) float s_red[kPoolWarps][H];
  __shared__ int s_wc[kPoolWarps];
  __shared__ float s_fred[kPoolWarps];

  // a programmatic dependent (the persistent chain kernel of a whole-step call) may start filling SMs as soon as the
  // last wave of this grid is resident; it waits for this grid's completion before it reads xhat
  pdl_launch();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // block -> (segment, sequence); host orders segments longest-first so short ones fill the tail
  int b = blockIdx.x, s = 0;
  while (s + 1 < p.nseg && b >= p.seg[s].B) {
    b -= p.seg[s].B;
    ++s;
  }
  const PoolSegDev sg = p.seg[s];
  const int L = sg.L;
  const size_t tok0 = (size_t)b * L;
  const TE* __restrict__ table = reinterpret_cast<const TE*>(sg.table);

  // ---- 1. compact the unmasked tokens of this sequence (order kept -> deterministic sums) ----
  int n_valid = 0;
  float cnt_local = 0.f;
  for (int base = 0; base < L; base += kPoolThreads) {
    const int t = base + tid;
    long long id = 0;
    float w = 0.f;
    if (t < L) {
      w = (float)load_index(sg.mask, p.mask_dtype, tok0 + t);
      if (w != 0.f) {
        id = load_index(sg.ids, p.ids_dtype, tok0 + t);
        if (id < 0 || id >= p.vocab) {
          if (p.err) atomicExch(p.err, 1);
          w = 0.f;
          id = 0;
        }
      }
    }
    cnt_local += w;
    const bool valid = (w != 0.f);
    const unsigned bal = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) s_wc[warp] = __popc(bal);
    __syncthreads();
    int off = n_valid, tot = 0;
#pragma unroll
    for (int i = 0; i < kPoolWarps; ++i) {
      const int c = s_wc[i];
      if (i < warp) off += c;
      tot += c;
    }
    if (valid) {
      const int pos = off + __popc(bal & ((1u << lane) - 1u));
      s_row[pos] = (unsigned)id;
      s_w[pos] = w;
    }
    n_valid += tot;
    __syncthreads();
  }
  // count = sum of mask values (model.py:71 `input_mask_expanded.sum(1)`)
  cnt_local = warp_sum(cnt_local);
  if (lane == 0) s_fred[warp] = cnt_local;

  // ---- 2. stream the rows: warp w takes entries w, w+4, ...; UNROLL rows in flight ----------
  float acc[NV * 4];
#pragma unroll
  for (int i = 0; i < NV * 4; ++i) acc[i] = 0.f;

  using RV = RowVec<TE>;
  // One batch of UNROLL rows in flight per warp; latency is hidden by the other resident warps.  A padding entry
  // re-reads row s_row[0] with weight 0 instead of predicating the load, which keeps each batch one unconditional run
  // of loads.
  for (int e0 = warp; e0 < n_valid; e0 += kPoolWarps * UNROLL) {
    typename RV::V v[UNROLL][NV];
    float wt[UNROLL];
    const TE* rows[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int e = e0 + u * kPoolWarps;
      const bool ok = e < n_valid;
      wt[u] = ok ? s_w[e] : 0.f;
      rows[u] = table + (size_t)s_row[ok ? e : 0] * H;
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u)
#pragma unroll
      for (int j = 0; j < NV; ++j) v[u][j] = RV::load(rows[u], j * 32 + lane);
#pragma unroll
    for (int u = 0; u < UNROLL; ++u)
#pragma unroll
      for (int j = 0; j < NV; ++j) RV::fma(wt[u], v[u][j], acc + j * 4);
  }

  // ---- 3. cross-warp reduction staged in shared memory --------------------------------------
#pragma unroll
  for (int j = 0; j < NV; ++j)
    *reinterpret_cast<float4*>(&s_red[warp][(j * 32 + lane) * 4]) =
        make_float4(acc[j * 4 + 0], acc[j * 4 + 1], acc[j * 4 + 2], acc[j * 4 + 3]);
  __syncthreads();

  float cnt = 0.f;
#pragma unroll
  for (int i = 0; i < kPoolWarps; ++i) cnt += s_fred[i];
  const float denom = fmaxf(cnt, 1e-9f);  // clamp(min=1e-9), model.py:70-72

  // thread tid owns the 4-column groups tid + k * kPoolThreads (k < kOwn) below NV * 32: columns [4*grp, 4*grp+4).
  // kOwn is 1 for H <= 512 and 2 for H = 768.
  constexpr int kOwn = (NV * 32 + kPoolThreads - 1) / kPoolThreads;
  float4 m[kOwn];
  float sq = 0.f;
#pragma unroll
  for (int k = 0; k < kOwn; ++k) {
    const int grp = tid + k * kPoolThreads;
    m[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (grp < NV * 32) {
#pragma unroll
      for (int i = 0; i < kPoolWarps; ++i) {
        const float4 t = *reinterpret_cast<const float4*>(&s_red[i][grp * 4]);
        m[k].x += t.x; m[k].y += t.y; m[k].z += t.z; m[k].w += t.w;
      }
      m[k].x = m[k].x / denom; m[k].y = m[k].y / denom; m[k].z = m[k].z / denom; m[k].w = m[k].w / denom;
      const float s = m[k].x * m[k].x + m[k].y * m[k].y + m[k].z * m[k].z + m[k].w * m[k].w;
      sq = k == 0 ? s : sq + s;
    }
  }
  __syncthreads();  // s_fred is reused below
  sq = warp_sum(sq);
  if (lane == 0) s_fred[warp] = sq;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < kPoolWarps; ++i) tot += s_fred[i];
  const float nrm = sqrtf(tot);
  const float dn = fmaxf(nrm, 1e-12f);  // F.normalize eps, model.py:56

  const int row_out = sg.row0 + b;
  float4 x[kOwn];
#pragma unroll
  for (int k = 0; k < kOwn; ++k) {
    x[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid + k * kPoolThreads < NV * 32) x[k] = make_float4(m[k].x / dn, m[k].y / dn, m[k].z / dn, m[k].w / dn);
  }
  // every output of one pooled row (each thread: its column groups; thread 0: the count and the norm)
  auto emit_row = [&](int row) {
#pragma unroll
    for (int k = 0; k < kOwn; ++k) {
      const int grp = tid + k * kPoolThreads;
      if (grp >= NV * 32) continue;
      store_pooled4(p, H, (size_t)row, grp * 4, x[k]);
    }
    if (tid == 0) {
      if (p.cnt) p.cnt[row] = cnt;
      if (p.nrm) p.nrm[row] = nrm;
    }
  };
  emit_row(row_out);
  if (p.alias && (int)blockIdx.x < p.alias_n && tid == 0) {  // every alias index is range-checked by some CTA
    const int a = __ldg(p.alias + blockIdx.x);
    if ((a < 0 || a >= p.alias_n) && p.err) atomicExch(p.err, 1);
  }
  // In-batch negatives (backend/data.py:113-137: a negative IS another item's positive document): rows that alias
  // this one get the same bits instead of a second gather of the same tokens.
  if (p.alias && row_out >= p.alias_src_row0 && row_out < p.alias_src_row0 + p.alias_n) {
    constexpr int kMatchCap = 32;
    __shared__ int s_match[kMatchCap];
    __shared__ int s_nmatch;
    const int j = row_out - p.alias_src_row0;
    if (tid == 0) s_nmatch = 0;
    __syncthreads();
    for (int i = tid; i < p.alias_n; i += kPoolThreads)
      if (__ldg(p.alias + i) == j) {
        const int k = atomicAdd(&s_nmatch, 1);
        if (k < kMatchCap) s_match[k] = i;
      }
    __syncthreads();
    const int nm = s_nmatch;
    if (nm <= kMatchCap) {
      for (int k = 0; k < nm; ++k) emit_row(p.alias_dst_row0 + s_match[k]);
    } else {  // (a document drawn as the negative of more than 32 items of one batch: plain rescan, CTA-uniform)
      for (int i = 0; i < p.alias_n; ++i)
        if (__ldg(p.alias + i) == j) emit_row(p.alias_dst_row0 + i);
    }
  }
}

// Rows in flight per warp: 8 for bf16 tables.  For fp32 tables 8 when the gather has the SMs to itself (whole-step
// calls: 100.5 vs 103 us per launch, 0.2373 vs 0.2407 ms per configs[1] step), 4 when it shares them with other kernels
// (p.share_sm: more, lighter warps interleave better).
template <typename TE, int NV>
int launch_pool(const PoolParams& p, int total, cudaStream_t st) {
  constexpr int kSharedUnroll = sizeof(TE) == 4 ? 4 : 8;
  if (p.share_sm)
    pool_fwd_kernel<TE, NV, kSharedUnroll><<<total, kPoolThreads, 0, st>>>(p);
  else
    pool_fwd_kernel<TE, NV, 8><<<total, kPoolThreads, 0, st>>>(p);
  TT_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int pool_fwd_launch(PoolParams p, int table_dtype, int H, cudaStream_t st) {
  if (p.row_index) {  // precomputed pooled rows: a copy with the epilogue's split instead of a gather of tokens
    TT_REQUIRE(p.rows_q && p.rows_d && p.rows_q_n >= 1 && p.rows_d_n >= 1,
               "tt_triplet_step: pooled_q / pooled_d need at least one row each");
    TT_REQUIRE(H >= 4 && H % 4 == 0, "tt_triplet_step: pooled rows need H a multiple of 4, got %d", H);
    TT_REQUIRE(((reinterpret_cast<uintptr_t>(p.rows_q) | reinterpret_cast<uintptr_t>(p.rows_d)) & 15) == 0,
               "tt_triplet_step: pooled_q / pooled_d must be 16-byte aligned");
    if (p.row_B == 0) return 0;
    constexpr int kRowsPerCta = kRowThreads / 32;
    pooled_rows_kernel<<<(3 * p.row_B + kRowsPerCta - 1) / kRowsPerCta, kRowThreads, 0, st>>>(p, H);
    TT_LAUNCH_CHECK();
    return 0;
  }
  TT_REQUIRE(p.nseg >= 1 && p.nseg <= 4, "tt_pool_fwd: nseg must be in [1,4], got %d", p.nseg);
  TT_REQUIRE(H == 128 || H == 256 || H == 384 || H == 768,
             "tt_pool_fwd: hidden size %d not supported (128, 256, 384, 768)", H);
  TT_REQUIRE(table_dtype == TT_F32 || table_dtype == TT_BF16, "tt_pool_fwd: table dtype must be f32 or bf16");
  TT_REQUIRE(p.ids_dtype == TT_I64 || p.ids_dtype == TT_I32 || p.ids_dtype == TT_U16,
             "tt_pool_fwd: ids dtype must be i64, i32 or u16");
  TT_REQUIRE(p.mask_dtype == TT_I64 || p.mask_dtype == TT_I32 || p.mask_dtype == TT_U8,
             "tt_pool_fwd: mask dtype must be i64, i32 or u8");
  // longest segments first (insertion sort, <= 4 entries)
  for (int i = 1; i < p.nseg; ++i)
    for (int j = i; j > 0 && p.seg[j].L > p.seg[j - 1].L; --j) {
      PoolSegDev t = p.seg[j];
      p.seg[j] = p.seg[j - 1];
      p.seg[j - 1] = t;
    }
  long long total = 0;
  for (int i = 0; i < p.nseg; ++i) {
    TT_REQUIRE(p.seg[i].L >= 1 && p.seg[i].L <= kMaxL, "tt_pool_fwd: L=%d outside [1,%d]", p.seg[i].L, kMaxL);
    TT_REQUIRE(p.seg[i].B >= 0, "tt_pool_fwd: negative batch");
    total += p.seg[i].B;
  }
  if (total == 0) return 0;
  const int NV = H / 128;
#define TT_POOL_CASE(TE)                                        \
  switch (NV) {                                                 \
    case 1: return launch_pool<TE, 1>(p, (int)total, st);       \
    case 2: return launch_pool<TE, 2>(p, (int)total, st);       \
    case 3: return launch_pool<TE, 3>(p, (int)total, st);       \
    default: return launch_pool<TE, 6>(p, (int)total, st);      \
  }
  if (table_dtype == TT_F32) { TT_POOL_CASE(float) }
  TT_POOL_CASE(__nv_bfloat16)
#undef TT_POOL_CASE
}

}  // namespace tt

extern "C" int tt_pool_fwd_multi(const tt_pool_seg* segs, int nseg, int table_dtype, int vocab, int H,
                                 int ids_dtype, int mask_dtype, float* xhat, float* cnt, float* nrm,
                                 int* err_flag, tt_stream_t stream) {
  TT_REQUIRE(segs != nullptr && nseg >= 1 && nseg <= 4, "tt_pool_fwd_multi: bad segment list");
  tt::PoolParams p{};
  p.nseg = nseg;
  for (int i = 0; i < nseg; ++i) {
    p.seg[i].table = segs[i].table;
    p.seg[i].ids = segs[i].ids;
    p.seg[i].mask = segs[i].mask;
    p.seg[i].B = segs[i].B;
    p.seg[i].L = segs[i].L;
    p.seg[i].row0 = segs[i].row0;
  }
  p.ids_dtype = ids_dtype;
  p.mask_dtype = mask_dtype;
  p.vocab = vocab;
  p.xhat = xhat;
  p.cnt = cnt;
  p.nrm = nrm;
  p.err = err_flag;
  return tt::pool_fwd_launch(p, table_dtype, H, tt::as_stream(stream));
}

extern "C" int tt_pool_fwd(const void* table, int table_dtype, int vocab, int H, const void* ids,
                           int ids_dtype, const void* mask, int mask_dtype, int B, int L, float* xhat,
                           float* cnt, float* nrm, int* err_flag, tt_stream_t stream) {
  tt_pool_seg s{table, ids, mask, B, L, 0, 0};
  return tt_pool_fwd_multi(&s, 1, table_dtype, vocab, H, ids_dtype, mask_dtype, xhat, cnt, nrm, err_flag,
                           stream);
}

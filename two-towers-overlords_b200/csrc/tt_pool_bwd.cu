// Backward of the pooled gather into the token table: deterministic sorted-segment scatter-add.
// (north_star config 3 "trainable table"; the reference freezes the backbone at backend/model.py:28-30,
// so this is the D2 extension of SURVEY.md — its oracle is autograd through nn.Embedding.)
//
//   1. prep:    g[seq] = d(loss)/d(masked sum) = normalize-backward(dxhat) / max(cnt,1e-9)
//      fold:    (in-batch negatives named by index) g_p[j] += g_n[i] for every negative i naming positive j, in
//               ascending i; the document table then sums over the positives' tokens only
//   2. sort:   stable LSD radix sort (8-bit digits) of (token id, position) pairs; masked tokens get
//               the sentinel key `vocab`.  Warp-private contiguous chunks + __match_any_sync ranking keep
//               the sort stable, hence the reduction order (ascending position) is fixed.
//   3. reduce:  one warp per table row sums mask_t * g[seq(t)] over its run in sorted order and writes
//               the row once (zero rows for untouched ids).  Runs longer than kHeavy entries go to a
//               second kernel that splits them over the 8 warps of a CTA in a fixed order.
//               Adam variant (trainable tables with their optimiser in the step): the warp that formed a row's
//               gradient takes the row's dense Adam step itself (read + write p, m, v: 24 B per element instead of
//               the 4 B gradient write + 28 B of a separate dense Adam pass), and dtable is not written.
// No float atomics anywhere; two runs give bit-identical tables.
#include "tt_pool.cuh"

namespace tt {

namespace {

constexpr int kSortWarpItems = 1024;  // contiguous items owned by one warp
constexpr int kSortBlockWarps = 4;
constexpr int kHeavy = 256;

struct BwdSegs {
  PoolBwdSeg seg[4];
  long long base[5];  // cumulative token offsets
  int nseg;
  int ids_dtype, mask_dtype;
};

__device__ __forceinline__ int seg_of(const BwdSegs& S, long long pos) {
  int s = 0;
  while (s + 1 < S.nseg && pos >= S.base[s + 1]) ++s;
  return s;
}

// ---- 1. prep -----------------------------------------------------------------------------------
template <int NV>
__global__ void pool_bwd_prep_kernel(const float* __restrict__ dxhat, const float* __restrict__ xhat,
                                     const float* __restrict__ cnt, const float* __restrict__ nrm, int rows,
                                     float* __restrict__ g) {
  constexpr int H = NV * 128;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float4 d[NV], x[NV];
  float dot = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    d[j] = *reinterpret_cast<const float4*>(dxhat + (size_t)row * H + (j * 32 + lane) * 4);
    x[j] = *reinterpret_cast<const float4*>(xhat + (size_t)row * H + (j * 32 + lane) * 4);
    dot += d[j].x * x[j].x + d[j].y * x[j].y + d[j].z * x[j].z + d[j].w * x[j].w;
  }
  dot = warp_sum(dot);
  const float n = nrm[row];
  const float c = fmaxf(cnt[row], 1e-9f);
  // x / max(||x||, eps): below eps the denominator is a constant (clamp blocks the gradient)
  const bool clamped = n < 1e-12f;
  const float inv = 1.f / (fmaxf(n, 1e-12f) * c);
  const float k = clamped ? 0.f : dot;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    float4 o;
    o.x = (d[j].x - x[j].x * k) * inv;
    o.y = (d[j].y - x[j].y * k) * inv;
    o.z = (d[j].z - x[j].z * k) * inv;
    o.w = (d[j].w - x[j].w * k) * inv;
    *reinterpret_cast<float4*>(g + (size_t)row * H + (j * 32 + lane) * 4) = o;
  }
}

// ---- 1b. fold of the in-batch negatives --------------------------------------------------------
// Negative row i is the token sequence of positive row neg_index[i], so its share of the table gradient is that
// positive's with g_n[i] in place of g_p[j]: add it into g_p[j] and the scatter walks the positives' tokens only.
// One warp per positive j; the CTA stages neg_index in shared tiles and every warp ballots over them in ascending i,
// so g'_p[j] = ((g_p[j] + g_n[i1]) + g_n[i2]) + ... for i1 < i2 < ...  Indices outside [0, B) match no positive.
constexpr int kFoldWarps = 8;
constexpr int kFoldTile = 1024;

template <int NV>
__global__ void __launch_bounds__(kFoldWarps * 32)
    pool_bwd_fold_kernel(const int* __restrict__ neg_index, int B, const float* __restrict__ g_n,
                         float* __restrict__ g_p) {
  constexpr int H = NV * 128;
  __shared__ int s_idx[kFoldTile];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = blockIdx.x * kFoldWarps + warp;  // j >= B: a spare warp of the last CTA, which writes nothing
  const float* src = g_p + (size_t)min(j, B - 1) * H;
  float4 acc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) acc[k] = *(reinterpret_cast<const float4*>(src) + k * 32 + lane);
  bool any = false;
  for (int t0 = 0; t0 < B; t0 += kFoldTile) {
    const int n = min(kFoldTile, B - t0);
    __syncthreads();
    for (int t = threadIdx.x; t < n; t += kFoldWarps * 32) s_idx[t] = __ldg(neg_index + t0 + t);
    __syncthreads();
    for (int c = 0; c < n; c += 32) {
      unsigned hit = __ballot_sync(0xffffffffu, c + lane < n && s_idx[c + lane] == j);
      any |= hit != 0u;
      while (hit) {
        const int i = t0 + c + __ffs(hit) - 1;
        hit &= hit - 1u;
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(g_n + (size_t)i * H) + k * 32 + lane);
          acc[k].x += v.x; acc[k].y += v.y; acc[k].z += v.z; acc[k].w += v.w;
        }
      }
    }
  }
  if (j < B && any) {
#pragma unroll
    for (int k = 0; k < NV; ++k) *(reinterpret_cast<float4*>(g_p + (size_t)j * H) + k * 32 + lane) = acc[k];
  }
}

// ---- 2. radix sort -----------------------------------------------------------------------------
__global__ void make_keys_kernel(const BwdSegs S, int vocab, long long N, unsigned* __restrict__ keys,
                                 unsigned* __restrict__ vals) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int s = seg_of(S, i);
  const size_t local = (size_t)(i - S.base[s]);
  unsigned key = (unsigned)vocab;
  if (load_index(S.seg[s].mask, S.mask_dtype, local) != 0) {
    const long long id = load_index(S.seg[s].ids, S.ids_dtype, local);
    if (id >= 0 && id < vocab) key = (unsigned)id;
  }
  keys[i] = key;
  vals[i] = (unsigned)i;
}

// id_off[k] = number of sorted keys < k, for k in [0, vocab + 1]: read off the run boundaries of the sorted keys (no
// atomics: a Zipf head or the masked-token sentinel would put millions of increments on one address)
__global__ void id_offsets_kernel(const unsigned* __restrict__ keys, long long N, int vocab, int* __restrict__ id_off) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > N) return;
  const int prev = i == 0 ? -1 : (int)keys[i - 1];
  const int cur = i == N ? vocab + 1 : (int)keys[i];
  for (int k = prev + 1; k <= cur; ++k) id_off[k] = (int)i;
}

__global__ void __launch_bounds__(kSortBlockWarps * 32) radix_hist_kernel(const unsigned* __restrict__ keys,
                                                                         long long N, int shift, int W,
                                                                         int* __restrict__ hist) {
  __shared__ int s_h[kSortBlockWarps][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * kSortBlockWarps + warp;
  for (int d = lane; d < 256; d += 32) s_h[warp][d] = 0;
  __syncwarp();
  if (w < W) {
    const long long beg = (long long)w * kSortWarpItems;
    const long long end = min(beg + (long long)kSortWarpItems, N);
    for (long long i = beg + lane; i < end; i += 32) atomicAdd(&s_h[warp][(keys[i] >> shift) & 255u], 1);
  }
  __syncwarp();
  if (w < W)
    for (int d = lane; d < 256; d += 32) hist[(size_t)d * W + w] = s_h[warp][d];
}

// hist[d][0..W) -> exclusive prefix within digit d (in place), tot[d] = the digit's total.  One CTA per digit.
__global__ void __launch_bounds__(1024) digit_scan_kernel(int* __restrict__ hist, int W, int* __restrict__ tot) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  int* h = hist + (size_t)blockIdx.x * W;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (t == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < W; base += 1024) {
    const int i = base + t;
    const int v = i < W ? h[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      s_warp[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const int carry = s_carry;
    const int before = (warp ? s_warp[warp - 1] : 0) + carry;
    if (i < W) h[i] = before + x - v;
    __syncthreads();
    if (t == 1023) s_carry = carry + s_warp[31];
    __syncthreads();
  }
  if (t == 0) tot[blockIdx.x] = s_carry;
}

__global__ void __launch_bounds__(kSortBlockWarps * 32)
    radix_scatter_kernel(const unsigned* __restrict__ keys_in, const unsigned* __restrict__ vals_in, long long N,
                         int shift, int W, const int* __restrict__ hist, const int* __restrict__ tot,
                         unsigned* __restrict__ keys_out, unsigned* __restrict__ vals_out) {
  __shared__ int s_off[kSortBlockWarps][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * kSortBlockWarps + warp;
  if (w >= W) return;
  {  // first slot of digit d for this warp = (sum of the totals of smaller digits) + (this warp's prefix inside d)
    int t8[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      t8[k] = tot[lane * 8 + k];
      sum += t8[k];
    }
    int x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    int run = x - sum;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      s_off[warp][lane * 8 + k] = run + hist[(size_t)(lane * 8 + k) * W + w];
      run += t8[k];
    }
  }
  __syncwarp();
  const long long beg = (long long)w * kSortWarpItems;
  const long long end = min(beg + (long long)kSortWarpItems, N);
  const unsigned lt = (1u << lane) - 1u;
  for (long long i0 = beg; i0 < end; i0 += 32) {
    const long long i = i0 + lane;
    const bool act = i < end;
    const unsigned active = __ballot_sync(0xffffffffu, act);
    if (act) {
      const unsigned key = keys_in[i], val = vals_in[i];
      const int d = (key >> shift) & 255u;
      const unsigned peers = __match_any_sync(active, d);
      const int rank = __popc(peers & lt);
      const int base = s_off[warp][d];
      __syncwarp(active);
      if (rank == 0) s_off[warp][d] = base + __popc(peers);
      __syncwarp(active);
      keys_out[base + rank] = key;
      vals_out[base + rank] = val;
    }
  }
}

// ---- 3. segment reduce ---------------------------------------------------------------------------
template <int NV>
__device__ __forceinline__ void run_sum(const BwdSegs& S, const unsigned* __restrict__ vals, long long beg,
                                        long long end, const float* __restrict__ g, int lane, float* acc) {
  constexpr int H = NV * 128;
  for (long long b0 = beg; b0 < end; b0 += 32) {
    const long long e = b0 + lane;
    int row = 0;
    float w = 0.f;
    if (e < end) {
      const long long pos = vals[e];
      const int s = seg_of(S, pos);
      const size_t local = (size_t)(pos - S.base[s]);
      row = S.seg[s].row0 + (int)(local / (size_t)S.seg[s].L);
      w = (float)load_index(S.seg[s].mask, S.mask_dtype, local);
    }
    const int cntj = (int)min((long long)32, end - b0);
#pragma unroll 4
    for (int j = 0; j < cntj; ++j) {
      const int r = __shfl_sync(0xffffffffu, row, j);
      const float ww = __shfl_sync(0xffffffffu, w, j);
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(g + (size_t)r * H) + k * 32 + lane);
        acc[k * 4 + 0] = fmaf(ww, v.x, acc[k * 4 + 0]);
        acc[k * 4 + 1] = fmaf(ww, v.y, acc[k * 4 + 1]);
        acc[k * 4 + 2] = fmaf(ww, v.z, acc[k * 4 + 2]);
        acc[k * 4 + 3] = fmaf(ww, v.w, acc[k * 4 + 3]);
      }
    }
  }
}

constexpr int kChunk = 2048;  // entries of a heavy row summed by one CTA

// The finished gradient o of four consecutive elements of row `id`: written to dtable, or (ADAM) one Adam step on the
// table's p / m / v with it.  o already holds the old dtable row when accumulating.
template <bool ADAM>
__device__ __forceinline__ void finish_row4(float4 o, int id, int H, int col4, float* __restrict__ dtable,
                                            const TableAdam& ta, float step_size, float bc2_sqrt) {
  const size_t off = (size_t)id * H + (size_t)col4 * 4;
  if (!ADAM) {
    *reinterpret_cast<float4*>(dtable + off) = o;
    return;
  }
  float4 p = *reinterpret_cast<const float4*>(ta.p + off);
  float4 m = *reinterpret_cast<const float4*>(ta.m + off);
  float4 v = *reinterpret_cast<const float4*>(ta.v + off);
  adam_element(p.x, m.x, v.x, o.x, ta.beta1, ta.beta2, ta.eps, step_size, bc2_sqrt);
  adam_element(p.y, m.y, v.y, o.y, ta.beta1, ta.beta2, ta.eps, step_size, bc2_sqrt);
  adam_element(p.z, m.z, v.z, o.z, ta.beta1, ta.beta2, ta.eps, step_size, bc2_sqrt);
  adam_element(p.w, m.w, v.w, o.w, ta.beta1, ta.beta2, ta.eps, step_size, bc2_sqrt);
  *reinterpret_cast<float4*>(ta.p + off) = p;
  *reinterpret_cast<float4*>(ta.m + off) = m;
  *reinterpret_cast<float4*>(ta.v + off) = v;
}

// heavy bookkeeping (ints): [0] number of heavy ids, [1] number of chunks, then per heavy id {id, first chunk, chunks},
// then per chunk {id, index of the chunk inside its row}
// ADAM: every light row, touched or not (g = 0 exactly), takes its Adam step here; heavy rows take theirs in
// heavy_final_kernel, so each row of [0, vocab) is updated exactly once
template <int NV, bool ADAM>
__global__ void __launch_bounds__(256)
    seg_reduce_kernel(const BwdSegs S, const unsigned* __restrict__ vals, const int* __restrict__ id_off, int vocab,
                      const float* __restrict__ g, float* __restrict__ dtable, int accumulate, int* __restrict__ hv,
                      int max_heavy, const TableAdam ta) {
  constexpr int H = NV * 128;
  const int id = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (id >= vocab) return;
  const long long beg = id_off[id], end = id_off[id + 1];
  if (end - beg > kHeavy) {
    // rows named by many tokens (Zipf heads, [CLS]/[SEP]) are cut into chunks of kChunk entries, one CTA each; which
    // slots a row gets depends on scheduling, the summation order (chunk order, fixed split inside a chunk) does not
    if (lane == 0) {
      const int nch = (int)((end - beg + kChunk - 1) / kChunk);
      const int h = atomicAdd(&hv[0], 1);
      const int base = atomicAdd(&hv[1], nch);
      int* rec = hv + 2 + 3 * h;
      rec[0] = id; rec[1] = base; rec[2] = nch;
      int* ch = hv + 2 + 3 * max_heavy;
      for (int c = 0; c < nch; ++c) {
        ch[2 * (base + c)] = id;
        ch[2 * (base + c) + 1] = c;
      }
    }
    return;
  }
  float acc[NV * 4];
#pragma unroll
  for (int i = 0; i < NV * 4; ++i) acc[i] = 0.f;
  const float step_size = ADAM ? adam_step_size(ta.state, ta.lr) : 0.f;
  const float bc2_sqrt = ADAM ? adam_bc2_sqrt(ta.state) : 0.f;
  run_sum<NV>(S, vals, beg, end, g, lane, acc);
  float* out = dtable + (size_t)id * H;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    float4 o = make_float4(acc[k * 4], acc[k * 4 + 1], acc[k * 4 + 2], acc[k * 4 + 3]);
    float4* dst = reinterpret_cast<float4*>(out) + k * 32 + lane;
    if (accumulate) {
      const float4 old = *dst;
      o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
    }
    finish_row4<ADAM>(o, id, H, k * 32 + lane, dtable, ta, step_size, bc2_sqrt);
  }
}

// stage 1: one CTA per chunk; warp w sums a fixed 32-aligned slice, the eight slices are added in warp order
template <int NV>
__global__ void __launch_bounds__(256)
    heavy_chunk_kernel(const BwdSegs S, const unsigned* __restrict__ vals, const int* __restrict__ id_off,
                       const float* __restrict__ g, const int* __restrict__ hv, int max_heavy,
                       float* __restrict__ partial) {
  constexpr int H = NV * 128;
  __shared__ __align__(16) float s_part[8][H];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_chunks = hv[1];
  const int* ch = hv + 2 + 3 * max_heavy;
  for (int slot = blockIdx.x; slot < n_chunks; slot += gridDim.x) {
    const int id = ch[2 * slot], c = ch[2 * slot + 1];
    const long long beg = (long long)id_off[id] + (long long)c * kChunk;
    const long long end = min((long long)id_off[id + 1], beg + kChunk);
    constexpr long long per = kChunk / 8;
    const long long b = min(beg + warp * per, end), e = min(b + per, end);
    float acc[NV * 4];
#pragma unroll
    for (int i = 0; i < NV * 4; ++i) acc[i] = 0.f;
    run_sum<NV>(S, vals, b, e, g, lane, acc);
#pragma unroll
    for (int k = 0; k < NV; ++k)
      *reinterpret_cast<float4*>(&s_part[warp][(k * 32 + lane) * 4]) =
          make_float4(acc[k * 4], acc[k * 4 + 1], acc[k * 4 + 2], acc[k * 4 + 3]);
    __syncthreads();
    for (int col = threadIdx.x; col < H; col += 256) {
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) sum += s_part[w][col];
      partial[(size_t)slot * H + col] = sum;
    }
    __syncthreads();
  }
}

// stage 2: one warp per heavy row adds its chunk sums in chunk order (ADAM: then takes the row's Adam step)
template <int NV, bool ADAM>
__global__ void __launch_bounds__(256)
    heavy_final_kernel(const int* __restrict__ hv, const float* __restrict__ partial, float* __restrict__ dtable,
                       int accumulate, const TableAdam ta) {
  constexpr int H = NV * 128;
  const int lane = threadIdx.x & 31;
  const int n_heavy = hv[0];
  const float step_size = ADAM ? adam_step_size(ta.state, ta.lr) : 0.f;
  const float bc2_sqrt = ADAM ? adam_bc2_sqrt(ta.state) : 0.f;
  for (int h = blockIdx.x * 8 + (threadIdx.x >> 5); h < n_heavy; h += gridDim.x * 8) {
    const int id = hv[2 + 3 * h], base = hv[2 + 3 * h + 1], nch = hv[2 + 3 * h + 2];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int c = 0; c < nch; ++c) {
        const float4 t = *(reinterpret_cast<const float4*>(partial + (size_t)(base + c) * H) + k * 32 + lane);
        acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
      }
      if (accumulate) {
        const float4 old = *(reinterpret_cast<const float4*>(dtable + (size_t)id * H) + k * 32 + lane);
        acc.x += old.x; acc.y += old.y; acc.z += old.z; acc.w += old.w;
      }
      finish_row4<ADAM>(acc, id, H, k * 32 + lane, dtable, ta, step_size, bc2_sqrt);
    }
  }
}

}  // namespace

static inline long long max_heavy_rows(long long n_tokens) { return n_tokens / kHeavy + 1; }
static inline long long max_heavy_chunks(long long n_tokens) { return n_tokens / kChunk + max_heavy_rows(n_tokens); }

size_t pool_bwd_ws_bytes(long long n_tokens, int vocab) {
  const long long W = (n_tokens + kSortWarpItems - 1) / kSortWarpItems;
  size_t b = 0;
  b += 4 * ws_round((size_t)n_tokens * 4);         // keys A/B, vals A/B
  b += ws_round((size_t)256 * (W + 1) * 4);        // digit histograms
  b += ws_round((size_t)256 * 4);                  // digit totals
  b += ws_round((size_t)(vocab + 2) * 4);          // id offsets
  b += ws_round((size_t)(2 + 3 * max_heavy_rows(n_tokens) + 2 * max_heavy_chunks(n_tokens)) * 4);  // heavy bookkeeping
  b += ws_round((size_t)max_heavy_chunks(n_tokens) * 768 * 4);  // chunk sums (H <= 768)
  return b + 2048;
}

int pool_bwd_prep(const float* dxhat, const float* xhat, const float* cnt, const float* nrm, int rows, int H,
                  float* g, cudaStream_t st) {
  if (rows == 0) return 0;
  const int blocks = (rows + 3) / 4;
  switch (H / 128) {
    case 1: pool_bwd_prep_kernel<1><<<blocks, 128, 0, st>>>(dxhat, xhat, cnt, nrm, rows, g); break;
    case 2: pool_bwd_prep_kernel<2><<<blocks, 128, 0, st>>>(dxhat, xhat, cnt, nrm, rows, g); break;
    case 3: pool_bwd_prep_kernel<3><<<blocks, 128, 0, st>>>(dxhat, xhat, cnt, nrm, rows, g); break;
    default: pool_bwd_prep_kernel<6><<<blocks, 128, 0, st>>>(dxhat, xhat, cnt, nrm, rows, g); break;
  }
  TT_LAUNCH_CHECK();
  return 0;
}

int pool_bwd_fold_neg(const int* neg_index, int B, int H, const float* g_n, float* g_p, cudaStream_t st) {
  if (B == 0) return 0;
  const int blocks = (B + kFoldWarps - 1) / kFoldWarps;
  switch (H / 128) {
    case 1: pool_bwd_fold_kernel<1><<<blocks, kFoldWarps * 32, 0, st>>>(neg_index, B, g_n, g_p); break;
    case 2: pool_bwd_fold_kernel<2><<<blocks, kFoldWarps * 32, 0, st>>>(neg_index, B, g_n, g_p); break;
    case 3: pool_bwd_fold_kernel<3><<<blocks, kFoldWarps * 32, 0, st>>>(neg_index, B, g_n, g_p); break;
    default: pool_bwd_fold_kernel<6><<<blocks, kFoldWarps * 32, 0, st>>>(neg_index, B, g_n, g_p); break;
  }
  TT_LAUNCH_CHECK();
  return 0;
}

int pool_bwd_scatter(const PoolBwdSeg* segs, int nseg, int ids_dtype, int mask_dtype, const float* g, int vocab,
                     int H, float* dtable, int accumulate, void* ws, size_t ws_bytes, cudaStream_t st,
                     const TableAdam* adam) {
  TT_REQUIRE(nseg >= 1 && nseg <= 4, "tt_pool_bwd: nseg must be in [1,4]");
  TT_REQUIRE(H == 128 || H == 256 || H == 384 || H == 768, "tt_pool_bwd: hidden size %d not supported", H);
  BwdSegs S{};
  S.nseg = nseg;
  S.ids_dtype = ids_dtype;
  S.mask_dtype = mask_dtype;
  long long N = 0;
  for (int i = 0; i < nseg; ++i) {
    S.seg[i] = segs[i];
    S.base[i] = N;
    N += (long long)segs[i].B * segs[i].L;
  }
  S.base[nseg] = N;
  TT_REQUIRE(N < (1ll << 31), "tt_pool_bwd: too many tokens (%lld)", N);
  TT_REQUIRE(ws_bytes >= pool_bwd_ws_bytes(N, vocab), "tt_pool_bwd: workspace too small (%zu < %zu)", ws_bytes,
             pool_bwd_ws_bytes(N, vocab));
  const int W = (int)((N + kSortWarpItems - 1) / kSortWarpItems);
  char* p = reinterpret_cast<char*>(ws);
  unsigned* keyA = ws_take<unsigned>(p, N);
  unsigned* keyB = ws_take<unsigned>(p, N);
  unsigned* valA = ws_take<unsigned>(p, N);
  unsigned* valB = ws_take<unsigned>(p, N);
  int* hist = ws_take<int>(p, (size_t)256 * (W + 1));
  int* tot = ws_take<int>(p, 256);
  int* id_off = ws_take<int>(p, vocab + 2);
  const int max_heavy = (int)max_heavy_rows(N);
  int* hv = ws_take<int>(p, (size_t)2 + 3 * max_heavy + 2 * max_heavy_chunks(N));
  float* partial = ws_take<float>(p, (size_t)max_heavy_chunks(N) * H);

  TT_CUDA(cudaMemsetAsync(hv, 0, 8, st));
  if (N > 0) {
    make_keys_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(S, vocab, N, keyA, valA);
    TT_LAUNCH_CHECK();
    int bits = 1;
    while ((1ll << bits) < (long long)vocab + 1) ++bits;
    const int passes = (bits + 7) / 8;
    const int blocks = (W + kSortBlockWarps - 1) / kSortBlockWarps;
    for (int ps = 0; ps < passes; ++ps) {
      radix_hist_kernel<<<blocks, kSortBlockWarps * 32, 0, st>>>(keyA, N, ps * 8, W, hist);
      TT_LAUNCH_CHECK();
      digit_scan_kernel<<<256, 1024, 0, st>>>(hist, W, tot);
      TT_LAUNCH_CHECK();
      radix_scatter_kernel<<<blocks, kSortBlockWarps * 32, 0, st>>>(keyA, valA, N, ps * 8, W, hist, tot, keyB, valB);
      TT_LAUNCH_CHECK();
      unsigned* t = keyA; keyA = keyB; keyB = t;
      t = valA; valA = valB; valB = t;
    }
  }
  id_offsets_kernel<<<(unsigned)((N + 1 + 255) / 256), 256, 0, st>>>(keyA, N, vocab, id_off);
  TT_LAUNCH_CHECK();
  const int rblocks = (vocab + 7) / 8;
  const int hblocks = 4 * sm_count();
  const TableAdam ta = adam ? *adam : TableAdam{};
#define TT_SEG_CASE(NV, ADAM)                                                                                         \
  seg_reduce_kernel<NV, ADAM><<<rblocks, 256, 0, st>>>(S, valA, id_off, vocab, g, dtable, accumulate, hv, max_heavy,  \
                                                       ta);                                                          \
  TT_LAUNCH_CHECK();                                                                                                  \
  heavy_chunk_kernel<NV><<<hblocks, 256, 0, st>>>(S, valA, id_off, g, hv, max_heavy, partial);                          \
  TT_LAUNCH_CHECK();                                                                                                  \
  heavy_final_kernel<NV, ADAM><<<sm_count(), 256, 0, st>>>(hv, partial, dtable, accumulate, ta);                        \
  TT_LAUNCH_CHECK();
#define TT_SEG_H(ADAM)                       \
  switch (H / 128) {                         \
    case 1: { TT_SEG_CASE(1, ADAM) } break;  \
    case 2: { TT_SEG_CASE(2, ADAM) } break;  \
    case 3: { TT_SEG_CASE(3, ADAM) } break;  \
    default: { TT_SEG_CASE(6, ADAM) } break; \
  }
  if (adam) {
    TT_SEG_H(true)
  } else {
    TT_SEG_H(false)
  }
#undef TT_SEG_H
#undef TT_SEG_CASE
  return 0;
}

}  // namespace tt

extern "C" size_t tt_pool_bwd_ws_bytes(int B, int L, int vocab, int H) {
  return tt::pool_bwd_ws_bytes((long long)B * L, vocab) + tt::ws_round((size_t)B * H * 4);
}

extern "C" int tt_pool_bwd(const float* dxhat, const float* xhat, const float* cnt, const float* nrm,
                           const void* ids, int ids_dtype, const void* mask, int mask_dtype, int B, int L, int vocab,
                           int H, float* dtable, int accumulate, void* ws, size_t ws_bytes, tt_stream_t stream) {
  TT_REQUIRE(ws_bytes >= tt_pool_bwd_ws_bytes(B, L, vocab, H), "tt_pool_bwd: workspace too small");
  cudaStream_t st = tt::as_stream(stream);
  char* p = reinterpret_cast<char*>(ws);
  float* g = tt::ws_take<float>(p, (size_t)B * H);
  int rc = tt::pool_bwd_prep(dxhat, xhat, cnt, nrm, B, H, g, st);
  if (rc) return rc;
  tt::PoolBwdSeg s{ids, mask, B, L, 0};
  const size_t used = (size_t)(p - reinterpret_cast<char*>(ws));
  return tt::pool_bwd_scatter(&s, 1, ids_dtype, mask_dtype, g, vocab, H, dtable, accumulate, p, ws_bytes - used, st);
}

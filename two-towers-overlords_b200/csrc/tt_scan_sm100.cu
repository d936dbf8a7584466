// Tensor-core corpus scan (TT_PREC_BF16 / TT_PREC_BF16X3 on tt_scan_topk): query x document dot products on
// tcgen05.mma with a per-tile top-K' selection fused into the epilogue, so the score matrix lives only in TMEM.
// Restates backend/training.py:297-304 (one `cosine_similarity` row + ranking per query) as a batched exhaustive scan.
//
//   1. scan_candidates_kernel — one CTA = 128 queries (bf16 tile resident in shared memory) x one document range.
//      warp 0 streams 128-document x 64-k bf16 tiles by TMA through an mbarrier ring; warp 1 issues
//      128x128x16 MMAs into a double-buffered TMEM accumulator; warps 2-5 read finished score tiles with
//      tcgen05.ld (thread = query, columns = documents) and keep the KC best (approximate score, doc) per query
//      in shared memory behind a register threshold — an insertion happens ~KC*ln(n/KC) times per query, so the
//      epilogue is one compare per score and hides under the MMAs of the next tile.
//   2. refine_kernel — drops candidates whose approximate score is more than 2 eps below the k-th best approximate
//      score (they provably cannot enter the top k), exact fp32 dot products (CUDA cores) of the rest, top-k by
//      (score desc, id asc), plus a completeness proof: every non-candidate of split s has approximate score <=
//      bound_s (the KC-th best of that split), and |approx - exact| <= eps for unit-norm rows, so the list is
//      exact if max_s bound_s + eps < k-th exact score.  Queries that fail the proof are listed and re-scanned
//      exactly in fp32 (scan_topk_fp32_listed), so the returned ids never depend on bf16 rounding.
#include <stdlib.h>

#include "tt_ptx.cuh"
#include "tt_scan.cuh"
#include "tt_sm100.cuh"
#include "tt_tma.cuh"

namespace tt {

namespace {

using bf16 = __nv_bfloat16;
using namespace ptx;

constexpr int TQ = 128, TD = 128, BK = 64;
constexpr int kScanThreads = 192;  // warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 epilogue
constexpr uint32_t kTileBytes = TD * BK * 2;  // 16 KB: one 128-row x 64-k bf16 tile (queries or documents)
constexpr int kMaxKC = 48;
constexpr int kSlack = 64;  // append room beyond KC: a compaction runs when fewer than 32 (one TMEM chunk) slots remain
constexpr int kMaxSplits = 148;
constexpr int kTmemCols = 512;  // [0,256): two 128-column score accumulators, [256, 256 + P/2): the query tile
constexpr size_t kSmemLimit = 227 * 1024;
// |bf16(q).bf16(d) - q.d| <= |q - q~||d| + |q~||d - d~| <= 2^-9 + 2^-9 (1 + 2^-9) for rows of norm <= 1, plus the
// tensor-core accumulation error (< 1e-6): a rigorous, deliberately loose bound
constexpr float kScanEps = 4e-3f;
constexpr int kScanStagger = 4;  // document tiles between the starting points of neighbouring CTAs

struct alignas(64) ScanParams {
  CUtensorMap d_map;
  const bf16* Qb;  // [Q, P] normalised queries, bf16
  int Q, P, KB, KC, stages, stagger;
  long long N, docs_per_split;
  float* cand_s;   // [S, Q, KC] approximate scores (diagnostic / tie information)
  int* cand_i;     // [S, Q, KC] local document index, -1 = empty
  float* bound;    // [S, Q] final append threshold of the split: every document outside its list scored <= this
  // Shared floor of the append thresholds, one per query (float bits; 0xffffffff = none yet).  A split that has seen k
  // documents publishes its k-th best approximate score t: at least k documents of the corpus score >= t, so the exact
  // k-th best is >= t - eps and a document whose approximate score is below t - 3 eps can be neither in the result nor
  // needed for the completeness proof (refine_kernel checks max bound + eps < exact k-th best; here bound + eps <=
  // t - 2 eps).  Every split raises its own threshold to the floor, so short splits stop appending as soon as ANY
  // split has found good documents (without it a split of a few thousand documents never settles).
  unsigned* gthr;  // [Q]
  int k;
  float eps;
};

__device__ __forceinline__ void atomic_max_float(unsigned* addr, float v) {  // works from the 0xffffffff start value
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(addr, __float_as_uint(v));
}

// PAIR = true: two CTAs (a cluster of 2 along the query tiles) drive one cta_group::2 MMA of 256 queries x 128 documents:
// each CTA holds its own 128 queries in TMEM and streams only 64 of the 128 documents of a tile, so the L2 and
// shared-memory traffic per flop is half of the single-CTA kernel's.  The leader (cluster rank 0) issues the MMAs and
// multicast commits; data-ready barriers live in the leader, slot-free / accumulator-ready barriers in both CTAs.
template <bool PAIR>
__global__ void __launch_bounds__(kScanThreads, 1) scan_candidates_kernel(const __grid_constant__ ScanParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * TQ, split = blockIdx.y;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  constexpr uint32_t kSlotBytes = PAIR ? kTileBytes / 2 : kTileBytes;  // documents of a tile held by this CTA x 64 k
  constexpr int kOwnDocs = PAIR ? TD / 2 : TD;
  constexpr uint32_t kEpiArrivals = PAIR ? 8 : 4;  // epilogue warps that must report to the MMA issuer
  const long long d_beg = (long long)split * p.docs_per_split;
  const long long d_end = min(d_beg + p.docs_per_split, p.N);
  const int n_tiles = d_end > d_beg ? (int)((d_end - d_beg + TD - 1) / TD) : 0;
  const int KB = p.KB, NS = p.stages, KC = p.KC;
  // CTAs of one wave share a document range through L2; starting each a few tiles apart keeps them inside an
  // L2-sized window (so HBM still sees every tile once per wave) without all SMs hitting the same lines at once
  const int stagger =
      n_tiles > 0 ? (int)(((blockIdx.x / (PAIR ? 2u : 1u)) % 148u) * (unsigned)p.stagger) % n_tiles : 0;

  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* d_ring = smem;                               // NS slots
  float* list_s = reinterpret_cast<float*>(d_ring + (size_t)NS * kSlotBytes);  // [KC + kSlack][128]
  int* list_i = reinterpret_cast<int*>(list_s + (KC + kSlack) * TQ);           // [KC + kSlack][128]
  uint64_t* full = reinterpret_cast<uint64_t*>(list_i + (KC + kSlack) * TQ);
  uint64_t* empty = full + NS;
  uint64_t* q_full = empty + NS;
  uint64_t* tmem_full = q_full + 1;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(q_full, kEpiArrivals);  // one arrive per epilogue warp once its 32 query rows sit in TMEM
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], kEpiArrivals);  // one arrive per epilogue warp
    }
    fence_barrier_init();
    prefetch_tensormap(&p.d_map);
  }
  if (warp == 1) {
    if (PAIR) {
      tmem_alloc_pair(tmem_slot, kTmemCols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_slot, kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // The producer and issuer loops run on ONE lane chosen by elect.sync.  (Inside a `lane == 0` region the compiler cannot
  // prove single-thread execution and wraps every UTMALDG / UTCHMMA / UTCBAR in an ELECT + BRA.U.ANY loop, ~80 clk per
  // MMA, which made the issuing thread the bottleneck of the whole kernel; under an elect.sync predicate they issue
  // back to back.)
  if (warp == 0) {
    if (n_tiles > 0 && elect_one()) {  // ---- TMA producer (both CTAs of a pair): ONE elected lane runs the loop -------
      int s = 0;            // ring slot and its phase, advanced incrementally (no integer division in the hot loops)
      uint32_t ph = 0;
      int tt_ = stagger;
      for (int t = 0; t < n_tiles; ++t) {
        const int d0 = (int)(d_beg + (long long)tt_ * TD) + (int)rank * kOwnDocs;
        if (++tt_ == n_tiles) tt_ = 0;
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&empty[s], ph ^ 1u);
          if (PAIR) {
            if (leader) mbar_arrive_expect_tx(&full[s], kTileBytes);  // both halves complete on the leader's barrier
            tma_load_2d_pair(d_ring + (size_t)s * kSlotBytes, &p.d_map, mapa_shared(smem_u32(&full[s]), 0), kb * BK, d0);
          } else {
            mbar_arrive_expect_tx(&full[s], kTileBytes);
            tma_load_2d(d_ring + (size_t)s * kSlotBytes, &p.d_map, &full[s], kb * BK, d0);
          }
          if (++s == NS) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // (A second issuing thread on alternating tiles was tried: no gain — the batched scan runs at the power cap —
    // and with parity-only mbarrier waits an issuer that gets a whole ring round ahead of the other mistakes an old
    // phase of a slot for the new one, so there is exactly one issuer.)
    if (n_tiles > 0 && leader && elect_one()) {  // ---- MMA issuer (leader CTA only), ONE elected lane -------------------
      constexpr uint32_t idesc = make_idesc_bf16(PAIR ? 2 * TQ : TQ, TD);
      mbar_wait(q_full, 0);
      tc_fence_after();
      const uint32_t r_addr = smem_u32(d_ring);
      const uint32_t a_tmem = tmem_base + (uint32_t)(2 * TD);
      int s = 0;
      uint32_t ph = 0;
      for (int t = 0; t < n_tiles; ++t) {
        const int buf = t & 1;
        mbar_wait(&tmem_empty[buf], ((uint32_t)(t >> 1) & 1u) ^ 1u);  // epilogue(s) drained this accumulator
        tc_fence_after();
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint64_t db = make_smem_desc_sw128(r_addr + (uint32_t)s * kSlotBytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            if (PAIR)
              mma_bf16_ts_pair(tmem_base + (uint32_t)(buf * TD), a_tmem + (uint32_t)(kb * 32 + k * 8), db + 2 * k, idesc,
                               (kb | k) != 0);
            else
              mma_bf16_ts(tmem_base + (uint32_t)(buf * TD), a_tmem + (uint32_t)(kb * 32 + k * 8), db + 2 * k, idesc,
                          (kb | k) != 0);
          }
          if (PAIR) mma_commit_pair(&empty[s], 3); else mma_commit(&empty[s]);
          if (++s == NS) {
            s = 0;
            ph ^= 1u;
          }
        }
        if (PAIR) mma_commit_pair(&tmem_full[buf], 3); else mma_commit(&tmem_full[buf]);
      }
    }
  } else {  // ---- epilogue: thread = query row, walks the 128 document scores of each finished tile ---------------
    // Per query an append buffer of CAP = KC + kSlack entries behind a register threshold: a score above the
    // threshold is appended (two shared stores); when any lane of the warp runs out of room the whole warp
    // compacts together — a selection pass keeps each lane's KC best and raises its threshold to the KC-th.
    // The threshold only ever rises, so every document not in the final list scored <= the final threshold.
    const int qd = warp & 3;
    const int t_row = qd * 32 + lane;
    const bool q_ok = q0 + t_row < p.Q;
    const int CAP = KC + kSlack;
    float* ls = list_s + t_row;
    int* li = list_i + t_row;
    float thr = q_ok ? -INFINITY : INFINITY;  // rows past Q never append
    int cnt = 0;
    {  // A operand: this thread's query row -> its TMEM lane, two bf16 per 32-bit column, zero beyond P / past Q
      const uint4* qrow = reinterpret_cast<const uint4*>(p.Qb + (size_t)(q0 + t_row) * p.P);
      const int n_vec = p.P / 8;  // uint4 = 8 bf16
      for (int c = 0; c < KB * 2; ++c) {  // 16 columns = 32 bf16 = 4 uint4 per store
        uint32_t r[16];
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
          const int vi = c * 4 + v4;
          uint4 x = make_uint4(0u, 0u, 0u, 0u);
          if (q_ok && vi < n_vec) x = __ldg(qrow + vi);
          r[v4 * 4 + 0] = x.x; r[v4 * 4 + 1] = x.y; r[v4 * 4 + 2] = x.z; r[v4 * 4 + 3] = x.w;
        }
        tmem_st16(tmem_base + (uint32_t)(2 * TD) + ((uint32_t)(qd * 32) << 16) + (uint32_t)(c * 16), r);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(q_full, 0); else mbar_arrive(q_full);
      }
    }
    auto compact = [&]() {
      const int nmax = __reduce_max_sync(0xffffffffu, cnt);
      const int rounds = min(KC, nmax);
      for (int r = 0; r < rounds; ++r) {
        float best = -INFINITY;
        int bp = r;
        for (int e = r; e < nmax; ++e) {
          const float sv = (e < cnt) ? ls[e * TQ] : -INFINITY;
          if (sv > best) {
            best = sv;
            bp = e;
          }
        }
        if (r < cnt && bp != r) {
          const float s0 = ls[r * TQ];
          const int i0 = li[r * TQ];
          ls[r * TQ] = best;
          li[r * TQ] = li[bp * TQ];
          ls[bp * TQ] = s0;
          li[bp * TQ] = i0;
        }
      }
      if (cnt >= KC) {
        cnt = KC;
        thr = fmaxf(thr, ls[(KC - 1) * TQ]);
      }
      if (q_ok && cnt >= p.k) atomic_max_float(p.gthr + q0 + t_row, ls[(p.k - 1) * TQ]);  // (the list is sorted now)
    };
    const float floor_margin = 3.f * p.eps;
    for (int t = 0; t < n_tiles; ++t) {
      const int buf = t & 1;
      // the shared floor is looked at after tiles 1, 2, 4, 8 and then every 16th (it moves fast only at the start); the
      // load is issued before the wait for the accumulator so that its latency is not on the tile's path
      const bool floor_due = q_ok && (((t & (t - 1)) == 0 && t < 16) || (t & 15) == 0);
      float floor_g = 0.f;
      if (floor_due) floor_g = __uint_as_float(*reinterpret_cast<volatile const unsigned*>(p.gthr + q0 + t_row));
      mbar_wait(&tmem_full[buf], (uint32_t)(t >> 1) & 1u);
      tc_fence_after();
      int tt_ = t + stagger;
      if (tt_ >= n_tiles) tt_ -= n_tiles;
      const int d0 = tt_ * TD;  // local to the split
      const int nd = (int)min((long long)TD, d_end - d_beg - d0);
      if (floor_due) thr = fmaxf(thr, floor_g - floor_margin);  // (a NaN start value leaves thr alone)
      // 4 chunks of 32 scores, double-buffered in registers: the TMEM load of chunk c+1 flies while chunk c is scanned
      const uint32_t t_addr = tmem_base + (uint32_t)(buf * TD) + ((uint32_t)(qd * 32) << 16);
      uint32_t ra[32], rb[32];
      auto scan32 = [&](const uint32_t* r, int c) {
        // group maxima first (four independent 8-long chains instead of one 32-long one); on a hit only the
        // groups that hold a score above the threshold are walked
        float gm[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float m = __uint_as_float(r[g * 8]);
#pragma unroll
          for (int j = 1; j < 8; ++j) m = fmaxf(m, __uint_as_float(r[g * 8 + j]));
          gm[g] = m;
        }
        if (fmaxf(fmaxf(gm[0], gm[1]), fmaxf(gm[2], gm[3])) > thr) {  // rare once the threshold has settled
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            if (gm[g] > thr) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const int dj = c * 32 + g * 8 + j;
                const float vj = __uint_as_float(r[g * 8 + j]);
                if (vj > thr && dj < nd) {
                  ls[cnt * TQ] = vj;
                  li[cnt * TQ] = d0 + dj;
                  ++cnt;
                }
              }
            }
          }
        }
        if (__any_sync(0xffffffffu, cnt > CAP - 32)) compact();  // warp-uniform: no lane can overflow next chunk
      };
      tmem_ld32_async(t_addr, ra);
      tmem_ld_wait32(ra);
      tmem_ld32_async(t_addr + 32, rb);
      scan32(ra, 0);
      tmem_ld_wait32(rb);
      tmem_ld32_async(t_addr + 64, ra);
      scan32(rb, 1);
      tmem_ld_wait32(ra);
      tmem_ld32_async(t_addr + 96, rb);
      scan32(ra, 2);
      tmem_ld_wait32(rb);
      scan32(rb, 3);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(&tmem_empty[buf], 0); else mbar_arrive(&tmem_empty[buf]);
      }
    }
    compact();
    if (q_ok) {
      const size_t o = ((size_t)split * p.Q + q0 + t_row) * KC;
      const int base = (int)(d_beg);  // candidates are stored as indices local to the shard (0-based over N)
      for (int j = 0; j < KC; ++j) {
        const bool have = j < cnt;
        p.cand_s[o + j] = have ? ls[j * TQ] : -INFINITY;
        p.cand_i[o + j] = have ? base + li[j * TQ] : -1;
      }
      p.bound[(size_t)split * p.Q + q0 + t_row] = thr;  // -inf until KC documents have been seen
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync(); else __syncthreads();
  if (warp == 1) {
    if (PAIR) tmem_dealloc_pair(tmem_base, kTmemCols); else tmem_dealloc(tmem_base, kTmemCols);
  }
}

__device__ __forceinline__ bool better(float s1, long long i1, float s2, long long i2) {
  return s1 > s2 || (s1 == s2 && i1 < i2);
}

// Refinement of one query's S*KC candidates (one CTA per query):
//   a. tk = k-th best APPROXIMATE score among the candidates; since |approx - exact| <= eps, the k documents that
//      lead by approximate score all have exact score >= tk - eps, so the k-th best exact score is >= tk - eps;
//   b. a candidate with approx < tk - 2 eps has exact < tk - eps and can never enter the top k: only candidates
//      at or above t = tk - 2 eps are re-scored exactly (a few dozen instead of S*KC row gathers);
//   c. exact fp32 dot products (one warp per candidate, the same lane-strided fmaf chain as the fp32 scan),
//      top-k by (score desc, id asc);
//   d. completeness proof against the documents that never became candidates: every such document of split s
//      has approx <= bound_s, so the list is exact if max_s bound_s + eps < k-th exact score.  Queries that fail
//      (or select more than kSelCap candidates) are flagged for the exact fp32 re-scan.
constexpr int kSelCap = 256;
constexpr int kRefineThreads = 128;
__global__ void __launch_bounds__(kRefineThreads)
    refine_kernel(const float* __restrict__ Qn, const float* __restrict__ Dn, const float* __restrict__ cand_s,
                  const int* __restrict__ cand_i, const float* __restrict__ bound, int S, int Q, int KC, int P, int k,
                  long long id_base, float eps, float* __restrict__ top_score, long long* __restrict__ top_id,
                  int* __restrict__ flag) {
  extern __shared__ float approx[];  // [C]
  __shared__ float red_v[4];
  __shared__ int red_c[4];
  __shared__ int sel_c[kSelCap];
  __shared__ float sel_s[kSelCap];
  __shared__ int sel_id[kSelCap];
  __shared__ int n_sel;
  __shared__ float s_last_v, s_bmax;
  __shared__ int s_last_c, s_found;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = blockIdx.x, C = S * KC;
  for (int c0 = tid; c0 < C; c0 += 4 * kRefineThreads) {  // four slots per trip: eight independent loads in flight
    int ci[4];
    float cs[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + u * kRefineThreads;
      const int cc = c < C ? c : tid;  // (a slot of this thread that exists: keeps the loads unconditional)
      const int s = cc / KC, j = cc - s * KC;
      const size_t idx = ((size_t)s * Q + q) * KC + j;
      ci[u] = __ldg(cand_i + idx);
      cs[u] = __ldg(cand_s + idx);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + u * kRefineThreads;
      if (c < C) approx[c] = ci[u] >= 0 ? cs[u] : -INFINITY;
    }
  }
  float bm = -INFINITY;
  for (int s = tid; s < S; s += kRefineThreads) bm = fmaxf(bm, bound[(size_t)s * Q + q]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, o));
  if (lane == 0) red_v[warp] = bm;
  if (tid == 0) {
    n_sel = 0;
    s_found = 0;
    s_last_v = INFINITY;
    s_last_c = -1;
  }
  __syncthreads();
  if (tid == 0) s_bmax = fmaxf(fmaxf(red_v[0], red_v[1]), fmaxf(red_v[2], red_v[3]));
  __syncthreads();
  // a. k-th best approximate score.  Every warp first lists the k best of its own slots by itself — k rounds of "best
  //    element after the previous one" in (value desc, slot asc) order, shuffles only, no block barrier — then warp 0
  //    takes the k-th best of the 4k listed entries (the k best overall are among them).
  {
    float* wl_v = sel_s;  // [4][k] (the selection buffers are not in use yet; 4k <= kSelCap as k <= 32)
    int* wl_c = sel_c;
    float lv = INFINITY;
    int lc = -1;
    for (int r = 0; r < k; ++r) {
      float bv = -INFINITY;
      int bc = -1;
      for (int c = tid; c < C; c += kRefineThreads) {
        const float v = approx[c];
        if (v == -INFINITY) continue;
        const bool after = v < lv || (v == lv && c > lc);
        if (after && (bc < 0 || v > bv)) {  // slots ascend within a thread, so the first maximum wins ties
          bv = v;
          bc = c;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
        const int c2 = __shfl_xor_sync(0xffffffffu, bc, o);
        if (c2 >= 0 && (bc < 0 || v2 > bv || (v2 == bv && c2 < bc))) {
          bv = v2;
          bc = c2;
        }
      }
      if (lane == 0) {
        wl_v[warp * k + r] = bv;
        wl_c[warp * k + r] = bc;
      }
      if (bc >= 0) {
        lv = bv;
        lc = bc;
      } else {  // this warp's slots are exhausted: its remaining entries stay empty
        lv = -INFINITY;
        lc = C;
      }
    }
    __syncthreads();
    if (warp == 0) {
      const int n = 4 * k;  // <= 128: up to four entries per lane
      float mv = INFINITY;
      int mc = -1, found = 0;
      for (int r = 0; r < k; ++r) {
        float bv = -INFINITY;
        int bc = -1;
        for (int i = lane; i < n; i += 32) {
          const float v = wl_v[i];
          const int c = wl_c[i];
          if (c < 0) continue;
          const bool after = v < mv || (v == mv && c > mc);
          if (after && (bc < 0 || v > bv || (v == bv && c < bc))) {
            bv = v;
            bc = c;
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
          const int c2 = __shfl_xor_sync(0xffffffffu, bc, o);
          if (c2 >= 0 && (bc < 0 || v2 > bv || (v2 == bv && c2 < bc))) {
            bv = v2;
            bc = c2;
          }
        }
        if (bc < 0) break;  // fewer than k candidates exist
        mv = bv;
        mc = bc;
        ++found;
      }
      if (lane == 0) {
        s_last_v = mv;
        s_found = found;
      }
    }
    __syncthreads();
  }
  // b. candidates that can still reach the top k
  const float t = (s_found == k) ? s_last_v - 2.f * eps : -INFINITY;
  for (int c = tid; c < C; c += kRefineThreads) {
    const float v = approx[c];
    if (v != -INFINITY && v >= t) {
      const int pos = atomicAdd(&n_sel, 1);
      if (pos < kSelCap) sel_c[pos] = c;
    }
  }
  __syncthreads();
  const int total_sel = n_sel;
  const int ns = min(total_sel, kSelCap);
  // c. exact scores
  {
    float qv[16];  // P <= 512
    const float* qr = Qn + (size_t)q * P;
#pragma unroll
    for (int i = 0; i < 16; ++i) qv[i] = (lane + 32 * i < P) ? qr[lane + 32 * i] : 0.f;
    // two candidates per trip: their document rows (random 4 P-byte reads from HBM) are requested together
    constexpr int kW = kRefineThreads / 32;
    for (int i = warp; i < ns; i += 2 * kW) {
      const int i2 = i + kW;
      const bool two = i2 < ns;
      const int c0 = sel_c[i], c1 = sel_c[two ? i2 : i];
      const int s0 = c0 / KC, s1 = c1 / KC;
      const int id0 = cand_i[((size_t)s0 * Q + q) * KC + (c0 - s0 * KC)];
      const int id1 = cand_i[((size_t)s1 * Q + q) * KC + (c1 - s1 * KC)];
      const float* d0 = Dn + (size_t)id0 * P;
      const float* d1 = Dn + (size_t)id1 * P;
      float x0[16], x1[16];
#pragma unroll
      for (int ii = 0; ii < 16; ++ii) {
        const bool in = lane + 32 * ii < P;
        x0[ii] = in ? __ldg(d0 + lane + 32 * ii) : 0.f;
        x1[ii] = in ? __ldg(d1 + lane + 32 * ii) : 0.f;
      }
      float dot0 = 0.f, dot1 = 0.f;
#pragma unroll
      for (int ii = 0; ii < 16; ++ii) {  // same order of the products as one row at a time: same bits
        dot0 = fmaf(qv[ii], x0[ii], dot0);
        dot1 = fmaf(qv[ii], x1[ii], dot1);
      }
      dot0 = warp_sum(dot0);
      dot1 = warp_sum(dot1);
      if (lane == 0) {
        sel_s[i] = dot0;
        sel_id[i] = id0;
        if (two) {
          sel_s[i2] = dot1;
          sel_id[i2] = id1;
        }
      }
    }
  }
  __syncthreads();
  if (warp != 0) return;
  float last_s = INFINITY, kth = -INFINITY;
  long long last_i = -1;
  int found = 0;
  for (int r = 0; r < k; ++r) {
    float bs = -INFINITY;
    long long bi = -1;
    for (int i = lane; i < ns; i += 32) {
      const float sv = sel_s[i];
      const long long id = sel_id[i];
      const bool after = (r == 0) || better(last_s, last_i, sv, id);
      if (after && (bi < 0 || better(sv, id, bs, bi))) {
        bs = sv;
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
      top_score[(size_t)q * k + r] = (bi >= 0) ? bs : -INFINITY;
      top_id[(size_t)q * k + r] = (bi >= 0) ? bi + id_base : -1;
    }
    if (bi >= 0) {
      last_s = bs;
      last_i = bi;
      kth = bs;
      ++found;
    } else {
      last_s = -INFINITY;
      last_i = -1;
    }
  }
  // d. a document outside the candidate lists could only matter if its exact score can reach the k-th best
  if (lane == 0) {
    const float bmax = s_bmax;
    flag[q] = (total_sel > kSelCap || (found == k && bmax + eps >= kth) || (found < k && bmax > -INFINITY)) ? 1 : 0;
  }
}

// ordered compaction of the flagged query rows (single CTA: Q is at most a few hundred thousand)
__global__ void __launch_bounds__(1024) compact_flags_kernel(const int* __restrict__ flag, int Q, int* __restrict__ qlist,
                                                             int* __restrict__ qcount) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int q0 = 0; q0 < Q; q0 += 1024) {
    const int q = q0 + threadIdx.x;
    const bool f = q < Q && flag[q] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    if (f) qlist[off + __popc(bal & ((1u << lane) - 1u))] = q;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < 32; ++w) tot += s_warp[w];
      s_base += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *qcount = s_base;
}

int scan_pair_enabled(int Q, long long N);
float scan_eps();

struct ScanPlan {
  int n_qtiles, S, KC, KB, stages, cap;
  int pair;  // 1: cta_group::2 kernel, grid.x = n_qtiles rounded up to even, clusters of 2
  long long docs_per_split;
  size_t smem;
};

int make_plan(int Q, long long N, int P, int k, ScanPlan* out) {
  ScanPlan pl{};
  pl.n_qtiles = (Q + TQ - 1) / TQ;
  pl.pair = (pl.n_qtiles >= 2 && scan_pair_enabled(Q, N)) ? 1 : 0;
  if (pl.pair) pl.n_qtiles = (pl.n_qtiles + 1) / 2 * 2;
  pl.KB = (P + BK - 1) / BK;
  const long long tiles = (N + TD - 1) / TD;
  // document splits.  One CTA per SM, so the n_qtiles x S CTAs run in strict waves of `sms`; a CTA costs its
  // document tiles plus a fixed prologue/epilogue worth ~6 tiles, and every split adds candidate handling.  Take
  // the S that minimises  waves(S) x (tiles / S + 6)  (+ a small handicap per split).
  int S = 1;
  const int sms = sm_count();
  if (pl.n_qtiles == 1) {
    S = sms;
  } else {
    double best = 0.0;
    const int smax = (int)(tiles / 8 < 1 ? 1 : (tiles / 8 > kMaxSplits ? kMaxSplits : tiles / 8));
    for (int c = 1; c <= smax; ++c) {
      const long long waves = ((long long)pl.n_qtiles * c + sms - 1) / sms;
      const double cost = (double)waves * ((double)tiles / c + 6.0) * (1.0 + 0.004 * (c - 1));
      if (c == 1 || cost < best) {
        best = cost;
        S = c;
      }
    }
  }
  if (S > tiles) S = (int)tiles;
  if (S > kMaxSplits) S = kMaxSplits;
  if (S < 1) S = 1;
  pl.docs_per_split = ((tiles + S - 1) / S) * TD;
  S = (int)((N + pl.docs_per_split - 1) / pl.docs_per_split);
  pl.S = S;
  int kc = S >= 6 ? 16 : (S >= 3 ? 32 : kMaxKC);
  while (kc < k + 6 && kc < kMaxKC) kc += 16;
  // shared memory: candidate buffers + document slots (16 KB, or 8 KB per CTA of a pair)
  const size_t slot = pl.pair ? kTileBytes / 2 : kTileBytes;
  const size_t fixed = 1024 + 512 + (size_t)(kc + kSlack) * TQ * 8;
  int stages = (int)((kSmemLimit - fixed) / slot);
  pl.KC = kc;
  if (stages > (pl.pair ? 16 : 12)) stages = pl.pair ? 16 : 12;
  pl.stages = stages;
  pl.smem = fixed + (size_t)stages * slot;
  pl.cap = Q < 8192 ? Q : 8192;
  *out = pl;
  return 0;
}

// cta_group::2 scan tiles (256 queries per CTA pair, each document tile loaded once per pair and multicast): measured on
// B200 with 100k queries (ms per pass, pair vs one CTA) — 8.8 M documents 577 vs 634 (the scan sits at the power cap, and
// the pair moves half the bytes per flop from L2: 52 GB instead of 1.3 TB of DRAM traffic), 4.4 M 292 vs 321-345,
// 2.2 M 153 vs 153, 1.1 M 79 vs 68 (the pair halves the number of CTAs, and short shards cannot fill the waves with
// them).  So: pairs for shards of 3 M documents and more with many query tiles.  TT_SCAN_PAIR=0 / 1 forces either.
int scan_pair_enabled(int Q, long long N) {
  const char* e = getenv("TT_SCAN_PAIR");
  if (e) return atoi(e);
  return (N >= 3000000 && Q >= 4096) ? 1 : 0;
}

float scan_eps() {
  const char* e = getenv("TT_SCAN_EPS");  // test hook: a huge value forces every query through the exact re-scan
  return e ? (float)atof(e) : kScanEps;
}

struct ScanWs {
  float* exact;
  float* cand_s;
  int* cand_i;
  float* bound;
  int *flag, *qlist, *qcount;
  unsigned* gthr;
  void* listed;
};

size_t carve_scan(char* base, const ScanPlan& pl, int Q, int k, ScanWs* out) {
  char* p = base;
  ScanWs w{};
  w.exact = ws_take<float>(p, (size_t)pl.S * Q * pl.KC);
  w.cand_s = ws_take<float>(p, (size_t)pl.S * Q * pl.KC);
  w.cand_i = ws_take<int>(p, (size_t)pl.S * Q * pl.KC);
  w.bound = ws_take<float>(p, (size_t)pl.S * Q);
  w.flag = ws_take<int>(p, Q);
  w.qlist = ws_take<int>(p, Q);
  w.qcount = ws_take<int>(p, 64);
  w.gthr = ws_take<unsigned>(p, Q);
  w.listed = ws_take<char>(p, scan_listed_ws_bytes(pl.cap, k));
  if (out) *out = w;
  return (size_t)(p - base) + 256;
}

}  // namespace

size_t scan_sm100_ws_bytes(int Q, long long N, int P, int k) {
  ScanPlan pl;
  make_plan(Q, N, P, k, &pl);
  return carve_scan(nullptr, pl, Q, k, nullptr);
}

int scan_topk_sm100(const float* Qn, const float* Dn, const void* Qb, const void* Db, int Q, long long N, int P, int k,
                    long long id_base, float* top_score, long long* top_id, void* ws, size_t ws_bytes,
                    cudaStream_t st) {
  TT_REQUIRE(P % 8 == 0 && P <= 512, "tt_scan_topk: the tensor-core scan needs P %% 8 == 0 and P <= 512 (P=%d)", P);
  TT_REQUIRE(k <= 32, "tt_scan_topk: the tensor-core scan keeps at most 32 results per query (k=%d)", k);
  TT_REQUIRE(N < (1ll << 31), "tt_scan_topk: a shard holds at most 2^31 documents");
  ScanPlan pl;
  make_plan(Q, N, P, k, &pl);
  TT_REQUIRE(pl.stages >= 2, "tt_scan_topk: not enough shared memory for P=%d", P);
  TT_REQUIRE(ws_bytes >= carve_scan(nullptr, pl, Q, k, nullptr), "tt_scan_topk: workspace too small");
  ScanWs w;
  carve_scan(reinterpret_cast<char*>(ws), pl, Q, k, &w);

  static bool attr_done = false;
  if (!attr_done) {
    TT_CUDA(cudaFuncSetAttribute(scan_candidates_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    TT_CUDA(cudaFuncSetAttribute(scan_candidates_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    attr_done = true;
  }
  ScanParams sp{};
  int rc;
  if ((rc = make_map_bf16_kmajor(&sp.d_map, Db, (uint64_t)N, P, P, pl.pair ? TD / 2 : TD))) return rc;
  sp.Qb = reinterpret_cast<const bf16*>(Qb);
  sp.stagger = kScanStagger;
  sp.Q = Q; sp.P = P; sp.KB = pl.KB; sp.KC = pl.KC; sp.stages = pl.stages;
  sp.N = N; sp.docs_per_split = pl.docs_per_split;
  sp.cand_s = w.cand_s; sp.cand_i = w.cand_i; sp.bound = w.bound;
  sp.gthr = w.gthr; sp.k = k; sp.eps = scan_eps();
  TT_CUDA(cudaMemsetAsync(w.gthr, 0xff, (size_t)Q * sizeof(unsigned), st));
  if (pl.pair) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(pl.n_qtiles, pl.S);
    cfg.blockDim = dim3(kScanThreads);
    cfg.dynamicSmemBytes = pl.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    TT_CUDA(cudaLaunchKernelEx(&cfg, scan_candidates_kernel<true>, sp));
    note_launch();
  } else {
    scan_candidates_kernel<false><<<dim3(pl.n_qtiles, pl.S), kScanThreads, pl.smem, st>>>(sp);
    TT_LAUNCH_CHECK();
  }

  const int C = pl.S * pl.KC;
  refine_kernel<<<Q, kRefineThreads, (size_t)C * sizeof(float), st>>>(Qn, Dn, w.cand_s, w.cand_i, w.bound, pl.S, Q, pl.KC, P,
                                                                     k, id_base, scan_eps(), top_score, top_id, w.flag);
  TT_LAUNCH_CHECK();
  compact_flags_kernel<<<1, 1024, 0, st>>>(w.flag, Q, w.qlist, w.qcount);
  TT_LAUNCH_CHECK();
  return scan_topk_fp32_listed(Qn, Dn, Q, N, P, k, id_base, w.qlist, w.qcount, pl.cap, top_score, top_id, w.listed, st);
}

}  // namespace tt

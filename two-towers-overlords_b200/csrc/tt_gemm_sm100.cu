// Tensor-core projection path (TT_PREC_BF16X3 / TT_PREC_BF16): every contraction of the tower MLP, forward and
// backward, runs on tcgen05.mma with TMA-fed, 128-byte-swizzled shared-memory operands and fp32 accumulators in
// TMEM.  Replaces backend/model.py:33-38,59 and what autograd does for it inside backend/training.py:50.
//
// One kernel, gemm_tn_kernel:   C[m,n] = epi( sum_pairs sum_k A_pair[m,k] * B_pair[n,k] )
//   * both operands K-major bf16 (row-major with K contiguous); transposed copies are produced by the upstream
//     epilogues / a tiled transpose kernel so that no contraction needs an MN-major descriptor;
//   * bf16x3: fp32 values are carried as (hi, lo) bf16 pairs and the product is hi*hi + hi*lo + lo*hi, three MMAs
//     into the same TMEM accumulator (~2^-17 relative error: inside the 1e-4 loss / 1e-3 gradient gates);
//   * warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer, warps 2-5 = epilogue
//     (tcgen05.ld 32 lanes x 16 columns per warp quarter), STAGES-deep mbarrier ring between producer and issuer;
//   * up to two problem groups per launch (query tower | document tower) and split-K over blockIdx.z for the
//     weight-gradient contractions (K = batch rows), reduced afterwards in a fixed order (deterministic).
#include "tt_ptx.cuh"
#include "tt_simt.cuh"
#include "tt_sm100.cuh"
#include "tt_step_ws.cuh"
#include "tt_tma.cuh"

namespace tt {

namespace {

using namespace ptx;

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int kMaxStages = 6;
constexpr int kGemmThreads = 192;
constexpr uint32_t kABytes = BM * BK * 2, kBBytes = BN * BK * 2, kStageBytes = kABytes + kBBytes;
constexpr size_t gemm_smem(int stages) { return (size_t)stages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/; }

struct alignas(64) GemmGroup {
  CUtensorMap a[3], b[3];  // bf16 terms of each operand: hi, lo (= fp32 - hi), lo2 (= fp32 - hi - lo)
  int M, N, K, relu;   // relu: 0 none, 1 ReLU, 2 GELU (erf)
  const float* bias;   // [N] nullable
  const float* gate;   // [M, ldc] nullable: result is zeroed where gate <= 0 (ReLU backward)
  float* C;            // [M, ldc] nullable
  float* partial;      // [splits, M, N] when splits > 1 (raw sums, no epilogue)
  bf16 *C_hi, *C_lo;   // [M, ldc] nullable: bf16 split of the result
  bf16 *Ct_hi, *Ct_lo; // [N, ldt] nullable: transposed split, column = m
  int ldc, ldt;
  int pad[2];
};

struct alignas(64) GemmParams {
  GemmGroup g[2];
  int ngroups, splits, n_pairs;
  int stages;  // ring of 32 KB (A tile, B tile) slots; a k-block occupies `terms` consecutive slots
};

__global__ void __launch_bounds__(kGemmThreads, 2) gemm_tn_kernel(const __grid_constant__ GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gi = blockIdx.z / p.splits, split = blockIdx.z - gi * p.splits;
  const GemmGroup& g = p.g[gi];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (m0 >= g.M || n0 >= g.N) return;  // CTA-uniform: the grid is sized for the larger group

  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const int NS = p.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NS * kStageBytes);
  uint64_t* empty = full + kMaxStages;
  uint64_t* tmem_full = empty + kMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int kb_total = (g.K + BK - 1) / BK;
  const int kb_per = (kb_total + p.splits - 1) / p.splits;
  const int kb0 = split * kb_per;
  const int n_kb = min(kb0 + kb_per, kb_total) - kb0;  // >= 1: the host never creates an empty split
  // Each k-block brings every bf16 term of both operands exactly once: slot j of the block holds (A term j, B term j);
  // the MMAs then combine terms across slots (hi*hi, hi*lo, lo*hi | lo*lo, hi*lo2, lo2*hi).
  const int T = p.n_pairs == 1 ? 1 : (p.n_pairs == 3 ? 2 : 3);

  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
    for (int j = 0; j < T; ++j) {
      prefetch_tensormap(&g.a[j]);
      prefetch_tensormap(&g.b[j]);
    }
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Producer and issuer loops run on one lane chosen by elect.sync: in a `lane == 0` region every UTMALDG / UTCHMMA /
  // UTCBAR is wrapped in an ELECT + BRA.U.ANY loop (~80 clk each); under an elect.sync predicate they issue directly.
  if (warp == 0) {
    if (elect_one()) {  // ---- TMA producer ------------------------------------------------------------------------
      int s = 0;  // ring slot and its phase, advanced incrementally (no integer division in the hot loops)
      uint32_t ph = 0;
      for (int kbi = 0; kbi < n_kb; ++kbi) {
        for (int j = 0; j < T; ++j) {
          mbar_wait(&empty[s], ph ^ 1u);
          mbar_arrive_expect_tx(&full[s], kStageBytes);
          tma_load_2d(smem + s * kStageBytes, &g.a[j], &full[s], (kb0 + kbi) * BK, m0);
          tma_load_2d(smem + s * kStageBytes + kABytes, &g.b[j], &full[s], (kb0 + kbi) * BK, n0);
          if (++s == NS) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {  // ---- MMA issuer --------------------------------------------------------------------------
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN);
      const uint32_t ring = smem_u32(smem);
      int s = 0;
      uint32_t ph = 0;
      for (int kbi = 0; kbi < n_kb; ++kbi) {
        uint32_t slot_addr[3];
        int slot_id[3];
        for (int j = 0; j < T; ++j) {
          mbar_wait(&full[s], ph);
          slot_id[j] = s;
          slot_addr[j] = ring + (uint32_t)s * kStageBytes;
          if (++s == NS) {
            s = 0;
            ph ^= 1u;
          }
        }
        tc_fence_after();
        for (int pair = 0; pair < p.n_pairs; ++pair) {
          const int ai = (0x201100 >> (4 * pair)) & 3, bi = (0x021010 >> (4 * pair)) & 3;
          const uint64_t da = make_smem_desc_sw128(slot_addr[ai]), db = make_smem_desc_sw128(slot_addr[bi] + kABytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)  // +32 B per 16-element K slice inside the swizzled 128 B row
            mma_bf16(tmem_base, da + 2 * k, db + 2 * k, idesc, (kbi | pair | k) != 0);
        }
        for (int j = 0; j < T; ++j) mma_commit(&empty[slot_id[j]]);  // frees the slots once these MMAs have read them
      }
      mma_commit(tmem_full);
    }
  } else {  // ---- epilogue: warp quarter q owns TMEM lanes [32q, 32q+32) -----------------------------------
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int q = warp & 3;
    const int m = m0 + q * 32 + lane;
    const bool row_ok = m < g.M;
    const bool raw_out = g.partial != nullptr;
    for (int c = 0; c < BN / 16; ++c) {
      float v[16];
      tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 16), v);
      const int n = n0 + c * 16;
      if (n >= g.N) break;  // warp-uniform
      if (raw_out) {
        if (row_ok) {
          float4* dst = reinterpret_cast<float4*>(g.partial + ((size_t)split * g.M + m) * g.N + n);
#pragma unroll
          for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        continue;
      }
      if (g.bias) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] += __ldg(g.bias + n + j);
      }
      if (g.relu == 1) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
      } else if (g.relu == 2) {  // exact (erf) GELU: the frozen encoder's intermediate activation
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0.5f * v[j] * (1.f + erff(v[j] * 0.70710678118654752f));
      }
      const size_t o = (size_t)m * g.ldc + n;
      if (g.gate && row_ok) {
        const float4* gp = reinterpret_cast<const float4*>(g.gate + o);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 t = __ldg(gp + j);
          v[4 * j + 0] = t.x > 0.f ? v[4 * j + 0] : 0.f;
          v[4 * j + 1] = t.y > 0.f ? v[4 * j + 1] : 0.f;
          v[4 * j + 2] = t.z > 0.f ? v[4 * j + 2] : 0.f;
          v[4 * j + 3] = t.w > 0.f ? v[4 * j + 3] : 0.f;
        }
      }
      if (!row_ok) continue;
      if (g.C) {
        float4* dst = reinterpret_cast<float4*>(g.C + o);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
      if (g.C_hi || g.Ct_hi) {
        alignas(16) bf16 hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) split_bf16(v[j], hi[j], lo[j]);
        if (g.C_hi) {
          uint4* dh = reinterpret_cast<uint4*>(g.C_hi + o);
          uint4* dl = reinterpret_cast<uint4*>(g.C_lo + o);
          dh[0] = reinterpret_cast<const uint4*>(hi)[0];
          dh[1] = reinterpret_cast<const uint4*>(hi)[1];
          dl[0] = reinterpret_cast<const uint4*>(lo)[0];
          dl[1] = reinterpret_cast<const uint4*>(lo)[1];
        }
        if (g.Ct_hi) {  // lanes hold consecutive m: each store is one coalesced 64 B run per column
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            g.Ct_hi[(size_t)(n + j) * g.ldt + m] = hi[j];
            g.Ct_lo[(size_t)(n + j) * g.ldt + m] = lo[j];
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BN);
}

// out[i] = (accumulate ? out[i] : 0) + sum_z partial[z][i], z ascending: fixed order, no atomics.  blockIdx.y = group.
// accumulate == kAccumAfterSum: out[i] = fl(out[i] + sum_z partial[z][i]), the sum taken in the same order as for 0.
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ partial0, float* __restrict__ out0,
                                                            size_t n0, const float* __restrict__ partial1,
                                                            float* __restrict__ out1, size_t n1, int splits,
                                                            int accumulate) {
  const float* partial = blockIdx.y ? partial1 : partial0;
  float* out = blockIdx.y ? out1 : out0;
  const size_t n = blockIdx.y ? n1 : n0;
  const size_t i = ((size_t)blockIdx.x * 256 + threadIdx.x) * 4;
  if (i >= n) return;
  const bool old_first = accumulate && accumulate != kAccumAfterSum;
  float4 acc = old_first ? *reinterpret_cast<const float4*>(out + i) : make_float4(0.f, 0.f, 0.f, 0.f);
  for (int z = 0; z < splits; ++z) {
    const float4 t = *reinterpret_cast<const float4*>(partial + (size_t)z * n + i);
    acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
  }
  if (accumulate == kAccumAfterSum) {
    const float4 old = *reinterpret_cast<const float4*>(out + i);
    acc.x = old.x + acc.x; acc.y = old.y + acc.y; acc.z = old.z + acc.z; acc.w = old.w + acc.w;
  }
  *reinterpret_cast<float4*>(out + i) = acc;
}

// fp32 [R, C] (pitch ld) -> bf16 terms hi/lo[/lo2] [R, C] and, optionally, transposed hi/lo [C, ldt] (column = row
// index + tcol0).  Up to 4 matrices per launch (blockIdx.z = job): all projection weights of a step in one go.
struct SplitJob {
  const float* X;
  int R, C;
  long long ld;
  bf16 *hi, *lo, *lo2, *thi, *tlo;
  int ldt, tcol0;
};
struct SplitJobs {
  SplitJob j[4];
};

__global__ void __launch_bounds__(256) split_transpose_kernel(const SplitJobs jobs) {
  __shared__ bf16 s_hi[32][33], s_lo[32][33];
  const SplitJob& J = jobs.j[blockIdx.z];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  if (r0 >= J.R || c0 >= J.C) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + i * 8, c = c0 + tx;
    bf16 h = __float2bfloat16_rn(0.f), l = h;
    if (r < J.R && c < J.C) {
      const float xv = J.X[(size_t)r * J.ld + c];
      split_bf16(xv, h, l);
      if (J.hi) {
        J.hi[(size_t)r * J.C + c] = h;
        J.lo[(size_t)r * J.C + c] = l;
      }
      if (J.lo2) J.lo2[(size_t)r * J.C + c] = __float2bfloat16_rn((xv - __bfloat162float(h)) - __bfloat162float(l));
    }
    s_hi[ty + i * 8][tx] = h;
    s_lo[ty + i * 8][tx] = l;
  }
  if (!J.thi) return;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + i * 8, r = r0 + tx;
    if (r < J.R && c < J.C) {
      J.thi[(size_t)c * J.ldt + J.tcol0 + r] = s_hi[tx][ty + i * 8];
      J.tlo[(size_t)c * J.ldt + J.tcol0 + r] = s_lo[tx][ty + i * 8];
    }
  }
}

// bf16 hi/lo [R, C] -> transposed hi/lo [C, ldt], column = tcol0 + r + (r >= split_row ? shift : 0): the query rows and
// the document rows of a step land in their own 64-aligned column ranges with one launch
__global__ void __launch_bounds__(256) transpose_pair_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo,
                                                             int R, int C, bf16* __restrict__ thi,
                                                             bf16* __restrict__ tlo, int ldt, int tcol0, int split_row,
                                                             int shift) {
  __shared__ bf16 s[2][32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + i * 8, c = c0 + tx;
    if (r < R && c < C) {
      s[0][ty + i * 8][tx] = hi[(size_t)r * C + c];
      s[1][ty + i * 8][tx] = lo[(size_t)r * C + c];
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + i * 8, r = r0 + tx;
    if (r < R && c < C) {
      const int col = tcol0 + r + (r >= split_row ? shift : 0);
      thi[(size_t)c * ldt + col] = s[0][tx][ty + i * 8];
      tlo[(size_t)c * ldt + col] = s[1][tx][ty + i * 8];
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------------------
struct Operand {  // a K-major bf16 (hi, lo[, lo2]) split: [rows, K] with pitch ld
  const bf16* hi;
  const bf16* lo;
  long long ld;
  const bf16* lo2 = nullptr;
};

struct GemmDesc {
  Operand A, B;
  int M, N, K;
  const float* bias = nullptr;
  int relu = 0;
  const float* gate = nullptr;
  float* C = nullptr;
  int ldc = 0;
  bf16 *C_hi = nullptr, *C_lo = nullptr, *Ct_hi = nullptr, *Ct_lo = nullptr;
  int ldt = 0;
};

int fill_group(GemmGroup& g, const GemmDesc& d, int n_pairs) {
  int rc;
  const bf16* at[3] = {d.A.hi, d.A.lo, d.A.lo2};
  const bf16* bt[3] = {d.B.hi, d.B.lo, d.B.lo2};
  const int terms = n_pairs == 1 ? 1 : (n_pairs == 3 ? 2 : 3);
  for (int i = 0; i < 3; ++i) {
    if (i < terms) {
      TT_REQUIRE(at[i] && bt[i], "gemm: operand term %d missing for a %d-product contraction", i, n_pairs);
      if ((rc = make_map_bf16_kmajor(&g.a[i], at[i], d.M, d.K, d.A.ld, BM))) return rc;
      if ((rc = make_map_bf16_kmajor(&g.b[i], bt[i], d.N, d.K, d.B.ld, BN))) return rc;
    } else {
      g.a[i] = g.a[0];
      g.b[i] = g.b[0];
    }
  }
  g.M = d.M; g.N = d.N; g.K = d.K; g.relu = d.relu;
  g.bias = d.bias; g.gate = d.gate; g.C = d.C; g.partial = nullptr;
  g.C_hi = d.C_hi; g.C_lo = d.C_lo; g.Ct_hi = d.Ct_hi; g.Ct_lo = d.Ct_lo;
  g.ldc = d.ldc ? d.ldc : d.N;
  g.ldt = d.ldt;
  return 0;
}

int ensure_gemm_attr() {
  static bool done = false;
  if (done) return 0;
  TT_CUDA(cudaFuncSetAttribute(gemm_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem(kMaxStages)));
  done = true;
  return 0;
}

// ring depth: 3 slots (98 KB) keep two CTAs per SM, so one CTA's epilogue overlaps the other's main loop
constexpr int kGemmStages = 3;

// Launches 1 or 2 problem groups.  partial != nullptr: every group is a split-K contraction whose raw partial sums
// go to `partial` ([group][split][M*N], groups packed back to back) and are then reduced into d.C (+= if accumulate).
int launch_gemm(const GemmDesc* d, int ngroups, int n_pairs, int splits, float* partial, int accumulate,
                cudaStream_t st) {
  int rc;
  if ((rc = ensure_gemm_attr())) return rc;
  GemmParams p{};
  p.ngroups = ngroups;
  p.n_pairs = n_pairs;
  int tiles_m = 0, tiles_n = 0;
  for (int i = 0; i < ngroups; ++i) {
    TT_REQUIRE(d[i].M >= 1 && d[i].N >= 16 && d[i].N % 16 == 0 && d[i].K >= 1, "gemm: bad shape M=%d N=%d K=%d", d[i].M,
               d[i].N, d[i].K);
    if ((rc = fill_group(p.g[i], d[i], n_pairs))) return rc;
    tiles_m = max(tiles_m, (d[i].M + BM - 1) / BM);
    tiles_n = max(tiles_n, (d[i].N + BN - 1) / BN);
  }
  const bool use_partial = partial != nullptr;
  if (!use_partial) splits = 1;
  if (splits > 1) {
    // all groups of a split-K launch share K (same batch rows) up to the tower split; clamp to the smallest
    int kb_min = 1 << 30;
    for (int i = 0; i < ngroups; ++i) kb_min = min(kb_min, (d[i].K + BK - 1) / BK);
    splits = min(splits, kb_min);
    // no empty split for any group: ceil(kb/ceil(kb/splits)) must equal splits for every group
    for (bool ok = false; !ok && splits > 1;) {
      ok = true;
      for (int i = 0; i < ngroups; ++i) {
        const int kb = (d[i].K + BK - 1) / BK, per = (kb + splits - 1) / splits;
        if ((kb + per - 1) / per != splits) ok = false;
      }
      if (!ok) --splits;
    }
  }
  p.splits = splits;
  if (use_partial) {
    size_t off = 0;
    for (int i = 0; i < ngroups; ++i) {
      p.g[i].partial = partial + off;
      off += (size_t)splits * d[i].M * d[i].N;
    }
  }
  p.stages = kGemmStages;
  dim3 grid(tiles_n, tiles_m, ngroups * splits);
  gemm_tn_kernel<<<grid, kGemmThreads, gemm_smem(p.stages), st>>>(p);
  TT_LAUNCH_CHECK();
  if (use_partial) {
    size_t n[2] = {0, 0};
    for (int i = 0; i < ngroups; ++i) {
      n[i] = (size_t)d[i].M * d[i].N;
      TT_REQUIRE(d[i].ldc == 0 || d[i].ldc == d[i].N, "gemm: split-K output must be dense");
    }
    const size_t nmax = n[0] > n[1] ? n[0] : n[1];
    splitk_reduce_kernel<<<dim3((unsigned)((nmax / 4 + 255) / 256), ngroups), 256, 0, st>>>(
        p.g[0].partial, d[0].C, n[0], ngroups > 1 ? p.g[1].partial : nullptr, ngroups > 1 ? d[1].C : nullptr, n[1],
        splits, accumulate);
    TT_LAUNCH_CHECK();
  } else {
    TT_REQUIRE(!accumulate, "gemm: accumulate needs the split-K path");  // checked before the launch in practice
  }
  return 0;
}

int choose_splits(int tiles, int K) {
  const int kb = (K + BK - 1) / BK;
  int s = (2 * sm_count() + tiles - 1) / tiles;
  s = min(s, kb);
  s = min(s, 32);
  return max(s, 2);  // weight-gradient GEMMs always take the split-K path (it also implements `accumulate`)
}

int split_jobs(const SplitJob* jobs, int n, cudaStream_t st) {
  SplitJobs J{};
  int rmax = 0, cmax = 0;
  for (int i = 0; i < n; ++i) {
    J.j[i] = jobs[i];
    rmax = max(rmax, jobs[i].R);
    cmax = max(cmax, jobs[i].C);
  }
  split_transpose_kernel<<<dim3((cmax + 31) / 32, (rmax + 31) / 32, n), 256, 0, st>>>(J);
  TT_LAUNCH_CHECK();
  return 0;
}

int split_transpose(const float* X, int R, int C, long long ld, bf16* hi, bf16* lo, bf16* thi, bf16* tlo, int ldt,
                    int tcol0, cudaStream_t st, bf16* lo2 = nullptr) {
  SplitJob j{X, R, C, ld, hi, lo, lo2, thi, tlo, ldt, tcol0};
  return split_jobs(&j, 1, st);
}

int transpose_pair(const bf16* hi, const bf16* lo, int R, int C, bf16* thi, bf16* tlo, int ldt, int tcol0,
                   int split_row, int shift, cudaStream_t st) {
  dim3 grid((C + 31) / 32, (R + 31) / 32);
  transpose_pair_kernel<<<grid, 256, 0, st>>>(hi, lo, R, C, thi, tlo, ldt, tcol0, split_row, shift);
  TT_LAUNCH_CHECK();
  return 0;
}

// ---- workspace of one tower pass (standalone tt_encode_fwd / tt_encode_bwd) --------------------------------
struct MlpWs {
  bf16 *x_hi, *x_lo, *x_lo2, *xt_hi, *xt_lo;  // [M,H], [H,ldm]
  bf16 *w1_hi, *w1_lo, *w1_lo2, *w1t_hi, *w1t_lo;  // [P,H], [H,P]
  bf16 *w2_hi, *w2_lo, *w2t_hi, *w2t_lo;      // [P,P], [P,P]
  bf16 *h_hi, *h_lo, *ht_hi, *ht_lo;          // [M,P], [P,ldm]
  bf16 *dy_hi, *dy_lo, *dyt_hi, *dyt_lo;      // [M,P], [P,ldm]
  bf16 *dz_hi, *dz_lo, *dzt_hi, *dzt_lo;      // [M,P], [P,ldm]
  float *hbuf, *dz1, *partial, *colsum;
  int ldm;
};

size_t carve_mlp_ws(char* base, int M, int H, int P, MlpWs* out) {
  char* p = base;
  MlpWs w{};
  const int ldm = round64(M);
  w.ldm = ldm;
  const size_t MH = (size_t)M * H, MP = (size_t)M * P, HL = (size_t)H * ldm, PL = (size_t)P * ldm;
  w.x_hi = ws_take<bf16>(p, MH); w.x_lo = ws_take<bf16>(p, MH); w.x_lo2 = ws_take<bf16>(p, MH);
  w.xt_hi = ws_take<bf16>(p, HL); w.xt_lo = ws_take<bf16>(p, HL);
  w.w1_hi = ws_take<bf16>(p, (size_t)P * H); w.w1_lo = ws_take<bf16>(p, (size_t)P * H);
  w.w1_lo2 = ws_take<bf16>(p, (size_t)P * H);
  w.w1t_hi = ws_take<bf16>(p, (size_t)P * H); w.w1t_lo = ws_take<bf16>(p, (size_t)P * H);
  w.w2_hi = ws_take<bf16>(p, (size_t)P * P); w.w2_lo = ws_take<bf16>(p, (size_t)P * P);
  w.w2t_hi = ws_take<bf16>(p, (size_t)P * P); w.w2t_lo = ws_take<bf16>(p, (size_t)P * P);
  w.h_hi = ws_take<bf16>(p, MP); w.h_lo = ws_take<bf16>(p, MP);
  w.ht_hi = ws_take<bf16>(p, PL); w.ht_lo = ws_take<bf16>(p, PL);
  w.dy_hi = ws_take<bf16>(p, MP); w.dy_lo = ws_take<bf16>(p, MP);
  w.dyt_hi = ws_take<bf16>(p, PL); w.dyt_lo = ws_take<bf16>(p, PL);
  w.dz_hi = ws_take<bf16>(p, MP); w.dz_lo = ws_take<bf16>(p, MP);
  w.dzt_hi = ws_take<bf16>(p, PL); w.dzt_lo = ws_take<bf16>(p, PL);
  w.hbuf = ws_take<float>(p, MP);
  w.dz1 = ws_take<float>(p, MP);
  w.partial = ws_take<float>(p, (size_t)32 * P * max(P, H));
  w.colsum = ws_take<float>(p, (size_t)2 * kColsumSlices * P);
  if (out) *out = w;
  return (size_t)(p - base) + 256;
}

}  // namespace

size_t mlp_sm100_ws_bytes(int M, int H, int P) { return carve_mlp_ws(nullptr, M, H, P, nullptr); }

int mlp_fwd_sm100(const float* x, int M, int H, int P, const float* W1, const float* b1, const float* W2,
                  const float* b2, float* h, float* y, int precision, void* ws, size_t ws_bytes, cudaStream_t st) {
  TT_REQUIRE(ws_bytes >= mlp_sm100_ws_bytes(M, H, P), "tt_encode_fwd: workspace too small");
  MlpWs w;
  carve_mlp_ws(reinterpret_cast<char*>(ws), M, H, P, &w);
  const int np = precision == TT_PREC_BF16X3 ? 3 : 1;
  // the first layer feeds the ReLU whose sign gates the backward: it gets the 6-product (fp32-exact) split
  const int np1 = precision == TT_PREC_BF16X3 ? 6 : 1;
  int rc;
  if ((rc = split_transpose(x, M, H, H, w.x_hi, w.x_lo, nullptr, nullptr, 0, 0, st, w.x_lo2))) return rc;
  if ((rc = split_transpose(W1, P, H, H, w.w1_hi, w.w1_lo, nullptr, nullptr, 0, 0, st, w.w1_lo2))) return rc;
  if ((rc = split_transpose(W2, P, P, P, w.w2_hi, w.w2_lo, nullptr, nullptr, 0, 0, st))) return rc;
  GemmDesc g1{};
  g1.A = {w.x_hi, w.x_lo, H, w.x_lo2}; g1.B = {w.w1_hi, w.w1_lo, H, w.w1_lo2};
  g1.M = M; g1.N = P; g1.K = H; g1.bias = b1; g1.relu = 1;
  g1.C = h ? h : w.hbuf; g1.ldc = P; g1.C_hi = w.h_hi; g1.C_lo = w.h_lo;
  if ((rc = launch_gemm(&g1, 1, np1, 1, nullptr, 0, st))) return rc;
  GemmDesc g2{};
  g2.A = {w.h_hi, w.h_lo, P}; g2.B = {w.w2_hi, w.w2_lo, P};
  g2.M = M; g2.N = P; g2.K = P; g2.bias = b2; g2.C = y; g2.ldc = P;
  return launch_gemm(&g2, 1, np, 1, nullptr, 0, st);
}

int mlp_bwd_sm100(const float* dy, const float* x, const float* h, const float* W1, const float* W2, int M, int H,
                  int P, float* dW1, float* db1, float* dW2, float* db2, float* dx, int accumulate, int precision,
                  void* ws, size_t ws_bytes, cudaStream_t st) {
  TT_REQUIRE(ws_bytes >= mlp_sm100_ws_bytes(M, H, P), "tt_encode_bwd: workspace too small");
  MlpWs w;
  carve_mlp_ws(reinterpret_cast<char*>(ws), M, H, P, &w);
  const int np = precision == TT_PREC_BF16X3 ? 3 : 1;
  const int ldm = w.ldm;
  int rc;
  // operands: dy, h, x (row-major + transposed), W2^T, W1^T
  if ((rc = split_transpose(dy, M, P, P, w.dy_hi, w.dy_lo, w.dyt_hi, w.dyt_lo, ldm, 0, st))) return rc;
  if ((rc = split_transpose(h, M, P, P, nullptr, nullptr, w.ht_hi, w.ht_lo, ldm, 0, st))) return rc;
  if ((rc = split_transpose(x, M, H, H, nullptr, nullptr, w.xt_hi, w.xt_lo, ldm, 0, st))) return rc;
  if ((rc = split_transpose(W2, P, P, P, nullptr, nullptr, w.w2t_hi, w.w2t_lo, P, 0, st))) return rc;
  // db2, dW2 = dy^T h
  if ((rc = colsum2(dy, M, db2, nullptr, 0, nullptr, P, P, accumulate, w.colsum, st))) return rc;
  GemmDesc gw2{};
  gw2.A = {w.dyt_hi, w.dyt_lo, ldm}; gw2.B = {w.ht_hi, w.ht_lo, ldm};
  gw2.M = P; gw2.N = P; gw2.K = M; gw2.C = dW2;
  const int tiles2 = ((P + BM - 1) / BM) * ((P + BN - 1) / BN);
  if ((rc = launch_gemm(&gw2, 1, np, choose_splits(tiles2, M), w.partial, accumulate, st))) return rc;
  // dz1 = (dy W2) * (h > 0)
  GemmDesc gz{};
  gz.A = {w.dy_hi, w.dy_lo, P}; gz.B = {w.w2t_hi, w.w2t_lo, P};
  gz.M = M; gz.N = P; gz.K = P; gz.gate = h; gz.C = w.dz1; gz.ldc = P;
  gz.C_hi = dx ? w.dz_hi : nullptr; gz.C_lo = dx ? w.dz_lo : nullptr;
  gz.Ct_hi = w.dzt_hi; gz.Ct_lo = w.dzt_lo; gz.ldt = ldm;
  if ((rc = launch_gemm(&gz, 1, np, 1, nullptr, 0, st))) return rc;
  if ((rc = colsum2(w.dz1, M, db1, nullptr, 0, nullptr, P, P, accumulate, w.colsum, st))) return rc;
  // dW1 = dz1^T x
  GemmDesc gw1{};
  gw1.A = {w.dzt_hi, w.dzt_lo, ldm}; gw1.B = {w.xt_hi, w.xt_lo, ldm};
  gw1.M = P; gw1.N = H; gw1.K = M; gw1.C = dW1;
  const int tiles1 = ((P + BM - 1) / BM) * ((H + BN - 1) / BN);
  if ((rc = launch_gemm(&gw1, 1, np, choose_splits(tiles1, M), w.partial, accumulate, st))) return rc;
  if (dx) {  // dx = dz1 W1
    if ((rc = split_transpose(W1, P, H, H, nullptr, nullptr, w.w1t_hi, w.w1t_lo, P, 0, st))) return rc;
    GemmDesc gx{};
    gx.A = {w.dz_hi, w.dz_lo, P}; gx.B = {w.w1t_hi, w.w1t_lo, P};
    gx.M = M; gx.N = H; gx.K = P; gx.C = dx; gx.ldc = H;
    if ((rc = launch_gemm(&gx, 1, np, 1, nullptr, 0, st))) return rc;
  }
  return 0;
}

// ================================================================================================================
// whole triplet step on the tensor cores: rows [0,B) = queries (query tower), rows [B,3B) = positives | negatives
// (document tower).  Every GEMM launch carries both towers as two problem groups.
// ================================================================================================================

size_t step_sm100_ws_bytes(int B, int H, int P, int train_table) { return carve_step(nullptr, B, H, P, train_table, nullptr); }

// Auxiliary streams + events for the independent branches of the backward chain.  Created on first use (the first
// call is never inside a stream capture: FusedTrainer warms up eagerly); fork()/join() are capture-legal, so in a
// CUDA graph the branches become parallel paths of the DAG.
struct Forks {
  cudaStream_t aux[2] = {nullptr, nullptr};
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int device = -1;
};
static int get_forks(Forks** out) {
  static thread_local Forks f;
  int dev = 0;
  TT_CUDA(cudaGetDevice(&dev));
  if (f.device != dev) {
    for (auto& a : f.aux) TT_CUDA(cudaStreamCreateWithFlags(&a, cudaStreamNonBlocking));
    for (auto& e : f.ev) TT_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    f.device = dev;
  }
  *out = &f;
  return 0;
}
int step_sm100(const StepSm100& s, cudaStream_t st) {
  const int B = s.B, H = s.H, P = s.P, np = s.n_split;
  TT_REQUIRE(s.ws && s.ws_bytes >= step_sm100_ws_bytes(B, H, P, s.dxhat != nullptr), "tt_triplet_step: tensor-core workspace too small");
  StepWs w;
  carve_step(reinterpret_cast<char*>(s.ws), B, H, P, s.dxhat != nullptr, &w);
  int rc;
  const float* W1[2] = {s.Wq1, s.Wd1};
  const float* W2[2] = {s.Wq2, s.Wd2};
  const float* b1[2] = {s.bq1, s.bd1};
  const float* b2[2] = {s.bq2, s.bd2};
  float* dW1[2] = {s.dWq1, s.dWd1};
  float* db1[2] = {s.dbq1, s.dbd1};
  float* dW2[2] = {s.dWq2, s.dWd2};
  float* db2[2] = {s.dbq2, s.dbd2};
  const int row0[2] = {0, B}, rows[2] = {B, 2 * B}, tcol[2] = {0, w.dcol};

  // 1. pooled gather: fp32 xhat + its bf16 split (row-major); the transposed copy comes from a tiled transpose
  const bool front = s.phases == 0 || (s.phases & TT_STEP_FRONT), back = s.phases == 0 || (s.phases & TT_STEP_BACK);
  if (front) {
    PoolParams pp = s.pool;
    pp.x_hi = w.x_hi; pp.x_lo = w.x_lo; pp.x_lo2 = (np == 3) ? w.x_lo2 : nullptr;
    pp.share_sm = (s.phases == TT_STEP_FRONT) ? 1 : 0;  // gather-only call = the pipelined trainer's look-ahead gather
    if ((rc = pool_fwd_launch(pp, s.table_dtype, H, st))) return rc;
    // (the persistent chain kernel transposes the xhat terms itself)
    if (!s.chain && (rc = transpose_pair(w.x_hi, w.x_lo, 3 * B, H, w.xt_hi, w.xt_lo, w.ldt, 0, B, w.dcol - B, st))) return rc;
  }
  if (!back) return 0;
  if (s.chain) return chain_sm100(s, /*after_gather=*/front, st);
  // 2. weights of both towers -> bf16 terms (+ transposes for the backward contractions), one launch
  {
    SplitJob jobs[4];
    for (int t = 0; t < 2; ++t) {
      jobs[2 * t] = SplitJob{W1[t], P, H, H, w.w1_hi[t], w.w1_lo[t], np == 3 ? w.w1_lo2[t] : nullptr,
                             s.dxhat ? w.w1t_hi[t] : nullptr, s.dxhat ? w.w1t_lo[t] : nullptr, P, 0};
      jobs[2 * t + 1] = SplitJob{W2[t], P, P, P, w.w2_hi[t], w.w2_lo[t], nullptr, w.w2t_hi[t], w.w2t_lo[t], P, 0};
    }
    if ((rc = split_jobs(jobs, 4, st))) return rc;
  }
  // 3. h = relu(x W1^T + b1)  (fp32 + split + transposed split)
  GemmDesc g[2];
  for (int t = 0; t < 2; ++t) {
    g[t] = GemmDesc{};
    g[t].A = {w.x_hi + (size_t)row0[t] * H, w.x_lo + (size_t)row0[t] * H, H, w.x_lo2 + (size_t)row0[t] * H};
    g[t].B = {w.w1_hi[t], w.w1_lo[t], H, w.w1_lo2[t]};
    g[t].M = rows[t]; g[t].N = P; g[t].K = H; g[t].bias = b1[t]; g[t].relu = 1;
    g[t].C = s.h + (size_t)row0[t] * P; g[t].ldc = P;
    g[t].C_hi = w.h_hi + (size_t)row0[t] * P; g[t].C_lo = w.h_lo + (size_t)row0[t] * P;
    g[t].Ct_hi = w.ht_hi + tcol[t]; g[t].Ct_lo = w.ht_lo + tcol[t]; g[t].ldt = w.ldt;
  }
  // (6-product split for this layer only: its ReLU sign gates the backward, see mlp_fwd_sm100)
  if ((rc = launch_gemm(g, 2, np == 3 ? 6 : 1, 1, nullptr, 0, st))) return rc;
  // 4. y = h W2^T + b2
  for (int t = 0; t < 2; ++t) {
    g[t] = GemmDesc{};
    g[t].A = {w.h_hi + (size_t)row0[t] * P, w.h_lo + (size_t)row0[t] * P, P};
    g[t].B = {w.w2_hi[t], w.w2_lo[t], P};
    g[t].M = rows[t]; g[t].N = P; g[t].K = P; g[t].bias = b2[t];
    g[t].C = s.y + (size_t)row0[t] * P; g[t].ldc = P;
  }
  if ((rc = launch_gemm(g, 2, np, 1, nullptr, 0, st))) return rc;
  // 5. loss and its gradient (fp32 CUDA-core kernels; dY leaves as fp32 + bf16 split)
  const float* yq = s.y;
  const float* yp = s.y + (size_t)B * P;
  const float* yn = s.y + (size_t)2 * B * P;
  LossSplitOut so{};
  so.dy_hi = w.dy_hi; so.dy_lo = w.dy_lo;
  if ((rc = triplet_loss_fused(yq, yp, yn, B, P, s.margin, s.inv_batch, s.grad_scale, s.stats, s.loss, s.dy,
                               s.dy + (size_t)B * P, s.dy + (size_t)2 * B * P, &so, w.loss_scratch, st)))
    return rc;
  // From here the chain forks: {dY^T -> dW2}, {db2, db1} and {dz1 -> dW1} only share inputs.
  Forks* fk = nullptr;
  if ((rc = get_forks(&fk))) return rc;
  cudaStream_t sA = fk->aux[0], sB = fk->aux[1];
  TT_CUDA(cudaEventRecord(fk->ev[0], st));
  TT_CUDA(cudaStreamWaitEvent(sA, fk->ev[0], 0));
  TT_CUDA(cudaStreamWaitEvent(sB, fk->ev[0], 0));
  // 6a. (branch A) dY^T, then dW2 = dY^T h   (split-K over the batch rows)
  if ((rc = transpose_pair(w.dy_hi, w.dy_lo, 3 * B, P, w.dyt_hi, w.dyt_lo, w.ldt, 0, B, w.dcol - B, sA))) return rc;
  for (int t = 0; t < 2; ++t) {
    g[t] = GemmDesc{};
    g[t].A = {w.dyt_hi + tcol[t], w.dyt_lo + tcol[t], w.ldt};
    g[t].B = {w.ht_hi + tcol[t], w.ht_lo + tcol[t], w.ldt};
    g[t].M = P; g[t].N = P; g[t].K = rows[t]; g[t].C = dW2[t];
  }
  const int tiles2 = 2 * ((P + BM - 1) / BM) * ((P + BN - 1) / BN);
  // (s.grad_accumulate: every gradient output is fl(old + the sum a call without it writes))
  const int acc = s.grad_accumulate ? kAccumAfterSum : 0;
  if ((rc = launch_gemm(g, 2, np, choose_splits(tiles2, B), w.partial2, acc, sA))) return rc;
  // 6b. (branch B) db2
  if ((rc = colsum2(s.dy, rows[0], db2[0], s.dy + (size_t)row0[1] * P, rows[1], db2[1], P, P, acc, w.colsum2, sB))) return rc;
  // 7. (main) dz1 = (dY W2) * (h > 0)
  for (int t = 0; t < 2; ++t) {
    g[t] = GemmDesc{};
    g[t].A = {w.dy_hi + (size_t)row0[t] * P, w.dy_lo + (size_t)row0[t] * P, P};
    g[t].B = {w.w2t_hi[t], w.w2t_lo[t], P};
    g[t].M = rows[t]; g[t].N = P; g[t].K = P; g[t].gate = s.h + (size_t)row0[t] * P;
    g[t].C = w.dz1 + (size_t)row0[t] * P; g[t].ldc = P;
    if (s.dxhat) {
      g[t].C_hi = w.dz_hi + (size_t)row0[t] * P; g[t].C_lo = w.dz_lo + (size_t)row0[t] * P;
    }
    g[t].Ct_hi = w.dzt_hi + tcol[t]; g[t].Ct_lo = w.dzt_lo + tcol[t]; g[t].ldt = w.ldt;
  }
  if ((rc = launch_gemm(g, 2, np, 1, nullptr, 0, st))) return rc;
  // branch B continues with db1 once dz1 exists
  TT_CUDA(cudaEventRecord(fk->ev[1], st));
  TT_CUDA(cudaStreamWaitEvent(sB, fk->ev[1], 0));
  if ((rc = colsum2(w.dz1, rows[0], db1[0], w.dz1 + (size_t)row0[1] * P, rows[1], db1[1], P, P, acc, w.colsum, sB)))
    return rc;
  // 8. (main) dW1 = dz1^T x
  for (int t = 0; t < 2; ++t) {
    g[t] = GemmDesc{};
    g[t].A = {w.dzt_hi + tcol[t], w.dzt_lo + tcol[t], w.ldt};
    g[t].B = {w.xt_hi + tcol[t], w.xt_lo + tcol[t], w.ldt};
    g[t].M = P; g[t].N = H; g[t].K = rows[t]; g[t].C = dW1[t];
  }
  const int tiles1 = 2 * ((P + BM - 1) / BM) * ((H + BN - 1) / BN);
  if ((rc = launch_gemm(g, 2, np, choose_splits(tiles1, B), w.partial, acc, st))) return rc;
  // join
  TT_CUDA(cudaEventRecord(fk->ev[2], sA));
  TT_CUDA(cudaEventRecord(fk->ev[3], sB));
  TT_CUDA(cudaStreamWaitEvent(st, fk->ev[2], 0));
  TT_CUDA(cudaStreamWaitEvent(st, fk->ev[3], 0));
  // 9. dxhat = dz1 W1 (only when the token tables train)
  if (s.dxhat) {
    for (int t = 0; t < 2; ++t) {
      g[t] = GemmDesc{};
      g[t].A = {w.dz_hi + (size_t)row0[t] * P, w.dz_lo + (size_t)row0[t] * P, P};
      g[t].B = {w.w1t_hi[t], w.w1t_lo[t], P};
      g[t].M = rows[t]; g[t].N = H; g[t].K = P; g[t].C = s.dxhat + (size_t)row0[t] * H; g[t].ldc = H;
    }
    if ((rc = launch_gemm(g, 2, np, 1, nullptr, 0, st))) return rc;
  }
  return 0;
}

// One contraction C = act(A B^T + bias) on the tensor cores for other parts of the library (the frozen encoder):
// operands as bf16 (hi, lo) terms, K-major; outputs fp32 and / or bf16 terms (each nullable).
int gemm_terms_sm100(const bf16* A_hi, const bf16* A_lo, long long lda, const bf16* B_hi, const bf16* B_lo, long long ldb,
                     int M, int N, int K, const float* bias, int act, float* C, int ldc, bf16* C_hi, bf16* C_lo,
                     cudaStream_t st) {
  GemmDesc d{};
  d.A = {A_hi, A_lo, lda};
  d.B = {B_hi, B_lo, ldb};
  d.M = M; d.N = N; d.K = K; d.bias = bias; d.relu = act;
  d.C = C; d.ldc = ldc; d.C_hi = C_hi; d.C_lo = C_lo;
  return launch_gemm(&d, 1, A_lo ? 3 : 1, 1, nullptr, 0, st);
}

int split_terms_sm100(const float* X, int R, int C, bf16* hi, bf16* lo, cudaStream_t st) {
  return split_transpose(X, R, C, C, hi, lo, nullptr, nullptr, 0, 0, st);
}

}  // namespace tt

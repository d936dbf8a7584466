// Workspace of the tensor-core triplet step (shared by the per-kernel chain in tt_gemm_sm100.cu and the persistent
// chain kernel in tt_chain_sm100.cu).
#pragma once
#include "tt_simt.cuh"
#include "tt_sm100.cuh"

namespace tt {

using bf16 = __nv_bfloat16;
static inline int round64(int x) { return (x + 63) / 64 * 64; }

struct StepWs {
  int ldt, dcol;  // transposed buffers: query rows at columns [0,B), document rows at [dcol, dcol+2B)
  bf16 *x_hi, *x_lo, *x_lo2, *xt_hi, *xt_lo;  // [3B,H], [H,ldt]
  bf16 *h_hi, *h_lo, *ht_hi, *ht_lo;        // [3B,P], [P,ldt]
  bf16 *dy_hi, *dy_lo, *dyt_hi, *dyt_lo;    // [3B,P], [P,ldt]
  bf16 *dz_hi, *dz_lo, *dzt_hi, *dzt_lo;    // [3B,P], [P,ldt]
  bf16 *w1_hi[2], *w1_lo[2], *w1_lo2[2], *w1t_hi[2], *w1t_lo[2];  // per tower: [P,H], [H,P]
  bf16 *w2_hi[2], *w2_lo[2], *w2t_hi[2], *w2t_lo[2];  // per tower: [P,P], [P,P]
  float *dz1, *partial, *partial2, *colsum, *colsum2, *loss_scratch;
  // persistent chain kernel (tt_chain_sm100.cu): per-(triplet tile, column half) loss partial sums, per-row-tile
  // column sums for the bias gradients, per-tile hinge sums, dependency counters
  float *stat_part, *cs1, *cs2, *hinge_part, *ybuf;
  unsigned* counters;
  int n_counters;
  unsigned long long* trace;  // TT_CHAIN_TRACE=1: [CTA][kTraceSlots] x {task index << 4 | event, globaltimer ns}
};
constexpr int kTraceSlots = 128, kTraceCtas = 160;

static inline size_t carve_step(char* base, int B, int H, int P, int train_table, StepWs* out) {
  char* p = base;
  StepWs w{};
  w.dcol = round64(B);
  w.ldt = w.dcol + round64(2 * B);
  const size_t R = (size_t)3 * B;
  w.x_hi = ws_take<bf16>(p, R * H); w.x_lo = ws_take<bf16>(p, R * H); w.x_lo2 = ws_take<bf16>(p, R * H);
  w.xt_hi = ws_take<bf16>(p, (size_t)H * w.ldt); w.xt_lo = ws_take<bf16>(p, (size_t)H * w.ldt);
  w.h_hi = ws_take<bf16>(p, R * P); w.h_lo = ws_take<bf16>(p, R * P);
  w.ht_hi = ws_take<bf16>(p, (size_t)P * w.ldt); w.ht_lo = ws_take<bf16>(p, (size_t)P * w.ldt);
  w.dy_hi = ws_take<bf16>(p, R * P); w.dy_lo = ws_take<bf16>(p, R * P);
  w.dyt_hi = ws_take<bf16>(p, (size_t)P * w.ldt); w.dyt_lo = ws_take<bf16>(p, (size_t)P * w.ldt);
  w.dz_hi = ws_take<bf16>(p, R * P); w.dz_lo = ws_take<bf16>(p, R * P);
  w.dzt_hi = ws_take<bf16>(p, (size_t)P * w.ldt); w.dzt_lo = ws_take<bf16>(p, (size_t)P * w.ldt);
  for (int t = 0; t < 2; ++t) {
    w.w1_hi[t] = ws_take<bf16>(p, (size_t)P * H); w.w1_lo[t] = ws_take<bf16>(p, (size_t)P * H);
    w.w1_lo2[t] = ws_take<bf16>(p, (size_t)P * H);
    w.w1t_hi[t] = ws_take<bf16>(p, (size_t)P * H); w.w1t_lo[t] = ws_take<bf16>(p, (size_t)P * H);
    w.w2_hi[t] = ws_take<bf16>(p, (size_t)P * P); w.w2_lo[t] = ws_take<bf16>(p, (size_t)P * P);
    w.w2t_hi[t] = ws_take<bf16>(p, (size_t)P * P); w.w2t_lo[t] = ws_take<bf16>(p, (size_t)P * P);
  }
  w.dz1 = ws_take<float>(p, R * P);
  w.partial = ws_take<float>(p, (size_t)2 * 32 * P * max(P, H));
  w.partial2 = ws_take<float>(p, (size_t)2 * 32 * P * P);  // dW2's split-K sums: it runs beside the dW1 branch
  w.colsum = ws_take<float>(p, (size_t)2 * kColsumSlices * P);
  w.colsum2 = ws_take<float>(p, (size_t)2 * kColsumSlices * P);
  w.loss_scratch = ws_take<float>(p, (size_t)(B + 3) / 4 + 8);
  {
    const int RTB = (B + 127) / 128, NC = (P + 127) / 128;
    w.stat_part = ws_take<float>(p, (size_t)RTB * 2 * (P / 64 + 1) * 5 * 128);
    w.cs1 = ws_take<float>(p, (size_t)3 * RTB * P);
    w.cs2 = ws_take<float>(p, (size_t)3 * RTB * P);
    w.ybuf = ws_take<float>(p, (size_t)3 * RTB * 128 * P);  // layer-2 outputs exchanged between the q | p | n tasks
    w.hinge_part = ws_take<float>(p, (size_t)RTB + 8);
    w.n_counters = 10 * RTB + 8 + RTB * (P / 64 + 1);
    w.counters = ws_take<unsigned>(p, (size_t)w.n_counters);
    w.trace = ws_take<unsigned long long>(p, (size_t)kTraceCtas * kTraceSlots * 2);
  }
  (void)train_table;
  if (out) *out = w;
  return (size_t)(p - base) + 256;
}


}  // namespace tt

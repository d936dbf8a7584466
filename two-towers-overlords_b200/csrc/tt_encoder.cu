// The reference's ACTUAL backbone (SURVEY.md section 0, D1): the frozen 6-layer MiniLM BertModel that
// backend/model.py:24 loads and backend/model.py:51-52 runs under no_grad, forward only.  Its last hidden state feeds
// the same masked-mean pool kernel as the embedding-only backbone (the hidden states are pooled as a "table" indexed
// by token position).  Architecture = transformers' BertModel (absolute positions, post-LayerNorm, erf GELU):
//   embeddings  LN(word[id] + position[l] + token_type[0])
//   x 6         qkv = h Wqkv^T + b ; per head softmax(q k^T / sqrt(d) + key mask) v ; h = LN(ctx Wo^T + bo + h)
//               h = LN(gelu(h W1^T + b1) W2^T + b2 + h)
// The dense contractions run on the tcgen05 GEMM of tt_gemm_sm100.cu in split-bf16 arithmetic (weights are frozen,
// so their (hi, lo) terms are prepared once); LayerNorm, softmax attention and the embedding sum are fp32 CUDA-core
// kernels that emit the next contraction's operand terms directly.
#include <math.h>

#include "tt_sm100.cuh"

namespace tt {

namespace {

using bf16 = __nv_bfloat16;

// one warp per token; H = NV * 128, lane owns float4 k*32 + lane for k < NV
template <int NV>
__device__ __forceinline__ void layer_norm_row(float (&x)[NV * 4], const float* __restrict__ gamma,
                                               const float* __restrict__ beta, float eps, int lane, float* out,
                                               bf16* out_hi, bf16* out_lo) {
  constexpr int H = NV * 128;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV * 4; ++i) s += x[i];
  const float mean = warp_sum(s) * (1.f / H);
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < NV * 4; ++i) {
    const float d = x[i] - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = rsqrtf(warp_sum(v) * (1.f / H) + eps);  // biased variance, as torch.nn.LayerNorm
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int c = (k * 32 + lane) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    float y[4] = {(x[k * 4] - mean) * rstd * g.x + b.x, (x[k * 4 + 1] - mean) * rstd * g.y + b.y,
                  (x[k * 4 + 2] - mean) * rstd * g.z + b.z, (x[k * 4 + 3] - mean) * rstd * g.w + b.w};
    if (out) *reinterpret_cast<float4*>(out + c) = make_float4(y[0], y[1], y[2], y[3]);
    if (out_hi) {
      alignas(8) bf16 hi[4], lo[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) split_bf16(y[j], hi[j], lo[j]);
      *reinterpret_cast<uint2*>(out_hi + c) = *reinterpret_cast<const uint2*>(hi);
      *reinterpret_cast<uint2*>(out_lo + c) = *reinterpret_cast<const uint2*>(lo);
    }
  }
}

// h0 = LN(word[id] + position[l] + token_type[0])   (modeling_bert.BertEmbeddings; token_type_ids are all zero for
// single-sentence input, backend/model.py:43-45)
template <int NV>
__global__ void __launch_bounds__(128)
    embed_ln_kernel(const void* __restrict__ ids, int ids_dtype, int T, int L, int vocab, const float* __restrict__ word,
                    const float* __restrict__ pos, const float* __restrict__ type0, const float* __restrict__ gamma,
                    const float* __restrict__ beta, float eps, float* __restrict__ h, bf16* __restrict__ h_hi,
                    bf16* __restrict__ h_lo, int* __restrict__ err) {
  constexpr int H = NV * 128;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (t >= T) return;
  long long id = load_index(ids, ids_dtype, (size_t)t);
  if (id < 0 || id >= vocab) {
    if (err && lane == 0) *err = 1;
    id = 0;
  }
  const int l = t % L;
  float x[NV * 4];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int c = (k * 32 + lane) * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(word + (size_t)id * H + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(pos + (size_t)l * H + c));
    const float4 d = __ldg(reinterpret_cast<const float4*>(type0 + c));
    // same association as BertEmbeddings: (inputs_embeds + token_type_embeddings) + position_embeddings
    x[k * 4] = (a.x + d.x) + b.x; x[k * 4 + 1] = (a.y + d.y) + b.y;
    x[k * 4 + 2] = (a.z + d.z) + b.z; x[k * 4 + 3] = (a.w + d.w) + b.w;
  }
  layer_norm_row<NV>(x, gamma, beta, eps, lane, h + (size_t)t * H, h_hi + (size_t)t * H, h_lo + (size_t)t * H);
}

// out = LN(a + b)   (BertSelfOutput / BertOutput: dense output + residual)
template <int NV>
__global__ void __launch_bounds__(128)
    add_ln_kernel(const float* __restrict__ a, const float* __restrict__ b, int T, const float* __restrict__ gamma,
                  const float* __restrict__ beta, float eps, float* __restrict__ out, bf16* __restrict__ out_hi,
                  bf16* __restrict__ out_lo) {
  constexpr int H = NV * 128;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (t >= T) return;
  float x[NV * 4];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int c = (k * 32 + lane) * 4;
    const float4 u = *reinterpret_cast<const float4*>(a + (size_t)t * H + c);
    const float4 v = *reinterpret_cast<const float4*>(b + (size_t)t * H + c);
    x[k * 4] = u.x + v.x; x[k * 4 + 1] = u.y + v.y; x[k * 4 + 2] = u.z + v.z; x[k * 4 + 3] = u.w + v.w;
  }
  layer_norm_row<NV>(x, gamma, beta, eps, lane, out + (size_t)t * H, out_hi + (size_t)t * H, out_lo + (size_t)t * H);
}

// One CTA per (sequence, head): K and V of the head in shared memory, one query row per thread, streaming softmax in
// fp32.  Masked keys get weight exactly 0, as the additive finfo.min mask of BertSelfAttention does in fp32; a
// sequence without any unmasked key averages V over all positions (the softmax of equal scores).
template <int D>
__global__ void __launch_bounds__(128)
    attention_kernel(const float* __restrict__ qkv, const void* __restrict__ mask, int mask_dtype, int L, int H,
                     float scale, bf16* __restrict__ ctx_hi, bf16* __restrict__ ctx_lo) {
  extern __shared__ float sm[];
  float* Ks = sm;
  float* Vs = sm + (size_t)L * D;
  unsigned char* valid = reinterpret_cast<unsigned char*>(Vs + (size_t)L * D);
  __shared__ int s_any;
  const int b = blockIdx.x, hd = blockIdx.y, tid = threadIdx.x;
  const size_t row0 = (size_t)b * L, ld = (size_t)3 * H;
  if (tid == 0) s_any = 0;
  __syncthreads();
  for (int idx = tid; idx < L * D; idx += blockDim.x) {
    const int j = idx / D, d = idx - j * D;
    const float* src = qkv + (row0 + j) * ld + (size_t)hd * D + d;
    Ks[idx] = src[H];
    Vs[idx] = src[2 * H];
  }
  for (int j = tid; j < L; j += blockDim.x) {
    const unsigned char ok = load_index(mask, mask_dtype, row0 + j) != 0;
    valid[j] = ok;
    if (ok) s_any = 1;
  }
  __syncthreads();
  const bool any = s_any != 0;
  for (int i = tid; i < L; i += blockDim.x) {
    float q[D], acc[D];
    const float* qs = qkv + (row0 + i) * ld + (size_t)hd * D;
#pragma unroll
    for (int d = 0; d < D; d += 4) {
      const float4 t = *reinterpret_cast<const float4*>(qs + d);
      q[d] = t.x * scale; q[d + 1] = t.y * scale; q[d + 2] = t.z * scale; q[d + 3] = t.w * scale;
    }
#pragma unroll
    for (int d = 0; d < D; ++d) acc[d] = 0.f;
    float m = -INFINITY, l = 0.f;
    for (int j = 0; j < L; ++j) {
      if (any && !valid[j]) continue;  // CTA-uniform
      float s = 0.f;
      if (any) {
        const float4* kr = reinterpret_cast<const float4*>(Ks + (size_t)j * D);
#pragma unroll
        for (int d4 = 0; d4 < D / 4; ++d4) {
          const float4 t = kr[d4];
          s = fmaf(q[4 * d4], t.x, s); s = fmaf(q[4 * d4 + 1], t.y, s);
          s = fmaf(q[4 * d4 + 2], t.z, s); s = fmaf(q[4 * d4 + 3], t.w, s);
        }
      }
      if (s > m) {
        const float c = expf(m - s);  // exp(-inf) = 0 on the first key
        l *= c;
#pragma unroll
        for (int d = 0; d < D; ++d) acc[d] *= c;
        m = s;
      }
      const float pr = expf(s - m);
      l += pr;
      const float4* vr = reinterpret_cast<const float4*>(Vs + (size_t)j * D);
#pragma unroll
      for (int d4 = 0; d4 < D / 4; ++d4) {
        const float4 t = vr[d4];
        acc[4 * d4] = fmaf(pr, t.x, acc[4 * d4]); acc[4 * d4 + 1] = fmaf(pr, t.y, acc[4 * d4 + 1]);
        acc[4 * d4 + 2] = fmaf(pr, t.z, acc[4 * d4 + 2]); acc[4 * d4 + 3] = fmaf(pr, t.w, acc[4 * d4 + 3]);
      }
    }
    const float inv = 1.f / l;
    alignas(16) bf16 hi[D], lo[D];
#pragma unroll
    for (int d = 0; d < D; ++d) split_bf16(acc[d] * inv, hi[d], lo[d]);
    uint4* dh = reinterpret_cast<uint4*>(ctx_hi + (row0 + i) * H + (size_t)hd * D);
    uint4* dl = reinterpret_cast<uint4*>(ctx_lo + (row0 + i) * H + (size_t)hd * D);
#pragma unroll
    for (int v = 0; v < D / 8; ++v) {
      dh[v] = reinterpret_cast<const uint4*>(hi)[v];
      dl[v] = reinterpret_cast<const uint4*>(lo)[v];
    }
  }
}

struct EncWs {
  float *h, *h1, *tmp, *qkv;
  bf16 *h_hi, *h_lo, *h1_hi, *h1_lo, *ctx_hi, *ctx_lo, *ff_hi, *ff_lo;
};

size_t carve_enc(char* base, size_t T, int H, int I, EncWs* out) {
  char* p = base;
  EncWs w{};
  w.h = ws_take<float>(p, T * H); w.h1 = ws_take<float>(p, T * H); w.tmp = ws_take<float>(p, T * H);
  w.qkv = ws_take<float>(p, T * 3 * H);
  w.h_hi = ws_take<bf16>(p, T * H); w.h_lo = ws_take<bf16>(p, T * H);
  w.h1_hi = ws_take<bf16>(p, T * H); w.h1_lo = ws_take<bf16>(p, T * H);
  w.ctx_hi = ws_take<bf16>(p, T * H); w.ctx_lo = ws_take<bf16>(p, T * H);
  w.ff_hi = ws_take<bf16>(p, T * I); w.ff_lo = ws_take<bf16>(p, T * I);
  if (out) *out = w;
  return (size_t)(p - base) + 256;
}

// attention_kernel<32> keeps K and V of one head plus one mask byte per position in dynamic shared memory
size_t attention_smem(int L) { return (size_t)2 * L * 32 * sizeof(float) + L; }

// Dynamic shared memory attention_kernel<32> may use: the device's opt-in limit less the kernel's static shared
// memory (257 B per position: L <= 904 on a B200).  Opted into on the first call.
int attention_smem_limit(size_t* out) {
  static size_t limit = 0;
  if (!limit) {
    int dev = 0, optin = 0;
    TT_CUDA(cudaGetDevice(&dev));
    TT_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cudaFuncAttributes fa{};
    TT_CUDA(cudaFuncGetAttributes(&fa, attention_kernel<32>));
    const size_t lim = (size_t)optin - fa.sharedSizeBytes;
    TT_CUDA(cudaFuncSetAttribute(attention_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lim));
    limit = lim;
  }
  *out = limit;
  return 0;
}

template <int NV>
int encoder_fwd(const tt_encoder_weights* W, const void* ids, int ids_dtype, const void* mask, int mask_dtype, int B,
                int L, float* hidden_out, const EncWs& w, int* err, cudaStream_t st) {
  const int H = W->hidden, I = W->inter, T = B * L, D = H / W->heads;
  const int tb = (T + 3) / 4;
  // without layers the last hidden state is the embedding output, as in BertModel
  embed_ln_kernel<NV><<<tb, 128, 0, st>>>(ids, ids_dtype, T, L, W->vocab, W->word_emb, W->pos_emb, W->type_emb, W->emb_ln_g,
                                        W->emb_ln_b, W->ln_eps, W->n_layers ? w.h : hidden_out, w.h_hi, w.h_lo, err);
  TT_LAUNCH_CHECK();
  const size_t att_smem = attention_smem(L);
  int rc;
  for (int l = 0; l < W->n_layers; ++l) {
    const tt_encoder_layer& Y = W->layers[l];
    const bool last = l + 1 == W->n_layers;
    // self-attention block
    if ((rc = gemm_terms_sm100(w.h_hi, w.h_lo, H, reinterpret_cast<const bf16*>(Y.wqkv_hi),
                               reinterpret_cast<const bf16*>(Y.wqkv_lo), H, T, 3 * H, H, Y.bqkv, 0, w.qkv, 3 * H, nullptr,
                               nullptr, st)))
      return rc;
    attention_kernel<32><<<dim3(B, W->heads), 128, att_smem, st>>>(w.qkv, mask, mask_dtype, L, H, 1.f / sqrtf((float)D),
                                                               w.ctx_hi, w.ctx_lo);
    TT_LAUNCH_CHECK();
    if ((rc = gemm_terms_sm100(w.ctx_hi, w.ctx_lo, H, reinterpret_cast<const bf16*>(Y.wo_hi),
                               reinterpret_cast<const bf16*>(Y.wo_lo), H, T, H, H, Y.bo, 0, w.tmp, H, nullptr, nullptr, st)))
      return rc;
    add_ln_kernel<NV><<<tb, 128, 0, st>>>(w.tmp, w.h, T, Y.ln1_g, Y.ln1_b, W->ln_eps, w.h1, w.h1_hi, w.h1_lo);
    TT_LAUNCH_CHECK();
    // feed-forward block
    if ((rc = gemm_terms_sm100(w.h1_hi, w.h1_lo, H, reinterpret_cast<const bf16*>(Y.w1_hi),
                               reinterpret_cast<const bf16*>(Y.w1_lo), H, T, I, H, Y.b1, 2, nullptr, I, w.ff_hi, w.ff_lo, st)))
      return rc;
    if ((rc = gemm_terms_sm100(w.ff_hi, w.ff_lo, I, reinterpret_cast<const bf16*>(Y.w2_hi),
                               reinterpret_cast<const bf16*>(Y.w2_lo), I, T, H, I, Y.b2, 0, w.tmp, H, nullptr, nullptr, st)))
      return rc;
    add_ln_kernel<NV><<<tb, 128, 0, st>>>(w.tmp, w.h1, T, Y.ln2_g, Y.ln2_b, W->ln_eps, last ? hidden_out : w.h, w.h_hi,
                                        w.h_lo);
    TT_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace
}  // namespace tt

using namespace tt;

extern "C" size_t tt_encoder_ws_bytes(int tokens, int hidden, int inter) {
  return carve_enc(nullptr, (size_t)(tokens > 0 ? tokens : 0), hidden, inter, nullptr);
}

extern "C" int tt_split_bf16_terms(const float* x, int rows, int cols, void* hi, void* lo, tt_stream_t stream) {
  TT_REQUIRE(x && hi && lo && rows >= 1 && cols >= 1, "tt_split_bf16_terms: bad arguments");
  return split_terms_sm100(x, rows, cols, reinterpret_cast<bf16*>(hi), reinterpret_cast<bf16*>(lo), as_stream(stream));
}

extern "C" int tt_encoder_fwd(const tt_encoder_weights* w, const void* ids, int ids_dtype, const void* mask, int mask_dtype,
                              int B, int L, float* hidden_out, int* err_flag, void* ws, size_t ws_bytes,
                              tt_stream_t stream) {
  TT_REQUIRE(w && ids && mask && hidden_out, "tt_encoder_fwd: null argument");
  TT_REQUIRE(w->n_layers >= 0 && (w->n_layers == 0 || w->layers), "tt_encoder_fwd: bad layers (%d layers)", w->n_layers);
  TT_REQUIRE(B >= 0 && L >= 1 && L <= w->max_pos, "tt_encoder_fwd: bad shape B=%d L=%d (max positions %d)", B, L, w->max_pos);
  TT_REQUIRE(w->heads >= 1 && w->hidden >= 128 && w->hidden % 128 == 0 && w->hidden <= 768 &&
                 w->hidden / w->heads == 32 && w->inter >= 64 && w->inter % 64 == 0,
             "tt_encoder_fwd: supports hidden sizes 128..768 in steps of 128 with 32-wide heads and intermediate sizes "
             "in steps of 64 (hidden %d, heads %d, intermediate %d)",
             w->hidden, w->heads, w->inter);
  if (B == 0) return 0;
  TT_REQUIRE(ws_bytes >= tt_encoder_ws_bytes(B * L, w->hidden, w->inter), "tt_encoder_fwd: workspace too small");
  if (w->n_layers > 0) {
    size_t limit = 0;
    int rc = attention_smem_limit(&limit);
    if (rc) return rc;
    TT_REQUIRE(attention_smem(L) <= limit,
               "tt_encoder_fwd: sequence length L=%d needs %zu bytes of shared memory in attention, this device allows "
               "%zu (L <= %zu)", L, attention_smem(L), limit, limit / attention_smem(1));
  }
  EncWs e;
  carve_enc(reinterpret_cast<char*>(ws), (size_t)B * L, w->hidden, w->inter, &e);
  cudaStream_t st = as_stream(stream);
  switch (w->hidden / 128) {
    case 1: return encoder_fwd<1>(w, ids, ids_dtype, mask, mask_dtype, B, L, hidden_out, e, err_flag, st);
    case 2: return encoder_fwd<2>(w, ids, ids_dtype, mask, mask_dtype, B, L, hidden_out, e, err_flag, st);
    case 3: return encoder_fwd<3>(w, ids, ids_dtype, mask, mask_dtype, B, L, hidden_out, e, err_flag, st);
    case 4: return encoder_fwd<4>(w, ids, ids_dtype, mask, mask_dtype, B, L, hidden_out, e, err_flag, st);
    case 5: return encoder_fwd<5>(w, ids, ids_dtype, mask, mask_dtype, B, L, hidden_out, e, err_flag, st);
    case 6: return encoder_fwd<6>(w, ids, ids_dtype, mask, mask_dtype, B, L, hidden_out, e, err_flag, st);
    default: TT_REQUIRE(false, "tt_encoder_fwd: hidden size %d not supported", w->hidden);
  }
  return 0;
}

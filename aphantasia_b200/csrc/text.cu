// text.cu -- CLIP text encoder handle (forward only): fp32 token table, packed bf16 layer weights, activation buffers.
//
// Restates OpenAI clip/model.py CLIP.encode_text (third-party, SURVEY.md A5):
//   x = token_embedding[ids] + positional_embedding -> layers x { x += out_proj(causal MHA(ln_1 x)); x += c_proj(QuickGELU(c_fc(ln_2 x))) }
//   -> ln_final(x[s, argmax_t ids[s, t]]) @ text_projection
// Built from the image encoder's pieces: the tcgen05 GEMM with its fused epilogues (tc_gemm.cuh), the one-warp-per-row
// LayerNorm (ln_rows.cuh) and the mma.sync attention with a causal mask (vit_attn_tc.cuh, instantiated in vit.cu). It runs
// once per prompt before the optimisation loop, so there is no graph cache and no backward (no transposed weight copies).
#include "ln_rows.cuh"
#include <limits.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <string>
#include <vector>

namespace aph {

int pack(const float* src, bf16* dst, int rows, int cols, int transpose, cudaStream_t st);                  // vit.cu
int attn_fwd_causal(const bf16* qkv, bf16* out, int S, int T, int D, int heads, cudaStream_t st);          // vit.cu

struct TextLayerW {
  float *ln1_w = nullptr, *ln1_b = nullptr, *ln2_w = nullptr, *ln2_b = nullptr;
  float *b_qkv = nullptr, *b_o = nullptr, *b_fc = nullptr, *b_proj = nullptr;
  bf16 *w_qkv = nullptr, *w_o = nullptr, *w_fc = nullptr, *w_proj = nullptr;   // [3D, D], [D, D], [4D, D], [D, 4D]
};

struct TextImpl {
  aph_text_config cfg;
  int D;
  int64_t bytes = 0;
  std::vector<void*> allocs;
  // weights
  float* tok = nullptr;          // token_embedding [vocab, D] fp32 (rows are gathered, never a GEMM operand)
  float* pos = nullptr;          // [ctx, D]
  float *lnf_w = nullptr, *lnf_b = nullptr;
  bf16* w_out = nullptr;         // text_projection^T [out, D]
  std::vector<TextLayerW> L;
  std::map<std::string, bool> loaded;
  bool finalized = false;
  // activations (sized for max_batch * ctx rows)
  float *xa = nullptr, *xb = nullptr;          // residual stream [M, D]: a -> (attention) b -> (MLP) a
  bf16* ln_out = nullptr;        // [M, D]
  bf16* qkv = nullptr;           // [M, 3D]
  bf16* attn_out = nullptr;      // [M, D]
  bf16* h_pre = nullptr;         // [M, 4D] pre-activation the bias+QuickGELU epilogue writes (not needed later: reused)
  bf16* h_act = nullptr;         // [M, 4D]
  float *mean = nullptr, *rstd = nullptr;      // [M] (k_ln_fwd writes them; unused without a backward)
  bf16* eot_ln = nullptr;        // [max_batch, D]
};

template <typename Tp>
static int text_alloc(TextImpl* t, Tp** p, size_t count) {
  void* q = nullptr;
  APH_CUDA_OK(cudaMalloc(&q, count * sizeof(Tp)));
  t->allocs.push_back(q);
  t->bytes += (int64_t)(count * sizeof(Tp));
  *p = reinterpret_cast<Tp*>(q);
  return 0;
}

// x[row] = token_embedding[ids[row]] + positional_embedding[row % ctx], one warp per row. An id outside [0, vocab)
// contributes a zero row instead of reading outside the table (the Python layer rejects such ids before the call).
template <int NCH>
__global__ void __launch_bounds__(256) k_text_embed(const int64_t* __restrict__ ids, const float* __restrict__ table,
                                                    const float* __restrict__ pos, float* __restrict__ x, int rows, int ctx,
                                                    int vocab, int D) {
  pdl_trigger(); pdl_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= rows) return;
  constexpr int N = 4 * NCH;
  const int64_t id = ids[row];
  float v[N], pz[N];
  load_row(pos + (size_t)(row % ctx) * D, pz, lane);
  if (id >= 0 && id < vocab) {
    load_row(table + (size_t)id * D, v, lane);
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] += pz[i];
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = pz[i];
  }
  store_row_f32(x + (size_t)row * D, v, lane);
}

// EOT pooling fused with ln_final: per sample (one warp) the position of the first maximum id (torch.argmax: the
// end-of-text token has the largest id of the vocabulary), and y[s] = LN(x[s*ctx + that position]) as bf16.
template <int NCH>
__global__ void __launch_bounds__(256) k_text_eot_ln(const int64_t* __restrict__ ids, const float* __restrict__ x,
                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     bf16* __restrict__ y, int n, int ctx, int D) {
  pdl_trigger(); pdl_wait();
  const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (s >= n) return;
  constexpr int N = 4 * NCH;
  long long best = LLONG_MIN;
  int at = INT_MAX;
  for (int t = lane; t < ctx; t += 32) {                 // ascending t: a strict '>' keeps this lane's first maximum
    const long long v = ids[(size_t)s * ctx + t];
    if (v > best) { best = v; at = t; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const long long ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oa = __shfl_xor_sync(0xffffffffu, at, o);
    if (ob > best || (ob == best && oa < at)) { best = ob; at = oa; }
  }
  float v[N], gm[N], bt[N];
  load_row(x + ((size_t)s * ctx + at) * D, v, lane);
  const RowStats st = row_stats(v, D);
  load_row(gamma, gm, lane); load_row(beta, bt, lane);
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = (v[i] - st.mean) * st.rstd * gm[i] + bt[i];
  store_row_bf16(y + (size_t)s * D, v, lane);
}

}  // namespace aph

using namespace aph;

extern "C" int aph_text_destroy(aph_text* text) {
  if (!text) return 0;
  TextImpl* t = reinterpret_cast<TextImpl*>(text);
  for (void* p : t->allocs) cudaFree(p);
  delete t;
  return 0;
}

extern "C" int aph_text_create(aph_text** out, const aph_text_config* cfg) {
  APH_REQUIRE(out && cfg, "aph_text_create: null argument");
  APH_REQUIRE(cfg->width == 256 || cfg->width == 512 || cfg->width == 768, "aph_text_create: width %d unsupported (256, 512, 768)", cfg->width);
  APH_REQUIRE(cfg->heads * 64 == cfg->width, "aph_text_create: head dim must be 64 (width %d, heads %d)", cfg->width, cfg->heads);
  APH_REQUIRE(cfg->ctx > 0 && cfg->ctx <= 112, "aph_text_create: context length %d outside (0, 112]", cfg->ctx);
  APH_REQUIRE(cfg->vocab > 0 && cfg->layers > 0 && cfg->max_batch > 0, "aph_text_create: vocab %d, layers %d, max_batch %d must be positive",
              cfg->vocab, cfg->layers, cfg->max_batch);
  APH_REQUIRE(cfg->out_dim > 0 && cfg->out_dim % 128 == 0, "aph_text_create: out_dim %d must be a multiple of 128", cfg->out_dim);
  TextImpl* t = new TextImpl();
  t->cfg = *cfg;
  t->D = cfg->width;
  const int D = t->D, O = cfg->out_dim;
  const size_t M = (size_t)cfg->max_batch * cfg->ctx;
  int e = 0;
  e |= text_alloc(t, &t->tok, (size_t)cfg->vocab * D); e |= text_alloc(t, &t->pos, (size_t)cfg->ctx * D);
  e |= text_alloc(t, &t->lnf_w, D); e |= text_alloc(t, &t->lnf_b, D); e |= text_alloc(t, &t->w_out, (size_t)O * D);
  t->L.resize(cfg->layers);
  for (auto& l : t->L) {
    e |= text_alloc(t, &l.ln1_w, D); e |= text_alloc(t, &l.ln1_b, D); e |= text_alloc(t, &l.ln2_w, D); e |= text_alloc(t, &l.ln2_b, D);
    e |= text_alloc(t, &l.b_qkv, 3 * D); e |= text_alloc(t, &l.b_o, D); e |= text_alloc(t, &l.b_fc, 4 * D); e |= text_alloc(t, &l.b_proj, D);
    e |= text_alloc(t, &l.w_qkv, (size_t)3 * D * D); e |= text_alloc(t, &l.w_o, (size_t)D * D);
    e |= text_alloc(t, &l.w_fc, (size_t)4 * D * D); e |= text_alloc(t, &l.w_proj, (size_t)4 * D * D);
  }
  e |= text_alloc(t, &t->xa, M * D); e |= text_alloc(t, &t->xb, M * D); e |= text_alloc(t, &t->ln_out, M * D);
  e |= text_alloc(t, &t->qkv, M * 3 * D); e |= text_alloc(t, &t->attn_out, M * D);
  e |= text_alloc(t, &t->h_pre, M * 4 * D); e |= text_alloc(t, &t->h_act, M * 4 * D);
  e |= text_alloc(t, &t->mean, M); e |= text_alloc(t, &t->rstd, M);
  e |= text_alloc(t, &t->eot_ln, (size_t)cfg->max_batch * D);
  if (e) { aph_text_destroy(reinterpret_cast<aph_text*>(t)); return 1; }
  *out = reinterpret_cast<aph_text*>(t);
  return 0;
}

extern "C" int64_t aph_text_bytes(const aph_text* text) { return text ? reinterpret_cast<const TextImpl*>(text)->bytes : 0; }

extern "C" int aph_text_load_tensor(aph_text* text, const char* key, const float* data, int64_t numel, void* stream) {
  APH_REQUIRE(text && key && data, "aph_text_load_tensor: null argument");
  TextImpl* t = reinterpret_cast<TextImpl*>(text);
  cudaStream_t st = (cudaStream_t)stream;
  const int D = t->D, O = t->cfg.out_dim;
  const std::string k(key);
  auto need = [&](int64_t n) -> int { APH_REQUIRE(numel == n, "aph_text_load_tensor(%s): expected %lld elements, got %lld", key, (long long)n, (long long)numel); return 0; };
  auto copy = [&](float* dst, int64_t n) -> int {
    if (int e = need(n)) return e;
    APH_CUDA_OK(cudaMemcpyAsync(dst, data, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  auto packw = [&](bf16* dst, int rows, int cols, int transpose) -> int {
    if (int e = need((int64_t)rows * cols)) return e;
    return pack(data, dst, rows, cols, transpose, st);
  };
  int e = 0;
  if (k == "token_embedding.weight") e = copy(t->tok, (int64_t)t->cfg.vocab * D);
  else if (k == "positional_embedding") e = copy(t->pos, (int64_t)t->cfg.ctx * D);
  else if (k == "ln_final.weight") e = copy(t->lnf_w, D);
  else if (k == "ln_final.bias") e = copy(t->lnf_b, D);
  else if (k == "text_projection") e = packw(t->w_out, D, O, 1);        // [D, out] -> forward B operand [out, D]
  else if (k.rfind("transformer.resblocks.", 0) == 0) {
    const char* rest = k.c_str() + strlen("transformer.resblocks.");
    char* endp = nullptr;
    const long li = strtol(rest, &endp, 10);
    APH_REQUIRE(endp && endp != rest && *endp == '.' && li >= 0 && li < t->cfg.layers, "aph_text_load_tensor: bad layer index in %s", key);
    TextLayerW& l = t->L[li];
    const std::string f(endp + 1);
    if (f == "ln_1.weight") e = copy(l.ln1_w, D);
    else if (f == "ln_1.bias") e = copy(l.ln1_b, D);
    else if (f == "ln_2.weight") e = copy(l.ln2_w, D);
    else if (f == "ln_2.bias") e = copy(l.ln2_b, D);
    else if (f == "attn.in_proj_weight") e = packw(l.w_qkv, 3 * D, D, 0);
    else if (f == "attn.in_proj_bias") e = copy(l.b_qkv, 3 * D);
    else if (f == "attn.out_proj.weight") e = packw(l.w_o, D, D, 0);
    else if (f == "attn.out_proj.bias") e = copy(l.b_o, D);
    else if (f == "mlp.c_fc.weight") e = packw(l.w_fc, 4 * D, D, 0);
    else if (f == "mlp.c_fc.bias") e = copy(l.b_fc, 4 * D);
    else if (f == "mlp.c_proj.weight") e = packw(l.w_proj, D, 4 * D, 0);
    else if (f == "mlp.c_proj.bias") e = copy(l.b_proj, D);
    else { set_error("aph_text_load_tensor: unknown tensor %s", key); return 2; }
  } else { set_error("aph_text_load_tensor: unknown tensor %s", key); return 2; }
  if (e) return e;
  t->loaded[k] = true;
  return 0;
}

extern "C" int aph_text_finalize(aph_text* text) {
  APH_REQUIRE(text, "aph_text_finalize: null handle");
  TextImpl* t = reinterpret_cast<TextImpl*>(text);
  std::vector<std::string> want = {"token_embedding.weight", "positional_embedding", "ln_final.weight", "ln_final.bias", "text_projection"};
  const char* per[] = {"ln_1.weight", "ln_1.bias", "ln_2.weight", "ln_2.bias", "attn.in_proj_weight", "attn.in_proj_bias",
                       "attn.out_proj.weight", "attn.out_proj.bias", "mlp.c_fc.weight", "mlp.c_fc.bias", "mlp.c_proj.weight", "mlp.c_proj.bias"};
  for (int i = 0; i < t->cfg.layers; ++i)
    for (const char* p : per) want.push_back("transformer.resblocks." + std::to_string(i) + "." + p);
  for (const auto& w : want) APH_REQUIRE(t->loaded.count(w), "aph_text_finalize: tensor %s was never loaded", w.c_str());
  t->finalized = true;
  return 0;
}

extern "C" int aph_text_fwd(aph_text* text, const int64_t* tokens, int n, float* emb, void* stream) {
  APH_REQUIRE(text && tokens && emb, "aph_text_fwd: null argument");
  TextImpl* t = reinterpret_cast<TextImpl*>(text);
  APH_REQUIRE(t->finalized, "aph_text_fwd: weights not finalized");
  APH_REQUIRE(n > 0 && n <= t->cfg.max_batch, "aph_text_fwd: n=%d outside (0, max_batch=%d]", n, t->cfg.max_batch);
  cudaStream_t st = (cudaStream_t)stream;
  const int D = t->D, T = t->cfg.ctx, H = t->cfg.heads, O = t->cfg.out_dim, M = n * T;
  int e;
  NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_text_embed<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, tokens, t->tok, t->pos, t->xa,
                                       M, T, t->cfg.vocab, D)));
  APH_LAUNCH_OK();
  for (const TextLayerW& w : t->L) {
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_fwd<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, t->xa, (size_t)D, w.ln1_w, w.ln1_b, t->ln_out,
                                         t->mean, t->rstd, M, D)));
    APH_LAUNCH_OK();
    { GemmEpi ep; ep.bias = w.b_qkv; ep.out_bf16 = t->qkv;
      if ((e = launch_gemm(t->ln_out, w.w_qkv, GemmShape{M, 3 * D, D}, ep, st))) return e; }
    if ((e = attn_fwd_causal(t->qkv, t->attn_out, n, T, D, H, st))) return e;
    { GemmEpi ep; ep.bias = w.b_o; ep.resid = t->xa; ep.out_f32 = t->xb;
      if ((e = launch_gemm(t->attn_out, w.w_o, GemmShape{M, D, D}, ep, st))) return e; }
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_fwd<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, t->xb, (size_t)D, w.ln2_w, w.ln2_b, t->ln_out,
                                         t->mean, t->rstd, M, D)));
    APH_LAUNCH_OK();
    { GemmEpi ep; ep.bias = w.b_fc; ep.out_pre = t->h_pre; ep.act = 1; ep.out_bf16 = t->h_act;
      if ((e = launch_gemm(t->ln_out, w.w_fc, GemmShape{M, 4 * D, D}, ep, st))) return e; }
    { GemmEpi ep; ep.bias = w.b_proj; ep.resid = t->xb; ep.out_f32 = t->xa;
      if ((e = launch_gemm(t->h_act, w.w_proj, GemmShape{M, D, 4 * D}, ep, st))) return e; }
  }
  NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_text_eot_ln<NCH>, dim3(rows_grid(n)), dim3(256), (size_t)0, st, 1, tokens, t->xa, t->lnf_w, t->lnf_b,
                                       t->eot_ln, n, T, D)));
  APH_LAUNCH_OK();
  GemmEpi ep; ep.out_f32 = emb;
  return launch_gemm(t->eot_ln, t->w_out, GemmShape{n, O, D}, ep, st);
}

// vit.cu -- CLIP ViT-B image encoder handle: packed bf16 weights, activation arena, forward and
// data-gradient backward built from the tcgen05 GEMM (tc_gemm.cuh) and the kernels of vit_ops.cuh.
//
// Restates OpenAI clip/model.py VisionTransformer.forward (third-party, SURVEY.md A5):
//   conv1 (patch-embed GEMM) -> [cls; tok] + pos -> ln_pre -> 12 x { x += out_proj(MHA(ln_1 x)); x += c_proj(QuickGELU(c_fc(ln_2 x))) }
//   -> ln_post(x[:,0]) @ proj
// The residual stream is fp32; GEMM operands are bf16; every x_l is kept (out-of-place residual) so the
// LayerNorm backward can recompute x-hat. No weight gradients (the reference computes and discards them).
#include "vit_ops.cuh"
#include "vit_attn_tc.cuh"
#include "vit_attn_umma.cuh"
#include <stdlib.h>
#include <string>
#include <vector>
#include <map>
#include <string.h>

namespace aph {

struct LayerW {
  float *ln1_w = nullptr, *ln1_b = nullptr, *ln2_w = nullptr, *ln2_b = nullptr;
  float *b_qkv = nullptr, *b_o = nullptr, *b_fc = nullptr, *b_proj = nullptr;
  bf16 *w_qkv = nullptr, *w_qkv_t = nullptr;     // [3D, D], [D, 3D]
  bf16 *w_o = nullptr, *w_o_t = nullptr;         // [D, D]
  bf16 *w_fc = nullptr, *w_fc_t = nullptr;       // [4D, D], [D, 4D]
  bf16 *w_proj = nullptr, *w_proj_t = nullptr;   // [D, 4D], [4D, D]
};

struct VitImpl {
  aph_vit_config cfg;
  int g, T, D, Kp;
  int64_t bytes = 0;
  std::vector<void*> allocs;
  // weights
  bf16 *w_conv = nullptr, *w_conv_t = nullptr;   // [D, Kp], [Kp, D]
  float *cls = nullptr, *pos = nullptr, *lnpre_w = nullptr, *lnpre_b = nullptr, *lnpost_w = nullptr, *lnpost_b = nullptr;
  bf16 *w_out = nullptr, *w_out_t = nullptr;     // proj^T [out, D] (forward B operand), proj [D, out] (dgrad B operand)
  std::vector<LayerW> L;
  std::map<std::string, bool> loaded;
  bool finalized = false;
  // activations (sized for max_batch)
  bf16* patches = nullptr;       // [S*g*g, Kp]
  float* tok = nullptr;          // [S*g*g, D]
  float* e = nullptr;            // [M, D] pre-ln_pre
  std::vector<float*> xs;        // 2*layers+1 residual-stream snapshots, fp32 [M, D]
  bf16* ln_out = nullptr;        // [M, D]
  std::vector<bf16*> qkv;        // per layer [M, 3D]
  bf16* attn_out = nullptr;      // [M, D]
  std::vector<bf16*> h_pre;      // per layer [M, 4D]
  bf16* h_act = nullptr;         // [M, 4D]
  float *st_mean = nullptr, *st_rstd = nullptr;   // [(2*layers+2)][M]
  bf16* cls_ln = nullptr;        // [S, D]
  float* emb_int = nullptr;      // [S, out] (copied to the caller's buffer outside the graph)
  // backward scratch
  bf16* d_emb = nullptr;         // [S, out]
  float* d_cls = nullptr;        // [S, D]
  float* dx = nullptr;           // [M, D]
  bf16* dx_bf = nullptr;         // [M, D]
  bf16* dh = nullptr;            // [M, 4D]
  bf16* d_ln = nullptr;          // [M, D] gradient entering a LayerNorm backward (bf16: it is the output of a bf16-operand GEMM and is consumed once)
  bf16* d_attn = nullptr;        // [M, D]
  bf16* d_qkv = nullptr;         // [M, 3D]
  bf16* d_tok = nullptr;         // [S*g*g, D]
  int last_S = -1;
  // CUDA-graph cache: the ~90 launches of a forward (or backward) are replayed as one graph when the call repeats with the
  // same batch size and the same input/output pointers (the optimisation loop does); keyed, small LRU
  struct GraphEntry { const void* in; const void* out; int S; int flag; cudaGraphExec_t exec; unsigned long long stamp; int nodes; };
  std::vector<GraphEntry> fwd_graphs, bwd_graphs;
  std::map<int, int> warm_fwd, warm_bwd;
  unsigned long long stamp = 0;
  int graph_misses = 0;          // captures in a row that were never replayed (e.g. the caller re-allocates its tensors every step)
};

bool gemm_profiling_on();      // vit_gemm.cu

static bool graphs_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("APH_VIT_GRAPH"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1 && !gemm_profiling_on();
}

// Runs `body` through the graph cache: 1st call with a key runs eagerly (lazy one-time initialisations are not capturable),
// 2nd call captures + instantiates, later calls replay.
template <typename Body>
static int run_cached(std::vector<VitImpl::GraphEntry>& cache, std::map<int, int>& warm, unsigned long long& stamp, int& misses,
                      const void* in, const void* out, int S, int flag, cudaStream_t& st, Body body) {
  // a caller whose buffers move every step (clip_fft.py calls torch.cuda.empty_cache() per step) would re-capture forever:
  // after 6 never-replayed captures in a row the handle stays eager
  if (!graphs_enabled() || misses > 6) return body();
  for (auto& g : cache)
    if (g.in == in && g.out == out && g.S == S && g.flag == flag) {
      g.stamp = ++stamp;
      misses = 0;
      APH_CUDA_OK(cudaGraphLaunch(g.exec, st));
      count_launch(g.nodes);           // kernels replayed by the graph
      return 0;
    }
  if (!warm[S]) { warm[S] = 1; return body(); }
  // The caller's stream is often the legacy default stream (torch's default), which cannot be captured: record the launch
  // sequence on a private stream (`st` is what the body launches on -- capture enqueues nothing), replay on the caller's.
  static cudaStream_t cap = nullptr;
  if (!cap) APH_CUDA_OK(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
  cudaStream_t user = st;
  st = cap;
  if (cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); st = user; return body(); }
  const int rc = body();
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(cap, &graph);
  st = user;
  if (rc != 0 || ce != cudaSuccess || graph == nullptr) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    if (rc != 0) return rc;
    return body();                                                 // capture refused: stay eager
  }
  size_t nodes = 0;
  cudaGraphGetNodes(graph, nullptr, &nodes);
  g_launches.fetch_sub((long long)nodes, std::memory_order_relaxed);   // the capture pass enqueued nothing; the replay below counts
  cudaGraphExec_t exec = nullptr;
  if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { cudaGraphDestroy(graph); cudaGetLastError(); return body(); }
  cudaGraphDestroy(graph);
  if (cache.size() >= 4) {                                         // evict the least recently used
    size_t lru = 0;
    for (size_t i = 1; i < cache.size(); ++i) if (cache[i].stamp < cache[lru].stamp) lru = i;
    cudaGraphExecDestroy(cache[lru].exec);
    cache.erase(cache.begin() + lru);
  }
  ++misses;
  cache.push_back({in, out, S, flag, exec, ++stamp, (int)nodes});
  APH_CUDA_OK(cudaGraphLaunch(exec, st));
  count_launch((int)nodes);
  return 0;
}

template <typename Tp>
static int dev_alloc(VitImpl* v, Tp** p, size_t count) {
  void* q = nullptr;
  APH_CUDA_OK(cudaMalloc(&q, count * sizeof(Tp)));
  v->allocs.push_back(q);
  v->bytes += (int64_t)(count * sizeof(Tp));
  *p = reinterpret_cast<Tp*>(q);
  return 0;
}

// fp32 [rows, cols] -> bf16 [rows, cols] (transpose = 0) or bf16 [cols, rows] (transpose = 1)
__global__ void __launch_bounds__(256) k_pack_weight(const float* __restrict__ in, bf16* __restrict__ out, int rows, int cols, int transpose) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i - (size_t)r * cols);
    const bf16 v = __float2bfloat16_rn(in[i]);
    if (transpose) out[(size_t)c * rows + r] = v; else out[i] = v;
  }
}

int pack(const float* src, bf16* dst, int rows, int cols, int transpose, cudaStream_t st) {     // also text.cu
  const size_t n = (size_t)rows * cols;
  const int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)kNumSMs * 16);
  k_pack_weight<<<blocks, 256, 0, st>>>(src, dst, rows, cols, transpose);
  APH_LAUNCH_OK();
  return 0;
}

static int copy_f32(const float* src, float* dst, size_t n, cudaStream_t st) {
  APH_CUDA_OK(cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

// APH_ATTN_SIMT=1 selects the fp32 SIMT attention kernels (debug / comparison); default = tensor-core kernels.
static bool attn_simt() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("APH_ATTN_SIMT"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

// APH_ATTN_UMMA=0 falls back to the mma.sync forward for T <= 64 (default: the tcgen05 / TMEM kernel of vit_attn_umma.cuh)
static bool attn_umma() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("APH_ATTN_UMMA"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// Causal self-attention of the CLIP text tower (text.cu): the mma.sync forward with keys j > i masked, one CTA per
// (sample, head), T = context length <= 112.
int attn_fwd_causal(const bf16* qkv, bf16* out, int S, int T, int D, int heads, cudaStream_t st) {
  APH_REQUIRE(T > 0 && T <= 112, "causal attention: T=%d outside (0, 112]", T);
  constexpr size_t smem = attn_tc_fwd_smem<8, 7>();
  static bool cfg = false;
  if (!cfg) {
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_fwd_tc<8, 7, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cfg = true;
  }
  APH_CUDA_OK(launch_k(k_attn_fwd_tc<8, 7, true>, dim3(S * heads), dim3(8 * 32), smem, st, 1, qkv, out, T, D, heads));
  APH_LAUNCH_OK();
  return 0;
}

}  // namespace aph

using namespace aph;

extern "C" int aph_vit_create(aph_vit** out, const aph_vit_config* cfg) {
  APH_REQUIRE(out && cfg, "aph_vit_create: null argument");
  APH_REQUIRE(cfg->width % 128 == 0 && (cfg->width / 128 == 1 || cfg->width / 128 == 2 || cfg->width / 128 == 6 || cfg->width / 128 == 8),
              "aph_vit_create: width %d unsupported (128, 256, 768, 1024)", cfg->width);
  APH_REQUIRE(cfg->heads * 64 == cfg->width, "aph_vit_create: head dim must be 64 (width %d, heads %d)", cfg->width, cfg->heads);
  APH_REQUIRE(cfg->res % cfg->patch == 0 && cfg->patch % 8 == 0, "aph_vit_create: res %d / patch %d", cfg->res, cfg->patch);
  APH_REQUIRE(cfg->out_dim % 128 == 0 && cfg->max_batch > 0 && cfg->layers > 0, "aph_vit_create: out_dim %d must be a multiple of 128", cfg->out_dim);
  VitImpl* v = new VitImpl();
  v->cfg = *cfg;
  v->g = cfg->res / cfg->patch; v->T = v->g * v->g + 1; v->D = cfg->width; v->Kp = 3 * cfg->patch * cfg->patch;
  APH_REQUIRE(v->T <= 256 && v->Kp % 128 == 0, "aph_vit_create: T=%d (max 256) Kp=%d", v->T, v->Kp);
  const int D = v->D, T = v->T, S = cfg->max_batch, Ly = cfg->layers, O = cfg->out_dim;
  const size_t M = (size_t)S * T, Mp = (size_t)S * v->g * v->g;
  int e = 0;
  // weights
  e |= dev_alloc(v, &v->w_conv, (size_t)D * v->Kp); e |= dev_alloc(v, &v->w_conv_t, (size_t)D * v->Kp);
  e |= dev_alloc(v, &v->cls, D); e |= dev_alloc(v, &v->pos, (size_t)T * D);
  e |= dev_alloc(v, &v->lnpre_w, D); e |= dev_alloc(v, &v->lnpre_b, D); e |= dev_alloc(v, &v->lnpost_w, D); e |= dev_alloc(v, &v->lnpost_b, D);
  e |= dev_alloc(v, &v->w_out, (size_t)D * O); e |= dev_alloc(v, &v->w_out_t, (size_t)D * O);
  v->L.resize(Ly);
  for (auto& l : v->L) {
    e |= dev_alloc(v, &l.ln1_w, D); e |= dev_alloc(v, &l.ln1_b, D); e |= dev_alloc(v, &l.ln2_w, D); e |= dev_alloc(v, &l.ln2_b, D);
    e |= dev_alloc(v, &l.b_qkv, 3 * D); e |= dev_alloc(v, &l.b_o, D); e |= dev_alloc(v, &l.b_fc, 4 * D); e |= dev_alloc(v, &l.b_proj, D);
    e |= dev_alloc(v, &l.w_qkv, (size_t)3 * D * D); e |= dev_alloc(v, &l.w_qkv_t, (size_t)3 * D * D);
    e |= dev_alloc(v, &l.w_o, (size_t)D * D); e |= dev_alloc(v, &l.w_o_t, (size_t)D * D);
    e |= dev_alloc(v, &l.w_fc, (size_t)4 * D * D); e |= dev_alloc(v, &l.w_fc_t, (size_t)4 * D * D);
    e |= dev_alloc(v, &l.w_proj, (size_t)4 * D * D); e |= dev_alloc(v, &l.w_proj_t, (size_t)4 * D * D);
  }
  // activations
  e |= dev_alloc(v, &v->patches, Mp * v->Kp); e |= dev_alloc(v, &v->tok, Mp * D); e |= dev_alloc(v, &v->e, M * D);
  v->xs.resize(2 * Ly + 1); for (auto& x : v->xs) e |= dev_alloc(v, &x, M * D);
  e |= dev_alloc(v, &v->ln_out, M * D); e |= dev_alloc(v, &v->attn_out, M * D); e |= dev_alloc(v, &v->h_act, M * 4 * D);
  v->qkv.resize(Ly); v->h_pre.resize(Ly);
  for (int i = 0; i < Ly; ++i) { e |= dev_alloc(v, &v->qkv[i], M * 3 * D); e |= dev_alloc(v, &v->h_pre[i], M * 4 * D); }
  e |= dev_alloc(v, &v->st_mean, (size_t)(2 * Ly + 2) * M); e |= dev_alloc(v, &v->st_rstd, (size_t)(2 * Ly + 2) * M);
  e |= dev_alloc(v, &v->cls_ln, (size_t)S * D); e |= dev_alloc(v, &v->emb_int, (size_t)S * O);
  e |= dev_alloc(v, &v->d_emb, (size_t)S * O); e |= dev_alloc(v, &v->d_cls, (size_t)S * D);
  e |= dev_alloc(v, &v->dx, M * D); e |= dev_alloc(v, &v->dx_bf, M * D); e |= dev_alloc(v, &v->dh, M * 4 * D);
  e |= dev_alloc(v, &v->d_ln, M * D); e |= dev_alloc(v, &v->d_attn, M * D); e |= dev_alloc(v, &v->d_qkv, M * 3 * D);
  e |= dev_alloc(v, &v->d_tok, Mp * D);
  if (e) { aph_vit_destroy(reinterpret_cast<aph_vit*>(v)); return 1; }
  APH_CUDA_OK(cudaFuncSetAttribute(k_attn_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_fwd_smem(T)));
  APH_CUDA_OK(cudaFuncSetAttribute(k_attn_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_bwd_smem(T)));
  *out = reinterpret_cast<aph_vit*>(v);
  return 0;
}

extern "C" int aph_vit_destroy(aph_vit* vit) {
  if (!vit) return 0;
  VitImpl* v = reinterpret_cast<VitImpl*>(vit);
  for (auto& g : v->fwd_graphs) cudaGraphExecDestroy(g.exec);
  for (auto& g : v->bwd_graphs) cudaGraphExecDestroy(g.exec);
  for (void* p : v->allocs) cudaFree(p);
  delete v;
  return 0;
}

extern "C" int64_t aph_vit_bytes(const aph_vit* vit) { return vit ? reinterpret_cast<const VitImpl*>(vit)->bytes : 0; }

extern "C" int aph_vit_load_tensor(aph_vit* vit, const char* key, const float* data, int64_t numel, void* stream) {
  APH_REQUIRE(vit && key && data, "aph_vit_load_tensor: null argument");
  VitImpl* v = reinterpret_cast<VitImpl*>(vit);
  cudaStream_t st = (cudaStream_t)stream;
  const int D = v->D, O = v->cfg.out_dim;
  std::string k(key);
  if (k.rfind("visual.", 0) == 0) k = k.substr(7);
  auto need = [&](int64_t n) -> int { APH_REQUIRE(numel == n, "aph_vit_load_tensor(%s): expected %lld elements, got %lld", key, (long long)n, (long long)numel); return 0; };
  int e = 0;
  if (k == "conv1.weight") { if ((e = need((int64_t)D * v->Kp))) return e; e = pack(data, v->w_conv, D, v->Kp, 0, st) | pack(data, v->w_conv_t, D, v->Kp, 1, st); }
  else if (k == "class_embedding") { if ((e = need(D))) return e; e = copy_f32(data, v->cls, D, st); }
  else if (k == "positional_embedding") { if ((e = need((int64_t)v->T * D))) return e; e = copy_f32(data, v->pos, (size_t)v->T * D, st); }
  else if (k == "ln_pre.weight") { if ((e = need(D))) return e; e = copy_f32(data, v->lnpre_w, D, st); }
  else if (k == "ln_pre.bias") { if ((e = need(D))) return e; e = copy_f32(data, v->lnpre_b, D, st); }
  else if (k == "ln_post.weight") { if ((e = need(D))) return e; e = copy_f32(data, v->lnpost_w, D, st); }
  else if (k == "ln_post.bias") { if ((e = need(D))) return e; e = copy_f32(data, v->lnpost_b, D, st); }
  else if (k == "proj") {   // [D, out]: forward B operand is proj^T [out, D]; dgrad B operand is proj [D, out]
    if ((e = need((int64_t)D * O))) return e;
    e = pack(data, v->w_out, D, O, 1, st) | pack(data, v->w_out_t, D, O, 0, st);
  } else if (k.rfind("transformer.resblocks.", 0) == 0) {
    const char* rest = k.c_str() + strlen("transformer.resblocks.");
    char* endp = nullptr;
    const long li = strtol(rest, &endp, 10);
    APH_REQUIRE(endp && *endp == '.' && li >= 0 && li < v->cfg.layers, "aph_vit_load_tensor: bad layer index in %s", key);
    LayerW& l = v->L[li];
    const std::string f(endp + 1);
    if (f == "ln_1.weight") { if ((e = need(D))) return e; e = copy_f32(data, l.ln1_w, D, st); }
    else if (f == "ln_1.bias") { if ((e = need(D))) return e; e = copy_f32(data, l.ln1_b, D, st); }
    else if (f == "ln_2.weight") { if ((e = need(D))) return e; e = copy_f32(data, l.ln2_w, D, st); }
    else if (f == "ln_2.bias") { if ((e = need(D))) return e; e = copy_f32(data, l.ln2_b, D, st); }
    else if (f == "attn.in_proj_weight") { if ((e = need((int64_t)3 * D * D))) return e; e = pack(data, l.w_qkv, 3 * D, D, 0, st) | pack(data, l.w_qkv_t, 3 * D, D, 1, st); }
    else if (f == "attn.in_proj_bias") { if ((e = need(3 * D))) return e; e = copy_f32(data, l.b_qkv, 3 * D, st); }
    else if (f == "attn.out_proj.weight") { if ((e = need((int64_t)D * D))) return e; e = pack(data, l.w_o, D, D, 0, st) | pack(data, l.w_o_t, D, D, 1, st); }
    else if (f == "attn.out_proj.bias") { if ((e = need(D))) return e; e = copy_f32(data, l.b_o, D, st); }
    else if (f == "mlp.c_fc.weight") { if ((e = need((int64_t)4 * D * D))) return e; e = pack(data, l.w_fc, 4 * D, D, 0, st) | pack(data, l.w_fc_t, 4 * D, D, 1, st); }
    else if (f == "mlp.c_fc.bias") { if ((e = need(4 * D))) return e; e = copy_f32(data, l.b_fc, 4 * D, st); }
    else if (f == "mlp.c_proj.weight") { if ((e = need((int64_t)4 * D * D))) return e; e = pack(data, l.w_proj, D, 4 * D, 0, st) | pack(data, l.w_proj_t, D, 4 * D, 1, st); }
    else if (f == "mlp.c_proj.bias") { if ((e = need(D))) return e; e = copy_f32(data, l.b_proj, D, st); }
    else { set_error("aph_vit_load_tensor: unknown tensor %s", key); return 2; }
  } else { set_error("aph_vit_load_tensor: unknown tensor %s", key); return 2; }
  if (e) return e;
  v->loaded[k] = true;
  return 0;
}

extern "C" int aph_vit_finalize(aph_vit* vit) {
  APH_REQUIRE(vit, "aph_vit_finalize: null handle");
  VitImpl* v = reinterpret_cast<VitImpl*>(vit);
  std::vector<std::string> want = {"conv1.weight", "class_embedding", "positional_embedding", "ln_pre.weight", "ln_pre.bias",
                                   "ln_post.weight", "ln_post.bias", "proj"};
  const char* per[] = {"ln_1.weight", "ln_1.bias", "ln_2.weight", "ln_2.bias", "attn.in_proj_weight", "attn.in_proj_bias",
                       "attn.out_proj.weight", "attn.out_proj.bias", "mlp.c_fc.weight", "mlp.c_fc.bias", "mlp.c_proj.weight", "mlp.c_proj.bias"};
  for (int i = 0; i < v->cfg.layers; ++i)
    for (const char* p : per) want.push_back("transformer.resblocks." + std::to_string(i) + "." + p);
  for (const auto& w : want) APH_REQUIRE(v->loaded.count(w), "aph_vit_finalize: tensor visual.%s was never loaded", w.c_str());
  v->finalized = true;
  return 0;
}

static int vit_fwd_impl(aph_vit* vit, const float* images, int S, float* emb, int save_for_bwd, void* stream);

extern "C" int aph_vit_fwd(aph_vit* vit, const float* images, int S, float* emb, int save_for_bwd, void* stream) {
  APH_REQUIRE(vit && images && emb, "aph_vit_fwd: null argument");
  return vit_fwd_impl(vit, images, S, emb, save_for_bwd, stream);
}

// The sampler can write the patch-embedding operand itself (aph_sample_fwd_patches): this is where it goes ...
extern "C" int aph_vit_patch_operand(aph_vit* vit, int S, void** patches_bf16, int* patch, int* grid) {
  APH_REQUIRE(vit && patches_bf16 && patch && grid, "aph_vit_patch_operand: null argument");
  VitImpl* v = reinterpret_cast<VitImpl*>(vit);
  APH_REQUIRE(v->finalized, "aph_vit_patch_operand: weights not finalized");
  APH_REQUIRE(S > 0 && S <= v->cfg.max_batch, "aph_vit_patch_operand: S=%d outside (0, max_batch=%d]", S, v->cfg.max_batch);
  *patches_bf16 = v->patches; *patch = v->cfg.patch; *grid = v->g;
  return 0;
}

// ... and the forward that consumes it as it is (no k_patchify: the fp32 images are not read)
extern "C" int aph_vit_fwd_prepatched(aph_vit* vit, int S, float* emb, int save_for_bwd, void* stream) {
  APH_REQUIRE(vit && emb, "aph_vit_fwd_prepatched: null argument");
  return vit_fwd_impl(vit, nullptr, S, emb, save_for_bwd, stream);
}

static int vit_fwd_impl(aph_vit* vit, const float* images, int S, float* emb, int save_for_bwd, void* stream) {
  VitImpl* v = reinterpret_cast<VitImpl*>(vit);
  APH_REQUIRE(v->finalized, "aph_vit_fwd: weights not finalized");
  APH_REQUIRE(S > 0 && S <= v->cfg.max_batch, "aph_vit_fwd: S=%d outside (0, max_batch=%d]", S, v->cfg.max_batch);
  cudaStream_t st = (cudaStream_t)stream;
  // The only kernels that touch caller-owned memory (k_patchify reads `images`, the last copy writes `emb`) run OUTSIDE the cached
  // graph, so the graph is keyed on the batch size alone: a caller whose tensors move every step (clip_fft.py:285 calls
  // torch.cuda.empty_cache() per step) still replays it.
  if (images) {
    const int g = v->g, Mp = S * g * g;
    const size_t n8 = (size_t)Mp * v->Kp / 8;
    APH_CUDA_OK(launch_k(k_patchify, dim3((unsigned)std::min<size_t>((n8 + 255) / 256, (size_t)kNumSMs * 16)), dim3(256), (size_t)0, st, 1, images, v->patches, S, v->cfg.patch, g));
    APH_LAUNCH_OK();
  }
  const int rc = run_cached(v->fwd_graphs, v->warm_fwd, v->stamp, v->graph_misses, nullptr, nullptr, S, save_for_bwd, st, [&]() -> int {
  const int D = v->D, T = v->T, g = v->g, Ly = v->cfg.layers, O = v->cfg.out_dim, H = v->cfg.heads;
  const int M = S * T, Mp = S * g * g;
  const size_t Mmax = (size_t)v->cfg.max_batch * T;
  int e;
  // patch embedding
  {
    GemmEpi ep; ep.out_f32 = v->tok;
    if ((e = launch_gemm(v->patches, v->w_conv, GemmShape{Mp, D, v->Kp}, ep, st))) return e;
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_embed_lnpre<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, v->tok, v->cls, v->pos, v->lnpre_w, v->lnpre_b, v->e, v->xs[0],
                                                                      v->st_mean, v->st_rstd, S, T, D)));
    APH_LAUNCH_OK();
  }
  for (int l = 0; l < Ly; ++l) {
    const LayerW& w = v->L[l];
    float* x_in = v->xs[2 * l]; float* x_mid = v->xs[2 * l + 1]; float* x_out = v->xs[2 * l + 2];
    float* mean1 = v->st_mean + (size_t)(1 + 2 * l) * Mmax; float* rstd1 = v->st_rstd + (size_t)(1 + 2 * l) * Mmax;
    float* mean2 = mean1 + Mmax; float* rstd2 = rstd1 + Mmax;
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_fwd<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, x_in, (size_t)D, w.ln1_w, w.ln1_b, v->ln_out, mean1, rstd1, M, D)));
    APH_LAUNCH_OK();
    { GemmEpi ep; ep.bias = w.b_qkv; ep.out_bf16 = v->qkv[l];
      if ((e = launch_gemm(v->ln_out, w.w_qkv, GemmShape{M, 3 * D, D}, ep, st))) return e; }
    if (attn_simt()) { k_attn_fwd<<<S * H, 256, attn_fwd_smem(T), st>>>(v->qkv[l], v->attn_out, T, D, H); APH_LAUNCH_OK(); }
    else if (T <= 64 && attn_umma()) { if ((e = attn_fwd_umma_launch(v->qkv[l], v->attn_out, S, T, D, H, st))) return e; }
    else if ((e = attn_dispatch(true, v->qkv[l], nullptr, v->attn_out, S, T, D, H, st))) return e;
    { GemmEpi ep; ep.bias = w.b_o; ep.resid = x_in; ep.out_f32 = x_mid;
      if ((e = launch_gemm(v->attn_out, w.w_o, GemmShape{M, D, D}, ep, st))) return e; }
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_fwd<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, x_mid, (size_t)D, w.ln2_w, w.ln2_b, v->ln_out, mean2, rstd2, M, D)));
    APH_LAUNCH_OK();
    { GemmEpi ep; ep.bias = w.b_fc; ep.out_pre = v->h_pre[l]; ep.act = 1; ep.out_bf16 = v->h_act;
      if ((e = launch_gemm(v->ln_out, w.w_fc, GemmShape{M, 4 * D, D}, ep, st))) return e; }
    { GemmEpi ep; ep.bias = w.b_proj; ep.resid = x_mid; ep.out_f32 = x_out;
      if ((e = launch_gemm(v->h_act, w.w_proj, GemmShape{M, D, 4 * D}, ep, st))) return e; }
  }
  {
    float* meanp = v->st_mean + (size_t)(2 * Ly + 1) * Mmax; float* rstdp = v->st_rstd + (size_t)(2 * Ly + 1) * Mmax;
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_fwd<NCH>, dim3(rows_grid(S)), dim3(256), (size_t)0, st, 1, v->xs[2 * Ly], (size_t)T * D, v->lnpost_w, v->lnpost_b, v->cls_ln,
                                                                 meanp, rstdp, S, D)));
    APH_LAUNCH_OK();
    GemmEpi ep; ep.out_f32 = v->emb_int;
    if ((e = launch_gemm(v->cls_ln, v->w_out, GemmShape{S, O, D}, ep, st))) return e;
  }
  return 0;
  });
  if (rc) return rc;
  APH_CUDA_OK(cudaMemcpyAsync(emb, v->emb_int, (size_t)S * v->cfg.out_dim * sizeof(float), cudaMemcpyDeviceToDevice, st));
  v->last_S = save_for_bwd ? S : -1;
  return 0;
}

extern "C" int aph_vit_bwd(aph_vit* vit, const float* grad_emb, int S, float* grad_images, void* stream) {
  APH_REQUIRE(vit && grad_emb && grad_images, "aph_vit_bwd: null argument");
  VitImpl* v = reinterpret_cast<VitImpl*>(vit);
  APH_REQUIRE(v->last_S == S, "aph_vit_bwd: no saved forward for S=%d (last saved S=%d)", S, v->last_S);
  cudaStream_t st = (cudaStream_t)stream;
  {   // caller-owned input: converted outside the cached graph (see aph_vit_fwd)
    const size_t n = (size_t)S * v->cfg.out_dim;
    APH_CUDA_OK(launch_k(k_f32_to_bf16, dim3((int)std::min<size_t>((n + 255) / 256, (size_t)kNumSMs * 8)), dim3(256), (size_t)0, st, 1, grad_emb, v->d_emb, n));
    APH_LAUNCH_OK();
  }
  const int rc = run_cached(v->bwd_graphs, v->warm_bwd, v->stamp, v->graph_misses, nullptr, nullptr, S, 0, st, [&]() -> int {
  const int D = v->D, T = v->T, Ly = v->cfg.layers, O = v->cfg.out_dim, H = v->cfg.heads;
  const int M = S * T;
  const size_t Mmax = (size_t)v->cfg.max_batch * T;
  int e;
  {
    GemmEpi ep; ep.out_f32 = v->d_cls;
    if ((e = launch_gemm(v->d_emb, v->w_out_t, GemmShape{S, D, O}, ep, st))) return e;
    APH_CUDA_OK(cudaMemsetAsync(v->dx, 0, (size_t)M * D * sizeof(float), st));
    APH_CUDA_OK(cudaMemsetAsync(v->dx_bf, 0, (size_t)M * D * sizeof(bf16), st));
    float* meanp = v->st_mean + (size_t)(2 * Ly + 1) * Mmax; float* rstdp = v->st_rstd + (size_t)(2 * Ly + 1) * Mmax;
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_bwd<NCH>, dim3(rows_grid(S)), dim3(256), (size_t)0, st, 1, v->d_cls, v->xs[2 * Ly], meanp, rstdp, v->lnpost_w, v->dx, v->dx_bf,
                                                                 S, T, D, 1, 0)));
    APH_LAUNCH_OK();
  }
  for (int l = Ly - 1; l >= 0; --l) {
    const LayerW& w = v->L[l];
    float* x_in = v->xs[2 * l]; float* x_mid = v->xs[2 * l + 1];
    float* mean1 = v->st_mean + (size_t)(1 + 2 * l) * Mmax; float* rstd1 = v->st_rstd + (size_t)(1 + 2 * l) * Mmax;
    float* mean2 = mean1 + Mmax; float* rstd2 = rstd1 + Mmax;
    // MLP branch: dh = (dx . W_proj) * gelu'(h); d_ln2 = dh . W_fc
    { GemmEpi ep; ep.gelu_in = v->h_pre[l]; ep.out_bf16 = v->dh;
      if ((e = launch_gemm(v->dx_bf, w.w_proj_t, GemmShape{M, 4 * D, D}, ep, st))) return e; }
    { GemmEpi ep; ep.out_bf16 = v->d_ln;
      if ((e = launch_gemm(v->dh, w.w_fc_t, GemmShape{M, D, 4 * D}, ep, st))) return e; }
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_bwd<NCH, bf16>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, v->d_ln, x_mid, mean2, rstd2, w.ln2_w, v->dx, v->dx_bf, M, T, D, 0, 1)));
    APH_LAUNCH_OK();
    // attention branch: d_attn = dx . W_o; (dq,dk,dv) = attn'(...); d_ln1 = d_qkv . W_qkv
    { GemmEpi ep; ep.out_bf16 = v->d_attn;
      if ((e = launch_gemm(v->dx_bf, w.w_o_t, GemmShape{M, D, D}, ep, st))) return e; }
    if (attn_simt()) { k_attn_bwd<<<S * H, 256, attn_bwd_smem(T), st>>>(v->qkv[l], v->d_attn, v->d_qkv, T, D, H); APH_LAUNCH_OK(); }
    else if ((e = attn_dispatch(false, v->qkv[l], v->d_attn, v->d_qkv, S, T, D, H, st))) return e;
    { GemmEpi ep; ep.out_bf16 = v->d_ln;
      if ((e = launch_gemm(v->d_qkv, w.w_qkv_t, GemmShape{M, D, 3 * D}, ep, st))) return e; }
    NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_bwd<NCH, bf16>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, v->d_ln, x_in, mean1, rstd1, w.ln1_w, v->dx, v->dx_bf, M, T, D, 0, 1)));
    APH_LAUNCH_OK();
  }
  // ln_pre backward (cls rows dropped) and patch-embed data gradient scattered back to NCHW
  NCH_DISPATCH(D, APH_CUDA_OK(launch_k(k_ln_bwd<NCH>, dim3(rows_grid(M)), dim3(256), (size_t)0, st, 1, v->dx, v->e, v->st_mean, v->st_rstd, v->lnpre_w, nullptr, v->d_tok, M, T, D, 2, 0)));
  APH_LAUNCH_OK();
  return 0;
  });
  if (rc) return rc;
  // caller-owned output: the patch-embed data gradient (un-patchify epilogue writes NCHW) is launched outside the graph
  { const int g = v->g, Mp = S * g * g;
    GemmEpi ep; ep.out_f32 = grad_images; ep.unpatch_p = v->cfg.patch; ep.unpatch_g = g;
    if (int e = launch_gemm(v->d_tok, v->w_conv_t, GemmShape{Mp, v->Kp, v->D}, ep, st)) return e; }
  return 0;
}

/* aphb200.h -- C ABI of libaphb200.so: the B200-native (sm_100a) hot path of eps696/aphantasia.
 *
 * Drop-in boundary (SURVEY.md section 8b). Plain pointers and sizes only; no torch types. Every compute entry
 * point is asynchronous on the caller's `stream` (pass torch.cuda.current_stream().cuda_stream as void*),
 * returns 0 on success / non-zero on error (message: aph_last_error(), thread-local), and never owns
 * user-visible memory: inputs/outputs are caller-owned DEVICE pointers (fp32 unless stated). Scratch lives
 * in library-owned handles so it survives the reference's per-step torch.cuda.empty_cache()
 * (/root/reference/clip_fft.py:285).
 *
 * Each entry point cites the reference interface it replaces (paths relative to /root/reference).
 * The Python binding (ctypes) is aphantasia_b200/_lib.py; INTEGRATION.md shows the reference-side stub.
 */
#ifndef APHB200_H_
#define APHB200_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APH_ABI_VERSION 1

/* ---- crop parameter table: one row per crop, APH_CROP_PARAM_FLOATS float32 values.
 * Built on the host by replaying the reference's RNG order (aphantasia_b200/_rng.py).               */
#define APH_CROP_PARAM_FLOATS 24
#define APH_F_OFFY   0   /* crop top-left y in the sampling frame (integer-valued)   utils.py:247 */
#define APH_F_OFFX   1   /* crop top-left x                                          utils.py:246 */
#define APH_F_CSIZE  2   /* crop side in canvas pixels                                utils.py:245 */
#define APH_F_FLAGS  3   /* bit0 perspective, bit1 erase, bit2 rotate                              */
#define APH_F_PERSP  4   /* 8 coeffs a..h, output->input (torchvision _get_perspective_coeffs)     */
#define APH_F_ER_I   12  /* erase rect top, left, height, width (torchvision RandomErasing)        */
#define APH_F_ER_J   13
#define APH_F_ER_H   14
#define APH_F_ER_W   15
#define APH_F_ROT    16  /* theta00, theta01, theta10, theta11 of the inverse affine matrix        */
#define APH_F_ANGLE  20  /* degrees, informational                                                 */
#define APH_FLAG_PERSP 1
#define APH_FLAG_ERASE 2
#define APH_FLAG_ROT   4

/* sampler transform kinds (what `transform=` of slice_imgs was)                                  */
#define APH_TF_NONE      0   /* bicubic resize only                                                */
#define APH_TF_NORMALIZE 1   /* + transforms.normalize()            transforms.py:102-109          */
#define APH_TF_FAST      2   /* transforms.transforms_fast          transforms.py:165-170          */

/* similarity kinds (sim_func `type`)                                         utils.py:276-295    */
#define APH_SIM_COS 0
#define APH_SIM_MIX 1

int         aph_version(void);
const char* aph_last_error(void);

/* ================= L3: spectrum -> RGB synthesis =============================================
 * Replaces fft_image.inner (aphantasia/image.py:164-175) and, fused, to_valid_rgb.inner
 * (aphantasia/image.py:21-28):   x = irfftn(scale*(P [+shift]), s=(H,W), 'ortho');
 *                                 img = x*contrast/std(x);  out = sigmoid(colmat . img)            */
typedef struct aph_fft_plan aph_fft_plan;
int aph_fft_plan_create(aph_fft_plan** plan, int H, int W);   /* H, W: prime factors <= 13 */
int aph_fft_plan_destroy(aph_fft_plan* plan);

/* params [3,H,Wh,2], scale [H,Wh] (Wh = W/2+1).  shift_mode 0: none; 1: shift [H,Wh] (the script's
 * --noise, clip_fft.py:238); 2: shift [3,H,Wh,2] (illustra.py:334).
 * colmat: 9 floats, HOST pointer, row-major Mn[d][c] (out_d = sum_c Mn[d][c] img_c) or NULL = no
 * decorrelation. apply_sigmoid 0/1.
 * Outputs: x_raw [3,H,W] (un-normalised irfft, saved for backward), stats double[4] on device
 * {sum x, sum x^2, sum g.x (bwd scratch), unused}, out [3,H,W].                                    */
int aph_synth_fft_fwd(aph_fft_plan* plan, const float* params, const float* scale,
                      const float* shift, int shift_mode, float contrast,
                      const float* colmat_host, int apply_sigmoid,
                      float* x_raw, double* stats, float* out, void* stream);
/* grad_out [3,H,W] = dL/d out  ->  grad_params [3,H,Wh,2] (overwritten).                           */
int aph_synth_fft_bwd(aph_fft_plan* plan, const float* grad_out, const float* out,
                      const float* x_raw, double* stats, const float* scale, float contrast,
                      const float* colmat_host, int apply_sigmoid,
                      float* grad_params, void* stream);

/* Wavelet parameterisation (BASELINE config 3). Replaces dwt_image.inner (aphantasia/image.py:66-69):
 *   img = DWTInverse((Yl, [Yh_i * scale_i])) * contrast / std, fused with to_valid_rgb like the FFT path.
 * DWTInverse is pytorch_wavelets' (third-party, mode 'symmetric'); rec_lo / rec_hi (HOST, L taps) are the
 * PyWavelets reconstruction filters. J = floor(log2(min(H, W))) levels (image.py:35-36).                        */
typedef struct aph_dwt_plan aph_dwt_plan;
int aph_dwt_plan_create(aph_dwt_plan** plan, int H, int W, const float* rec_lo_host, const float* rec_hi_host, int L);
int aph_dwt_plan_destroy(aph_dwt_plan* plan);
/* J; dims[2*i], dims[2*i+1] = band height/width of level i+1 (finest first); out_hw = synthesised image size      */
int aph_dwt_plan_levels(const aph_dwt_plan* plan, int* J, int* dims, int* out_hw);
/* Ys: HOST array of J+1 DEVICE pointers {Yl [3,hJ,wJ], Yh_1 [3,3,h1,w1] (finest), ..., Yh_J}; scales_host [J]
 * (aphantasia/image.py:73-80). Outputs as aph_synth_fft_fwd (x_raw / out are [3,out_h,out_w]).                    */
int aph_synth_dwt_fwd(aph_dwt_plan* plan, const float* const* Ys, const float* scales_host, float contrast,
                      const float* colmat_host, int apply_sigmoid, float* x_raw, double* stats, float* out,
                      void* stream);
/* grad_Ys: HOST array of J+1 DEVICE pointers receiving d loss / d Ys (overwritten).                               */
int aph_synth_dwt_bwd(aph_dwt_plan* plan, const float* grad_out, const float* out, const float* x_raw,
                      double* stats, const float* scales_host, float contrast, const float* colmat_host,
                      int apply_sigmoid, float* const* grad_Ys, void* stream);

/* Direct RGB parameterisation: pixel_image.inner (aphantasia/image.py:112-118): img = x*contrast/std(x) (or /3.3 with
 * fixcontrast), fused with to_valid_rgb. x / out / grad_x are [3,H,W]; stats as above.                             */
int aph_pixel_fwd(const float* x, int64_t hw, float contrast, int fixcontrast, const float* colmat_host,
                  int apply_sigmoid, double* stats, float* out, void* stream);
int aph_pixel_bwd(const float* grad_out, const float* out, const float* x, double* stats, int64_t hw, float contrast,
                  int fixcontrast, const float* colmat_host, int apply_sigmoid, float* grad_x, void* stream);

/* Stand-alone to_valid_rgb for a foreign image_f (aphantasia/image.py:21-28): img [3,H,W] -> out.  */
int aph_valid_rgb_fwd(const float* img, int64_t hw, const float* colmat_host, float* out, void* stream);
int aph_valid_rgb_bwd(const float* grad_out, const float* out, int64_t hw, const float* colmat_host,
                      float* grad_img, void* stream);

/* ================= L2: multi-crop sampler =====================================================
 * Replaces the per-crop Python loop of slice_imgs (aphantasia/utils.py:243-253) + transforms_fast
 * (aphantasia/transforms.py:165-170): bicubic(A=-0.75, align_corners, crop-clamped) -> perspective
 * (bilinear, zeros, x coverage) -> erase -> rotate (bilinear, zeros, x coverage) -> normalise.
 * canvas [3,H,W]; the sampling frame is the canvas wrap-padded by (pad_top, pad_left)
 * ('over*' aligns, utils.py:152-187; 0,0 otherwise); table: DEVICE [S, APH_CROP_PARAM_FLOATS];
 * out [S,3,size,size]. the resized crop, its tap tables and the per-warp strips must fit one CTA's shared memory (size <= 224).           */
int aph_sample_fwd(const float* canvas, int H, int W, int pad_top, int pad_left,
                   const float* table, int S, int size, int kind, float* out, void* stream);
/* Same, and the last stage also writes the batch as the encoder's patch operand (bf16, patch-major: see
 * aph_vit_patch_operand below); size must be a multiple of patch. *patches_written = 1 when it did (0: the one-kernel
 * fallback form ran and the caller has to use aph_vit_fwd on `out`).                                 */
int aph_sample_fwd_patches(const float* canvas, int H, int W, int pad_top, int pad_left,
                           const float* table, int S, int size, int kind, float* out,
                           void* patches_bf16, int patch, int* patches_written, void* stream);
/* grad_out [S,3,size,size] -> grad_canvas [3,H,W] (zeroed here, then accumulated).                 */
int aph_sample_bwd(const float* grad_out, int H, int W, int pad_top, int pad_left,
                   const float* table, int S, int size, int kind, float* grad_canvas, void* stream);

/* Same with every contribution multiplied by gscale (the weight S_local / S of this rank's shard in the all-reduced
 * gradient under torchrun: folded into the scatter instead of a separate pass over the canvas).     */
int aph_sample_bwd_scaled(const float* grad_out, int H, int W, int pad_top, int pad_left,
                          const float* table, int S, int size, int kind, float gscale, float* grad_canvas, void* stream);

/* HOST function (no GPU work): exact native replay of the reference's per-crop random draws (utils.py:244-247,
 * torchvision RandomPerspective/RandomErasing.get_params, transforms.py:75) continuing torch's CPU generator
 * (torch_state = the torch.get_rng_state() blob, updated in place) and NumPy's legacy MT19937 (np_key[624], *np_pos,
 * updated in place). rnd_size/offx/offy are the [count] vectors slice_imgs draws first (utils.py:222-228).
 * Writes tables [n_imgs][count][APH_CROP_PARAM_FLOATS] (HOST memory).                                              */
int aph_rng_crop_tables(uint8_t* torch_state, int64_t torch_state_bytes, uint32_t* np_key, int32_t* np_pos,
                        const float* rnd_size, const float* rnd_offx, const float* rnd_offy, int count,
                        int H, int W, int frame_h, int frame_w, int size, int kind, float macro, int n_imgs,
                        float* tables);

/* ================= L1: CLIP ViT-B image encoder ===============================================
 * Replaces clip.model.CLIP.encode_image / VisionTransformer.forward (third-party OpenAI clip; call
 * sites clip_fft.py:216,254,276) and its autograd data-gradient. Weights are frozen: no weight
 * gradients are computed (the reference computes and discards them, clip_fft.py:293-295).           */
typedef struct aph_vit aph_vit;
typedef struct {
  int32_t patch;      /* 32 or 16                                   */
  int32_t width;      /* 768                                        */
  int32_t layers;     /* 12                                         */
  int32_t heads;      /* 12 (head dim must be 64)                   */
  int32_t out_dim;    /* 512                                        */
  int32_t res;        /* input resolution, 224                      */
  int32_t max_batch;  /* largest S a call will pass                 */
  int32_t reserved;
} aph_vit_config;
int aph_vit_create(aph_vit** vit, const aph_vit_config* cfg);
int aph_vit_destroy(aph_vit* vit);
/* One tensor of the OpenAI state dict, by its key ("visual.conv1.weight", "visual.transformer.
 * resblocks.3.attn.in_proj_weight", ...), fp32 DEVICE pointer; converted/transposed to the packed
 * bf16 operand layout on device. aph_vit_finalize checks every tensor arrived.                     */
int aph_vit_load_tensor(aph_vit* vit, const char* key, const float* data, int64_t numel, void* stream);
int aph_vit_finalize(aph_vit* vit);
/* images [S,3,res,res] fp32 (already normalised) -> emb [S,out_dim] fp32. save_for_bwd 0/1.        */
int aph_vit_fwd(aph_vit* vit, const float* images, int S, float* emb, int save_for_bwd, void* stream);
/* Patch operand hand-over (SURVEY 2.4 k10-k12: the sampler emits the patch-major bf16 A operand of conv1, replacing the
 * fp32 round trip x.type(dtype) -> conv1's im2col of the reference's clip/model.py VisionTransformer.forward):
 * aph_vit_patch_operand returns the handle's operand buffer [S*grid*grid, 3*patch*patch] bf16 (row = s*grid*grid + gy*grid + gx,
 * col = c*patch*patch + py*patch + px) for aph_sample_fwd_patches to fill; aph_vit_fwd_prepatched then runs the forward on it.  */
int aph_vit_patch_operand(aph_vit* vit, int S, void** patches_bf16, int* patch, int* grid);
int aph_vit_fwd_prepatched(aph_vit* vit, int S, float* emb, int save_for_bwd, void* stream);
/* grad_emb [S,out_dim] -> grad_images [S,3,res,res] (overwritten). Uses activations of the last
 * aph_vit_fwd(save_for_bwd=1) with the same S.                                                     */
int aph_vit_bwd(aph_vit* vit, const float* grad_emb, int S, float* grad_images, void* stream);
/* bytes of device memory owned by the handle (weights + activation arena)                          */
int64_t aph_vit_bytes(const aph_vit* vit);

/* ================= CLIP text encoder (forward only) ===========================================
 * Replaces clip.model.CLIP.encode_text (third-party OpenAI clip; call site clip_fft.py:150), run once per prompt
 * before the optimisation loop:  x = token_embedding[ids] + positional_embedding;  `layers` residual attention
 * blocks with a causal mask (query i sees keys j <= i);  emb = ln_final(x[s, argmax_t ids[s,t]]) @ text_projection.
 * Same block as the image encoder (QuickGELU, LayerNorm eps 1e-5, head dim 64); the residual stream is fp32,
 * GEMM operands bf16.                                                                                            */
typedef struct aph_text aph_text;
typedef struct {
  int32_t width;      /* 256, 512 or 768 (ViT-B text towers: 512) */
  int32_t layers;     /* 12                                        */
  int32_t heads;      /* width / 64                                */
  int32_t ctx;        /* context length, <= 112 (77)               */
  int32_t vocab;      /* 49408                                     */
  int32_t out_dim;    /* 512 (multiple of 128)                     */
  int32_t max_batch;  /* largest n a call will pass                */
} aph_text_config;
int aph_text_create(aph_text** text, const aph_text_config* cfg);
int aph_text_destroy(aph_text* text);
/* One tensor of the OpenAI state dict by its key, without prefix ("token_embedding.weight", "positional_embedding",
 * "ln_final.weight", "text_projection", "transformer.resblocks.3.attn.in_proj_weight", ...), fp32 DEVICE pointer.
 * aph_text_finalize names the first tensor that never arrived.                                                    */
int aph_text_load_tensor(aph_text* text, const char* key, const float* data, int64_t numel, void* stream);
int aph_text_finalize(aph_text* text);
/* tokens: int64 DEVICE [n, ctx] (clip.tokenize(...).cuda()) -> emb fp32 [n, out_dim]. An id outside [0, vocab)
 * contributes a zero embedding row (the table is never read out of bounds).                                       */
int aph_text_fwd(aph_text* text, const int64_t* tokens, int n, float* emb, void* stream);
/* bytes of device memory owned by the handle (weights + activations)                                              */
int64_t aph_text_bytes(const aph_text* text);

/* Stand-alone tcgen05 GEMM used by the encoder (exported for tests / profiling):
 * C[M,N] (fp32) = A[M,K] (bf16, row-major) . B[N,K]^T (bf16, row-major). K % 64 == 0, N % 128 == 0. */
int aph_gemm_bf16_tn(const void* A, const void* B, float* C, int M, int N, int K, void* stream);

/* Test entries. aph_gemm_epi_test: the same GEMM with the encoder's fused epilogues on caller-supplied operands
 * (NULL = unused; the combination selects the kind as the encoder's own calls do: +bias, QuickGELU saving the
 * pre-activation (act=1, out_pre), x gelu'(gelu_in), +fp32 resid, fp32 / bf16 outputs, NCHW un-patchify).
 * aph_gemm_variant_launches: launches so far of tile variant 0 (128x128, one CTA), 1 (256x192 pair tiles, two exact waves at
 * N = 768, remainder rows in-kernel), 2 (256x256, cta_group::2 pair) or 3 (256x384 one-wave pair tiles) with epilogue kind epi (0 f32, 1 bf16, 2 bias-bf16, 3 bias-gelu, 4 bias-resid,
 * 5 gelu-grad, 6 un-patchify; -1 = any).                                                             */
int aph_gemm_epi_test(const void* A, const void* B, int M, int N, int K, const float* bias, const float* resid,
                      const void* gelu_in, int act, float* out_f32, void* out_bf16, void* out_pre,
                      int unpatch_p, int unpatch_g, void* stream);
int64_t aph_gemm_variant_launches(int variant, int epi);

/* Profiling aid: enable=1 records a CUDA-event pair around every GEMM launch of this library; enable=0 stops and returns
 * the summed kernel time (ms), FLOPs (sum of 2MNK) and launch count since enabling (bench.py's roofline).            */
int aph_prof_gemm(int enable, double* total_ms, double* total_flops, int* launches);

/* ================= L1: similarity loss ========================================================
 * Replaces sim_func(v1, v2, type) for type in {None/'cossim', 'mix'} (aphantasia/utils.py:276-282,
 * 295). v1 [n1,D] with n1 in {1,S}; v2 [S,D]. value (device scalar) = mean_s f(v1, v2_s).
 * grad_v1 / grad_v2 may be NULL; they receive d value / d v (not yet multiplied by the upstream
 * gradient).                                                                                       */
int aph_sim_fwd(const float* v1, int n1, const float* v2, int S, int D, int kind,
                float* value, float* grad_v1, float* grad_v2, void* stream);

/* ---- optional loss heads (SURVEY.md 8 row f4) ---------------------------------------------------
 * derivat(img, mode='naiv') (aphantasia/utils.py:256-268; clip_fft.py:271-272 --sharp): img [C,H,W];
 * value = 0.5*(mean|d/dx| + mean|d/dy|); sums = double[2] device scratch. The backward multiplies by the
 * upstream gradient read from a DEVICE scalar.                                                      */
int aph_derivat_fwd(const float* img, int C, int H, int W, double* sums, float* value, void* stream);
int aph_derivat_bwd(const float* img, int C, int H, int W, const float* upstream, float* grad_img, void* stream);
/* Linear head on the embeddings: the LAION aesthetic predictor of --aest is nn.Linear(D, 1)
 * (aphantasia/utils.py:402-413; clip_fft.py:255-256). out[s] = <emb_s, w> + b[0] (b may be NULL).   */
int aph_head_fwd(const float* emb, int S, int D, const float* w, const float* b, float* out, void* stream);
int aph_head_bwd(const float* grad_out, const float* w, int S, int D, float* grad_emb, void* stream);

/* ================= step glue ==================================================================
 * torch.optim.Adam(betas=(b1,b2)) single-tensor update (clip_fft.py:108-115,295), bias-corrected. */
int aph_adam_step(float* p, const float* g, float* m, float* v, int64_t n,
                  float lr, float b1, float b2, float eps, int step, void* stream);

/* SURVEY.md 8 row f2: aph_synth_fft_bwd with the Adam update of the spectrum fused into its last pass (the data
 * gradient dP is in registers there): params / m / v [3,H,Wh,2] are updated in place; grad_params may be NULL
 * (nothing is written) or receives dP as aph_synth_fft_bwd does. Same arithmetic as aph_adam_step.              */
int aph_synth_fft_bwd_adam(aph_fft_plan* plan, const float* grad_out, const float* out, const float* x_raw,
                           double* stats, const float* scale, float contrast, const float* colmat_host,
                           int apply_sigmoid, float* grad_params, float* params, float* m, float* v,
                           float lr, float b1, float b2, float eps, int step, void* stream);

/* ================= multi-GPU exchange (SURVEY.md 8e) ==========================================
 * In-place all-reduce(SUM) of a fp32 buffer in SYMMETRIC memory (the canvas gradient dRGB [3,H,W], replacing the
 * single NCCL all-reduce of the path): one kernel, two shots over NVSwitch multicast (multimem.ld_reduce / multimem.st;
 * mc_ptr = multicast address) or, with mc_ptr == 0, over the peers' mapped pointers. peer_ptrs: HOST array[world] of
 * every rank's device mapping of the buffer; signal_pads_dev: DEVICE array[world] of pointers to zero-initialised
 * uint32 signal pads (>= 32*world words each); numel % 4 == 0. err_flag (device int) is set if a barrier timed out.  */
int aph_allreduce_sym(uint64_t mc_ptr, const uint64_t* peer_ptrs, const uint64_t* signal_pads_dev, int rank, int world,
                      int64_t numel, int* err_flag, void* stream);

/* number of kernels this library has launched since load (bench.py's gpu_launches)                 */
int64_t aph_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* APHB200_H_ */

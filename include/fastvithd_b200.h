/* fastvithd_b200.h -- C ABI of the B200-native FastViTHD vision tower + mm_projector.
 *
 * Drop-in boundary for ONE path of apple/ml-fastvlm: `LlavaMetaForCausalLM.encode_images`
 * (llava/model/llava_arch.py:141-144) == mm_projector(vision_tower(images)).  The reference has no
 * FFI of its own (pure Python); these entry points are what a binding for that path needs and each
 * cites the reference interface it replaces.  Plain pointers and sizes only -- no torch types.
 *
 * Conventions
 *   - every function returns FVHD_OK (0) or a negative fvhd_status; fvhd_last_error(h) gives the
 *     message (the Python wrapper raises RuntimeError with it).  There is NO CPU fallback.
 *   - device pointers are CUDA device memory of the current device; `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream).  Calls enqueue work and do not synchronise,
 *     except the *_host entry points, which synchronise `stream` before returning.
 *   - activations are NHWC bf16 inside the library; images enter as NCHW [B,3,R,R]
 *     (fp32 / fp16 / bf16, processor output: mean 0, std 1, range [0,1), mobileclip_encoder.py:45-49);
 *     tokens leave as row-major [B, (R/64)^2, C] bf16.
 */
#ifndef FASTVITHD_B200_H
#define FASTVITHD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FVHD_API_VERSION 1

typedef enum {
    FVHD_OK = 0,
    FVHD_ERR_INVALID = -1,      /* bad argument / unsupported configuration */
    FVHD_ERR_WEIGHTS = -2,      /* missing / mis-shaped weight tensor */
    FVHD_ERR_CUDA = -3,         /* CUDA runtime / driver error */
    FVHD_ERR_WORKSPACE = -4,    /* workspace missing or too small */
    FVHD_ERR_STATE = -5         /* call order (e.g. forward before load_weights) */
} fvhd_status;

typedef enum { FVHD_F32 = 0, FVHD_F16 = 1, FVHD_BF16 = 2 } fvhd_dtype;

/* Architecture constants of `fastvithd()` (mobileclip/mci.py:1454-1478); not configurable. */
#define FVHD_EMBED_DIM 3072     /* mobileclip_l.json image_cfg.embed_dim == tower.hidden_size */
#define FVHD_PATCH 64           /* mobileclip_l.json image_cfg.patch_size */

typedef struct {
    int image_size;             /* R: from the tower name suffix `mobileclip_l_<R>` (mobileclip_encoder.py:20); R % 64 == 0 */
    int projector_hidden;       /* H = config.hidden_size of the LLM (multimodal_projector/builder.py:26); 0 = tower only */
    int projector_depth;        /* N of `mlp{N}x_gelu` (builder.py:23-30); 1 or 2; ignored when projector_hidden == 0 */
    int max_batch;              /* images processed per internal pass; larger batches are chunked */
} fvhd_config;

/* One packed weight tensor (produced by the host-side packer from the reference state-dict keys
 * `model.vision_tower.vision_tower.model.*` / `model.mm_projector.{0,2}.*`, SURVEY.md 2.2). */
typedef struct {
    const char* name;           /* packed name, e.g. "network.2.5.fc1.w" */
    const void* data;           /* device pointer, 16-byte aligned */
    int dtype;                  /* FVHD_F32 or FVHD_BF16 */
    int64_t numel;
} fvhd_tensor;

/* Decoder configuration of the LLM whose prefill follows encode_images (row f3): the fields of transformers' Qwen2Config that
 * Qwen2ForCausalLM.forward reads (llava/model/language_model/llava_qwen.py:33-55: LlavaQwen2ForCausalLM subclasses it unchanged). */
typedef struct {
    int hidden;                 /* hidden_size */
    int layers;                 /* num_hidden_layers */
    int heads;                  /* num_attention_heads */
    int kv_heads;               /* num_key_value_heads (grouped-query attention) */
    int head_dim;               /* hidden_size / num_attention_heads: 64 or 128 */
    int intermediate;           /* intermediate_size */
    int vocab;                  /* vocab_size */
    int max_seq;                /* longest prompt (text + visual tokens) a prefill may have */
    float rope_theta;
    float rms_eps;
} fvhd_llm_config;

typedef struct fvhd_handle_s* fvhd_handle;

/* replaces: MobileCLIPVisionTower.__init__ / load_model (mobileclip_encoder.py:14-58) and
 * build_vision_projector (multimodal_projector/builder.py:17-35): builds the execution plan. */
int fvhd_create(const fvhd_config* cfg, fvhd_handle* out);
int fvhd_destroy(fvhd_handle h);
const char* fvhd_last_error(fvhd_handle h);    /* h may be NULL: error of the last failed fvhd_create */
int fvhd_api_version(void);

/* Names of the packed tensors the plan requires, in order (for the packer / for error reporting). */
int fvhd_num_weights(fvhd_handle h);
int fvhd_weight_spec(fvhd_handle h, int i, const char** name, int* dtype, int64_t* numel);

/* replaces: from_pretrained / load_state_dict of tower + projector (llava/model/builder.py:131,169-174).
 * The caller keeps ownership of the device buffers and must keep them alive. */
int fvhd_load_weights(fvhd_handle h, const fvhd_tensor* table, int n);

/* Caller-owned scratch.  Bytes needed for `batch` images per pass (batch <= cfg.max_batch). */
size_t fvhd_workspace_bytes(fvhd_handle h, int batch);
int fvhd_set_workspace(fvhd_handle h, void* dptr, size_t bytes);

/* replaces: MobileCLIPVisionTower.forward_images + feature_select (mobileclip_encoder.py:60-88) and,
 * when `projected` != NULL, mm_projector (multimodal_projector/builder.py:23-30) == encode_images
 * (llava_arch.py:141-144).
 *   images     device, NCHW [B,3,R,R] of `img_dtype`
 *   tokens     device, [B,(R/64)^2,3072] bf16, or NULL
 *   projected  device, [B,(R/64)^2,H] bf16, or NULL (requires projector_hidden > 0) */
int fvhd_forward(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch,
                 void* tokens, void* projected);

/* fvhd_forward whose FINAL output (projected tokens, or tower tokens for a projector-less plan) is written with
 * `out_image_stride` ELEMENTS between consecutive images (0 = dense).  With projected = embeds + pos*H and
 * out_image_stride = L*H the visual tokens land directly inside a [B, L, H] LLM input-embedding buffer: the token
 * splice of prepare_inputs_labels_for_multimodal (llava_arch.py:251-271) becomes the projector's store, no copy. */
int fvhd_forward_strided(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch,
                         void* tokens, void* projected, long long out_image_stride);

/* Batch-sharded encode_images whose projector epilogue IS the all-gather (SURVEY 8e; the exchange step that
 * follows mobileclip_encoder.py:84-86 + llava_arch.py:141-144 when one LLM prefill consumes the whole batch):
 * this rank encodes its `batch` images and every 16-byte output vector is stored (a) at local_out and (b) at the same
 * element offset of each peer_out[i] -- peer-mapped device pointers (CUDA IPC / symmetric memory, NVLink P2P) to the
 * slot `[first_image_of_this_rank, +batch)` of GPU i's gathered [B_total, N, H] buffer.  No collective pass follows;
 * the caller only has to order readers after all ranks' kernels (a barrier).  n_peers <= 8; requires a projector. */
int fvhd_forward_gather(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch,
                        void* local_out, void* const* peer_out, int n_peers);

/* encode_images whose projector epilogue stores image i's [N, H] token block (dense rows) at dst_per_image[i]: the general
 * splice of prepare_inputs_labels_for_multimodal (llava_arch.py:233-271) -- several <image> tokens per sample, a different
 * position in every sample, ragged sequence lengths -- with no intermediate feature tensor and no torch.cat.  The host
 * computes the destinations (Python: glue.prepare_inputs_embeds).  `dst_per_image`: HOST array of `batch` device pointers,
 * 16-B aligned; requires a projector and cfg.max_batch <= 64. */
int fvhd_forward_scatter(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch,
                         void* const* dst_per_image);

/* Same call with HOST buffers: H2D of the images, the forward, D2H of the result, one stream sync.
 * `host_out` receives `projected` when the plan has a projector, else `tokens` (bf16). */
int fvhd_encode_images_host(fvhd_handle h, void* stream, const void* host_images, int img_dtype, int batch,
                            void* host_out);

/* Geometry helpers (mobileclip_encoder.py:103-116). */
int fvhd_num_tokens(fvhd_handle h);             /* (R/64)^2 == tower.num_patches */
int fvhd_out_dim(fvhd_handle h);                /* H if projector else 3072 */

/* ---- unit-level access (parity tests and per-unit roofline; units follow the reference modules:
 * "stem", "network.<i>.<b>" / "network.<i>", "conv_exp", "projector") ---- */
int fvhd_num_units(fvhd_handle h);
/* in/out element counts are per image; activations NHWC bf16 ([H*W, C] row-major). */
int fvhd_unit_info(fvhd_handle h, int u, const char** name, int64_t* in_elems, int64_t* out_elems,
                   int* out_h, int* out_w, int* out_c, double* flops_per_image, double* min_bytes_per_image);
/* Run units [first, last] on `batch` images: `in` is the bf16 NHWC input of unit `first`
 * (for first == 0 the NCHW image of `img_dtype`), `out` receives the bf16 output of unit `last`. */
int fvhd_run_units(fvhd_handle h, void* stream, int first, int last, const void* in, int img_dtype,
                   int batch, void* out);
/* Forward with a cudaEvent around every unit; ms[u] = milliseconds of unit u (synchronises). */
int fvhd_profile_units(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch,
                       float* ms, int n_ms);
/* Kernel-level view of the plan for `batch` images per pass: one step == one kernel launch.
 * kernel = __global__ function name, unit = owning unit, flops/bytes = ALGORITHMIC work of that launch
 * (2*MACs; operands read once + result written once).  fvhd_profile_steps brackets every launch with
 * cudaEvents on `stream` (ms[i], synchronises) -- the live per-kernel times bench.py's roofline uses. */
int fvhd_num_steps(fvhd_handle h, int batch);
int fvhd_step_info(fvhd_handle h, int batch, int i, const char** kernel, int* unit, double* flops, double* bytes);
int fvhd_profile_steps(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch,
                       float* ms, int n_ms);
/* Number of kernel launches one forward of `batch` images enqueues. */
int fvhd_launches_per_forward(fvhd_handle h, int batch);

/* ---- row f1: the reference's CPU preprocessing on the GPU, bit-exact ----
 * replaces: process_images (llava/mm_utils.py:168-184) -> CLIPImageProcessor.preprocess as configured by
 * mobileclip_encoder.py:45-49 (pinned transformers 4.48.3 = PIL path): resize shortest edge to R with PIL BICUBIC, centre crop
 * R x R, x 1/255, mean 0 / std 1, CHW; pad_to_square = the 'pad' aspect mode (expand2square, mm_utils.py:154-165).
 *   rgb   uint8 RGB, HWC [H, W, 3]; device memory, or host memory when src_on_host != 0 (copied with cudaMemcpyAsync)
 *   out   device, [3, R, R] of out_dtype (one image of the tower's input batch) */
int fvhd_preprocess(fvhd_handle h, void* stream, const void* rgb, int src_on_host, int H, int W, int pad_to_square,
                    void* out, int out_dtype);
/* 'anyres' building block (llava/mm_utils.py:46-98, 121-147: resize_and_pad_image + divide_to_patches + processor.preprocess):
 * PIL-resize the image to new_h x new_w (BICUBIC, bit-exact), paste it at (pad_y, pad_x) on a black canvas and emit the canvas as
 * tiles_y x tiles_x row-major tiles of R x R (pixels beyond the pasted image are 0), x 1/255.  out: device, [tiles_y*tiles_x, 3, R, R].
 * The global view of process_anyres_image is the call new_h = new_w = R, pad 0, one tile. */
int fvhd_preprocess_tiles(fvhd_handle h, void* stream, const void* rgb, int src_on_host, int H, int W, int new_h, int new_w,
                          int pad_y, int pad_x, int tiles_y, int tiles_x, void* out, int out_dtype);
/* Host-only: Pillow's fixed-point bicubic coefficient table for resampling in_size -> out_size (Resample.c precompute_coeffs +
 * normalize_coeffs_8bpc).  bounds [out][2] = (first source index, tap count); kk [out][ksize]; returns ksize (or < 0). */
int fvhd_resample_coeffs(int in_size, int out_size, int* bounds, int* kk, int kk_capacity);

/* Debug: subsequent fvhd_gemm calls write 16 globaltimer stamps per CTA into `dev_buf` (NULL = off), optionally with a
 * forced N tile (0 = cost model) and a cluster-size cap (1/2/4).  Process-global; not for production use. */
int fvhd_debug_gemm_trace(void* dev_buf_16_u64_per_cta, int force_bn, int max_cs);

/* Debug: every RepMixer depthwise launch writes 8 globaltimer stamps per CTA into `dev_buf` (NULL = off); the buffer holds
 * the most recent launch.  Process-global; not for production use. */
int fvhd_debug_mixer_trace(void* dev_buf_8_u64_per_cta);

/* Stand-alone GEMM entry (tests): D[M,N] = act(A[M,K] W[N,K]^T + bias) + residual, bf16. */
int fvhd_gemm(fvhd_handle h, void* stream, const void* A, const void* W, const void* bias, const void* residual,
              void* D, int M, int N, int K, int act);

/* Test entry: the MHSA core softmax((q 32^-1/2) k^T) v of one attention block (mci.py:675-679) on qkv = [B*N, 3C] bf16 (q | k | v,
 * heads of 32) -> out [B*N, C] bf16; kernel per FVHD_ATTN as read by fvhd_create for this handle (u: tcgen05/TMEM, attention_umma.cuh;
 * default: mma.sync). */
int fvhd_attention(fvhd_handle h, void* stream, const void* qkv, void* out, int batch, int N, int C);

/* Test entry: the second-generation fused ConvFFN kernel (convffn.cuh; one CTA per 128-row tile, packed-half GELU, f16 hidden),
 * same operands as fvhd_convffn except w2: f16 [C, 4C] when w2_is_f16 (the production format, packer `fc2.wh`), else bf16;
 * C in {96, 192, 384}, any M. */
int fvhd_convffn_half(fvhd_handle h, void* stream, const void* z, const void* w1, const void* b1, const void* w2, int w2_is_f16, const void* b2,
                  const void* resid, void* out, int M, int C);

/* Test entry: the RepMixer depthwise pair of one block, mci.py:808-811 + :921, on the kernel FVHD_MIXER selected for this handle at
 * fvhd_create (default: Toeplitz tcgen05, mixer_tz.cuh):
 *   y = dw3x3(x) + b3,  z = dw7x7(y) + b7;  x, y, z device bf16 NHWC [B,H,W,C]; w3 [9][C], w7 [49][C], b3, b7 [C] fp32 (tap-major,
 *   BN folded).  C % 16 == 0. */
int fvhd_mixer(fvhd_handle h, void* stream, const void* x, const void* w3, const void* b3, const void* w7, const void* b7,
               void* y, void* z, int batch, int H, int W, int C);

/* Stand-alone fused ConvFFN entry (tests, traces): out[M,C] = resid + fc2(GELU(fc1(z) + b1)) + b2  (mci.py:922-926 with the
 * layer scale folded into w2 / b2), bf16 operands, fp32 biases; w1 [4C, C], w2 [C, 4C] row-major.  C = 96 / 192 run the
 * single-CTA kernel, C = 384 the 4-CTA-cluster kernel (hidden split across the cluster, DSMEM reduction); `trace` (C = 384
 * only, may be NULL) receives 64 globaltimer stamps per CTA. */
int fvhd_convffn(fvhd_handle h, void* stream, const void* z, const void* w1, const void* b1, const void* w2, const void* b2,
                 const void* resid, void* out, int M, int C, void* trace_64_u64_per_cta);

/* ---- row f3: LLM prefill (time to first token) ------------------------------------------------------------------------------
 * replaces: the first call of LlavaQwen2ForCausalLM.forward inside generate() (llava_qwen.py:57-103 -> transformers
 * Qwen2ForCausalLM.forward -> Qwen2Model.forward: 24 x [RMSNorm, q/k/v proj + bias, RoPE, causal GQA attention, o proj, RMSNorm,
 * SwiGLU MLP], final RMSNorm, lm_head on the last position; predict.py:58-65) for ONE sequence of L spliced embeddings.
 * The four GEMMs of a layer run on the tower's tcgen05 GEMM kernel; RMSNorm / RoPE / attention / SwiGLU / argmax are llm.cuh.
 *
 * fvhd_llm_load: `weights` are caller-owned DEVICE pointers, 7 per layer then 2:
 *     ln1 f32[H] | wqkv bf16[(heads+2kv)*D, H] (q rows, k rows, v rows) | bqkv f32[(heads+2kv)*D] | wo bf16[H, heads*D] | ln2 f32[H] |
 *     wgu bf16[2I, H] (gate rows then up rows) | wd bf16[H, I]      ...      final_norm f32[H] | lm_head bf16[V, H]
 * Activations, the RoPE table and a KV cache [layers, max_seq, kv*D] x 2 are owned by the handle.
 * fvhd_llm_input: device buffer [max_seq, H] bf16 the caller fills with the spliced sequence (text embeddings + visual tokens; the
 *     projector epilogue can store straight into it: fvhd_forward_strided / _scatter).
 * fvhd_llm_prefill: runs the L-token prefill as one CUDA graph on `stream`; optionally copies the last position's logits
 *     (bf16 [V], device) and the argmax token (int32, device or pinned host) out.  Does not synchronise.
 * fvhd_llm_kv_cache: the K (post-RoPE) and V rows of every layer written by the last prefill, for the decode loop. */
int fvhd_llm_load(fvhd_handle h, const fvhd_llm_config* cfg, const void* const* weights, int n_weights);
void* fvhd_llm_input(fvhd_handle h);
int fvhd_llm_prefill(fvhd_handle h, void* stream, int L, void* logits_out, int* token_out);
int fvhd_llm_kv_cache(fvhd_handle h, void** k_out, void** v_out);
int fvhd_llm_launches(fvhd_handle h, int L);

#ifdef __cplusplus
}
#endif
#endif /* FASTVITHD_B200_H */

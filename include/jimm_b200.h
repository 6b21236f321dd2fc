/* jimm_b200 -- C ABI of the B200-native ViT / CLIP / SigLIP inference forward path.
 *
 * The reference (pythoncrazy/jimm) has no FFI boundary: its boundary is the Python class surface
 * (src/jimm/models/{vit,clip,siglip}.py, src/jimm/common/{vit,transformer}.py).  This header is the C-ABI
 * underneath the drop-in Python mirror in jimm_b200/ (ctypes binding: jimm_b200/_lib.py; the stub a reference
 * maintainer would add is shown in INTEGRATION.md).  Each entry point cites the reference interface it replaces.
 *
 * Conventions
 *   - one opaque jimm_model_t per GPU; a handle is not thread-safe, distinct handles are;
 *   - every call returns 0 on success or a negative jimm_status; the message is in jimm_last_error() (thread-local);
 *   - "device" pointers are CUDA device pointers on the model's GPU; "host" pointers are CPU memory (pinned memory
 *     makes the copies asynchronous);
 *   - all work is enqueued on the caller's stream (a cudaStream_t passed as void*; NULL = default stream) and the call
 *     returns without synchronising, like JAX's asynchronous dispatch (examples/vit_inference.py:54);
 *   - images are NHWC (tests/test_vit.py:46), token ids int32 [B,T];
 *   - no C++ exceptions cross this boundary.
 */
#ifndef JIMM_B200_H_
#define JIMM_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define JIMM_API __attribute__((visibility("default")))
#else
#define JIMM_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct jimm_model jimm_model_t;

enum jimm_status { JIMM_OK = 0, JIMM_EINVAL = -1, JIMM_ECUDA = -2, JIMM_EDRIVER = -3, JIMM_ESTATE = -4, JIMM_ENOMEM = -5 };
enum jimm_dtype { JIMM_F32 = 0, JIMM_F16 = 1, JIMM_BF16 = 2, JIMM_I32 = 3 };
enum jimm_kind {
  JIMM_VIT = 0, JIMM_CLIP = 1, JIMM_SIGLIP = 2, JIMM_TOWER = 3 /* bare VisionTransformerBase */,
  JIMM_ENCODER = 4 /* bare Transformer / TransformerEncoder stack (common/transformer.py:22-196) */,
  JIMM_MAPHEAD = 5 /* bare MultiHeadAttentionPoolingHead (common/vit.py:12-101) */
};
enum jimm_pool { JIMM_POOL_CLS = 0, JIMM_POOL_MAP = 1 };
enum jimm_act { JIMM_GELU_TANH = 0, JIMM_QUICK_GELU = 1 };
enum jimm_text_pool { JIMM_TPOOL_EOT_ARGMAX = 0, JIMM_TPOOL_LAST = 1 };

/* Mirrors the constructor kwargs of VisionTransformer (models/vit.py:23-40), VisionTransformerBase
 * (common/vit.py:107-126), CLIP (models/clip.py:16-31) and SigLIP (models/siglip.py:16-31). */
typedef struct jimm_config {
  int kind;                               /* jimm_kind */
  /* vision tower */
  int img_size, patch, in_ch, v_width, v_layers, v_heads, v_mlp;
  int pooling;                            /* jimm_pool */
  int pre_norm, patch_bias, v_act;        /* use_pre_norm, use_patch_bias, use_quick_gelu */
  float v_eps_outer;                      /* ln_pre / ln_post / MAP layernorm: 1e-12 ViT | 1e-5 CLIP | 1e-6 SigLIP */
  float v_eps_block;                      /* encoder-block LayerNorm eps: 1e-6 (common/transformer.py:142; never overridden) */
  int num_classes;                        /* ViT classifier width; 0 = no classifier (do_classification=False) */
  /* text tower (CLIP / SigLIP) */
  int ctx_len, vocab, t_width, t_heads, t_layers, t_mlp;
  int t_act, t_causal, t_pool, t_head_bias;
  float t_eps_outer, t_eps_block;
  /* numerics */
  int compute_dtype;                      /* jimm_dtype of the tensor-core operands: F32 (tf32 MMA) | F16 | BF16;
                                             accumulation, residual stream, LN statistics, softmax, logits are fp32 */
} jimm_config_t;

JIMM_API const char* jimm_last_error(void);
/* ABI version of this header (bumped on any signature change). */
JIMM_API int jimm_abi_version(void);

/* -- lifecycle: replaces Module.__init__ + from_pretrained's parameter hand-off (models/vit.py:171-257) ----------- */
JIMM_API int jimm_model_create(const jimm_config_t* cfg, int device, jimm_model_t** out);
/* Hand one parameter over in the reference's flax layout, keyed by the reference's flat-state path joined with '.'
 * (e.g. "encoder.transformer.blocks.layers.0.attn.query.kernel", shape (D,H,d); SURVEY.md 8b table).
 * `host` is read during the call.  dtype: JIMM_F32 | JIMM_F16 | JIMM_BF16. */
JIMM_API int jimm_model_set_param(jimm_model_t* m, const char* flax_path, const void* host, const int64_t* shape, int ndim, int dtype);
/* Zero-copy hand-off: `host` is BORROWED and must stay valid and unchanged until jimm_model_finalize returns (e.g. the mmap of a
 * safetensors file).  `shape` is still the reference's flax shape.  flags & JIMM_PARAM_TRANSPOSED: the memory holds the 2-D transpose
 * [N, K] of the flax kernel's (K, N) view -- a HuggingFace (out, in) weight exactly as stored in the checkpoint, i.e. the transform
 * `W.T.reshape(...)` of models/vit.py:241-250 is NOT applied by the caller; that is already the K-major operand layout of the GEMMs,
 * so finalize only casts it.  Casts, transposes and packing run on the GPU; bytes go through a pinned staging ring; finalize
 * synchronises once. */
enum jimm_param_flags { JIMM_PARAM_TRANSPOSED = 1 };
JIMM_API int jimm_model_set_param_ref(jimm_model_t* m, const char* flax_path, const void* host, const int64_t* shape, int ndim, int dtype,
                                      int flags);
/* Pack weights (fused [3D,D] QKV, K-major operands, dtype cast), build TMA descriptors, size the workspace for
 * `max_batch` samples per call.  Fails (JIMM_ESTATE) naming the first missing / unexpected / mis-shaped parameter --
 * the analogue of the reference's strict visit checks (models/vit.py:229-232,259-268). */
JIMM_API int jimm_model_finalize(jimm_model_t* m, int max_batch);
JIMM_API int jimm_model_destroy(jimm_model_t* m);
/* Introspection used by the Python mirror. */
JIMM_API int jimm_model_output_dim(const jimm_model_t* m, int* vision_out, int* text_out);
JIMM_API int jimm_model_max_batch(const jimm_model_t* m);

/* -- forward: device-resident inputs/outputs ---------------------------------------------------------------------- */
/* VisionTransformer.__call__ (models/vit.py:91-103) / VisionTransformerBase.__call__ (common/vit.py:216-248).
 * img: device NHWC [B,img,img,in_ch] of in_dtype; out: device fp32 [B, num_classes | v_width]. */
JIMM_API int jimm_vit_forward(jimm_model_t* m, const void* img, int in_dtype, int B, float* out, void* stream);
/* CLIP.encode_image (models/clip.py:135-146) / SigLIP.encode_image (models/siglip.py:123-133); out fp32 [B,E]. */
JIMM_API int jimm_encode_image(jimm_model_t* m, const void* img, int in_dtype, int B, float* out, void* stream);
/* CLIP.encode_text (models/clip.py:148-167) / SigLIP.encode_text (models/siglip.py:135-153); ids device int32 [B,T]. */
JIMM_API int jimm_encode_text(jimm_model_t* m, const int32_t* ids, int B, int T, float* out, void* stream);
/* L2-normalise + exp(logit_scale) * I . T^T (+ logit_bias) (models/clip.py:183-187, models/siglip.py:169-173).
 * img_e fp32 [Bi,E], txt_e fp32 [Bt,E] (un-normalised encoder outputs), logits fp32 [Bi,Bt] row stride Bt. */
JIMM_API int jimm_contrastive_logits(jimm_model_t* m, const float* img_e, int Bi, const float* txt_e, int Bt, float* logits, void* stream);
/* encode_image + encode_text of one CLIP / SigLIP call with the two (independent) towers running CONCURRENTLY: the text tower is forked onto
 * a side stream and joined back into `stream`, so the idle SMs of one tower's GEMM tail rounds are filled by the other tower.
 * img_e fp32 [Bi,E], txt_e fp32 [Bt,E] (un-normalised, as jimm_encode_image / jimm_encode_text return them). */
JIMM_API int jimm_dual_encode(jimm_model_t* m, const void* img, int in_dtype, int Bi, const int32_t* ids, int Bt, int T, float* img_e, float* txt_e,
                     void* stream);
/* CLIP.__call__ / SigLIP.__call__ (models/clip.py:169-188, models/siglip.py:155-174) on one GPU. */
JIMM_API int jimm_dual_forward(jimm_model_t* m, const void* img, int in_dtype, int Bi, const int32_t* ids, int Bt, int T, float* logits,
                      void* stream);

/* -- forward of a bare sub-module (kinds JIMM_ENCODER / JIMM_MAPHEAD; config fields used: v_width, v_heads, v_mlp, v_layers, v_act,
 *    v_eps_block, v_eps_outer, t_causal (attn_mask = tril), ctx_len = max tokens per sample, compute_dtype; parameters keyed
 *    "blocks.layers.{i}.<...>" resp. "probe", "attn.<...>", "layernorm.<...>", "mlp.layers.{0,2}.<...>") ---------------------------- */
/* Transformer.__call__ / TransformerEncoder.__call__ (common/transformer.py:116-132,190-196): x, out device fp32 [B,S,D]. */
JIMM_API int jimm_encoder_forward(jimm_model_t* m, const float* x, int B, int S, float* out, void* stream);
/* MultiHeadAttentionPoolingHead.__call__ (common/vit.py:87-101): x device fp32 [B,S,D] -> out device fp32 [B,D]. */
JIMM_API int jimm_map_head_forward(jimm_model_t* m, const float* x, int B, int S, float* out, void* stream);

/* -- forward: HOST buffers (the reference-facing call: host->device copy, forward, device->host copy, all enqueued on
 *    `stream`; the caller synchronises the stream before reading `out`).  examples/vit_inference.py:52-58. ----------- */
JIMM_API int jimm_vit_forward_host(jimm_model_t* m, const void* img_host, int in_dtype, int B, float* out_host, void* stream);
JIMM_API int jimm_dual_forward_host(jimm_model_t* m, const void* img_host, int in_dtype, int Bi, const int32_t* ids_host, int Bt, int T,
                           float* logits_host, void* stream);
/* The whole examples/vit_inference.py:27-58 pipeline from raw frames: host uint8 RGB [B,H,W,3] -> (bytes over PCIe, a quarter of the
 * fp32 pixel values) -> image front-end `pre` on the GPU (see jimm_preproc_* below; its output size must equal the model's input) ->
 * tower -> host fp32 [B, num_classes | v_width].  Same slicing / stream semantics as jimm_vit_forward_host. */
typedef struct jimm_preproc jimm_preproc_t;
JIMM_API int jimm_vit_forward_host_u8(jimm_model_t* m, jimm_preproc_t* pre, const uint8_t* img_host, int B, int H, int W, float* out_host,
                                      void* stream);

/* -- multi-GPU contrastive head: one process per GPU, embeddings exchanged over NVLink peer memory ------------------- */
/* Allocate this rank's symmetric gather buffer ([world*max_rows, 2E] fp32 + flags) and export its IPC handle
 * (64 bytes).  The handles of all ranks are exchanged by the caller (torch.distributed / any out-of-band channel). */
JIMM_API int jimm_comm_init(jimm_model_t* m, int rank, int world, int max_rows_per_rank, unsigned char* handle_out /*[64]*/);
JIMM_API int jimm_comm_connect(jimm_model_t* m, const unsigned char* handles /*[world*64]*/);
/* Fused: L2-normalise the local [B_local,E] image/text embeddings, store them straight into every peer's gather buffer
 * over NVLink (st.global on mapped peer pointers), device-side flag barrier, then the local rank's logits row block
 * logits_local fp32 [B_local, world*B_local] = exp(scale) * I_local . T_all^T (+ bias).  No host synchronisation. */
JIMM_API int jimm_comm_contrastive_logits(jimm_model_t* m, const float* img_e, const float* txt_e, int B_local, float* logits_local,
                                 void* stream);
/* The device-side wait for the peers is bounded (JIMM_COMM_TIMEOUT_MS, default 10 s) and every rank must pass the same B_local: a
 * missing or mismatched peer yields NaN logits and a sticky error, returned here (after the stream has been synchronised) and by the
 * next jimm_comm_contrastive_logits call. */
JIMM_API int jimm_comm_status(jimm_model_t* m);
/* Device pointer to this rank's gathered, normalised [world*B_local, 2E] buffer (valid after the call above). */
JIMM_API int jimm_comm_gathered(jimm_model_t* m, float** gathered, int* row_stride);

/* -- per-kernel entry points (device pointers; used by tests/ and the ncu harness so every kernel is individually
 *    parity- and profile-testable; SURVEY.md 8b) ------------------------------------------------------------------- */
/* Type codes of the per-kernel entries: dtype / io_type / in_type are JIMM_F32 | JIMM_F16 | JIMM_BF16 (JIMM_F32 operands of the GEMM are
 * read as tf32).  An out_type may also be 3 (the value of JIMM_I32), which here means "fp32 rounded to tf32": fp32 storage with the low 13
 * mantissa bits zero, the operand format the fp32 compute mode stores between layers.  Any other out_type is rejected (JIMM_EINVAL). */
/* C[M,N] = epi(A[M,K] . B[N,K]^T): impl 0 = tcgen05/TMA kernel, 1 = SIMT cross-check.
 * act: 0 none | 1 gelu_tanh | 2 quick_gelu; epi_mode 0 staged | 1 direct | 2 TMA store / reduce-add (0 when not applicable);
 * rows_in>0 remaps output rows. */
JIMM_API int jimm_k_gemm(int impl, int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias, int act,
                const float* rowadd, const float* residual, int ldr, void* out, int out_type, int ldo, int rows_in, int rows_out,
                int row_off, int epi_mode, void* stream);
/* The tcgen05 GEMM of jimm_k_gemm with the plan-time and run-time knobs of the model forward:
 *   - the plan is built for M rows and run on run_M rows (0 = M; 1 <= run_M <= M): the schedule (single CTA or CTA pair, tail split)
 *     follows run_M.  With the TMA epilogue (epi_mode 2) rows [run_M, min(M, ceil32(run_M))) are written too (see gemm_plan_run);
 *   - reverse = 1 walks the tiles from the end (same results, bit for bit);
 *   - tok_pad > 0: token-scatter reduce-add of the patch embedding.  A row b * tok_pad + p is added to out[b, p + tok_off, :] of an fp32
 *     [M / tok_pad, tok_S, N] tensor (row stride ldo); rows with p + tok_off >= tok_S are dropped.  Needs residual == out, ldr == ldo,
 *     out_type JIMM_F32, epi_mode 2, tok_pad a multiple of 32 dividing M, no rowadd / row remap. */
JIMM_API int jimm_k_gemm_ex(int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias, int act,
                            const float* rowadd, const float* residual, int ldr, void* out, int out_type, int ldo, int rows_in, int rows_out,
                            int row_off, int tok_pad, int tok_off, int tok_S, int run_M, int reverse, int epi_mode, void* stream);
JIMM_API int jimm_k_layernorm(const float* x, int ldx, int group, int row_off, const int32_t* row_index, const float* scale, const float* bias,
                     float eps, void* out, int out_type, int ldy, int rows, int D, void* stream);
/* reverse = 1: the same LayerNorm / attention with rows (resp. (sample, head) items) walked from the end, as every other launch of an
 * encoder block does; the results are bit-identical to reverse = 0. */
JIMM_API int jimm_k_layernorm_ex(const float* x, int ldx, int group, int row_off, const int32_t* row_index, const float* scale, const float* bias,
                                 float eps, void* out, int out_type, int ldy, int rows, int D, int reverse, void* stream);
JIMM_API int jimm_k_attention(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, void* stream);
JIMM_API int jimm_k_attention_ex(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, int reverse, void* stream);
JIMM_API int jimm_k_map_attention(const float* q, const void* kv, int io_type, void* out, int out_type, int B, int S, int H, void* stream);
JIMM_API int jimm_k_patchify(const void* img, int in_type, int B, int H, int W, int C, int P, void* out, int out_type, void* stream);
/* y = act(x) elementwise on device fp32 (act: 1 tanh-GELU == nnx.gelu, 2 QuickGELU == common/transformer.py:12-19). */
JIMM_API int jimm_k_activation(const float* x, float* y, long long n, int act, void* stream);
JIMM_API int jimm_k_embed(const int32_t* ids, const float* table, const float* pos, float* x, int B, int T, int D, int vocab, void* stream);
JIMM_API int jimm_k_l2_normalize(const float* x, float* out, int ldo, int B, int E, void* stream);
JIMM_API int jimm_k_logits(const float* img, const float* txt, const float* logit_scale, const float* logit_bias, float* logits, int Bi, int Bt,
                  int E, int ldl, void* stream);
/* ---- image front-end (SURVEY.md 8f.1): the HuggingFace image processor the reference's examples run on the host ----
 * Replaces `processor(images=..., return_tensors="np")["pixel_values"]` + the NCHW->NHWC transpose of
 * examples/vit_inference.py:27-37, examples/clip_inference.py:35-38 (transformers 4.53.0 slow processors on Pillow 11.3.0,
 * uv.lock:2679,1573): Pillow 8-bit resize with antialiasing (bilinear | bicubic) -> optional centre crop -> rescale ->
 * normalise, written NHWC in the dtype the tower consumes.  Bit-exact with that pipeline (integer resampling, IEEE fp32
 * rescale/normalise).  Mirrors `preprocessor_config.json`: size {height,width} | {shortest_edge}, crop_size, resample,
 * rescale_factor, image_mean, image_std. */
typedef struct jimm_preproc_config {
  int height, width;        /* exact output size (ViT, SigLIP: size = {height, width}) ... */
  int shortest_edge;        /* ... or, when non-zero, resize the shortest edge to this keeping the aspect ratio (CLIP) */
  int crop_h, crop_w;       /* centre crop after the resize (CLIP crop_size); 0 = none */
  int resample;             /* PIL code: 2 bilinear, 3 bicubic */
  double rescale_factor;    /* 1/255 */
  float mean[3], std[3];    /* image_mean, image_std */
} jimm_preproc_config_t;
JIMM_API int jimm_preproc_create(const jimm_preproc_config_t* cfg, int device, jimm_preproc_t** out);
JIMM_API int jimm_preproc_output_size(const jimm_preproc_t* p, int H, int W, int* out_h, int* out_w);
/* img: device uint8 [B,H,W,3] (same-sized RGB images); out: device [B,out_h,out_w,3] of out_dtype (JIMM_F32 | JIMM_F16 | JIMM_BF16). */
JIMM_API int jimm_preproc_run(jimm_preproc_t* p, const uint8_t* img, int B, int H, int W, void* out, int out_dtype, void* stream);
JIMM_API int jimm_preproc_destroy(jimm_preproc_t* p);
/* Host-only test entry: Pillow's resampling windows and 22-bit fixed-point weights for one axis. */
JIMM_API int jimm_k_resample_coeffs(int in_size, int out_size, int resample, int* ksize, int* first, int* count, int* kk, int kk_capacity);
/* ---- zero-shot / classification epilogue (SURVEY.md 8f.3): what the examples compute in JAX after the forward ----
 * logits: device fp32 [rows, cols] (leading dimension ld).  mode 0: probs = exp(x) / sum(exp(x)) per row, un-shifted like
 * examples/clip_inference.py:47; mode 1: probs = sigmoid(x) (SigLIP pair probabilities).  order (nullable, int32 [rows, cols]):
 * `argsort(x)[::-1]` per row -- descending, equal scores with the larger index first (examples/clip_inference.py:49);
 * argmax (nullable, int32 [rows]): first maximum per row (examples/vit_inference.py:58).  order / argmax need cols <= 4096. */
JIMM_API int jimm_postprocess(const float* logits, int rows, int cols, int ld, int mode, float* probs, int ldp, int32_t* order, int32_t* argmax,
                              void* stream);
/* Micro-benchmark (not on the product path): TMA fill bandwidth from L2 with `cluster` CTAs per cluster.  mode 0: every CTA loads
 * its own 16 KB tiles; 1: the CTAs of a cluster load the same tile each; 2: same tile, each loads 1/cluster of it and multicasts. */
JIMM_API int jimm_k_l2_probe(const void* buf, int rows, int mode, int cluster, int iters, float* ms, void* stream);
/* Live timing of the dominant kernel (the tcgen05 GEMM) inside a forward: between begin and end every GEMM launch is
 * bracketed by CUDA events on the launch stream; end synchronises and returns the summed device time (ms), the
 * algorithmic FLOPs (2*M*N*K per launch) and the number of launches.  Used by bench.py's roofline object. */
JIMM_API int jimm_profile_begin(jimm_model_t* m);
JIMM_API int jimm_profile_end(jimm_model_t* m, double* gemm_ms, double* gemm_flops, long long* gemm_launches);
/* Count of kernel launches issued by this library since process start (bench.py's gpu_launches). */
JIMM_API long long jimm_launch_count(void);
/* Count of tower forwards replayed from a captured CUDA graph (batches <= JIMM_GRAPH_MAX_BATCH, default 32, from the
 * second call of a shape on); their kernels are included in jimm_launch_count. */
JIMM_API long long jimm_graph_replay_count(void);

#ifdef __cplusplus
}
#endif
#endif /* JIMM_B200_H_ */

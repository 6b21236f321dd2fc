// Host-callable launchers for the non-GEMM kernels of the forward path (elementwise.cu, attention.cu).
// All enqueue on `stream` and return 0 / negative status (message via jimm_last_error()).
// `reverse`: walk the rows / tiles / items from the end.  Consecutive kernels of an encoder block alternate direction so each
// one starts on the data its producer wrote LAST -- the part still resident in the 126 MB L2 (the activations are 77-310 MB).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm.cuh"

namespace jimm {

// nnx.LayerNorm (fast variance, fp32 statistics) over fp32 rows.  SURVEY 8a row a3.
//   src row for output r:  r * group + (row_index ? row_index[r] : row_off)      (row stride ldx elements)
//   out[r, :] (type out_type, row stride ldy) = (x - mean) * rsqrt(max(0, E[x^2]-mean^2) + eps) * scale + bias
int layernorm_run(const float* x, int ldx, int group, int row_off, const int* row_index, const float* scale, const float* bias,
                  float eps, void* out, int out_type, int ldy, int rows, int D, cudaStream_t stream, int reverse = 0);

// Patchify: NHWC image (in_type fp32/fp16/bf16) -> A matrix [B*gh*gw, P*P*C] of out_type, row order (b,gy,gx), column
// order (ky,kx,c) == the HWIO kernel reshape (common/vit.py:153-165,228-230).  128-bit loads.
int patchify_run(const void* img, int in_type, int B, int H, int W, int C, int P, void* out, int out_type, cudaStream_t stream,
                 int rows_per_sample = 0 /* 0 = gh*gw; larger = padded row count per sample (pad rows untouched) */,
                 int ldk = 0 /* row stride in elements; 0 = P*P*C; larger = zero-padded K (any P / C through the generic kernel) */);

// x[b, s, :] = pos[s, :] (+ cls for s == 0)   -- initial value of the residual stream; the patch GEMM then reduce-adds the
// patch embeddings into rows tok_off.. (common/vit.py:231-236)
int tokens_init_run(float* x, const float* cls, const float* pos, int B, int S, int D, cudaStream_t stream);

// x[b, 0, :] = cls + pos[0]   (common/vit.py:231-236), fp32 residual stream [B, S, D]
int cls_row_run(float* x, const float* cls, const float* pos, int B, int S, int D, cudaStream_t stream);

// x[b,t,:] = table[ids[b,t], :] + pos[t, :]   (models/clip.py:159-160, models/siglip.py:146-147)
int embed_run(const int32_t* ids, const float* table, const float* pos, float* x, int B, int T, int D, int vocab, cudaStream_t stream);

// idx[b] = first argmax_t ids[b, t]    (models/clip.py:164)
int argmax_ids_run(const int32_t* ids, int* idx, int B, int T, cudaStream_t stream);

// rows /= ||row||_2  (no epsilon; models/clip.py:183-184), fp32 [B,E] -> out (row stride ldo)
int l2_normalize_run(const float* x, float* out, int ldo, int B, int E, cudaStream_t stream);

// logits[i,j] = exp(logit_scale) * <img[i], txt[j]> (+ logit_bias)   fp32 SIMT (models/clip.py:186-187, models/siglip.py:172-173)
int logits_run(const float* img, const float* txt, const float* logit_scale, const float* logit_bias, float* logits, int Bi, int Bt,
               int E, int ldl, cudaStream_t stream);

// dst[n*K + k] = cast(src[k*N + n])   (flax (in,out) kernel -> K-major [N,K] operand)
int transpose_cast_run(const float* src, int K, int N, void* dst, int out_type, int ldd, cudaStream_t stream);
int cast_run(const float* src, void* dst, int out_type, size_t n, cudaStream_t stream);

// ---- checkpoint ingestion (pack.cu) ----
// rows of K elements of src_type (DT_F32 | DT_F16 | DT_BF16), row-major -> dst[r * ldd + k] of out_type
int pack_rows_run(const void* src, int src_type, size_t rows, size_t K, void* dst, int out_type, size_t ldd, cudaStream_t stream);
// kc rows (starting at row k0) of a (K, N) row-major matrix of src_type -> dst[n * ldd + k0 + k] of out_type (K-major operand)
int pack_transpose_run(const void* src, int src_type, int kc, int N, void* dst, int out_type, size_t ldd, int k0, cudaStream_t stream);
// two pinned host slots + two device slots: memcpy of chunk i+1 overlaps the DMA and the pack kernel of chunk i
struct UploadRing {
  static constexpr size_t kCap = static_cast<size_t>(32) << 20;
  void* pinned[2] = {nullptr, nullptr};
  void* dev[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  bool busy[2] = {false, false};
  int cur = 0;
  bool ready = false;
  int init();
  void destroy();
  int stage(const void* src, size_t bytes, cudaStream_t s, void** dptr);  // host -> pinned slot -> device slot (async); *dptr = device slot
  int commit(cudaStream_t s);                                              // after the consuming kernel has been enqueued
};
int activation_run(const float* x, float* y, size_t n, int act /* 0 none, 1 gelu_tanh, 2 quick_gelu */, cudaStream_t stream);

// Multi-head softmax attention over the fused qkv buffer [B*S, 3D] (q | k | v, heads of 64).  SURVEY 8a row a5.
//   o[b*S+s, h*64+d] = softmax_k((q/8) k^T  masked) v ; causal: key <= query.  io_type fp16/bf16; out_type fp16/bf16/fp32
int attention_run(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, cudaStream_t stream, int reverse = 0);

// tcgen05 variant for S <= 256 (attention_tc.cu); returns 1 when the configuration is not handled (caller falls back).
int attention_tc_run(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, cudaStream_t stream, int reverse = 0);

// tcgen05 two-pass variant for S > 256, non-causal (attention_tc_long.cu); returns 1 when not handled.
int attention_tc_long_run(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, cudaStream_t stream, int reverse = 0);

// MAP-head attention with a single (input-independent) probe query (common/vit.py:96-97).
//   q: fp32 [H*64] (already projected + biased), kv: [B*S, 2D] (k | v) io_type, out [B, D] out_type
int map_attention_run(const float* q, const void* kv, int io_type, void* out, int out_type, int B, int S, int H, cudaStream_t stream);

}  // namespace jimm

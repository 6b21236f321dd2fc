// Host-side interface of the tcgen05/TMA GEMM (gemm.cu).
//
//   C[M,N] = epilogue( A[M,K] . B[N,K]^T )      A, B K-major ("TN"), fp32 accumulate in TMEM
//
// This one kernel serves every dense contraction on the jimm forward path
// (SURVEY.md 8a rows a1,a4,a6,a7,a9,a10): patch-embed, fused QKV, attention
// out-projection (+residual), MLP FC1 (+GELU/QuickGELU), FC2 (+residual), MAP-head
// k/v + MLP, classifier / projections.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace jimm {

// DT_TF32: stored as fp32 with the value rounded (to nearest) to tf32 -- the operand format of the fp32 compute mode, so the
// tensor core's truncation of the low 13 mantissa bits is exact.  Only ever an internal buffer / operand type.
enum DType : int { DT_F32 = 0, DT_F16 = 1, DT_BF16 = 2, DT_TF32 = 3 };
enum Act : int { ACT_NONE = 0, ACT_GELU_TANH = 1, ACT_QUICK_GELU = 2 };

inline size_t dtype_size(int dt) { return (dt == DT_F32 || dt == DT_TF32) ? 4 : 2; }

struct GemmEpilogue {
  const float* bias = nullptr;      // [N] fp32, added per output column
  int act = ACT_NONE;               // applied after bias
  const float* rowadd = nullptr;    // fp32 [*, N]; row (r % rows_in + row_off) added (position embeddings)
  const float* residual = nullptr;  // fp32, indexed like the output (out_row, ldr); may alias out
  int ldr = 0;
  void* out = nullptr;
  int out_type = DT_F32;
  int ldo = 0;                                   // output row stride (elements)
  // Token-scatter form of the fp32 reduce-add epilogue (patch embedding): A rows are (sample, padded patch index) with
  // tok_pad rows per sample (multiple of 32); row (b, p) is ADDED to out[b, p + tok_off, :] of a [B, tok_S, N] tensor through a
  // 3-D tensor map (rows p + tok_off >= tok_S are clipped by TMA).  Requires residual == out (pre-initialised with pos-emb).
  int tok_pad = 0, tok_off = 0, tok_S = 0;
  int reverse = 0;  // walk the M tiles from the end (L2-resident part of the A operand first; see kernels.cuh)
  int rows_in = 0, rows_out = 0, row_off = 0;    // out_row = (r / rows_in) * rows_out + r % rows_in + row_off (rows_in == 0: identity)
  // 2: TMA epilogue (swizzled smem box -> cp.async.bulk.tensor store, cp.reduce .add for the fp32 residual stream; needs
  //    no rowadd / row remap and residual == out) -- falls back to 0 when not applicable;
  // 0: smem-staged, coalesced LSU stores; 1: direct row-per-thread LSU stores
  int mode = 2;
};

struct GemmPlan {
  CUtensorMap map_a, map_b, map_b_pair, map_c;  // map_b_pair: 128-row B box (CTA-pair mode); map_c: output (mode 2 only)
  int M = 0, N = 0, K = 0;
  int dtype = DT_F16;  // operand type: DT_F16 / DT_BF16 / DT_F32 (tf32 MMA)
  GemmEpilogue epi;
};

// Build TMA descriptors for A [M,K] (row stride lda elements) and B [N,K] (row stride ldb).
// Returns 0 or a negative status (message in jimm_last_error()).
int gemm_plan_init(GemmPlan* plan, int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K,
                   const GemmEpilogue& epi);
// Enqueue on `stream`; M may be overridden (<= planned M) to run on fewer rows of the same buffers.  The schedule (single CTA or
// CTA pair, tail split) is chosen for the overriding M.  The TMA epilogue (mode 2) stores or reduce-adds whole 32-row boxes, clipped
// only at the PLANNED M (the output tensor map): rows [M_override, min(planned M, ceil32(M_override))) are written too, with the
// epilogue applied to the A rows there (whatever the buffer holds).  The LSU epilogues (modes 0 / 1) write rows < M_override only.
int gemm_plan_run(const GemmPlan* plan, int M_override, cudaStream_t stream, int reverse = 0);

// Simple SIMT reference GEMM (debug / bring-up cross-check on the GPU; never on the product path
// unless JIMM_GEMM_IMPL=simt is set for bisection).
int gemm_simt_run(int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K, const GemmEpilogue& epi,
                  cudaStream_t stream);

int device_sm_count();

}  // namespace jimm

// HBM-bound kernels of the forward path: LayerNorm, patchify, CLS row, token embedding, pooling helpers,
// L2-normalise, fp32 logits, weight packing.  128-bit vectorised loads/stores, warp-shuffle reductions.
#include <limits.h>
#include <stdio.h>

#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"
#include "logits_tile.cuh"

namespace jimm {

// ------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, row kept in registers (D <= 2048), fp32 statistics.
// ------------------------------------------------------------------------------------------
template <typename OutT, int MAXV>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* __restrict__ x, size_t ldx, int group, int row_off, const int* __restrict__ row_index,
                 const float* __restrict__ scale, const float* __restrict__ bias, float eps, OutT* __restrict__ out, size_t ldy,
                 int rows, int D, int reverse) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (warp >= rows) return;
  if (reverse) warp = rows - 1 - warp;
  const size_t src_row = static_cast<size_t>(warp) * group + (row_index ? row_index[warp] : row_off);
  const float4* xr = reinterpret_cast<const float4*>(x + src_row * ldx);
  const int nv = D >> 2;
  float4 v[MAXV];
  float s = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) {
      v[i] = xr[idx];
      s += v[i].x + v[i].y + v[i].z + v[i].w;
      s2 += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
    }
  }
  s = warp_sum(s);
  s2 = warp_sum(s2);
  const float inv_d = 1.0f / static_cast<float>(D);
  const float mean = s * inv_d;
  const float var = fmaxf(s2 * inv_d - mean * mean, 0.0f);  // flax use_fast_variance=True
  const float rstd = rsqrtf(var + eps);
  const float4* sc = reinterpret_cast<const float4*>(scale);
  const float4* bi = reinterpret_cast<const float4*>(bias);
  OutT* orow = out + static_cast<size_t>(warp) * ldy;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    if (idx < nv) {
      const float4 g = __ldg(sc + idx), b = __ldg(bi + idx);
      float4 y;
      y.x = (v[i].x - mean) * rstd * g.x + b.x;
      y.y = (v[i].y - mean) * rstd * g.y + b.y;
      y.z = (v[i].z - mean) * rstd * g.z + b.z;
      y.w = (v[i].w - mean) * rstd * g.w + b.w;
      if constexpr (std::is_same<OutT, tf32_t>::value) {
        reinterpret_cast<float4*>(orow)[idx] = make_float4(round_tf32(y.x), round_tf32(y.y), round_tf32(y.z), round_tf32(y.w));
      } else if constexpr (sizeof(OutT) == 4) {
        reinterpret_cast<float4*>(orow)[idx] = y;
      } else {
        uint2 p;
        constexpr int ot = std::is_same<OutT, __half>::value ? 1 : 2;
        p.x = pack2(y.x, y.y, ot);
        p.y = pack2(y.z, y.w, ot);
        reinterpret_cast<uint2*>(orow)[idx] = p;
      }
    }
  }
}

template <typename OutT>
static int ln_launch(const float* x, int ldx, int group, int row_off, const int* row_index, const float* scale, const float* bias,
                     float eps, void* out, int ldy, int rows, int D, cudaStream_t stream, int reverse) {
  const int threads = 256, wpb = threads / 32;
  const int grid = (rows + wpb - 1) / wpb;
  const int nv = D / 4;
  if (nv <= 32 * 8)
    JIMM_CUDA_CHECK(launch_k(layernorm_kernel<OutT, 8>, dim3(grid), dim3(threads), 0, stream, 1, true, x, ldx, group, row_off, row_index, scale, bias, eps,
                             static_cast<OutT*>(out), ldy, rows, D, reverse));
  else
    JIMM_CUDA_CHECK(launch_k(layernorm_kernel<OutT, 16>, dim3(grid), dim3(threads), 0, stream, 1, true, x, ldx, group, row_off, row_index, scale, bias, eps,
                             static_cast<OutT*>(out), ldy, rows, D, reverse));
  note_launch();
  return 0;
}

int layernorm_run(const float* x, int ldx, int group, int row_off, const int* row_index, const float* scale, const float* bias,
                  float eps, void* out, int out_type, int ldy, int rows, int D, cudaStream_t stream, int reverse) {
  if (D % 4 != 0 || D > 2048 || ldx % 4 != 0 || ldy % 4 != 0) {
    set_last_error("layernorm: D=%d must be a multiple of 4 and <= 2048 (ldx=%d ldy=%d)", D, ldx, ldy);
    return -1;
  }
  if (out_type < DT_F32 || out_type > DT_TF32) { set_last_error("layernorm: bad out_type %d", out_type); return -1; }
  if (rows <= 0) return 0;
  if (out_type == DT_F32) return ln_launch<float>(x, ldx, group, row_off, row_index, scale, bias, eps, out, ldy, rows, D, stream, reverse);
  if (out_type == DT_TF32) return ln_launch<tf32_t>(x, ldx, group, row_off, row_index, scale, bias, eps, out, ldy, rows, D, stream, reverse);
  if (out_type == DT_F16) return ln_launch<__half>(x, ldx, group, row_off, row_index, scale, bias, eps, out, ldy, rows, D, stream, reverse);
  return ln_launch<__nv_bfloat16>(x, ldx, group, row_off, row_index, scale, bias, eps, out, ldy, rows, D, stream, reverse);
}

// ------------------------------------------------------------------------------------------
// Patchify: each thread moves 4 consecutive source elements (one 128-bit load for fp32 input).
// ------------------------------------------------------------------------------------------
template <typename InT, typename OutT>
__global__ void __launch_bounds__(256)
patchify_kernel(const InT* __restrict__ img, OutT* __restrict__ out, int B, int H, int W, int C, int P, int gh, int gw, int per_img4, int rps) {
  // blockIdx.y = image, 32-bit index arithmetic inside the image (the 64-bit divisions of a flat index made this kernel XU-bound:
  // 61 us for 231 MB, profiles/r2_kernels.md)
  const int i4 = blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= per_img4) return;
  const int b = blockIdx.y;
  const int rem = i4 * 4;
  const int WC = W * C, PC = P * C;
  const size_t e = static_cast<size_t>(b) * H * WC + rem;
  const int y = rem / WC, xc = rem - y * WC;
  const int gx = xc / PC, kc = xc - gx * PC;
  const int gy = y / P, ky = y - gy * P;
  if (gy >= gh || gx >= gw) return;  // VALID conv drops the remainder
  float v[4];
  if constexpr (sizeof(InT) == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(img + e));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(img + e));
    const InT* h = reinterpret_cast<const InT*>(&t);
    for (int j = 0; j < 4; ++j) v[j] = to_float(h[j]);
  }
  const size_t dst = (static_cast<size_t>(b) * rps + static_cast<size_t>(gy) * gw + gx) * (static_cast<size_t>(P) * PC) +
                     static_cast<size_t>(ky) * PC + kc;
  if constexpr (std::is_same<OutT, tf32_t>::value) {
    *reinterpret_cast<float4*>(out + dst) = make_float4(round_tf32(v[0]), round_tf32(v[1]), round_tf32(v[2]), round_tf32(v[3]));
  } else if constexpr (sizeof(OutT) == 4) {
    *reinterpret_cast<float4*>(out + dst) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
    constexpr int ot = std::is_same<OutT, __half>::value ? 1 : 2;
    uint2 p;
    p.x = pack2(v[0], v[1], ot);
    p.y = pack2(v[2], v[3], ot);
    *reinterpret_cast<uint2*>(out + dst) = p;
  }
}

template <typename InT>
static int patchify_dispatch(const void* img, int B, int H, int W, int C, int P, void* out, int out_type, cudaStream_t stream, int rps) {
  const int gh = H / P, gw = W / P;
  if (rps <= 0) rps = gh * gw;
  const int per_img4 = H * W * C / 4;
  const int threads = 256;
  const InT* in = static_cast<const InT*>(img);
  for (int b0 = 0; b0 < B; b0 += 65535) {  // grid.y limit
    const int nb = B - b0 < 65535 ? B - b0 : 65535;
    const dim3 grid(static_cast<unsigned>((per_img4 + threads - 1) / threads), static_cast<unsigned>(nb));
    const InT* src = in + static_cast<size_t>(b0) * H * W * C;
    const size_t ooff = static_cast<size_t>(b0) * rps * P * P * C;
    if (out_type == DT_F32) patchify_kernel<InT, float><<<grid, threads, 0, stream>>>(src, static_cast<float*>(out) + ooff, nb, H, W, C, P, gh, gw, per_img4, rps);
    else if (out_type == DT_TF32) patchify_kernel<InT, tf32_t><<<grid, threads, 0, stream>>>(src, static_cast<tf32_t*>(out) + ooff, nb, H, W, C, P, gh, gw, per_img4, rps);
    else if (out_type == DT_F16) patchify_kernel<InT, __half><<<grid, threads, 0, stream>>>(src, static_cast<__half*>(out) + ooff, nb, H, W, C, P, gh, gw, per_img4, rps);
    else patchify_kernel<InT, __nv_bfloat16><<<grid, threads, 0, stream>>>(src, static_cast<__nv_bfloat16*>(out) + ooff, nb, H, W, C, P, gh, gw, per_img4, rps);
  }
  JIMM_LAUNCH_CHECK();
  return 0;
}

// Generic form (any patch size / channel count, zero-padded K): one thread per OUTPUT element (b, patch, k), k in [0, ldk); columns
// k >= P*P*C are written as zeros so that the row stride ldk can be rounded up to the 16 bytes TMA needs (patch 14 x 3 channels = 588
// elements -> 592: every ViT-L/14 / H/14 CLIP and patch14 SigLIP checkpoint the reference loads).
template <typename InT, typename OutT>
__global__ void __launch_bounds__(256)
patchify_generic_kernel(const InT* __restrict__ img, OutT* __restrict__ out, int H, int W, int C, int P, int gh, int gw, int rps, int ldk,
                        size_t total) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int k = static_cast<int>(i % ldk);
  const size_t r = i / ldk;
  const int n = gh * gw;
  const int b = static_cast<int>(r / n), pt = static_cast<int>(r - static_cast<size_t>(b) * n);
  const int gy = pt / gw, gx = pt - gy * gw;
  float v = 0.f;
  const int PC = P * C;
  if (k < P * PC) {
    const int ky = k / PC, kc = k - ky * PC;  // (kh, kw, c) order == the HWIO kernel reshape
    v = to_float(img[(static_cast<size_t>(b) * H + gy * P + ky) * W * C + static_cast<size_t>(gx) * PC + kc]);
  }
  out[(static_cast<size_t>(b) * rps + pt) * ldk + k] = from_float<OutT>(v);
}

template <typename InT>
static int patchify_generic_dispatch(const void* img, int B, int H, int W, int C, int P, void* out, int out_type, cudaStream_t stream, int rps, int ldk) {
  const int gh = H / P, gw = W / P;
  if (rps <= 0) rps = gh * gw;
  const size_t total = static_cast<size_t>(B) * gh * gw * ldk;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  const InT* in = static_cast<const InT*>(img);
  if (out_type == DT_F32) patchify_generic_kernel<InT, float><<<grid, 256, 0, stream>>>(in, static_cast<float*>(out), H, W, C, P, gh, gw, rps, ldk, total);
  else if (out_type == DT_TF32) patchify_generic_kernel<InT, tf32_t><<<grid, 256, 0, stream>>>(in, static_cast<tf32_t*>(out), H, W, C, P, gh, gw, rps, ldk, total);
  else if (out_type == DT_F16) patchify_generic_kernel<InT, __half><<<grid, 256, 0, stream>>>(in, static_cast<__half*>(out), H, W, C, P, gh, gw, rps, ldk, total);
  else patchify_generic_kernel<InT, __nv_bfloat16><<<grid, 256, 0, stream>>>(in, static_cast<__nv_bfloat16*>(out), H, W, C, P, gh, gw, rps, ldk, total);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ldk: row stride of `out` in elements (0 = P*P*C).  The vectorised kernel needs P*C and W*C to be multiples of 4 and an unpadded row.
int patchify_run(const void* img, int in_type, int B, int H, int W, int C, int P, void* out, int out_type, cudaStream_t stream, int rows_per_sample,
                 int ldk) {
  if (out_type < DT_F32 || out_type > DT_TF32) { set_last_error("patchify: bad out_type %d", out_type); return -1; }
  if (B <= 0) return 0;
  const int PPC = P * P * C;
  if (ldk <= 0) ldk = PPC;
  if (ldk < PPC) { set_last_error("patchify: row stride %d < patch_size^2*channels %d", ldk, PPC); return -1; }
  if ((P * C) % 4 != 0 || (W * C) % 4 != 0 || ldk != PPC) {
    if (in_type == DT_F32) return patchify_generic_dispatch<float>(img, B, H, W, C, P, out, out_type, stream, rows_per_sample, ldk);
    if (in_type == DT_F16) return patchify_generic_dispatch<__half>(img, B, H, W, C, P, out, out_type, stream, rows_per_sample, ldk);
    return patchify_generic_dispatch<__nv_bfloat16>(img, B, H, W, C, P, out, out_type, stream, rows_per_sample, ldk);
  }
  if (in_type == DT_F32) return patchify_dispatch<float>(img, B, H, W, C, P, out, out_type, stream, rows_per_sample);
  if (in_type == DT_F16) return patchify_dispatch<__half>(img, B, H, W, C, P, out, out_type, stream, rows_per_sample);
  return patchify_dispatch<__nv_bfloat16>(img, B, H, W, C, P, out, out_type, stream, rows_per_sample);
}

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
tokens_init_kernel(float4* __restrict__ x, const float4* __restrict__ cls, const float4* __restrict__ pos, size_t total4, int SD4, int D4) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int r = static_cast<int>(i % SD4);  // position inside the sample
  float4 v = __ldg(pos + r);
  if (cls != nullptr && r < D4) {
    const float4 c = __ldg(cls + r);
    v.x += c.x; v.y += c.y; v.z += c.z; v.w += c.w;
  }
  x[i] = v;
}
int tokens_init_run(float* x, const float* cls, const float* pos, int B, int S, int D, cudaStream_t stream) {
  if (B <= 0) return 0;
  if (D % 4 != 0) { set_last_error("tokens_init: D must be a multiple of 4"); return -1; }
  const size_t total4 = static_cast<size_t>(B) * S * D / 4;
  tokens_init_kernel<<<static_cast<unsigned>((total4 + 255) / 256), 256, 0, stream>>>(reinterpret_cast<float4*>(x), reinterpret_cast<const float4*>(cls),
                                                                                         reinterpret_cast<const float4*>(pos), total4, S * D / 4, D / 4);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
__global__ void cls_row_kernel(float* __restrict__ x, const float* __restrict__ cls, const float* __restrict__ pos, int B, size_t SD, int D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * D) return;
  const int b = i / D, d = i - b * D;
  x[static_cast<size_t>(b) * SD + d] = cls[d] + pos[d];
}
int cls_row_run(float* x, const float* cls, const float* pos, int B, int S, int D, cudaStream_t stream) {
  if (B <= 0) return 0;
  const int n = B * D;
  cls_row_kernel<<<(n + 255) / 256, 256, 0, stream>>>(x, cls, pos, B, static_cast<size_t>(S) * D, D);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
embed_kernel(const int32_t* __restrict__ ids, const float* __restrict__ table, const float* __restrict__ pos, float* __restrict__ x,
             int rows, int T, int D4, int vocab) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  int id = ids[warp];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);  // jnp take clamps out-of-range indices
  const int t = warp % T;
  const float4* e = reinterpret_cast<const float4*>(table) + static_cast<size_t>(id) * D4;
  const float4* p = reinterpret_cast<const float4*>(pos) + static_cast<size_t>(t) * D4;
  float4* o = reinterpret_cast<float4*>(x) + static_cast<size_t>(warp) * D4;
  for (int i = lane; i < D4; i += 32) {
    const float4 a = __ldg(e + i), b = __ldg(p + i);
    o[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}
int embed_run(const int32_t* ids, const float* table, const float* pos, float* x, int B, int T, int D, int vocab, cudaStream_t stream) {
  if (D % 4 != 0) { set_last_error("embed: D must be a multiple of 4"); return -1; }
  const int rows = B * T;
  if (rows <= 0) return 0;
  embed_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(ids, table, pos, x, rows, T, D / 4, vocab);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
__global__ void argmax_ids_kernel(const int32_t* __restrict__ ids, int* __restrict__ idx, int B, int T) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  int best = INT_MIN, bi = 0x7fffffff;
  for (int t = lane; t < T; t += 32) {
    const int v = ids[static_cast<size_t>(warp) * T + t];
    if (v > best) { best = v; bi = t; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const int ob = __shfl_xor_sync(0xffffffffu, best, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (lane == 0) idx[warp] = bi;
}
int argmax_ids_run(const int32_t* ids, int* idx, int B, int T, cudaStream_t stream) {
  if (B <= 0) return 0;
  argmax_ids_kernel<<<(B + 7) / 8, 256, 0, stream>>>(ids, idx, B, T);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
__global__ void l2_normalize_kernel(const float* __restrict__ x, float* __restrict__ out, size_t ldo, int B, int E) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  const float* r = x + static_cast<size_t>(warp) * E;
  float s = 0.f;
  for (int i = lane; i < E; i += 32) s += r[i] * r[i];
  s = warp_sum(s);
  const float n = sqrtf(s);
  for (int i = lane; i < E; i += 32) out[static_cast<size_t>(warp) * ldo + i] = r[i] / n;
}
int l2_normalize_run(const float* x, float* out, int ldo, int B, int E, cudaStream_t stream) {
  if (B <= 0) return 0;
  l2_normalize_kernel<<<(B + 7) / 8, 256, 0, stream>>>(x, out, ldo, B, E);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// fp32 logits: 64x64 tile per CTA, 16x16 threads, 4x4 micro-tile, K step 16.  Full fp32 FMA (no tensor cores):
// 2*B^2*E is micro-seconds of work and the parity budget is spent elsewhere.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
logits_kernel(const float* __restrict__ img, const float* __restrict__ txt, const float* __restrict__ logit_scale,
              const float* __restrict__ logit_bias, float* __restrict__ out, int Bi, int Bt, int E, size_t ldl) {
  __shared__ __align__(16) float As[16][LOGITS_LDS], Bs[16][LOGITS_LDS];
  const float sc = expf(*logit_scale);
  const float bs = logit_bias ? *logit_bias : 0.f;
  logits_tile<false>(img, E, txt, E, out, ldl, Bi, Bt, E, blockIdx.y * 64, blockIdx.x * 64, sc, bs, As, Bs);
}
int logits_run(const float* img, const float* txt, const float* logit_scale, const float* logit_bias, float* logits, int Bi, int Bt,
               int E, int ldl, cudaStream_t stream) {
  if (Bi <= 0 || Bt <= 0) return 0;
  dim3 grid((Bt + 63) / 64, (Bi + 63) / 64);
  logits_kernel<<<grid, 256, 0, stream>>>(img, txt, logit_scale, logit_bias, logits, Bi, Bt, E, ldl);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// weight packing (runs once at finalize)
// ------------------------------------------------------------------------------------------
template <typename OutT>
__global__ void transpose_cast_kernel(const float* __restrict__ src, int K, int N, OutT* __restrict__ dst, size_t ldd) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, n = n0 + threadIdx.x;
    tile[i][threadIdx.x] = (k < K && n < N) ? src[static_cast<size_t>(k) * N + n] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int n = n0 + i, k = k0 + threadIdx.x;
    if (n < N && k < K) dst[static_cast<size_t>(n) * ldd + k] = from_float<OutT>(tile[threadIdx.x][i]);
  }
}
int transpose_cast_run(const float* src, int K, int N, void* dst, int out_type, int ldd, cudaStream_t stream) {
  dim3 block(32, 8), grid((N + 31) / 32, (K + 31) / 32);
  if (out_type == DT_F32) transpose_cast_kernel<float><<<grid, block, 0, stream>>>(src, K, N, static_cast<float*>(dst), ldd);
  else if (out_type == DT_TF32) transpose_cast_kernel<tf32_t><<<grid, block, 0, stream>>>(src, K, N, static_cast<tf32_t*>(dst), ldd);
  else if (out_type == DT_F16) transpose_cast_kernel<__half><<<grid, block, 0, stream>>>(src, K, N, static_cast<__half*>(dst), ldd);
  else transpose_cast_kernel<__nv_bfloat16><<<grid, block, 0, stream>>>(src, K, N, static_cast<__nv_bfloat16*>(dst), ldd);
  JIMM_LAUNCH_CHECK();
  return 0;
}

// standalone activation (API parity for jimm.common.transformer.quickgelu; inside the towers the activation is the FC1 epilogue)
__global__ void activation_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n, int act) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) y[i] = act == 2 ? quick_gelu(x[i]) : (act == 1 ? gelu_tanh(x[i]) : x[i]);
}
int activation_run(const float* x, float* y, size_t n, int act, cudaStream_t stream) {
  if (n == 0) return 0;
  activation_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(x, y, n, act);
  JIMM_LAUNCH_CHECK();
  return 0;
}

template <typename OutT>
__global__ void cast_kernel(const float* __restrict__ src, OutT* __restrict__ dst, size_t n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = from_float<OutT>(src[i]);
}
int cast_run(const float* src, void* dst, int out_type, size_t n, cudaStream_t stream) {
  if (n == 0) return 0;
  const unsigned grid = static_cast<unsigned>((n + 255) / 256);
  if (out_type == DT_F32) cast_kernel<float><<<grid, 256, 0, stream>>>(src, static_cast<float*>(dst), n);
  else if (out_type == DT_TF32) cast_kernel<tf32_t><<<grid, 256, 0, stream>>>(src, static_cast<tf32_t*>(dst), n);
  else if (out_type == DT_F16) cast_kernel<__half><<<grid, 256, 0, stream>>>(src, static_cast<__half*>(dst), n);
  else cast_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(src, static_cast<__nv_bfloat16*>(dst), n);
  JIMM_LAUNCH_CHECK();
  return 0;
}

}  // namespace jimm

// Softmax attention kernels (SURVEY.md 8a row a5, a9).
//
// attention_kernel: flash-style fused softmax(q k^T / sqrt(d)) v over the fused qkv buffer, head_dim 64 (every
// jimm config: vision heads = width // 64, models/clip.py:60, models/siglip.py:59).  One CTA = 64 query rows of one
// (sample, head); 4 warps x 16 rows; K/V streamed in 64-key tiles through a double-buffered cp.async ring with
// XOR-swizzled 128-byte rows (conflict-free ldmatrix); scores and probabilities never leave registers; fp32
// online softmax with warp-quad shuffles.  Tensor path: mma.sync.m16n8k16 (legacy HMMA) -- the tcgen05 version
// of this kernel is listed as the next optimisation in DESIGN.md.
//
// map_attention_kernel: MAP-head pooling attention with a single precomputed probe query (common/vit.py:96-97).
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"

namespace jimm {

template <typename T>
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (std::is_same<T, __half>::value) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  } else {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

template <typename T>
__device__ __forceinline__ uint32_t pack_pair(float a, float b) {
  if constexpr (std::is_same<T, __half>::value) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}

static constexpr int QT = 64;   // query rows per CTA
static constexpr int KT = 64;   // keys per pipeline stage
static constexpr int HD = 64;   // head dim

// Copy a 64-row x 128-byte tile (rows s0.. of one head; row stride `ld` elements) into swizzled smem; rows >= S are
// clamped to S-1 (their scores are masked / their outputs are never stored).
template <typename T>
__device__ __forceinline__ void load_tile(uint32_t smem_base, const T* __restrict__ gbase, size_t ld, int s0, int S, int tid) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = tid + i * 128;
    const int row = c >> 3, ch = c & 7;
    int s = s0 + row;
    s = s < S ? s : S - 1;
    const T* src = gbase + static_cast<size_t>(s) * ld + ch * 8;
    cp_async16(smem_base + row * 128 + ((ch ^ (row & 7)) << 4), src);
  }
}

template <typename T, typename OutT, bool CAUSAL>
__global__ void __launch_bounds__(128)
attention_kernel(const T* __restrict__ qkv, OutT* __restrict__ out, int S, int H, float scale_log2, int reverse) {
  __shared__ __align__(128) uint8_t smem[QT * 128 + 2 * 2 * KT * 128];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = reverse ? static_cast<int>(gridDim.z) - 1 - static_cast<int>(blockIdx.z) : static_cast<int>(blockIdx.z);
  const int D = H * HD;
  const size_t ld = static_cast<size_t>(3) * D;
  const T* base = qkv + static_cast<size_t>(b) * S * ld + h * HD;
  const T* gq = base;
  const T* gk = base + D;
  const T* gv = base + 2 * D;
  const uint32_t sQ = smem_u32(smem);
  const uint32_t sK0 = sQ + QT * 128;
  const uint32_t sV0 = sK0 + 2 * KT * 128;
  const int q0 = qt * QT;
  pdl_launch_dependents();
  pdl_wait();
  int n_kv = (S + KT - 1) / KT;
  if (CAUSAL) n_kv = min(n_kv, qt + 1);

  load_tile<T>(sQ, gq, ld, q0, S, tid);
  load_tile<T>(sK0, gk, ld, 0, S, tid);
  load_tile<T>(sV0, gv, ld, 0, S, tid);
  cp_async_commit();

  uint32_t qf[4][4];
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  const int g = lane >> 2, t4 = lane & 3;
  const int row_lo = q0 + warp * 16 + g;  // this thread's two query rows: row_lo, row_lo + 8

  for (int j = 0; j < n_kv; ++j) {
    const int buf = j & 1;
    if (j + 1 < n_kv) {
      load_tile<T>(sK0 + (buf ^ 1) * KT * 128, gk, ld, (j + 1) * KT, S, tid);
      load_tile<T>(sV0 + (buf ^ 1) * KT * 128, gv, ld, (j + 1) * KT, S, tid);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (j == 0) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const int row = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
        const int ch = ks * 2 + (lane >> 4);
        ldsm_x4(qf[ks], sQ + row * 128 + ((ch ^ (row & 7)) << 4));
      }
    }
    const uint32_t sK = sK0 + buf * KT * 128, sV = sV0 + buf * KT * 128;

    // ---- S = Q K^T (16 x 64 per warp) ----
    float s[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) s[i][jj] = 0.f;
#pragma unroll
    for (int np = 0; np < 4; ++np) {
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t kf[4];
        const int mi = lane >> 3;
        const int row = np * 16 + (lane & 7) + (mi >> 1) * 8;
        const int ch = ks * 2 + (mi & 1);
        ldsm_x4(kf, sK + row * 128 + ((ch ^ (row & 7)) << 4));
        mma16816<T>(s[2 * np], qf[ks], kf[0], kf[1]);
        mma16816<T>(s[2 * np + 1], qf[ks], kf[2], kf[3]);
      }
    }
    // ---- mask + online softmax ----
    const int k0 = j * KT;
    const bool need_mask = (k0 + KT > S) || (CAUSAL && (k0 + KT - 1 > q0));
    if (need_mask) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = k0 + nt * 8 + t4 * 2 + (e & 1);
          const int qrow = row_lo + (e >> 1) * 8;
          const bool ok = key < S && (!CAUSAL || key <= qrow);
          if (!ok) s[nt][e] = -INFINITY;
        }
      }
    }
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
      mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
    }
    float alpha[2], moff[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float mnew = fmaxf(m_run[r], mx[r]);
      const float muse = (mnew == -INFINITY) ? 0.f : mnew;
      alpha[r] = exp2f((m_run[r] - muse) * scale_log2);  // m_run = -inf -> 0
      m_run[r] = mnew;
      moff[r] = muse * scale_log2;
      l_run[r] *= alpha[r];
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = exp2f(s[nt][0] * scale_log2 - moff[0]);
      s[nt][1] = exp2f(s[nt][1] * scale_log2 - moff[0]);
      s[nt][2] = exp2f(s[nt][2] * scale_log2 - moff[1]);
      s[nt][3] = exp2f(s[nt][3] * scale_log2 - moff[1]);
      l_run[0] += s[nt][0] + s[nt][1];
      l_run[1] += s[nt][2] + s[nt][3];
      o[nt][0] *= alpha[0]; o[nt][1] *= alpha[0];
      o[nt][2] *= alpha[1]; o[nt][3] *= alpha[1];
    }
    // ---- O += P V ----
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      uint32_t pf[4];
      pf[0] = pack_pair<T>(s[2 * kk][0], s[2 * kk][1]);
      pf[1] = pack_pair<T>(s[2 * kk][2], s[2 * kk][3]);
      pf[2] = pack_pair<T>(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pf[3] = pack_pair<T>(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t vf[4];
        const int mi = lane >> 3;
        const int row = kk * 16 + (lane & 7) + (mi & 1) * 8;
        const int ch = dp * 2 + (mi >> 1);
        ldsm_x4_trans(vf, sV + row * 128 + ((ch ^ (row & 7)) << 4));
        mma16816<T>(o[2 * dp], pf, vf[0], vf[1]);
        mma16816<T>(o[2 * dp + 1], pf, vf[2], vf[3]);
      }
    }
    __syncthreads();  // everyone done with buf before it is refilled two iterations later
  }

  // ---- finalise: O /= l, store ----
  float inv[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    float l = l_run[r];
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    inv[r] = 1.0f / l;
  }
  OutT* obase = out + static_cast<size_t>(b) * S * D + h * HD;
  if constexpr (sizeof(OutT) == 2) {
    // stage this warp's 16 x 64 tile through its (now free) Q rows so the global stores are 128-byte rows
    uint8_t* sq = smem;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int row = warp * 16 + g + r * 8;
        const int ch = nt;  // 8 columns (16 B) per n-tile
        const uint32_t v = pack_pair<OutT>(o[nt][2 * r] * inv[r], o[nt][2 * r + 1] * inv[r]);
        *reinterpret_cast<uint32_t*>(sq + row * 128 + ((ch ^ (row & 7)) << 4) + t4 * 4) = v;
      }
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = warp * 16 + i * 4 + (lane >> 3), ch = lane & 7;
      const int srow = q0 + row;
      if (srow < S) {
        const uint4 v = *reinterpret_cast<const uint4*>(sq + row * 128 + ((ch ^ (row & 7)) << 4));
        *reinterpret_cast<uint4*>(obase + static_cast<size_t>(srow) * D + ch * 8) = v;
      }
    }
  } else {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int srow = row_lo + r * 8;
        if (srow < S) {
          float2 v = make_float2(o[nt][2 * r] * inv[r], o[nt][2 * r + 1] * inv[r]);
          if constexpr (std::is_same<OutT, tf32_t>::value) v = make_float2(round_tf32(v.x), round_tf32(v.y));
          *reinterpret_cast<float2*>(reinterpret_cast<float*>(obase) + static_cast<size_t>(srow) * D + nt * 8 + t4 * 2) = v;
        }
      }
    }
  }
}

template <typename T, typename OutT>
static int attn_launch(const void* qkv, void* out, int B, int S, int H, int causal, cudaStream_t stream, int reverse) {
  dim3 grid((S + QT - 1) / QT, H, B);
  const float scale_log2 = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
  if (causal) JIMM_CUDA_CHECK(launch_k(attention_kernel<T, OutT, true>, grid, dim3(128), 0, stream, 1, true, static_cast<const T*>(qkv), static_cast<OutT*>(out), S, H, scale_log2, reverse));
  else JIMM_CUDA_CHECK(launch_k(attention_kernel<T, OutT, false>, grid, dim3(128), 0, stream, 1, true, static_cast<const T*>(qkv), static_cast<OutT*>(out), S, H, scale_log2, reverse));
  note_launch();
  return 0;
}

int attention_run(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, cudaStream_t stream, int reverse) {
  if (B <= 0 || S <= 0) return 0;
  const char* env = getenv("JIMM_ATTN_IMPL");  // "flash" forces the mma.sync flash kernel for every S (bisection)
  if (!(env && strcmp(env, "flash") == 0)) {
    int rc = attention_tc_run(qkv, io_type, out, out_type, B, S, H, causal, stream, reverse);
    if (rc <= 0) return rc;
    rc = attention_tc_long_run(qkv, io_type, out, out_type, B, S, H, causal, stream, reverse);
    if (rc <= 0) return rc;
  }
  if (B > 65535 || H > 65535) { set_last_error("attention: grid too large (B=%d H=%d)", B, H); return -1; }
  if (io_type == DT_F16 && out_type == DT_F16) return attn_launch<__half, __half>(qkv, out, B, S, H, causal, stream, reverse);
  if (io_type == DT_F16 && out_type == DT_F32) return attn_launch<__half, float>(qkv, out, B, S, H, causal, stream, reverse);
  if (io_type == DT_F16 && out_type == DT_TF32) return attn_launch<__half, tf32_t>(qkv, out, B, S, H, causal, stream, reverse);
  if (io_type == DT_BF16 && out_type == DT_BF16) return attn_launch<__nv_bfloat16, __nv_bfloat16>(qkv, out, B, S, H, causal, stream, reverse);
  if (io_type == DT_BF16 && out_type == DT_F32) return attn_launch<__nv_bfloat16, float>(qkv, out, B, S, H, causal, stream, reverse);
  set_last_error("attention: unsupported dtype combination io=%d out=%d", io_type, out_type);
  return -1;
}

// ------------------------------------------------------------------------------------------
// MAP-head attention: one CTA (256 threads) per (sample, head); scores in smem; HBM-bound on K/V.
// ------------------------------------------------------------------------------------------
template <typename T, typename OutT>
__global__ void __launch_bounds__(256)
map_attention_kernel(const float* __restrict__ q, const T* __restrict__ kv, OutT* __restrict__ out, int S, int H) {
  extern __shared__ float sm[];
  float* sq = sm;             // [64]
  float* red = sm + 64;       // [8 * 64] cross-group reduction / [8] block reductions
  float* sc = sm + 64 + 512;  // [S]
  const int h = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = H * HD;
  const size_t ld = static_cast<size_t>(2) * D;
  const T* kbase = kv + static_cast<size_t>(b) * S * ld + h * HD;
  const T* vbase = kbase + D;
  if (tid < 64) sq[tid] = q[h * HD + tid] * 0.125f;  // query / sqrt(depth)
  __syncthreads();
  // scores
  float lmax = -INFINITY;
  for (int s = tid; s < S; s += 256) {
    const uint4* kr = reinterpret_cast<const uint4*>(kbase + static_cast<size_t>(s) * ld);
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint4 u = __ldg(kr + c);
      const T* e = reinterpret_cast<const T*>(&u);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc = fmaf(to_float(e[i]), sq[c * 8 + i], acc);
    }
    sc[s] = acc;
    lmax = fmaxf(lmax, acc);
  }
  lmax = warp_max(lmax);
  if (lane == 0) red[warp] = lmax;
  __syncthreads();
  float bmax = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) bmax = fmaxf(bmax, red[w]);
  __syncthreads();
  float lsum = 0.f;
  for (int s = tid; s < S; s += 256) {
    const float p = __expf(sc[s] - bmax);
    sc[s] = p;
    lsum += p;
  }
  lsum = warp_sum(lsum);
  if (lane == 0) red[warp] = lsum;
  __syncthreads();
  float bsum = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) bsum += red[w];
  __syncthreads();
  // output: warp = key group, lane = dim pair
  float a0 = 0.f, a1 = 0.f;
  for (int s = warp; s < S; s += 8) {
    const float p = sc[s];
    const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(vbase + static_cast<size_t>(s) * ld) + lane);
    const T* e = reinterpret_cast<const T*>(&u);
    a0 = fmaf(p, to_float(e[0]), a0);
    a1 = fmaf(p, to_float(e[1]), a1);
  }
  red[warp * 64 + lane * 2] = a0;
  red[warp * 64 + lane * 2 + 1] = a1;
  __syncthreads();
  if (tid < 64) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w * 64 + tid];
    out[static_cast<size_t>(b) * D + h * HD + tid] = from_float<OutT>(v / bsum);
  }
}

template <typename T, typename OutT>
static int map_launch(const float* q, const void* kv, void* out, int B, int S, int H, cudaStream_t stream) {
  dim3 grid(H, B);
  const size_t smem = (64 + 512 + S) * sizeof(float);
  map_attention_kernel<T, OutT><<<grid, 256, smem, stream>>>(q, static_cast<const T*>(kv), static_cast<OutT*>(out), S, H);
  JIMM_LAUNCH_CHECK();
  return 0;
}

int map_attention_run(const float* q, const void* kv, int io_type, void* out, int out_type, int B, int S, int H, cudaStream_t stream) {
  if (B <= 0) return 0;
  if (S > 8192) { set_last_error("map_attention: S=%d too large", S); return -1; }
  if (io_type == DT_F16 && out_type == DT_F16) return map_launch<__half, __half>(q, kv, out, B, S, H, stream);
  if (io_type == DT_F16 && out_type == DT_F32) return map_launch<__half, float>(q, kv, out, B, S, H, stream);
  if (io_type == DT_F16 && out_type == DT_TF32) return map_launch<__half, tf32_t>(q, kv, out, B, S, H, stream);
  if (io_type == DT_BF16 && out_type == DT_BF16) return map_launch<__nv_bfloat16, __nv_bfloat16>(q, kv, out, B, S, H, stream);
  if (io_type == DT_BF16 && out_type == DT_F32) return map_launch<__nv_bfloat16, float>(q, kv, out, B, S, H, stream);
  set_last_error("map_attention: unsupported dtype combination io=%d out=%d", io_type, out_type);
  return -1;
}

}  // namespace jimm

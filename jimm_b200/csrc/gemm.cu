// Persistent, warp-specialised tcgen05 GEMM for sm_100a with fused epilogues.
//
//   C[M,N] = epi( A[M,K] . B[N,K]^T ),  A/B K-major fp16 | bf16 | fp32(tf32), fp32 accumulate in TMEM.
//
// CTA = 384 threads, 1 CTA / SM, grid = min(#tiles, #SMs), static round-robin tile schedule (n fastest).
//   warp 0    : TMA producer (one lane): 4-stage smem ring of {A 128x128B, B 256x128B} tiles, SWIZZLE_128B
//   warp 1    : MMA issuer  (one lane): tcgen05.mma.cta_group::1 128x256xUMMA_K, accumulators double-buffered
//               in TMEM (2 x 256 columns), tcgen05.commit releases smem stages / publishes accumulators
//   warp 2    : TMEM allocator (512 columns)
//   warps 4-11: epilogue.  warp % 4 = TMEM lane quarter, (warp-4)/4 = column half of the accumulator.
// Three mbarrier pipelines: smem full/empty (TMA<->MMA), TMEM full/empty (MMA<->epilogue).
//
// Epilogues are compile-time specialised (the first version branched at run time on dtype / activation inside 32-way
// unrolled loops: 174 KB of SASS, instruction-cache misses and exposed bias-load latency -- profiles/r1_a, r1_b):
//   OUT_H16 / OUT_BF16 / OUT_TF32 / OUT_F32 + ACT {none, tanh-GELU, QuickGELU}: thread = row; tcgen05.ld 32x32b.x32 with
//       the next chunk prefetched; bias from a per-tile smem copy; pack; 32 x 128 B swizzled box in smem;
//       cp.async.bulk.tensor store (bounds clipped by the tensor map).
//   OUT_F32_ADD: the fp32 residual stream x += acc + bias through cp.reduce.async.bulk.tensor .add (done in L2; the SM
//       never reads the residual).
//   OUT_GENERIC: everything else (position-embedding row-add + row remap of the patch GEMM, heads with unaligned N,
//       fp32 stores to caller buffers): LSU stores, run-time flags, 4 epilogue warps.
//
// Reference ops served (SURVEY.md 8a): a1 patch-embed conv-as-GEMM (common/vit.py:153-165,228-236),
// a4 fused q/k/v projections (common/transformer.py:67-79), a6 out-proj + residual (:130),
// a7 MLP (:90-114,131), a9 MAP-head linears (common/vit.py:42-85), a10 classifier / projections
// (models/vit.py:81-89, models/clip.py:82-90,166, models/siglip.py:111-119).
#include "gemm.cuh"

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace jimm {

static constexpr int BM = 128;
static constexpr int BN = 256;
static constexpr int STAGES = 4;
static constexpr int A_STAGE_BYTES = BM * 128;
static constexpr int B_STAGE_BYTES = BN * 128;
static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
static constexpr int EPI_PITCH = 36;  // floats; conflict-free for 128-bit accesses (generic staged path)
static constexpr int EPI_WARPS = 8;   // warps 4..11
static constexpr int EPI_BUF_BYTES = 32 * 128;                     // one 32-row x 128-byte swizzled TMA-store box per warp
static constexpr int EPI_STAGE_BYTES = EPI_WARPS * EPI_BUF_BYTES;  // 32 KB (the generic path uses 4 x 4608 B of it)
static constexpr int BIAS_BYTES = BN * 4;                          // per-tile bias copy
static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_STAGE_BYTES + BIAS_BYTES + 256 + 1024;
// CTA-pair mode (cta_group::2): the pair computes a 256 x 256 tile; each CTA stages its own 128 A rows and HALF of the B
// rows (128) per k-block -> 32 KB stages, 6 of them; the B operand traffic from L2 and the smem fill per SM drop by a third.
// Five of them, which frees 32 KB to double-buffer the epilogue's TMA-store boxes (wait_group.read 1 instead of 0).
static constexpr int P_STAGES = 5;
static constexpr int P_B_STAGE_BYTES = (BN / 2) * 128;
static constexpr int P_STAGE_BYTES = A_STAGE_BYTES + P_B_STAGE_BYTES;
static constexpr int P_EPI_BUFS = 2;
static_assert(P_STAGES * P_STAGE_BYTES + P_EPI_BUFS * EPI_WARPS * EPI_BUF_BYTES == STAGES * STAGE_BYTES + EPI_STAGE_BYTES,
              "pair and single modes share the smem carve-up");
static constexpr int NUM_THREADS = 384;
static constexpr uint32_t TMEM_COLS = 512;
static_assert(4 * 32 * EPI_PITCH * 4 <= EPI_STAGE_BYTES, "staging region too small");
static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");

enum OutKind : int { OUT_GENERIC = 0, OUT_H16 = 1, OUT_BF16 = 2, OUT_TF32 = 3, OUT_F32_ADD = 4, OUT_F32 = 5 };

struct EpiDev {
  const float* bias;
  const float* rowadd;
  const float* residual;
  void* out;
  int act, ldr, out_type, ldo, rows_in, rows_out, row_off, mode;
  int M, N;
  int debug;
  int reverse;
  int tok_pad, tok_off;  // > 0: 3-D token-scatter reduce-add (see GemmEpilogue)
  // Tail splitting (pair mode): the static round-robin schedule costs a whole round for the last `tail` tiles even when they occupy a
  // few of the CTA pairs.  When tail * parts <= #pairs those tiles are cut into `parts` (2 or 4) column slices of 256 / parts columns,
  // so the last round takes ~1 / parts of a round: virtual tiles [0, full) are whole tiles, [full, full + tail * parts) the slices.
  int full_tiles, tail_parts;
  int vec;  // 1: N / ldo / ldr multiples of 4 and 16-byte aligned pointers -> vector accesses allowed (generic path)
};

template <int ACT>
__device__ __forceinline__ float act_ct(float v) {
  if constexpr (ACT == ACT_GELU_TANH) return gelu_tanh(v);
  else if constexpr (ACT == ACT_QUICK_GELU) return quick_gelu(v);
  else return v;
}
__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == ACT_GELU_TANH) return gelu_tanh(v);
  if (act == ACT_QUICK_GELU) return quick_gelu(v);
  return v;
}

__device__ __forceinline__ void remap_row(const EpiDev& e, int row, int& out_row, int& add_row) {
  if (e.rows_in > 0) {
    int b = row / e.rows_in, p = row - b * e.rows_in;
    out_row = b * e.rows_out + p + e.row_off;
    add_row = p + e.row_off;
  } else {
    out_row = row;
    add_row = row;
  }
}

// Store 4 consecutive columns (col % 4 == 0, col + 3 < N guaranteed by caller).
__device__ __forceinline__ void store4(const EpiDev& e, int out_row, int col, float4 v) {
  size_t off = static_cast<size_t>(out_row) * e.ldo + col;
  if (e.out_type == DT_F32) {
    *reinterpret_cast<float4*>(static_cast<float*>(e.out) + off) = v;
  } else if (e.out_type == DT_TF32) {
    *reinterpret_cast<float4*>(static_cast<float*>(e.out) + off) = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
  } else {
    uint2 p;
    p.x = pack2(v.x, v.y, e.out_type);
    p.y = pack2(v.z, v.w, e.out_type);
    *reinterpret_cast<uint2*>(static_cast<uint16_t*>(e.out) + off) = p;
  }
}
__device__ __forceinline__ void store1(const EpiDev& e, int out_row, int col, float v) {
  size_t off = static_cast<size_t>(out_row) * e.ldo + col;
  if (e.out_type == DT_F32) static_cast<float*>(e.out)[off] = v;
  else if (e.out_type == DT_TF32) static_cast<float*>(e.out)[off] = round_tf32(v);
  else if (e.out_type == DT_F16) static_cast<__half*>(e.out)[off] = __float2half_rn(v);
  else static_cast<__nv_bfloat16*>(e.out)[off] = __float2bfloat16_rn(v);
}

template <typename T>
struct Traits;
template <>
struct Traits<__half> {
  static constexpr int KIND = 0, FMT = 0;
};
template <>
struct Traits<__nv_bfloat16> {
  static constexpr int KIND = 0, FMT = 1;
};
template <>
struct Traits<float> {
  static constexpr int KIND = 1, FMT = 2;
};

// ---- TMA epilogue for one 128 x 128 half-tile owned by one epilogue warp's lane quarter (thread = row) ------------
// 16-bit outputs: 64 columns per 32 x 128 B box (two x32 TMEM loads); 32-bit outputs: 32 columns per box.
// `release()` hands the accumulator back to the MMA issuer; it is called as soon as this warp's LAST tcgen05.ld has completed, i.e.
// before the math / staging / store of the last box (the data is in registers by then), not after the whole epilogue.
template <int OUT, int ACT, int NBUF, typename Release>
__device__ __forceinline__ void epilogue_tma(const CUtensorMap* map_c, const EpiDev& epi, uint32_t taddr, const float* sbias, uint8_t* tbuf0,
                                             int lane, int row_base, int n_tile0, int c_begin, int c_len, uint32_t& box_count, Release&& release) {
  constexpr bool OUT16 = (OUT == OUT_H16 || OUT == OUT_BF16);
  constexpr int COLS_PER_BOX = OUT16 ? 64 : 32;
  const int N = epi.N;
  uint32_t r[32], r2[32], pk[32];
  bool released = false;
  if (n_tile0 + c_begin < N) tmem_ld_32x32b_x32(taddr + c_begin, r);
#pragma unroll 1
  for (int c = c_begin; c < c_begin + c_len; c += COLS_PER_BOX) {
    const int n0 = n_tile0 + c;
    if (n0 >= N) break;
    const int cn = c + COLS_PER_BOX;
    const bool more = (cn < c_begin + c_len) && (n_tile0 + cn < N);
    tmem_ld_wait();
    if constexpr (OUT16) tmem_ld_32x32b_x32(taddr + c + 32, r2);  // second half of this box, in flight during the math below
    else if (!more) { release(); released = true; }
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      float4 b4;
      if constexpr (OUT == OUT_F32_ADD) {
        // straight from global (warp-uniform address, L1 broadcast): the residual epilogue has no per-tile bias staging and therefore no
        // CTA-wide barrier -- its warps run independently
        b4 = (sbias != nullptr && n_tile0 + c + j < N) ? __ldg(reinterpret_cast<const float4*>(sbias + n_tile0 + c + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        b4 = *reinterpret_cast<const float4*>(sbias + c + j);
      }
      const float v0 = act_ct<ACT>(__uint_as_float(r[j]) + b4.x), v1 = act_ct<ACT>(__uint_as_float(r[j + 1]) + b4.y);
      const float v2 = act_ct<ACT>(__uint_as_float(r[j + 2]) + b4.z), v3 = act_ct<ACT>(__uint_as_float(r[j + 3]) + b4.w);
      if constexpr (OUT16) {
        pk[j >> 1] = pack2(v0, v1, OUT == OUT_H16 ? 1 : 2);
        pk[(j >> 1) + 1] = pack2(v2, v3, OUT == OUT_H16 ? 1 : 2);
      } else if constexpr (OUT == OUT_TF32) {
        pk[j] = __float_as_uint(round_tf32(v0)); pk[j + 1] = __float_as_uint(round_tf32(v1));
        pk[j + 2] = __float_as_uint(round_tf32(v2)); pk[j + 3] = __float_as_uint(round_tf32(v3));
      } else {
        pk[j] = __float_as_uint(v0); pk[j + 1] = __float_as_uint(v1); pk[j + 2] = __float_as_uint(v2); pk[j + 3] = __float_as_uint(v3);
      }
    }
    if constexpr (OUT16) {
      tmem_ld_wait();
      if (more) tmem_ld_32x32b_x32(taddr + cn, r);  // prefetch the next box
      else { release(); released = true; }
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(sbias + c + 32 + j);
        const float v0 = act_ct<ACT>(__uint_as_float(r2[j]) + b4.x), v1 = act_ct<ACT>(__uint_as_float(r2[j + 1]) + b4.y);
        const float v2 = act_ct<ACT>(__uint_as_float(r2[j + 2]) + b4.z), v3 = act_ct<ACT>(__uint_as_float(r2[j + 3]) + b4.w);
        pk[16 + (j >> 1)] = pack2(v0, v1, OUT == OUT_H16 ? 1 : 2);
        pk[16 + (j >> 1) + 1] = pack2(v2, v3, OUT == OUT_H16 ? 1 : 2);
      }
    } else {
      if (more) tmem_ld_32x32b_x32(taddr + cn, r);  // prefetch the next box
    }
    // ---- stage + TMA store ----
    uint8_t* tbuf = tbuf0 + (NBUF > 1 ? (box_count & (NBUF - 1)) * EPI_BUF_BYTES : 0);
    const uint32_t tbuf_u32 = smem_u32(tbuf);
    ++box_count;
    if (lane == 0) {  // the box that last used this buffer has been read out of smem
      if constexpr (NBUF > 1) tma_store_wait_read1();
      else tma_store_wait_read();
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; ++j)
      *reinterpret_cast<uint4*>(tbuf + lane * 128 + ((j ^ (lane & 7)) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      if constexpr (OUT == OUT_F32_ADD) {
        if (epi.tok_pad > 0) {
          const int b = row_base / epi.tok_pad;
          tma_reduce_add_3d(map_c, tbuf_u32, n0, row_base - b * epi.tok_pad + epi.tok_off, b);
        } else {
          tma_reduce_add_2d(map_c, tbuf_u32, n0, row_base);
        }
      } else {
        tma_store_2d(map_c, tbuf_u32, n0, row_base);
      }
      tma_store_commit();
    }
  }
  if (!released) release();
}

// ---- generic LSU epilogue (4 warps; run-time flags; modes 0 = staged / 1 = direct) ---------------------------------
__device__ __noinline__ void epilogue_generic(const EpiDev& epi, uint32_t taddr, float* st, int lane, int row_base, int n_tile0) {
  const int M = epi.M, N = epi.N;
  for (int c = 0; c < BN / 32; ++c) {
    const int n0 = n_tile0 + c * 32;
    if (n0 >= N) break;
    uint32_t r[32];
    tmem_ld_32x32b_x32(taddr + c * 32, r);
    tmem_ld_wait();
    if (epi.mode == 1) {
      // direct: thread owns one row, 32 consecutive columns
      const int row = row_base + lane;
      if (row < M) {
        int out_row, add_row;
        remap_row(epi, row, out_row, add_row);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int col = n0 + j;
          if (col < N) {
            float v = __uint_as_float(r[j]);
            if (epi.bias) v += __ldg(epi.bias + col);
            v = apply_act(v, epi.act);
            if (epi.rowadd) v += __ldg(epi.rowadd + static_cast<size_t>(add_row) * N + col);
            if (epi.residual) v += epi.residual[static_cast<size_t>(out_row) * epi.ldr + col];
            store1(epi, out_row, col, v);
          }
        }
      }
    } else {
      // staged: transpose through smem so every global access is a full 128-byte line
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<uint4*>(st + lane * EPI_PITCH + j * 4) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
      __syncwarp();
      const int cq = (lane & 7) * 4;
      const int col = n0 + cq;
      const bool col_ok = epi.vec && (col + 3 < N);
      float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (epi.bias && col_ok) b4 = __ldg(reinterpret_cast<const float4*>(epi.bias + col));
#pragma unroll 2
      for (int i = 0; i < 8; ++i) {
        const int rr = i * 4 + (lane >> 3);
        const int row = row_base + rr;
        float4 v = *reinterpret_cast<const float4*>(st + rr * EPI_PITCH + cq);
        if (row < M) {
          int out_row, add_row;
          remap_row(epi, row, out_row, add_row);
          if (col_ok) {
            v.x = apply_act(v.x + b4.x, epi.act);
            v.y = apply_act(v.y + b4.y, epi.act);
            v.z = apply_act(v.z + b4.z, epi.act);
            v.w = apply_act(v.w + b4.w, epi.act);
            if (epi.rowadd) {
              const float4 a = __ldg(reinterpret_cast<const float4*>(epi.rowadd + static_cast<size_t>(add_row) * N + col));
              v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
            }
            if (epi.residual) {
              const float4 a = *reinterpret_cast<const float4*>(epi.residual + static_cast<size_t>(out_row) * epi.ldr + col);
              v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
            }
            store4(epi, out_row, col, v);
          } else {
            const float vv[4] = {v.x, v.y, v.z, v.w};
            for (int j = 0; j < 4; ++j) {
              const int cc = col + j;
              if (cc < N) {
                float x = vv[j];
                if (epi.bias) x += __ldg(epi.bias + cc);
                x = apply_act(x, epi.act);
                if (epi.rowadd) x += __ldg(epi.rowadd + static_cast<size_t>(add_row) * N + cc);
                if (epi.residual) x += epi.residual[static_cast<size_t>(out_row) * epi.ldr + cc];
                store1(epi, out_row, cc, x);
              }
            }
          }
        }
      }
      __syncwarp();
    }
  }
}

struct TileCoord {
  int m_blk, n_blk, n_off, width;  // columns [n_blk * BN + n_off, ... + width) of row block m_blk
};
// virtual tile index (already direction-adjusted) -> coordinates; identical in the three roles
__device__ __forceinline__ TileCoord decode_tile(const EpiDev& e, int tv, int n_tiles) {
  TileCoord t;
  int te = tv;
  t.n_off = 0;
  t.width = BN;
  if (tv >= e.full_tiles) {
    const int j = tv - e.full_tiles;
    te = e.full_tiles + j / e.tail_parts;
    t.width = BN / e.tail_parts;
    t.n_off = (j % e.tail_parts) * t.width;
  }
  t.m_blk = te / n_tiles;
  t.n_blk = te - t.m_blk * n_tiles;
  return t;
}

template <typename T, int OUT, int ACT, bool PAIR>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_c, const EpiDev epi, int K) {
  constexpr int BK = 128 / sizeof(T);  // one 128-byte swizzle atom along K per stage
  constexpr int UK = 32 / sizeof(T);   // UMMA K (16 for 16-bit, 8 for tf32)
  constexpr uint32_t IDESC = make_idesc(Traits<T>::FMT, PAIR ? 2 * BM : BM, BN);
  constexpr int NSTAGE = PAIR ? P_STAGES : STAGES;
  constexpr int B_BYTES = PAIR ? P_B_STAGE_BYTES : B_STAGE_BYTES;
  constexpr int TILE_M = PAIR ? 2 * BM : BM;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + NSTAGE * A_STAGE_BYTES;
  uint8_t* epi_stage = smem + (PAIR ? P_STAGES * P_STAGE_BYTES : STAGES * STAGE_BYTES);
  constexpr int EPI_BUFS = PAIR ? P_EPI_BUFS : 1;
  constexpr int EPI_REGION = EPI_BUFS * EPI_STAGE_BYTES;
  float* sbias = reinterpret_cast<float*>(epi_stage + EPI_REGION);
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_stage + EPI_REGION + BIAS_BYTES);
  uint64_t* full_bar = bars;                    // [NSTAGE]
  uint64_t* empty_bar = bars + NSTAGE;          // [NSTAGE]
  uint64_t* tmem_full_bar = bars + 2 * NSTAGE;  // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2; // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int M = epi.M, N = epi.N;
  const int m_tiles = (M + TILE_M - 1) / TILE_M, n_tiles = (N + BN - 1) / BN;
  const int real_tiles = m_tiles * n_tiles;
  const int num_tiles = epi.full_tiles + (real_tiles - epi.full_tiles) * epi.tail_parts;  // virtual tiles (== real_tiles without a split tail)
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;   // 0 = leader (issues the MMAs)
  const int tile0 = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int num_kb = (K + BK - 1) / BK;
  const bool dbg_no_epi = (epi.debug & 1) != 0, dbg_no_load = (epi.debug & 2) != 0;  // bring-up probes (JIMM_GEMM_DEBUG)

  pdl_launch_dependents();
  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    if constexpr (OUT != OUT_GENERIC) tma_prefetch_desc(&map_c);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], PAIR ? 2 * EPI_WARPS : EPI_WARPS);  // pair: both CTAs' epilogues release the leader's MMA
    }
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    if constexpr (PAIR) tmem_alloc_pair(tmem_ptr_smem, TMEM_COLS);
    else tmem_alloc(tmem_ptr_smem, TMEM_COLS);
  }
  tcgen05_fence_before();
  if constexpr (PAIR) cluster_sync_all();  // the peer's barriers must be initialised before any remote arrive / multicast commit
  else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();  // everything above (barrier init, TMEM allocation, descriptor prefetch) overlapped the previous kernel's tail

  if (warp_idx == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        const TileCoord tc = decode_tile(epi, epi.reverse ? num_tiles - 1 - tile : tile, n_tiles);
        const int m_blk = tc.m_blk;
        // B rows of this CTA: its half of the tile's `width` columns (the box always carries BN / 2 rows; a slice uses the first width / 2)
        const int b_row = tc.n_blk * BN + tc.n_off + (PAIR ? static_cast<int>(cta_rank) * (tc.width / 2) : 0);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if constexpr (PAIR) {
            // both CTAs credit the LEADER's full barrier; only the leader arms it (with the bytes of both CTAs)
            const uint32_t full_leader = mapa_shared(smem_u32(&full_bar[stage]), 0);
            if (cta_rank == 0) {
              if (dbg_no_load) mbar_arrive(&full_bar[stage]);
              else mbar_arrive_expect_tx(&full_bar[stage], 2 * P_STAGE_BYTES);
            }
            if (!dbg_no_load) {
              tma_load_2d_pair(smem_a + stage * A_STAGE_BYTES, &map_a, full_leader, kb * BK, m_blk * TILE_M + static_cast<int>(cta_rank) * BM);
              tma_load_2d_pair(smem_b + stage * B_BYTES, &map_b, full_leader, kb * BK, b_row);
            }
          } else if (dbg_no_load) {
            mbar_arrive(&full_bar[stage]);
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], STAGE_BYTES);
            tma_load_2d(smem_a + stage * A_STAGE_BYTES, &map_a, &full_bar[stage], kb * BK, m_blk * BM);
            tma_load_2d(smem_b + stage * B_BYTES, &map_b, &full_bar[stage], kb * BK, b_row);
          }
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer (pair mode: the leader CTA only) =====================
    // The whole warp runs the control flow (waits, counters and descriptors stay warp-uniform); only the elected lane issues.
    if (cta_rank == 0) {
      const bool leader = lane == 0;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        const int tv = epi.reverse ? num_tiles - 1 - tile : tile;
        const uint32_t idesc = tv >= epi.full_tiles ? make_idesc(Traits<T>::FMT, PAIR ? 2 * BM : BM, static_cast<uint32_t>(BN / epi.tail_parts)) : IDESC;
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          if (leader) {
            const uint64_t adesc = make_umma_desc_sw128(smem_u32(smem_a + stage * A_STAGE_BYTES));
            const uint64_t bdesc = make_umma_desc_sw128(smem_u32(smem_b + stage * B_BYTES));
#pragma unroll
            for (int k = 0; k < BK / UK; ++k) {  // descriptors advance by 32 bytes (>> 4) per UMMA K step
              if constexpr (PAIR) umma_ss_pair<Traits<T>::KIND>(tmem_d, adesc + static_cast<uint64_t>(2 * k), bdesc + static_cast<uint64_t>(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
              else umma_ss<Traits<T>::KIND>(tmem_d, adesc + static_cast<uint64_t>(2 * k), bdesc + static_cast<uint64_t>(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
            }
            if constexpr (PAIR) {
              tcgen05_commit_pair(&empty_bar[stage]);  // frees this stage in BOTH CTAs once the MMAs above retire
              if (kb == num_kb - 1) tcgen05_commit_pair(&tmem_full_bar[acc]);
            } else {
              tcgen05_commit(&empty_bar[stage]);
              if (kb == num_kb - 1) tcgen05_commit(&tmem_full_bar[acc]);
            }
          }
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp_idx >= 4) {
    // ===================== epilogue =====================
    const int q = warp_idx & 3;            // the TMEM lane quarter this warp may access (hardware rule: warp % 4)
    const int half = (warp_idx - 4) >> 2;  // column half of the 256-wide accumulator this warp drains
    int acc = 0;
    uint32_t acc_phase = 0, box_count = 0;
    const uint32_t tmem_empty_leader0 = PAIR ? mapa_shared(smem_u32(&tmem_empty_bar[0]), 0) : 0u;
    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
      const TileCoord tc = decode_tile(epi, epi.reverse ? num_tiles - 1 - tile : tile, n_tiles);
      const int m_blk = tc.m_blk;
      const int n_tile0 = tc.n_blk * BN + tc.n_off;  // first column of this (possibly sliced) tile
      const int c_len = tc.width / 2;                // accumulator columns per column half
      const int row_base = m_blk * TILE_M + static_cast<int>(cta_rank) * BM + q * 32;
      if constexpr (OUT != OUT_GENERIC && OUT != OUT_F32_ADD) {  // (OUT_F32_ADD: bias from global, so its warps need no barrier)
        // per-tile bias copy (one coalesced 128-bit load per lane of two warps), overlapped with the wait for the MMAs
        named_bar_sync(1, EPI_WARPS * 32);  // every epilogue warp is done with the previous tile's bias
        if (q == 0) {  // sbias[c] = bias[n_tile0 + c] for the accumulator columns c of this half
          const int c = half * c_len + lane * 4;
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (epi.bias && lane * 4 < c_len && n_tile0 + c < N) b4 = __ldg(reinterpret_cast<const float4*>(epi.bias + n_tile0 + c));
          if (lane * 4 < c_len) *reinterpret_cast<float4*>(sbias + c) = b4;
        }
        named_bar_sync(1, EPI_WARPS * 32);
      }
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN;
      // hand the accumulator back: all of this warp's tcgen05.ld's of the tile are complete (wait::ld) when this runs
      auto release = [&]() {
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (PAIR) mbar_arrive_cluster_relaxed(tmem_empty_leader0 + acc * 8);
          else mbar_arrive_relaxed(&tmem_empty_bar[acc]);
        }
      };
      if (dbg_no_epi) {
        release();
      } else if constexpr (OUT != OUT_GENERIC) {
        if (row_base < M) {
          epilogue_tma<OUT, ACT, EPI_BUFS>(&map_c, epi, taddr, OUT == OUT_F32_ADD ? epi.bias : sbias, epi_stage + (warp_idx - 4) * EPI_BUFS * EPI_BUF_BYTES,
                                           lane, row_base, n_tile0, half * c_len, c_len, box_count, release);
        } else {
          release();
        }
      } else {
        if (half == 0 && row_base < M)
          epilogue_generic(epi, taddr, reinterpret_cast<float*>(epi_stage) + q * 32 * EPI_PITCH, lane, row_base, n_tile0);
        release();
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if constexpr (OUT != OUT_GENERIC) {
      if (lane == 0) tma_store_wait_all();
    }
  }

  tcgen05_fence_before();
  if constexpr (PAIR) cluster_sync_all();  // neither CTA may exit (or free TMEM) while the pair's MMAs / remote arrives are in flight
  else __syncthreads();
  tcgen05_fence_after();
  if (warp_idx == 2) {
    if constexpr (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------
// SIMT reference GEMM (bring-up cross-check / JIMM_GEMM_IMPL=simt bisection only)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void gemm_simt_kernel(const T* __restrict__ A, int lda, const T* __restrict__ B, int ldb, int K, EpiDev epi) {
  __shared__ float As[16][17], Bs[16][17];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int row = blockIdx.y * 16 + ty, col = blockIdx.x * 16 + tx;
  float acc = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    const int ar = blockIdx.y * 16 + ty, ak = k0 + tx;
    As[ty][tx] = (ar < epi.M && ak < K) ? to_float(A[static_cast<size_t>(ar) * lda + ak]) : 0.f;
    const int br = blockIdx.x * 16 + ty, bk = k0 + tx;
    Bs[ty][tx] = (br < epi.N && bk < K) ? to_float(B[static_cast<size_t>(br) * ldb + bk]) : 0.f;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) acc += As[ty][k] * Bs[tx][k];
    __syncthreads();
  }
  if (row < epi.M && col < epi.N) {
    int out_row, add_row;
    remap_row(epi, row, out_row, add_row);
    float v = acc;
    if (epi.bias) v += epi.bias[col];
    v = apply_act(v, epi.act);
    if (epi.rowadd) v += epi.rowadd[static_cast<size_t>(add_row) * epi.N + col];
    if (epi.residual) v += epi.residual[static_cast<size_t>(out_row) * epi.ldr + col];
    store1(epi, out_row, col, v);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) {
    set_last_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed: %s", cudaGetErrorString(e));
    return nullptr;
  }
  fn = reinterpret_cast<PFN_encodeTiled>(p);
  return fn;
}

// 2-D K-major tensor map: dims {K, rows}, box {128 B worth of K, box_rows}, SWIZZLE_128B, zero OOB fill.
static int make_map(CUtensorMap* map, int dtype, const void* ptr, int rows, int K, int ld, int box_rows) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return -3;
  const size_t es = dtype_size(dtype);
  CUtensorMapDataType dt = (dtype == DT_F32 || dtype == DT_TF32) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                           : (dtype == DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * es};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / es), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (strides[0] & 15) != 0) {
    set_last_error("gemm: operand pointer/stride must be 16-byte aligned (ptr=%p, ld=%d)", ptr, ld);
    return -1;
  }
  CUresult r = enc(map, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed: CUresult %d (rows=%d K=%d ld=%d)", static_cast<int>(r), rows, K, ld);
    return -3;
  }
  return 0;
}

// 3-D tensor map over out[B, S, N] (dims {N, S, B}), box {128 B of columns, 32 rows, 1}, SWIZZLE_128B: rows >= S are clipped,
// so a 32-row box never spills into the next sample.
int make_tensor_map_3d(CUtensorMap* map, int dtype, const void* ptr, int B, int S, int N, int ld) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return -3;
  const size_t es = dtype_size(dtype);
  CUtensorMapDataType dt = (dtype == DT_F32 || dtype == DT_TF32) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                           : (dtype == DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(S), static_cast<cuuint64_t>(B)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(ld) * es, static_cast<cuuint64_t>(S) * ld * es};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(128 / es), 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, dt, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_last_error("cuTensorMapEncodeTiled(3d) failed: CUresult %d", static_cast<int>(r)); return -3; }
  return 0;
}
static int make_map_3d_f32(CUtensorMap* map, const void* ptr, int B, int S, int N, int ld) { return make_tensor_map_3d(map, DT_F32, ptr, B, S, N, ld); }

int make_tensor_map_2d(CUtensorMap* map, int dtype, const void* ptr, int rows, int cols, int ld, int box_rows) {
  return make_map(map, dtype, ptr, rows, cols, ld, box_rows);
}

int device_sm_count() {  // of the CURRENT device (cached per device: a process may drive several GPUs)
  static int sms[DeviceOnce::kMaxDevices] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= DeviceOnce::kMaxDevices) dev = 0;
  if (sms[dev] == 0) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    const char* env = getenv("JIMM_NUM_SMS");
    if (env && atoi(env) > 0) n = atoi(env);
    sms[dev] = n;
  }
  return sms[dev];
}

static int check_epi(const GemmEpilogue& e, int N) {
  if (e.out == nullptr) { set_last_error("gemm: null output"); return -1; }
  if (e.ldo < N) { set_last_error("gemm: ldo (%d) < N (%d)", e.ldo, N); return -1; }
  if (e.out_type < DT_F32 || e.out_type > DT_TF32) { set_last_error("gemm: bad out_type %d", e.out_type); return -1; }
  return 0;
}
// vector accesses need aligned rows; otherwise the generic epilogue takes its scalar path (tiny head GEMMs, N = 10 classes)
static int epi_vec_ok(const GemmEpilogue& e, int N) {
  if (N % 4 != 0 || e.ldo % 4 != 0) return 0;
  if (e.residual && e.ldr % 4 != 0) return 0;
  if ((reinterpret_cast<uintptr_t>(e.out) & 15) || (reinterpret_cast<uintptr_t>(e.bias) & 15) ||
      (reinterpret_cast<uintptr_t>(e.residual) & 15) || (reinterpret_cast<uintptr_t>(e.rowadd) & 15)) return 0;
  return 1;
}

int gemm_plan_init(GemmPlan* plan, int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K,
                   const GemmEpilogue& epi) {
  if (M <= 0 || N <= 0 || K <= 0) { set_last_error("gemm: bad shape %dx%dx%d", M, N, K); return -1; }
  if (int rc = check_epi(epi, N)) return rc;
  if (int rc = make_map(&plan->map_a, dtype, A, M, K, lda, BM)) return rc;
  if (int rc = make_map(&plan->map_b, dtype, B, N, K, ldb, BN)) return rc;
  if (int rc = make_map(&plan->map_b_pair, dtype, B, N, K, ldb, BN / 2)) return rc;
  plan->M = M; plan->N = N; plan->K = K; plan->dtype = dtype; plan->epi = epi;
  memset(&plan->map_c, 0, sizeof(plan->map_c));
  if (plan->epi.mode == 2) {
    const size_t es = dtype_size(epi.out_type);
    const bool ok = epi.rowadd == nullptr && epi.rows_in == 0 &&
                    (epi.residual == nullptr || (epi.residual == epi.out && epi.ldr == epi.ldo && epi.out_type == DT_F32)) &&
                    (static_cast<size_t>(epi.ldo) * es) % 16 == 0 && (reinterpret_cast<uintptr_t>(epi.out) & 15) == 0 &&
                    (epi.bias == nullptr || ((reinterpret_cast<uintptr_t>(epi.bias) & 15) == 0 && N % 4 == 0)) &&
                    !(epi.residual && epi.act != ACT_NONE);
    if (ok && epi.tok_pad > 0) {
      if (epi.tok_pad % 32 != 0 || M % epi.tok_pad != 0 || !epi.residual) { set_last_error("gemm: bad token-scatter epilogue"); return -1; }
      if (int rc = make_map_3d_f32(&plan->map_c, epi.out, M / epi.tok_pad, epi.tok_S, N, epi.ldo)) return rc;
    } else if (ok) {
      if (int rc = make_map(&plan->map_c, epi.out_type, epi.out, M, N, epi.ldo, 32)) return rc;
    } else {
      plan->epi.mode = 0;
    }
  }
  return 0;
}

static EpiDev to_dev(const GemmEpilogue& e, int M, int N) {
  EpiDev d;
  d.bias = e.bias; d.rowadd = e.rowadd; d.residual = e.residual; d.out = e.out;
  d.act = e.act; d.ldr = e.ldr; d.out_type = e.out_type; d.ldo = e.ldo;
  d.rows_in = e.rows_in; d.rows_out = e.rows_out; d.row_off = e.row_off; d.mode = e.mode;
  d.M = M; d.N = N;
  d.tok_pad = e.tok_pad; d.tok_off = e.tok_off;
  d.reverse = e.reverse;
  d.full_tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);  // overwritten by the pair-mode launch (its row blocks are 2 * BM)
  d.tail_parts = 1;
  d.vec = epi_vec_ok(e, N);
  static int dbg = -1;
  if (dbg < 0) { const char* env = getenv("JIMM_GEMM_DEBUG"); dbg = env ? atoi(env) : 0; }
  d.debug = dbg;
  return d;
}

static int tail_split_enabled() {
  static int v = -1;
  if (v < 0) { const char* env = getenv("JIMM_GEMM_TAIL_SPLIT"); v = env ? atoi(env) : 1; }
  return v;
}
static int pair_mode_enabled() {
  static int v = -1;
  if (v < 0) { const char* env = getenv("JIMM_GEMM_PAIR"); v = env ? atoi(env) : 1; }
  return v;
}

template <typename T, int OUT, int ACT>
static int launch_one(const GemmPlan* p, int M, cudaStream_t stream) {
  static DeviceOnce attr_set;
  if (attr_set.first()) {
    JIMM_CUDA_CHECK(cudaFuncSetAttribute(gemm_tcgen05_kernel<T, OUT, ACT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    JIMM_CUDA_CHECK(cudaFuncSetAttribute(gemm_tcgen05_kernel<T, OUT, ACT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  }
  const int n_tiles = (p->N + BN - 1) / BN;
  EpiDev d = to_dev(p->epi, M, p->N);
  if (OUT != OUT_GENERIC && pair_mode_enabled() && M >= 512) {
    // CTA pairs: 256 x 256 tiles, cluster (2,1,1), one pair per two SMs
    const int tiles = ((M + 2 * BM - 1) / (2 * BM)) * n_tiles;
    const int max_pairs = device_sm_count() / 2;
    // split the tail round into column slices when that shortens it (see EpiDev): 16-bit outputs store 64-column boxes, so a column
    // half must keep >= 64 columns (parts <= 2); 32-bit outputs store 32-column boxes (parts <= 4)
    int tail = tiles % max_pairs, parts = 1;
    constexpr int kMaxParts = (OUT == OUT_H16 || OUT == OUT_BF16) ? 2 : 4;
    if (tail_split_enabled() && tail > 0) {
      while (parts * 2 <= kMaxParts && tail * parts * 2 <= max_pairs) parts *= 2;
    }
    d.full_tiles = parts > 1 ? tiles - tail : tiles;
    d.tail_parts = parts;
    const int vtiles = d.full_tiles + (tiles - d.full_tiles) * parts;
    const int pairs = vtiles < max_pairs ? vtiles : max_pairs;
    JIMM_CUDA_CHECK(launch_k(gemm_tcgen05_kernel<T, OUT, ACT, true>, dim3(2 * pairs), dim3(NUM_THREADS), SMEM_BYTES, stream, 2, true,
                             p->map_a, p->map_b_pair, p->map_c, d, p->K));
    note_launch();
    return 0;
  }
  const int tiles = ((M + BM - 1) / BM) * n_tiles;
  const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
  JIMM_CUDA_CHECK(launch_k(gemm_tcgen05_kernel<T, OUT, ACT, false>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, stream, 1, true, p->map_a,
                           p->map_b, p->map_c, d, p->K));
  note_launch();
  return 0;
}

template <typename T, int OUT>
static int launch_act(const GemmPlan* p, int M, cudaStream_t stream) {
  switch (p->epi.act) {
    case ACT_GELU_TANH: return launch_one<T, OUT, ACT_GELU_TANH>(p, M, stream);
    case ACT_QUICK_GELU: return launch_one<T, OUT, ACT_QUICK_GELU>(p, M, stream);
    default: return launch_one<T, OUT, ACT_NONE>(p, M, stream);
  }
}

template <typename T>
static int launch_tc(const GemmPlan* p, int M, cudaStream_t stream) {
  const GemmEpilogue& e = p->epi;
  if (e.mode != 2) return launch_one<T, OUT_GENERIC, ACT_NONE>(p, M, stream);
  if (e.residual) return launch_one<T, OUT_F32_ADD, ACT_NONE>(p, M, stream);
  switch (e.out_type) {
    case DT_F16: return launch_act<T, OUT_H16>(p, M, stream);
    case DT_BF16: return launch_act<T, OUT_BF16>(p, M, stream);
    case DT_TF32: return launch_act<T, OUT_TF32>(p, M, stream);
    default: return launch_act<T, OUT_F32>(p, M, stream);
  }
}

int gemm_plan_run(const GemmPlan* p0, int M_override, cudaStream_t stream, int reverse) {
  const int M = (M_override > 0 && M_override <= p0->M) ? M_override : p0->M;
  GemmPlan local;
  const GemmPlan* p = p0;
  if (reverse != p0->epi.reverse) { local = *p0; local.epi.reverse = reverse; p = &local; }
  switch (p->dtype) {
    case DT_F16: return launch_tc<__half>(p, M, stream);
    case DT_BF16: return launch_tc<__nv_bfloat16>(p, M, stream);
    case DT_F32:
    case DT_TF32: return launch_tc<float>(p, M, stream);
  }
  set_last_error("gemm: bad dtype %d", p->dtype);
  return -1;
}

int gemm_simt_run(int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K, const GemmEpilogue& epi,
                  cudaStream_t stream) {
  if (int rc = check_epi(epi, N)) return rc;
  dim3 block(16, 16), grid((N + 15) / 16, (M + 15) / 16);
  EpiDev d = to_dev(epi, M, N);
  if (dtype == DT_F16) gemm_simt_kernel<__half><<<grid, block, 0, stream>>>(static_cast<const __half*>(A), lda, static_cast<const __half*>(B), ldb, K, d);
  else if (dtype == DT_BF16) gemm_simt_kernel<__nv_bfloat16><<<grid, block, 0, stream>>>(static_cast<const __nv_bfloat16*>(A), lda, static_cast<const __nv_bfloat16*>(B), ldb, K, d);
  else gemm_simt_kernel<float><<<grid, block, 0, stream>>>(static_cast<const float*>(A), lda, static_cast<const float*>(B), ldb, K, d);
  JIMM_LAUNCH_CHECK();
  return 0;
}

}  // namespace jimm

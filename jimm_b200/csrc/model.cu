// Model state, weight packing, forward orchestration and the C ABI (include/jimm_b200.h).
//
// Host-side structure mirrors the reference's module tree:
//   Tower (VisionTransformerBase, common/vit.py:104-248)  -> patch GEMM, cls/pos, [ln_pre], L x Block, ln_post, CLS | MAP head
//   Block (TransformerEncoder, common/transformer.py:22-132)
//   TextTower (nnx.Embed + Transformer + ln_final + pooling; models/clip.py:148-167, models/siglip.py:135-153)
//   heads (classifier / visual_projection / text_projection; contrastive logits)
// All arithmetic is in the kernels of gemm.cu / attention.cu / elementwise.cu / comm.cu; there is no CPU fallback.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <cmath>
#include <map>
#include <tuple>
#include <memory>
#include <string>
#include <vector>

#include "../../include/jimm_b200.h"
#include "comm.cuh"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

namespace jimm {

// ------------------------------------------------------------------------------------------
// error + launch accounting
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
static std::atomic<long long> g_launches{0};
static std::atomic<long long> g_graph_replays{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* env = getenv("JIMM_PDL"); v = env ? atoi(env) : 1; }
  return v;
}

#define JIMM_TRY(expr)          \
  do {                          \
    int _rc = (expr);           \
    if (_rc != 0) return _rc;   \
  } while (0)

// ------------------------------------------------------------------------------------------
// small RAII-free device memory pool (freed in model destroy)
// ------------------------------------------------------------------------------------------
struct DevPool {
  std::vector<void*> ptrs;
  size_t bytes = 0;
  int alloc(void** out, size_t n) {
    if (n == 0) n = 16;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, n);
    if (e != cudaSuccess) {
      set_last_error("cudaMalloc(%zu bytes) failed: %s", n, cudaGetErrorString(e));
      return JIMM_ENOMEM;
    }
    ptrs.push_back(p);
    bytes += n;
    *out = p;
    return 0;
  }
  void release() {
    for (void* p : ptrs) cudaFree(p);
    ptrs.clear();
    bytes = 0;
  }
};

struct HostParam {
  std::vector<int64_t> shape;   // the reference's flax shape
  std::vector<float> data;      // owned fp32 copy (jimm_model_set_param) ...
  const void* ref = nullptr;    // ... or a borrowed host pointer (jimm_model_set_param_ref), valid until finalize returns
  int dtype = DT_F32;           // element type behind ptr()
  bool transposed = false;      // ref holds the 2-D transpose [N, K] of the flax kernel's (K, N) view (a HuggingFace (out, in) weight as is)
  bool used = false;
  size_t n = 0;
  size_t numel() const { return n; }
  const void* ptr() const { return ref ? ref : static_cast<const void*>(data.data()); }
  size_t esize() const { return dtype == DT_F32 ? 4 : 2; }
  float at(size_t i) const {  // host-side read of element i of the STORED order
    if (dtype == DT_F32) return static_cast<const float*>(ptr())[i];
    const uint16_t h = static_cast<const uint16_t*>(ptr())[i];
    if (dtype == DT_BF16) { uint32_t u = static_cast<uint32_t>(h) << 16; float f; memcpy(&f, &u, 4); return f; }
    return __half2float(*reinterpret_cast<const __half*>(&h));
  }
};

struct LinearW {
  void* w = nullptr;   // [N, K] compute dtype, K-major
  float* b = nullptr;  // [N] fp32 or null
  int N = 0, K = 0;
};
struct LNW {
  float* scale = nullptr;
  float* bias = nullptr;
};
struct BlockW {
  LNW norm1, norm2;
  LinearW qkv, out, fc1, fc2;
  GemmPlan p_qkv, p_out, p_fc1, p_fc2;
};

struct EncoderCfg {  // one Transformer stack
  int D = 0, H = 0, M = 0, L = 0, act = 0, causal = 0;
  float eps = 1e-6f;
};

struct Encoder {
  EncoderCfg c;
  std::vector<BlockW> blocks;
};

struct VisionTower {
  bool present = false;
  int img = 0, P = 0, C = 0, D = 0, n = 0, n_pad = 0, S = 0, pooling = 0, pre_norm = 0, patch_bias = 0;
  int Kp = 0;  // patch GEMM K = P*P*C rounded up to a multiple of 8 (16-byte rows for TMA; the pad columns are zeros on both operands)
  bool patch_scatter = false;  // patch GEMM reduce-adds into the pos-initialised residual stream through a 3-D TMA map
  float eps_outer = 1e-5f;
  Encoder enc;
  LinearW patch;
  float* cls = nullptr;
  float* pos = nullptr;  // [S, D]
  LNW ln_pre, ln_post;
  // MAP head
  float* map_q = nullptr;  // [D] fp32: probe . Wq + bq (input independent)
  LinearW map_kv, map_out, map_fc1, map_fc2;
  LNW map_ln;
  // head after pooling (classifier / visual_projection); N == 0 -> none
  LinearW head;
  GemmPlan p_patch, p_head, p_map_kv, p_map_out, p_map_fc1, p_map_fc2;
};

struct TextTower {
  bool present = false;
  int T = 0, V = 0, D = 0, pool = 0;
  float eps_outer = 1e-5f;
  Encoder enc;
  float* table = nullptr;  // [V, D] fp32
  float* pos = nullptr;    // [T, D] fp32
  LNW ln_final;
  LinearW head;  // text_projection
  GemmPlan p_head;
};

// The text tower has its own residual stream / activation buffers so that the two towers of CLIP / SigLIP can run CONCURRENTLY on two
// streams (they are independent until the contrastive head): the tail rounds of one tower's persistent GEMMs and its small kernels are
// filled by the other tower's CTAs instead of leaving SMs idle.
struct TextWs {
  float* x = nullptr;     // fp32 residual stream [Bmax*T, Dt]
  void* h = nullptr;      // LN out / attention out
  void* big = nullptr;    // qkv | mlp hidden
  void* pooled = nullptr; // [Bmax, Dt]
  int* idx = nullptr;     // [Bmax] EOT positions
};

struct Workspace {
  float* x = nullptr;     // fp32 residual stream [Tmax, Dmax]
  void* h = nullptr;      // LN out / attention out (compute dtype) [Tmax, Dmax]
  void* big = nullptr;    // patches | qkv | mlp hidden | MAP kv (aliased; disjoint lifetimes)
  void* pooled = nullptr; // [Bmax, Dmax] compute dtype
  float* feat = nullptr;  // [Bmax, Dmax] fp32 (MAP attention out-proj / residual)
  void* mid2 = nullptr;   // [Bmax, 4*Dmax] compute dtype (MAP MLP hidden)
  int* idx = nullptr;     // [Bmax]
  float* emb_i = nullptr; // [Bmax, E] fp32 encoder outputs
  float* emb_t = nullptr;
  float* nrm_i = nullptr; // normalised
  float* nrm_t = nullptr;
  void* in_img = nullptr; // host-path staging: image batch (fp32 worst case)
  uint8_t* in_u8 = nullptr;  // host-path staging of raw uint8 RGB frames (jimm_vit_forward_host_u8); grown on demand
  size_t in_u8_bytes = 0;
  int32_t* in_ids = nullptr;
  float* out_dev = nullptr;  // host-path staging for results
  size_t out_dev_elems = 0;
};

}  // namespace jimm

using namespace jimm;

struct jimm_model {
  jimm_config_t cfg;
  int device = 0;
  bool finalized = false;
  int max_batch = 0;
  int cdt = DT_F16;    // compute dtype of GEMM operands
  int adt = DT_F16;    // dtype of the qkv / MAP-kv buffers consumed by the attention kernels (16-bit even in fp32 mode)
  std::map<std::string, HostParam> host;
  DevPool pool;
  VisionTower vis;
  TextTower txt;
  float* logit_scale = nullptr;
  float* logit_bias = nullptr;
  Workspace ws;
  TextWs wt;
  // two-stream execution of the dual towers (JIMM_DUAL_STREAMS=0 disables): text tower on `text_stream`, forked from / joined to the
  // caller's stream with events
  bool dual_streams = true;
  cudaStream_t text_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  float* graph_out_t = nullptr;  // text-tower twin of graph_out
  CommState comm;
  cudaStream_t copy_stream = nullptr;            // host path: H2D of chunk i+1 overlaps the forward of chunk i
  static constexpr int kHostSlices = 4;
  cudaEvent_t ev_copied[kHostSlices] = {};
  cudaEvent_t ev_consumed[kHostSlices] = {};
  cudaEvent_t ev_start = nullptr;
  // Back-to-back host-path calls on one stream are ordered slot by slot (a slot is free again once its slice has been through
  // patchify), so the copies of call k+1 run under the towers of call k: the asynchronous-dispatch pipeline of the reference.
  bool host_chain = false;            // the last toucher of the staging buffer was jimm_vit_forward_host ...
  cudaStream_t host_chain_stream = nullptr;  // ... on this stream ...
  int host_chain_sizes[kHostSlices] = {};    // ... with this slice layout
  int host_chain_kind = 0;                   // ... 0: float images into in_img, 1: uint8 frames into in_u8 (+ front-end into in_img)
  bool slot_recorded[kHostSlices] = {};
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;
  size_t prof_used = 0;
  double prof_flops = 0.0;
  long long prof_launches = 0;
  int epi_mode_16 = 2;  // epilogue mode for 16-bit no-residual outputs (2 = TMA store)
  int epi_mode_res = 2; // epilogue mode for fp32 residual outputs (2 = TMA reduce-add into the residual stream)
  bool l2_alternate = true;  // JIMM_L2_ALTERNATE=0 disables the alternating walk direction
  bool simt = false;    // JIMM_GEMM_IMPL=simt: bisection aid, routes every GEMM through the SIMT cross-check kernel
  // CUDA-graph replay of a whole tower for small batches (launch-bound regime; config 1 is B=4): the second call of a
  // (tower, batch, dtype | length) shape is stream-captured from fixed staging buffers, later calls replay it.
  struct GraphEntry {
    cudaGraphExec_t exec = nullptr;
    long long launches = 0;
    int seen = 0;
  };
  std::map<std::tuple<int, int, int>, GraphEntry> graphs;
  int graph_max_batch = 32;  // JIMM_GRAPH_MAX_BATCH (0 disables)
  float* graph_out = nullptr;  // [graph_max_batch, max(vision out, E)]
  cudaStream_t capture_stream = nullptr;
};

namespace jimm {

static size_t cdt_size(const jimm_model* m) { return dtype_size(m->cdt); }

// ------------------------------------------------------------------------------------------
// parameter upload / packing helpers (finalize)
// ------------------------------------------------------------------------------------------
struct Packer {
  jimm_model* m;
  UploadRing ring;
  cudaStream_t stream = 0;

  // one synchronisation for the whole finalize
  void done() {
    cudaStreamSynchronize(stream);
    ring.destroy();
  }

  HostParam* find(const std::string& name, std::initializer_list<int64_t> shape) {
    auto it = m->host.find(name);
    if (it == m->host.end()) {
      set_last_error("finalize: parameter '%s' was never set (the reference asserts every flax param is visited, models/vit.py:259)", name.c_str());
      return nullptr;
    }
    HostParam& hp = it->second;
    std::vector<int64_t> want(shape);
    if (hp.shape != want) {
      std::string got, exp;
      for (auto d : hp.shape) got += std::to_string(d) + ",";
      for (auto d : want) exp += std::to_string(d) + ",";
      set_last_error("finalize: shape mismatch for '%s': expected (%s) got (%s)", name.c_str(), exp.c_str(), got.c_str());
      return nullptr;
    }
    hp.used = true;
    return &hp;
  }

  // `rows` rows of K stored elements -> dst[r * ldd + k] of out_type, streamed through the ring in row chunks
  int rows_to_device(const HostParam* hp, size_t rows, size_t K, void* dst, int out_type, size_t ldd) {
    const size_t es = hp->esize(), row_bytes = K * es;
    if (row_bytes == 0 || rows == 0) return 0;
    const uint8_t* src = static_cast<const uint8_t*>(hp->ptr());
    const size_t out_es = dtype_size(out_type);
    if (row_bytes > UploadRing::kCap) {  // a single very long row (flat vectors): split it into pieces
      if (rows != 1 || ldd != K) { set_last_error("finalize: row of %zu bytes exceeds the staging slot", row_bytes); return JIMM_EINVAL; }
      const size_t per = UploadRing::kCap / es;
      for (size_t k0 = 0; k0 < K; k0 += per) {
        const size_t kc = K - k0 < per ? K - k0 : per;
        void* d = nullptr;
        JIMM_TRY(ring.stage(src + k0 * es, kc * es, stream, &d));
        JIMM_TRY(pack_rows_run(d, hp->dtype, 1, kc, static_cast<uint8_t*>(dst) + k0 * out_es, out_type, kc, stream));
        JIMM_TRY(ring.commit(stream));
      }
      return 0;
    }
    const size_t per = UploadRing::kCap / row_bytes;
    for (size_t r0 = 0; r0 < rows; r0 += per) {
      const size_t rc = rows - r0 < per ? rows - r0 : per;
      void* d = nullptr;
      JIMM_TRY(ring.stage(src + r0 * row_bytes, rc * row_bytes, stream, &d));
      JIMM_TRY(pack_rows_run(d, hp->dtype, rc, K, static_cast<uint8_t*>(dst) + r0 * ldd * out_es, out_type, ldd, stream));
      JIMM_TRY(ring.commit(stream));
    }
    return 0;
  }

  // fp32 vector / tensor uploaded element for element (biases, LayerNorm, cls, pos, embedding table, scalars)
  int upload_f32(const std::string& name, std::initializer_list<int64_t> shape, float** out) {
    HostParam* hp = find(name, shape);
    if (!hp) return JIMM_ESTATE;
    if (hp->transposed) { set_last_error("finalize: '%s' cannot be handed over transposed", name.c_str()); return JIMM_EINVAL; }
    void* d = nullptr;
    JIMM_TRY(m->pool.alloc(&d, hp->numel() * sizeof(float)));
    // 2-D tensors go row by row so that a long table streams through the ring in row chunks
    const size_t K = hp->shape.empty() ? 1 : static_cast<size_t>(hp->shape.back());
    const size_t rows = K ? hp->numel() / K : 0;
    JIMM_TRY(rows_to_device(hp, rows, K, d, DT_F32, K));
    *out = static_cast<float*>(d);
    return 0;
  }
  int upload_ln(const std::string& prefix, int D, LNW* ln) {
    JIMM_TRY(upload_f32(prefix + ".scale", {D}, &ln->scale));
    JIMM_TRY(upload_f32(prefix + ".bias", {D}, &ln->bias));
    return 0;
  }
  // flax kernel viewed as (K, N) row-major  ->  rows [n0, n0+N) of a packed [Ntot, ldd] K-major operand (ldd >= K: zero-padded K)
  int pack_kernel(const std::string& name, std::initializer_list<int64_t> shape, int K, int N, void* dst_base, int n0, int ldd = 0) {
    if (ldd <= 0) ldd = K;
    HostParam* hp = find(name, shape);
    if (!hp) return JIMM_ESTATE;
    if (hp->numel() != static_cast<size_t>(K) * N) { set_last_error("finalize: '%s' numel mismatch", name.c_str()); return JIMM_ESTATE; }
    uint8_t* dst = static_cast<uint8_t*>(dst_base) + static_cast<size_t>(n0) * ldd * cdt_size(m);
    if (hp->transposed) return rows_to_device(hp, N, K, dst, m->cdt, ldd);  // already [N, K]: cast-copy
    const size_t es = hp->esize(), row_bytes = static_cast<size_t>(N) * es;
    if (row_bytes > UploadRing::kCap) { set_last_error("finalize: '%s' row of %zu bytes exceeds the staging slot", name.c_str(), row_bytes); return JIMM_EINVAL; }
    const int per = static_cast<int>(UploadRing::kCap / row_bytes);
    const uint8_t* src = static_cast<const uint8_t*>(hp->ptr());
    for (int k0 = 0; k0 < K; k0 += per) {
      const int kc = K - k0 < per ? K - k0 : per;
      void* d = nullptr;
      JIMM_TRY(ring.stage(src + static_cast<size_t>(k0) * row_bytes, static_cast<size_t>(kc) * row_bytes, stream, &d));
      JIMM_TRY(pack_transpose_run(d, hp->dtype, kc, N, dst, m->cdt, ldd, k0, stream));
      JIMM_TRY(ring.commit(stream));
    }
    return 0;
  }
  int alloc_linear(LinearW* lw, int N, int K, bool bias) {
    lw->N = N; lw->K = K;
    JIMM_TRY(m->pool.alloc(&lw->w, static_cast<size_t>(N) * K * cdt_size(m)));
    if (bias) {
      void* b = nullptr;
      JIMM_TRY(m->pool.alloc(&b, static_cast<size_t>(N) * sizeof(float)));
      lw->b = static_cast<float*>(b);
    }
    return 0;
  }
  int upload_bias_at(const std::string& name, std::initializer_list<int64_t> shape, float* dst, size_t count) {
    HostParam* hp = find(name, shape);
    if (!hp) return JIMM_ESTATE;
    if (hp->numel() != count) { set_last_error("finalize: '%s' numel mismatch", name.c_str()); return JIMM_ESTATE; }
    return rows_to_device(hp, 1, count, dst, DT_F32, count);
  }
  // element (k, n) of a kernel's flax (K, N) view, whatever its stored order
  static float kn(const HostParam* hp, size_t k, size_t n, size_t K, size_t N) { return hp->transposed ? hp->at(n * K + k) : hp->at(k * N + n); }
  // nnx.Linear: kernel (K,N), optional bias (N)
  int linear(const std::string& prefix, int K, int N, bool bias, LinearW* lw) {
    JIMM_TRY(alloc_linear(lw, N, K, bias));
    JIMM_TRY(pack_kernel(prefix + ".kernel", {K, N}, K, N, lw->w, 0));
    if (bias) JIMM_TRY(upload_bias_at(prefix + ".bias", {N}, lw->b, N));
    return 0;
  }
  // nnx.MultiHeadAttention projections -> fused operand; names: subset of {"query","key","value"}
  int fused_proj(const std::string& attn_prefix, const std::vector<std::string>& names, int D, int H, LinearW* lw) {
    const int d = D / H;
    const int N = D * static_cast<int>(names.size());
    JIMM_TRY(alloc_linear(lw, N, D, true));
    for (size_t i = 0; i < names.size(); ++i) {
      JIMM_TRY(pack_kernel(attn_prefix + "." + names[i] + ".kernel", {D, H, d}, D, D, lw->w, static_cast<int>(i) * D));
      JIMM_TRY(upload_bias_at(attn_prefix + "." + names[i] + ".bias", {H, d}, lw->b + i * D, D));
    }
    return 0;
  }
  int out_proj(const std::string& attn_prefix, int D, int H, LinearW* lw) {
    const int d = D / H;
    JIMM_TRY(alloc_linear(lw, D, D, true));
    JIMM_TRY(pack_kernel(attn_prefix + ".out.kernel", {H, d, D}, D, D, lw->w, 0));
    JIMM_TRY(upload_bias_at(attn_prefix + ".out.bias", {D}, lw->b, D));
    return 0;
  }
  // MultiHeadAttentionPoolingHead parameters (common/vit.py:27-85) under `mp`
  int map_head(const std::string& mp, int D, int H, VisionTower* v) {
    const int d = D / H;
    JIMM_TRY(fused_proj(mp + "attn", {"key", "value"}, D, H, &v->map_kv));
    JIMM_TRY(out_proj(mp + "attn", D, H, &v->map_out));
    JIMM_TRY(upload_ln(mp + "layernorm", D, &v->map_ln));
    JIMM_TRY(linear(mp + "mlp.layers.0", D, 4 * D, true, &v->map_fc1));  // intermediate_size = 4*hidden (common/vit.py:175)
    JIMM_TRY(linear(mp + "mlp.layers.2", 4 * D, D, true, &v->map_fc2));
    // probe query is input independent: q = probe . Wq + bq  (common/vit.py:96-97), done once on the host in fp64
    HostParam* probe = find(mp + "probe", {1, 1, D});
    HostParam* wq = find(mp + "attn.query.kernel", {D, H, d});
    HostParam* bq = find(mp + "attn.query.bias", {H, d});
    if (!probe || !wq || !bq) return JIMM_ESTATE;
    std::vector<float> q(D);
    for (int o = 0; o < D; ++o) {
      double acc = bq->at(o);
      for (int i = 0; i < D; ++i) acc += static_cast<double>(probe->at(i)) * kn(wq, i, o, D, D);
      q[o] = static_cast<float>(acc);
    }
    void* dq = nullptr;
    JIMM_TRY(m->pool.alloc(&dq, D * sizeof(float)));
    JIMM_CUDA_CHECK(cudaMemcpy(dq, q.data(), D * sizeof(float), cudaMemcpyHostToDevice));
    v->map_q = static_cast<float*>(dq);
    return 0;
  }
  int encoder(const std::string& prefix, Encoder* enc) {
    const EncoderCfg& c = enc->c;
    enc->blocks.resize(c.L);
    for (int i = 0; i < c.L; ++i) {
      const std::string f = prefix + "blocks.layers." + std::to_string(i) + ".";
      BlockW& b = enc->blocks[i];
      JIMM_TRY(upload_ln(f + "norm1", c.D, &b.norm1));
      JIMM_TRY(upload_ln(f + "norm2", c.D, &b.norm2));
      JIMM_TRY(fused_proj(f + "attn", {"query", "key", "value"}, c.D, c.H, &b.qkv));
      JIMM_TRY(out_proj(f + "attn", c.D, c.H, &b.out));
      JIMM_TRY(linear(f + "mlp.layers.0", c.D, c.M, true, &b.fc1));
      JIMM_TRY(linear(f + "mlp.layers.3", c.M, c.D, true, &b.fc2));
    }
    return 0;
  }
};

// ------------------------------------------------------------------------------------------
// GEMM dispatch (plan-based tcgen05 path; optional SIMT bisection path)
// ------------------------------------------------------------------------------------------
static int run_gemm(jimm_model* m, const GemmPlan& p, const void* A, int lda, const LinearW& w, int M, cudaStream_t s, int reverse = 0) {
  if (M <= 0) return 0;
  if (m->simt) return gemm_simt_run(p.dtype, A, lda, w.w, w.K, M, p.N, p.K, p.epi, s);
  if (!m->prof_on) return gemm_plan_run(&p, M, s, reverse);
  if (m->prof_used + 2 > m->prof_ev.size()) {
    for (int i = 0; i < 256; ++i) {
      cudaEvent_t e;
      JIMM_CUDA_CHECK(cudaEventCreate(&e));
      m->prof_ev.push_back(e);
    }
  }
  JIMM_CUDA_CHECK(cudaEventRecord(m->prof_ev[m->prof_used], s));
  JIMM_TRY(gemm_plan_run(&p, M, s, reverse));
  JIMM_CUDA_CHECK(cudaEventRecord(m->prof_ev[m->prof_used + 1], s));
  m->prof_used += 2;
  m->prof_flops += 2.0 * M * static_cast<double>(p.N) * p.K;
  m->prof_launches += 1;
  return 0;
}

static GemmEpilogue epi_plain(const LinearW& w, int act, void* out, int out_type, int ldo, int mode) {
  GemmEpilogue e;
  e.bias = w.b; e.act = act; e.out = out; e.out_type = out_type; e.ldo = ldo; e.mode = mode;
  return e;
}
static GemmEpilogue epi_residual(const LinearW& w, float* x, int ld, int mode) {
  GemmEpilogue e;
  e.bias = w.b; e.residual = x; e.ldr = ld; e.out = x; e.out_type = DT_F32; e.ldo = ld; e.mode = mode;
  return e;
}

struct EncBufs {  // the activation buffers one encoder stack works in
  float* x;
  void* h;
  void* big;
};

static int plan_encoder(jimm_model* m, Encoder* enc, int Tmax, EncBufs ws) {
  const EncoderCfg& c = enc->c;
  const int act = c.act == JIMM_QUICK_GELU ? ACT_QUICK_GELU : ACT_GELU_TANH;
  for (BlockW& b : enc->blocks) {
    // QKV: h[T,D] x Wqkv[3D,D]^T + b -> qkv (16-bit) [T,3D]
    JIMM_TRY(gemm_plan_init(&b.p_qkv, m->cdt, ws.h, c.D, b.qkv.w, c.D, Tmax, 3 * c.D, c.D,
                            epi_plain(b.qkv, ACT_NONE, ws.big, m->adt, 3 * c.D, m->epi_mode_16)));
    // out-proj: attn[T,D] x Wo[D,D]^T + bo + x -> x
    JIMM_TRY(gemm_plan_init(&b.p_out, m->cdt, ws.h, c.D, b.out.w, c.D, Tmax, c.D, c.D, epi_residual(b.out, ws.x, c.D, m->epi_mode_res)));
    // FC1: h x W1^T + b1 -> act -> mid [T,M]
    JIMM_TRY(gemm_plan_init(&b.p_fc1, m->cdt, ws.h, c.D, b.fc1.w, c.D, Tmax, c.M, c.D,
                            epi_plain(b.fc1, act, ws.big, m->cdt, c.M, m->epi_mode_16)));
    // FC2: mid x W2^T + b2 + x -> x
    JIMM_TRY(gemm_plan_init(&b.p_fc2, m->cdt, ws.big, c.M, b.fc2.w, c.M, Tmax, c.D, c.M, epi_residual(b.fc2, ws.x, c.D, m->epi_mode_res)));
  }
  return 0;
}

static int plan_map_head(jimm_model* m, int Bm, int Tv) {
  VisionTower& v = m->vis;
  Workspace& ws = m->ws;
  const int D = v.D;
  JIMM_TRY(gemm_plan_init(&v.p_map_kv, m->cdt, ws.h, D, v.map_kv.w, D, Tv, 2 * D, D, epi_plain(v.map_kv, ACT_NONE, ws.big, m->adt, 2 * D, m->epi_mode_16)));
  JIMM_TRY(gemm_plan_init(&v.p_map_out, m->cdt, ws.pooled, D, v.map_out.w, D, Bm, D, D, epi_plain(v.map_out, ACT_NONE, ws.feat, DT_F32, D, 0)));
  JIMM_TRY(gemm_plan_init(&v.p_map_fc1, m->cdt, ws.pooled, D, v.map_fc1.w, D, Bm, 4 * D, D, epi_plain(v.map_fc1, ACT_GELU_TANH, ws.mid2, m->cdt, 4 * D, 0)));
  GemmEpilogue e = epi_plain(v.map_fc2, ACT_NONE, ws.out_dev, DT_F32, D, 0);
  e.residual = ws.feat; e.ldr = D;
  JIMM_TRY(gemm_plan_init(&v.p_map_fc2, m->cdt, ws.mid2, 4 * D, v.map_fc2.w, 4 * D, Bm, D, 4 * D, e));
  return 0;
}

// x: fp32 [B*S, D] residual stream in ws.x.  TransformerEncoder.__call__ x L (common/transformer.py:116-132,190-196).
static int run_encoder(jimm_model* m, Encoder* enc, int B, int S, cudaStream_t s, EncBufs ws) {
  const EncoderCfg& c = enc->c;
  const int T = B * S;
  // Boustrophedon schedule: every kernel walks its rows / tiles / items in the direction opposite to its producer, so it
  // starts on the data written last -- the part of the 77-310 MB activation still resident in the 126 MB L2.
  int dir = m->l2_alternate ? 1 : 0;  // the patch GEMM / embedding kernels ran forward -> the first LayerNorm runs backward
  auto flip = [&]() { const int d = dir; if (m->l2_alternate) dir ^= 1; return d; };
  for (BlockW& b : enc->blocks) {
    JIMM_TRY(layernorm_run(ws.x, c.D, 1, 0, nullptr, b.norm1.scale, b.norm1.bias, c.eps, ws.h, m->cdt, c.D, T, c.D, s, flip()));
    JIMM_TRY(run_gemm(m, b.p_qkv, ws.h, c.D, b.qkv, T, s, flip()));
    JIMM_TRY(attention_run(ws.big, m->adt, ws.h, m->cdt, B, S, c.H, c.causal, s, flip()));
    JIMM_TRY(run_gemm(m, b.p_out, ws.h, c.D, b.out, T, s, flip()));  // + residual
    JIMM_TRY(layernorm_run(ws.x, c.D, 1, 0, nullptr, b.norm2.scale, b.norm2.bias, c.eps, ws.h, m->cdt, c.D, T, c.D, s, flip()));
    JIMM_TRY(run_gemm(m, b.p_fc1, ws.h, c.D, b.fc1, T, s, flip()));
    JIMM_TRY(run_gemm(m, b.p_fc2, ws.big, c.M, b.fc2, T, s, flip()));  // + residual
  }
  return 0;
}

// MultiHeadAttentionPoolingHead.__call__ (common/vit.py:87-101) on the tokens in ws.h (compute dtype, [B*S, D]); out fp32 [B, D]
static int run_map_head(jimm_model* m, int B, int S, float* out, cudaStream_t s) {
  VisionTower& v = m->vis;
  Workspace& ws = m->ws;
  const int D = v.D, T = B * S;
  JIMM_TRY(run_gemm(m, v.p_map_kv, ws.h, D, v.map_kv, T, s));                                        // k | v  [T, 2D]
  JIMM_TRY(map_attention_run(v.map_q, ws.big, m->adt, ws.pooled, m->cdt, B, S, v.enc.c.H, s));     // [B, D]
  JIMM_TRY(run_gemm(m, v.p_map_out, ws.pooled, D, v.map_out, B, s));                                 // -> feat fp32 [B, D]
  JIMM_TRY(layernorm_run(ws.feat, D, 1, 0, nullptr, v.map_ln.scale, v.map_ln.bias, v.eps_outer, ws.pooled, m->cdt, D, B, D, s));
  JIMM_TRY(run_gemm(m, v.p_map_fc1, ws.pooled, D, v.map_fc1, B, s));                                 // gelu -> mid2 [B, 4D]
  GemmPlan p = v.p_map_fc2;  // + bias + residual(feat) -> out fp32 [B, D]
  p.epi.out = out;
  return run_gemm(m, p, ws.mid2, 4 * D, v.map_fc2, B, s);
}

// VisionTransformerBase.__call__ (common/vit.py:216-248) + the model's head.  out: fp32 [B, out_dim]
static int run_vision(jimm_model* m, const void* img, int in_dtype, int B, float* out, cudaStream_t s) {
  VisionTower& v = m->vis;
  Workspace& ws = m->ws;
  const int D = v.D, S = v.S, n = v.n;
  // patch embed + pos (+cls)
  if (v.patch_scatter) {
    JIMM_TRY(tokens_init_run(ws.x, v.pooling == JIMM_POOL_CLS ? v.cls : nullptr, v.pos, B, S, D, s));
    JIMM_TRY(patchify_run(img, in_dtype, B, v.img, v.img, v.C, v.P, ws.big, m->cdt, s, v.n_pad, v.Kp));
    JIMM_TRY(run_gemm(m, v.p_patch, ws.big, v.patch.K, v.patch, B * v.n_pad, s));
  } else {
    JIMM_TRY(patchify_run(img, in_dtype, B, v.img, v.img, v.C, v.P, ws.big, m->cdt, s, 0, v.Kp));
    JIMM_TRY(run_gemm(m, v.p_patch, ws.big, v.patch.K, v.patch, B * n, s));
    if (v.pooling == JIMM_POOL_CLS) JIMM_TRY(cls_row_run(ws.x, v.cls, v.pos, B, S, D, s));
  }
  if (v.pre_norm) JIMM_TRY(layernorm_run(ws.x, D, 1, 0, nullptr, v.ln_pre.scale, v.ln_pre.bias, v.eps_outer, ws.x, DT_F32, D, B * S, D, s));
  JIMM_TRY(run_encoder(m, &v.enc, B, S, s, EncBufs{ws.x, ws.h, ws.big}));
  if (v.pooling == JIMM_POOL_CLS) {
    // ln_post is per-row, only row 0 of each sample is consumed (common/vit.py:244-246)
    if (v.head.N > 0) {
      JIMM_TRY(layernorm_run(ws.x, D, S, 0, nullptr, v.ln_post.scale, v.ln_post.bias, v.eps_outer, ws.pooled, m->cdt, D, B, D, s));
      GemmPlan p = v.p_head;
      p.epi.out = out;
      JIMM_TRY(run_gemm(m, p, ws.pooled, D, v.head, B, s));
    } else {
      JIMM_TRY(layernorm_run(ws.x, D, S, 0, nullptr, v.ln_post.scale, v.ln_post.bias, v.eps_outer, out, DT_F32, D, B, D, s));
    }
    return 0;
  }
  // MAP head (common/vit.py:87-101)
  const int T = B * S;
  JIMM_TRY(layernorm_run(ws.x, D, 1, 0, nullptr, v.ln_post.scale, v.ln_post.bias, v.eps_outer, ws.h, m->cdt, D, T, D, s));
  return run_map_head(m, B, S, out, s);
}

// CLIP.encode_text (models/clip.py:148-167) / SigLIP.encode_text (models/siglip.py:135-153).  out fp32 [B, Dt]
static int run_text(jimm_model* m, const int32_t* ids, int B, int T, float* out, cudaStream_t s) {
  TextTower& t = m->txt;
  TextWs& ws = m->wt;
  JIMM_TRY(embed_run(ids, t.table, t.pos, ws.x, B, T, t.D, t.V, s));
  JIMM_TRY(run_encoder(m, &t.enc, B, T, s, EncBufs{ws.x, ws.h, ws.big}));
  if (t.pool == JIMM_TPOOL_EOT_ARGMAX) {
    JIMM_TRY(argmax_ids_run(ids, ws.idx, B, T, s));
    JIMM_TRY(layernorm_run(ws.x, t.D, T, 0, ws.idx, t.ln_final.scale, t.ln_final.bias, t.eps_outer, ws.pooled, m->cdt, t.D, B, t.D, s));
  } else {
    JIMM_TRY(layernorm_run(ws.x, t.D, T, T - 1, nullptr, t.ln_final.scale, t.ln_final.bias, t.eps_outer, ws.pooled, m->cdt, t.D, B, t.D, s));
  }
  GemmPlan p = t.p_head;
  p.epi.out = out;
  JIMM_TRY(run_gemm(m, p, ws.pooled, t.D, t.head, B, s));
  return 0;
}

static int check_ready(const jimm_model* m, int B) {
  if (!m) { set_last_error("null model"); return JIMM_EINVAL; }
  if (!m->finalized) { set_last_error("model not finalized"); return JIMM_ESTATE; }
  if (B < 0) { set_last_error("negative batch"); return JIMM_EINVAL; }
  return 0;
}
static int set_device(const jimm_model* m) {
  JIMM_CUDA_CHECK(cudaSetDevice(m->device));
  return 0;
}

static int vision_out_dim(const jimm_model* m) { return m->vis.head.N > 0 ? m->vis.head.N : m->vis.D; }

// ------------------------------------------------------------------------------------------
// CUDA-graph replay for small batches
// ------------------------------------------------------------------------------------------
static void graphs_release(jimm_model* m) {
  for (auto& kv : m->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  m->graphs.clear();
}

// Runs `body` (which enqueues a tower on `s`, reading and writing fixed workspace buffers only) eagerly the first time a key is
// seen, captures it into a graph the second time, and replays the graph afterwards.  Any capture problem disables graphs for
// the model and falls back to the eager launches -- the same kernels either way.
template <typename F>
static int run_graphed(jimm_model* m, std::tuple<int, int, int> key, cudaStream_t s, F&& body) {
  if (m->graph_max_batch <= 0 || m->prof_on || m->simt) return body(s);
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) {  // the caller is capturing already
    cudaGetLastError();
    return body(s);
  }
  jimm_model::GraphEntry& e = m->graphs[key];
  if (e.exec) {
    JIMM_CUDA_CHECK(cudaGraphLaunch(e.exec, s));
    g_launches.fetch_add(e.launches, std::memory_order_relaxed);
    g_graph_replays.fetch_add(1, std::memory_order_relaxed);
    return 0;
  }
  if (e.seen++ == 0) return body(s);
  // Capture on a private stream: the caller's stream may be the legacy default stream, which cannot be captured; nothing
  // executes during capture, and the instantiated graph is launched on the caller's stream.
  if (!m->capture_stream && cudaStreamCreateWithFlags(&m->capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    m->graph_max_batch = 0;
    return body(s);
  }
  const long long l0 = g_launches.load();
  if (cudaStreamBeginCapture(m->capture_stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
    cudaGetLastError();
    m->graph_max_batch = 0;
    return body(s);
  }
  const int rc = body(m->capture_stream);
  cudaGraph_t g = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(m->capture_stream, &g);
  const long long captured = g_launches.load() - l0;
  g_launches.fetch_sub(captured, std::memory_order_relaxed);  // captured launches have not run
  cudaGraphExec_t exec = nullptr;
  if (rc == 0 && ce == cudaSuccess && g && cudaGraphInstantiate(&exec, g, 0) == cudaSuccess) {
    cudaGraphDestroy(g);
    e.exec = exec;
    e.launches = captured;
    JIMM_CUDA_CHECK(cudaGraphLaunch(e.exec, s));
    g_launches.fetch_add(e.launches, std::memory_order_relaxed);
    g_graph_replays.fetch_add(1, std::memory_order_relaxed);
    return 0;
  }
  if (g) cudaGraphDestroy(g);
  cudaGetLastError();
  m->graph_max_batch = 0;
  if (rc != 0) return rc;
  return body(s);
}

// Vision tower of one chunk.  Small chunks go through the graph: input staged into ws.in_img, result from m->graph_out.
static int exec_vision(jimm_model* m, const void* img, int in_dtype, int n, float* out, cudaStream_t s) {
  if (n <= 0 || n > m->graph_max_batch || !m->graph_out) return run_vision(m, img, in_dtype, n, out, s);
  const size_t bytes = static_cast<size_t>(n) * m->vis.img * m->vis.img * m->vis.C * dtype_size(in_dtype);
  if (img != m->ws.in_img) {
    m->host_chain = false;  // the staging buffer is written outside the host path's slot protocol
    JIMM_CUDA_CHECK(cudaMemcpyAsync(m->ws.in_img, img, bytes, cudaMemcpyDeviceToDevice, s));
  }
  JIMM_TRY(run_graphed(m, std::make_tuple(0, n, in_dtype), s, [&](cudaStream_t cs) { return run_vision(m, m->ws.in_img, in_dtype, n, m->graph_out, cs); }));
  JIMM_CUDA_CHECK(cudaMemcpyAsync(out, m->graph_out, static_cast<size_t>(n) * vision_out_dim(m) * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

static int exec_text(jimm_model* m, const int32_t* ids, int n, int T, float* out, cudaStream_t s) {
  if (n <= 0 || n > m->graph_max_batch || !m->graph_out_t) return run_text(m, ids, n, T, out, s);
  if (ids != m->ws.in_ids) JIMM_CUDA_CHECK(cudaMemcpyAsync(m->ws.in_ids, ids, static_cast<size_t>(n) * T * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
  JIMM_TRY(run_graphed(m, std::make_tuple(1, n, T), s, [&](cudaStream_t cs) { return run_text(m, m->ws.in_ids, n, T, m->graph_out_t, cs); }));
  JIMM_CUDA_CHECK(cudaMemcpyAsync(out, m->graph_out_t, static_cast<size_t>(n) * m->txt.D * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

// Handle of a bare sub-module (kind JIMM_ENCODER: Transformer, parameters "blocks.layers.{i}.*", common/transformer.py:135-196;
// kind JIMM_MAPHEAD: MultiHeadAttentionPoolingHead, parameters "probe", "attn.*", "layernorm.*", "mlp.layers.{0,2}.*",
// common/vit.py:12-101).  cfg: v_width / v_heads / v_mlp / v_layers / v_act / v_eps_block (block LN) / v_eps_outer (MAP LN) / t_causal,
// ctx_len = max tokens per sample.  The same kernels and orchestration as inside a tower (run_encoder / run_map_head).
static int finalize_sub(jimm_model* m, int max_batch) {
  const jimm_config_t& c = m->cfg;
  Packer pk{m};
  int rc = 0;
  VisionTower& v = m->vis;
  v.present = false;
  v.D = c.v_width; v.S = c.ctx_len; v.n = v.S; v.pooling = JIMM_POOL_MAP; v.eps_outer = c.v_eps_outer;
  v.enc.c.D = c.v_width; v.enc.c.H = c.v_heads; v.enc.c.M = c.v_mlp; v.enc.c.L = c.kind == JIMM_ENCODER ? c.v_layers : 0;
  v.enc.c.act = c.v_act; v.enc.c.causal = c.t_causal; v.enc.c.eps = c.v_eps_block;
  const int D = v.D;
  if (c.kind == JIMM_ENCODER) rc = pk.encoder("", &v.enc);
  else rc = pk.map_head("", D, c.v_heads, &v);
  pk.done();
  if (rc) return rc;
  for (auto& kv : m->host) {
    if (!kv.second.used) { set_last_error("finalize: unexpected parameter '%s' was set but is not part of this module", kv.first.c_str()); return JIMM_ESTATE; }
  }
  m->host.clear();
  Workspace& ws = m->ws;
  const size_t cs = cdt_size(m), Bm = max_batch, Tv = Bm * v.S;
  size_t big = Tv * 3 * D * 2;
  if (Tv * static_cast<size_t>(c.v_mlp) * cs > big) big = Tv * static_cast<size_t>(c.v_mlp) * cs;
  void* p = nullptr;
  JIMM_TRY(m->pool.alloc(&p, Tv * D * sizeof(float))); ws.x = static_cast<float*>(p);
  JIMM_TRY(m->pool.alloc(&ws.h, Tv * D * cs));
  JIMM_TRY(m->pool.alloc(&ws.big, big));
  JIMM_TRY(m->pool.alloc(&ws.pooled, Bm * D * cs));
  JIMM_TRY(m->pool.alloc(&p, Bm * D * sizeof(float))); ws.feat = static_cast<float*>(p);
  JIMM_TRY(m->pool.alloc(&ws.mid2, Bm * 4 * D * cs));
  ws.out_dev_elems = Bm * D;
  JIMM_TRY(m->pool.alloc(&p, ws.out_dev_elems * sizeof(float))); ws.out_dev = static_cast<float*>(p);
  if (c.kind == JIMM_ENCODER) JIMM_TRY(plan_encoder(m, &v.enc, static_cast<int>(Tv), EncBufs{ws.x, ws.h, ws.big}));
  else JIMM_TRY(plan_map_head(m, static_cast<int>(Bm), static_cast<int>(Tv)));
  JIMM_CUDA_CHECK(cudaDeviceSynchronize());
  m->graph_max_batch = 0;
  m->max_batch = max_batch;
  m->finalized = true;
  return 0;
}

}  // namespace jimm

// ==========================================================================================
// C ABI
// ==========================================================================================
extern "C" {

const char* jimm_last_error(void) { return g_err; }
int jimm_abi_version(void) { return 2; }
long long jimm_launch_count(void) { return g_launches.load(); }
long long jimm_graph_replay_count(void) { return g_graph_replays.load(); }

int jimm_model_create(const jimm_config_t* cfg, int device, jimm_model_t** out) {
  if (!cfg || !out) { set_last_error("jimm_model_create: null argument"); return JIMM_EINVAL; }
  if (cfg->kind < JIMM_VIT || cfg->kind > JIMM_MAPHEAD) { set_last_error("bad kind %d", cfg->kind); return JIMM_EINVAL; }
  const bool sub = cfg->kind == JIMM_ENCODER || cfg->kind == JIMM_MAPHEAD;  // a bare Transformer / MultiHeadAttentionPoolingHead
  if (cfg->pooling != JIMM_POOL_CLS && cfg->pooling != JIMM_POOL_MAP) {
    set_last_error("pooling_type must be either MAP or CLS.");  // common/vit.py:178
    return JIMM_EINVAL;
  }
  if (cfg->v_heads <= 0 || cfg->v_width != cfg->v_heads * 64) {
    set_last_error("vision head_dim must be 64 (width %d, heads %d): the attention kernels are specialised for it", cfg->v_width, cfg->v_heads);
    return JIMM_EINVAL;
  }
  const bool dual = cfg->kind == JIMM_CLIP || cfg->kind == JIMM_SIGLIP;
  if (dual && (cfg->t_heads <= 0 || cfg->t_width != cfg->t_heads * 64)) {
    set_last_error("text head_dim must be 64 (width %d, heads %d)", cfg->t_width, cfg->t_heads);
    return JIMM_EINVAL;
  }
  if (cfg->compute_dtype < JIMM_F32 || cfg->compute_dtype > JIMM_BF16) { set_last_error("bad compute_dtype"); return JIMM_EINVAL; }
  if (sub && cfg->ctx_len <= 0) { set_last_error("sub-module handle: ctx_len (max tokens per sample) must be positive"); return JIMM_EINVAL; }
  if (!sub && (cfg->patch <= 0 || cfg->img_size < cfg->patch || cfg->in_ch <= 0)) {
    set_last_error("unsupported patch/img/channels (%d/%d/%d)", cfg->patch, cfg->img_size, cfg->in_ch);
    return JIMM_EINVAL;
  }
  // limits of the kernels, reported at construction (not on the first forward): widths are TMA rows (16-byte multiples), LayerNorm keeps
  // a row in registers
  if (cfg->v_width % 8 != 0 || cfg->v_mlp % 8 != 0 || cfg->v_width > 2048) {
    set_last_error("vision width %d / mlp %d: must be multiples of 8 and width <= 2048", cfg->v_width, cfg->v_mlp);
    return JIMM_EINVAL;
  }
  if (dual && (cfg->t_width % 8 != 0 || cfg->t_mlp % 8 != 0 || cfg->t_width > 2048)) {
    set_last_error("text width %d / mlp %d: must be multiples of 8 and width <= 2048", cfg->t_width, cfg->t_mlp);
    return JIMM_EINVAL;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_last_error("no CUDA device available (%s): jimm_b200 has no CPU fallback", cudaGetErrorString(e));
    return JIMM_ECUDA;
  }
  if (device < 0 || device >= ndev) { set_last_error("bad device %d (have %d)", device, ndev); return JIMM_EINVAL; }
  cudaDeviceProp prop;
  JIMM_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error("device %d is sm_%d%d; jimm_b200 kernels are sm_100a only", device, prop.major, prop.minor);
    return JIMM_ECUDA;
  }
  jimm_model* m = new jimm_model();
  m->cfg = *cfg;
  m->device = device;
  m->cdt = cfg->compute_dtype == JIMM_F32 ? DT_TF32 : cfg->compute_dtype;  // fp32 mode: operands rounded to tf32 when produced
  m->adt = cfg->compute_dtype == JIMM_BF16 ? DT_BF16 : DT_F16;
  const char* env = getenv("JIMM_GEMM_IMPL");
  m->simt = env && strcmp(env, "simt") == 0;
  if ((env = getenv("JIMM_L2_ALTERNATE"))) m->l2_alternate = atoi(env) != 0;
  if ((env = getenv("JIMM_GRAPH_MAX_BATCH"))) m->graph_max_batch = atoi(env) > 0 ? atoi(env) : 0;
  if ((env = getenv("JIMM_DUAL_STREAMS"))) m->dual_streams = atoi(env) != 0;
  if ((env = getenv("JIMM_EPI_MODE_16"))) m->epi_mode_16 = atoi(env);
  if ((env = getenv("JIMM_EPI_MODE_RES"))) m->epi_mode_res = atoi(env);
  *out = m;
  return 0;
}

static int make_host_param(const int64_t* shape, int ndim, HostParam* hp) {
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    if (shape[i] < 0) { set_last_error("negative dim"); return JIMM_EINVAL; }
    hp->shape.push_back(shape[i]);
    n *= static_cast<size_t>(shape[i]);
  }
  hp->n = n;
  return 0;
}

int jimm_model_set_param(jimm_model_t* m, const char* flax_path, const void* host, const int64_t* shape, int ndim, int dtype) {
  if (!m || !flax_path || !host || (ndim > 0 && !shape)) { set_last_error("jimm_model_set_param: null argument"); return JIMM_EINVAL; }
  if (m->finalized) { set_last_error("model already finalized"); return JIMM_ESTATE; }
  if (dtype < JIMM_F32 || dtype > JIMM_BF16) { set_last_error("set_param: unsupported dtype %d", dtype); return JIMM_EINVAL; }
  HostParam hp;
  JIMM_TRY(make_host_param(shape, ndim, &hp));
  hp.dtype = dtype;  // kept in the caller's element type: the cast happens on the GPU at finalize
  const size_t bytes = hp.n * hp.esize();
  hp.data.resize((bytes + 3) / 4);
  memcpy(hp.data.data(), host, bytes);
  m->host[flax_path] = std::move(hp);
  return 0;
}

int jimm_model_set_param_ref(jimm_model_t* m, const char* flax_path, const void* host, const int64_t* shape, int ndim, int dtype, int flags) {
  if (!m || !flax_path || !host || (ndim > 0 && !shape)) { set_last_error("jimm_model_set_param_ref: null argument"); return JIMM_EINVAL; }
  if (m->finalized) { set_last_error("model already finalized"); return JIMM_ESTATE; }
  if (dtype < JIMM_F32 || dtype > JIMM_BF16) { set_last_error("set_param_ref: unsupported dtype %d", dtype); return JIMM_EINVAL; }
  HostParam hp;
  JIMM_TRY(make_host_param(shape, ndim, &hp));
  hp.dtype = dtype;
  hp.ref = host;
  hp.transposed = (flags & JIMM_PARAM_TRANSPOSED) != 0;
  if (hp.transposed && ndim < 2) { set_last_error("set_param_ref: '%s': only kernels (ndim >= 2) can be handed over transposed", flax_path); return JIMM_EINVAL; }
  m->host[flax_path] = std::move(hp);
  return 0;
}

int jimm_model_finalize(jimm_model_t* m, int max_batch) {
  if (!m) { set_last_error("null model"); return JIMM_EINVAL; }
  if (m->finalized) { set_last_error("model already finalized"); return JIMM_ESTATE; }
  if (max_batch <= 0) { set_last_error("max_batch must be positive"); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  const jimm_config_t& c = m->cfg;
  if (c.kind == JIMM_ENCODER || c.kind == JIMM_MAPHEAD) return finalize_sub(m, max_batch);
  const bool dual = c.kind == JIMM_CLIP || c.kind == JIMM_SIGLIP;
  const std::string vp = c.kind == JIMM_VIT ? "encoder." : (dual ? "vision_model." : "");
  Packer pk{m};
  int rc = 0;
  auto fail = [&](int code) { pk.done(); return code; };

  // ---- vision tower ----
  VisionTower& v = m->vis;
  v.present = true;
  v.img = c.img_size; v.P = c.patch; v.C = c.in_ch; v.D = c.v_width;
  v.n = (c.img_size / c.patch) * (c.img_size / c.patch);
  v.pooling = c.pooling; v.pre_norm = c.pre_norm; v.patch_bias = c.patch_bias; v.eps_outer = c.v_eps_outer;
  v.S = v.n + (v.pooling == JIMM_POOL_CLS ? 1 : 0);
  v.n_pad = ((v.n + 31) / 32) * 32;
  v.patch_scatter = !m->simt && m->epi_mode_res == 2;
  v.enc.c.D = c.v_width; v.enc.c.H = c.v_heads; v.enc.c.M = c.v_mlp; v.enc.c.L = c.v_layers;
  v.enc.c.act = c.v_act; v.enc.c.causal = 0; v.enc.c.eps = c.v_eps_block;
  const int D = v.D, PPC0 = c.patch * c.patch * c.in_ch;
  const int PPC = (PPC0 + 7) / 8 * 8;  // K of the patch GEMM, zero-padded (patch 14: 588 -> 592)
  v.Kp = PPC;
  if ((rc = pk.alloc_linear(&v.patch, D, PPC, c.patch_bias != 0))) return fail(rc);
  if (PPC != PPC0) JIMM_CUDA_CHECK(cudaMemsetAsync(v.patch.w, 0, static_cast<size_t>(D) * PPC * cdt_size(m), pk.stream));
  if ((rc = pk.pack_kernel(vp + "patch_embeddings.kernel", {c.patch, c.patch, c.in_ch, D}, PPC0, D, v.patch.w, 0, PPC))) return fail(rc);
  if (c.patch_bias && (rc = pk.upload_bias_at(vp + "patch_embeddings.bias", {D}, v.patch.b, D))) return fail(rc);
  if (v.pooling == JIMM_POOL_CLS && (rc = pk.upload_f32(vp + "cls_token", {1, 1, D}, &v.cls))) return fail(rc);
  if ((rc = pk.upload_f32(vp + "position_embeddings", {1, v.S, D}, &v.pos))) return fail(rc);
  if (c.pre_norm && (rc = pk.upload_ln(vp + "ln_pre", D, &v.ln_pre))) return fail(rc);
  if ((rc = pk.upload_ln(vp + "ln_post", D, &v.ln_post))) return fail(rc);
  if ((rc = pk.encoder(vp + "transformer.", &v.enc))) return fail(rc);
  if (v.pooling == JIMM_POOL_MAP && (rc = pk.map_head(vp + "MAPHead.", D, c.v_heads, &v))) return fail(rc);
  if (c.kind == JIMM_VIT && c.num_classes > 0) {
    if ((rc = pk.linear("classifier", D, c.num_classes, true, &v.head))) return fail(rc);
  } else if (c.kind == JIMM_CLIP) {
    if ((rc = pk.linear("visual_projection", D, c.t_width, false, &v.head))) return fail(rc);
  }

  // ---- text tower ----
  TextTower& t = m->txt;
  if (dual) {
    t.present = true;
    t.T = c.ctx_len; t.V = c.vocab; t.D = c.t_width; t.pool = c.t_pool; t.eps_outer = c.t_eps_outer;
    t.enc.c.D = c.t_width; t.enc.c.H = c.t_heads; t.enc.c.M = c.t_mlp; t.enc.c.L = c.t_layers;
    t.enc.c.act = c.t_act; t.enc.c.causal = c.t_causal; t.enc.c.eps = c.t_eps_block;
    if (t.D % 8 != 0 || c.t_mlp % 8 != 0) { set_last_error("text dims must be multiples of 8"); return fail(JIMM_EINVAL); }
    if ((rc = pk.upload_f32("token_embedding.embedding", {t.V, t.D}, &t.table))) return fail(rc);
    if ((rc = pk.upload_f32("positional_embedding", {t.T, t.D}, &t.pos))) return fail(rc);
    if ((rc = pk.upload_ln("ln_final", t.D, &t.ln_final))) return fail(rc);
    if ((rc = pk.encoder("text_model.", &t.enc))) return fail(rc);
    if ((rc = pk.linear("text_projection", t.D, t.D, c.t_head_bias != 0, &t.head))) return fail(rc);
    if ((rc = pk.upload_f32("logit_scale", {}, &m->logit_scale))) return fail(rc);
    if (c.kind == JIMM_SIGLIP && (rc = pk.upload_f32("logit_bias", {}, &m->logit_bias))) return fail(rc);
  }
  pk.done();
  for (auto& kv : m->host) {
    if (!kv.second.used) {
      set_last_error("finalize: unexpected parameter '%s' was set but is not part of this model", kv.first.c_str());
      return JIMM_ESTATE;
    }
  }
  m->host.clear();

  // ---- workspace ----
  Workspace& ws = m->ws;
  const size_t cs = cdt_size(m);
  const size_t Bm = max_batch;
  size_t Tv = Bm * v.S, Dmax = D, x_elems = Tv * D, big_bytes = 0;
  auto upd = [&](size_t b) { if (b > big_bytes) big_bytes = b; };
  upd(Bm * v.n_pad * PPC * cs);          // patches (rows per sample padded to a multiple of 32)
  upd(Tv * 3 * D * 2);                   // qkv (16-bit)
  upd(Tv * static_cast<size_t>(c.v_mlp) * cs);  // MLP hidden
  if (v.pooling == JIMM_POOL_MAP) upd(Tv * 2 * D * 2);
  if (dual) {  // the text tower's own buffers (it runs concurrently with the vision tower)
    const size_t Tt = Bm * t.T;
    size_t tb = Tt * 3 * t.D * 2;
    if (Tt * static_cast<size_t>(c.t_mlp) * cs > tb) tb = Tt * static_cast<size_t>(c.t_mlp) * cs;
    void* q = nullptr;
    if ((rc = m->pool.alloc(&q, Tt * t.D * sizeof(float)))) return rc; m->wt.x = static_cast<float*>(q);
    if ((rc = m->pool.alloc(&m->wt.h, Tt * t.D * cs))) return rc;
    if ((rc = m->pool.alloc(&m->wt.big, tb))) return rc;
    if ((rc = m->pool.alloc(&m->wt.pooled, Bm * t.D * cs))) return rc;
    if ((rc = m->pool.alloc(&q, Bm * sizeof(int)))) return rc; m->wt.idx = static_cast<int*>(q);
  }
  const size_t E = dual ? t.D : vision_out_dim(m);
  void* p = nullptr;
  if ((rc = m->pool.alloc(&p, x_elems * sizeof(float)))) return rc; ws.x = static_cast<float*>(p);
  if ((rc = m->pool.alloc(&ws.h, x_elems * cs))) return rc;
  if ((rc = m->pool.alloc(&ws.big, big_bytes))) return rc;
  if ((rc = m->pool.alloc(&ws.pooled, Bm * Dmax * cs))) return rc;
  if ((rc = m->pool.alloc(&p, Bm * Dmax * sizeof(float)))) return rc; ws.feat = static_cast<float*>(p);
  if ((rc = m->pool.alloc(&ws.mid2, Bm * 4 * Dmax * cs))) return rc;
  if ((rc = m->pool.alloc(&p, Bm * sizeof(int)))) return rc; ws.idx = static_cast<int*>(p);
  if ((rc = m->pool.alloc(&p, Bm * E * sizeof(float)))) return rc; ws.emb_i = static_cast<float*>(p);
  if ((rc = m->pool.alloc(&p, Bm * E * sizeof(float)))) return rc; ws.emb_t = static_cast<float*>(p);
  if ((rc = m->pool.alloc(&p, Bm * E * sizeof(float)))) return rc; ws.nrm_i = static_cast<float*>(p);
  if ((rc = m->pool.alloc(&p, Bm * E * sizeof(float)))) return rc; ws.nrm_t = static_cast<float*>(p);
  if ((rc = m->pool.alloc(&ws.in_img, Bm * v.img * v.img * v.C * sizeof(float)))) return rc;
  if (dual) { if ((rc = m->pool.alloc(&p, Bm * t.T * sizeof(int32_t)))) return rc; ws.in_ids = static_cast<int32_t*>(p); }
  ws.out_dev_elems = dual ? Bm * Bm : Bm * vision_out_dim(m);
  if (ws.out_dev_elems < Bm * E) ws.out_dev_elems = Bm * E;
  if ((rc = m->pool.alloc(&p, ws.out_dev_elems * sizeof(float)))) return rc; ws.out_dev = static_cast<float*>(p);
  if (m->graph_max_batch > 0) {
    const size_t gw = static_cast<size_t>(vision_out_dim(m)) > E ? vision_out_dim(m) : E;
    const size_t gb = static_cast<size_t>(m->graph_max_batch) < Bm ? m->graph_max_batch : Bm;
    if ((rc = m->pool.alloc(&p, gb * gw * sizeof(float)))) return rc;
    m->graph_out = static_cast<float*>(p);
    if (dual) { if ((rc = m->pool.alloc(&p, gb * gw * sizeof(float)))) return rc; m->graph_out_t = static_cast<float*>(p); }
  }

  // ---- GEMM plans (TMA descriptors bound to the fixed workspace / weight buffers) ----
  if (v.patch_scatter) {
    GemmEpilogue e;
    e.bias = v.patch.b; e.residual = ws.x; e.ldr = D; e.out = ws.x; e.out_type = DT_F32; e.ldo = D; e.mode = 2;
    e.tok_pad = v.n_pad; e.tok_off = v.pooling == JIMM_POOL_CLS ? 1 : 0; e.tok_S = v.S;
    JIMM_TRY(gemm_plan_init(&v.p_patch, m->cdt, ws.big, PPC, v.patch.w, PPC, static_cast<int>(Bm) * v.n_pad, D, PPC, e));
    if (v.p_patch.epi.mode != 2) { set_last_error("patch GEMM: token-scatter epilogue unavailable"); return JIMM_EINVAL; }
  } else {
    GemmEpilogue e;
    e.bias = v.patch.b; e.rowadd = v.pos; e.out = ws.x; e.out_type = DT_F32; e.ldo = D;
    e.rows_in = v.n; e.rows_out = v.S; e.row_off = v.pooling == JIMM_POOL_CLS ? 1 : 0; e.mode = 0;
    JIMM_TRY(gemm_plan_init(&v.p_patch, m->cdt, ws.big, PPC, v.patch.w, PPC, static_cast<int>(Bm) * v.n, D, PPC, e));
  }
  JIMM_TRY(plan_encoder(m, &v.enc, static_cast<int>(Tv), EncBufs{ws.x, ws.h, ws.big}));
  if (v.head.N > 0)
    JIMM_TRY(gemm_plan_init(&v.p_head, m->cdt, ws.pooled, D, v.head.w, D, static_cast<int>(Bm), v.head.N, D,
                            epi_plain(v.head, ACT_NONE, ws.out_dev, DT_F32, v.head.N, 0)));
  if (v.pooling == JIMM_POOL_MAP) JIMM_TRY(plan_map_head(m, static_cast<int>(Bm), static_cast<int>(Tv)));
  if (dual) {
    JIMM_TRY(plan_encoder(m, &t.enc, static_cast<int>(Bm) * t.T, EncBufs{m->wt.x, m->wt.h, m->wt.big}));
    JIMM_TRY(gemm_plan_init(&t.p_head, m->cdt, m->wt.pooled, t.D, t.head.w, t.D, static_cast<int>(Bm), t.D, t.D,
                            epi_plain(t.head, ACT_NONE, ws.out_dev, DT_F32, t.D, 0)));
  }
  JIMM_CUDA_CHECK(cudaDeviceSynchronize());
  m->max_batch = max_batch;
  m->finalized = true;
  return 0;
}

int jimm_model_destroy(jimm_model_t* m) {
  if (!m) return 0;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();
  comm_destroy(&m->comm);
  graphs_release(m);
  if (m->capture_stream) cudaStreamDestroy(m->capture_stream);
  if (m->text_stream) { cudaStreamDestroy(m->text_stream); cudaEventDestroy(m->ev_fork); cudaEventDestroy(m->ev_join); }
  for (cudaEvent_t e : m->prof_ev) cudaEventDestroy(e);
  if (m->copy_stream) {
    cudaStreamDestroy(m->copy_stream);
    for (int i = 0; i < jimm_model::kHostSlices; ++i) { cudaEventDestroy(m->ev_copied[i]); cudaEventDestroy(m->ev_consumed[i]); }
    cudaEventDestroy(m->ev_start);
  }
  if (m->ws.in_u8) cudaFree(m->ws.in_u8);
  m->pool.release();
  delete m;
  return 0;
}

int jimm_model_output_dim(const jimm_model_t* m, int* vision_out, int* text_out) {
  if (!m) { set_last_error("null model"); return JIMM_EINVAL; }
  if (vision_out) *vision_out = m->cfg.kind == JIMM_VIT && m->cfg.num_classes > 0 ? m->cfg.num_classes
                                : (m->cfg.kind == JIMM_CLIP ? m->cfg.t_width : m->cfg.v_width);
  if (text_out) *text_out = m->cfg.t_width;
  return 0;
}
int jimm_model_max_batch(const jimm_model_t* m) { return m ? m->max_batch : 0; }

// ---- forward, device buffers ----
static int vision_chunks(jimm_model* m, const void* img, int in_dtype, int B, float* out, cudaStream_t s) {
  const size_t img_elems = static_cast<size_t>(m->vis.img) * m->vis.img * m->vis.C;
  const size_t in_es = dtype_size(in_dtype);
  const int od = vision_out_dim(m);
  for (int b0 = 0; b0 < B; b0 += m->max_batch) {
    const int nb = B - b0 < m->max_batch ? B - b0 : m->max_batch;
    JIMM_TRY(exec_vision(m, static_cast<const uint8_t*>(img) + b0 * img_elems * in_es, in_dtype, nb, out + static_cast<size_t>(b0) * od, s));
  }
  return 0;
}
static int text_chunks(jimm_model* m, const int32_t* ids, int B, int T, float* out, cudaStream_t s) {
  for (int b0 = 0; b0 < B; b0 += m->max_batch) {
    const int nb = B - b0 < m->max_batch ? B - b0 : m->max_batch;
    JIMM_TRY(exec_text(m, ids + static_cast<size_t>(b0) * T, nb, T, out + static_cast<size_t>(b0) * m->txt.D, s));
  }
  return 0;
}

int jimm_vit_forward(jimm_model_t* m, const void* img, int in_dtype, int B, float* out, void* stream) {
  JIMM_TRY(check_ready(m, B));
  if (in_dtype < JIMM_F32 || in_dtype > JIMM_BF16) { set_last_error("bad image dtype %d", in_dtype); return JIMM_EINVAL; }
  if (m->cfg.kind != JIMM_VIT && m->cfg.kind != JIMM_TOWER) { set_last_error("jimm_vit_forward on a dual-tower model; use jimm_encode_image"); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  return vision_chunks(m, img, in_dtype, B, out, static_cast<cudaStream_t>(stream));
}

int jimm_encode_image(jimm_model_t* m, const void* img, int in_dtype, int B, float* out, void* stream) {
  JIMM_TRY(check_ready(m, B));
  if (in_dtype < JIMM_F32 || in_dtype > JIMM_BF16) { set_last_error("bad image dtype %d", in_dtype); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  return vision_chunks(m, img, in_dtype, B, out, static_cast<cudaStream_t>(stream));
}

int jimm_encode_text(jimm_model_t* m, const int32_t* ids, int B, int T, float* out, void* stream) {
  JIMM_TRY(check_ready(m, B));
  if (!m->txt.present) { set_last_error("model has no text tower"); return JIMM_EINVAL; }
  if (T <= 0 || T > m->txt.T) { set_last_error("sequence length %d outside (0, context_length=%d]", T, m->txt.T); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  return text_chunks(m, ids, B, T, out, static_cast<cudaStream_t>(stream));
}

int jimm_contrastive_logits(jimm_model_t* m, const float* img_e, int Bi, const float* txt_e, int Bt, float* logits, void* stream) {
  JIMM_TRY(check_ready(m, Bi));
  if (!m->txt.present) { set_last_error("model has no text tower"); return JIMM_EINVAL; }
  if (Bi > m->max_batch || Bt > m->max_batch) { set_last_error("contrastive_logits: batch (%d,%d) exceeds max_batch %d", Bi, Bt, m->max_batch); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int E = m->txt.D;
  JIMM_TRY(l2_normalize_run(img_e, m->ws.nrm_i, E, Bi, E, s));
  JIMM_TRY(l2_normalize_run(txt_e, m->ws.nrm_t, E, Bt, E, s));
  return logits_run(m->ws.nrm_i, m->ws.nrm_t, m->logit_scale, m->logit_bias, logits, Bi, Bt, E, Bt, s);
}

// Fork the text tower onto the model's side stream (ordered after everything already enqueued on `s`), returning the stream it runs
// on; join_text() makes `s` wait for it.  Profiling (per-GEMM events) and JIMM_DUAL_STREAMS=0 keep the towers on one stream.
static int fork_text(jimm_model* m, cudaStream_t s, cudaStream_t* ts) {
  *ts = s;
  if (!m->dual_streams || m->prof_on) return 0;
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) { cudaGetLastError(); return 0; }
  if (!m->text_stream) {
    JIMM_CUDA_CHECK(cudaStreamCreateWithFlags(&m->text_stream, cudaStreamNonBlocking));
    JIMM_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
    JIMM_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming));
  }
  JIMM_CUDA_CHECK(cudaEventRecord(m->ev_fork, s));
  JIMM_CUDA_CHECK(cudaStreamWaitEvent(m->text_stream, m->ev_fork, 0));
  *ts = m->text_stream;
  return 0;
}
static int join_text(jimm_model* m, cudaStream_t s, cudaStream_t ts) {
  if (ts == s) return 0;
  JIMM_CUDA_CHECK(cudaEventRecord(m->ev_join, ts));
  JIMM_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_join, 0));
  return 0;
}

// encode_image + encode_text of one call, the two towers running concurrently (device inputs); img_e fp32 [Bi,E], txt_e fp32 [Bt,E].
int jimm_dual_encode(jimm_model_t* m, const void* img, int in_dtype, int Bi, const int32_t* ids, int Bt, int T, float* img_e, float* txt_e,
                     void* stream) {
  JIMM_TRY(check_ready(m, Bi));
  if (!m->txt.present) { set_last_error("model has no text tower"); return JIMM_EINVAL; }
  if (in_dtype < JIMM_F32 || in_dtype > JIMM_BF16) { set_last_error("bad image dtype %d", in_dtype); return JIMM_EINVAL; }
  if (T <= 0 || T > m->txt.T) { set_last_error("sequence length %d outside (0, context_length=%d]", T, m->txt.T); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  cudaStream_t s = static_cast<cudaStream_t>(stream), ts = s;
  JIMM_TRY(fork_text(m, s, &ts));
  JIMM_TRY(text_chunks(m, ids, Bt, T, txt_e, ts));
  JIMM_TRY(vision_chunks(m, img, in_dtype, Bi, img_e, s));
  return join_text(m, s, ts);
}

int jimm_dual_forward(jimm_model_t* m, const void* img, int in_dtype, int Bi, const int32_t* ids, int Bt, int T, float* logits,
                      void* stream) {
  JIMM_TRY(check_ready(m, Bi));
  if (Bi > m->max_batch || Bt > m->max_batch) { set_last_error("dual_forward: batch (%d,%d) exceeds max_batch %d", Bi, Bt, m->max_batch); return JIMM_EINVAL; }
  JIMM_TRY(jimm_dual_encode(m, img, in_dtype, Bi, ids, Bt, T, m->ws.emb_i, m->ws.emb_t, stream));
  return jimm_contrastive_logits(m, m->ws.emb_i, Bi, m->ws.emb_t, Bt, logits, stream);
}

// ---- forward of a bare sub-module (device buffers) ----
static int check_sub(jimm_model_t* m, int kind, int B, int S, const void* x, const void* out) {
  JIMM_TRY(check_ready(m, B));
  if (m->cfg.kind != kind) { set_last_error("this handle is not a %s", kind == JIMM_ENCODER ? "Transformer (JIMM_ENCODER)" : "MAP head (JIMM_MAPHEAD)"); return JIMM_EINVAL; }
  if (S <= 0 || S > m->vis.S) { set_last_error("sequence length %d outside (0, %d]", S, m->vis.S); return JIMM_EINVAL; }
  if (!x || !out) { set_last_error("null buffer"); return JIMM_EINVAL; }
  return set_device(m);
}

int jimm_encoder_forward(jimm_model_t* m, const float* x, int B, int S, float* out, void* stream) {
  JIMM_TRY(check_sub(m, JIMM_ENCODER, B, S, x, out));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t row = static_cast<size_t>(S) * m->vis.D;
  for (int b0 = 0; b0 < B; b0 += m->max_batch) {
    const int nb = B - b0 < m->max_batch ? B - b0 : m->max_batch;
    JIMM_CUDA_CHECK(cudaMemcpyAsync(m->ws.x, x + b0 * row, nb * row * sizeof(float), cudaMemcpyDeviceToDevice, s));
    JIMM_TRY(run_encoder(m, &m->vis.enc, nb, S, s, EncBufs{m->ws.x, m->ws.h, m->ws.big}));
    JIMM_CUDA_CHECK(cudaMemcpyAsync(out + b0 * row, m->ws.x, nb * row * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  return 0;
}

int jimm_map_head_forward(jimm_model_t* m, const float* x, int B, int S, float* out, void* stream) {
  JIMM_TRY(check_sub(m, JIMM_MAPHEAD, B, S, x, out));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t row = static_cast<size_t>(S) * m->vis.D;
  for (int b0 = 0; b0 < B; b0 += m->max_batch) {
    const int nb = B - b0 < m->max_batch ? B - b0 : m->max_batch;
    JIMM_TRY(cast_run(x + b0 * row, m->ws.h, m->cdt, nb * row, s));  // the head's inputs are GEMM operands: compute dtype
    JIMM_TRY(run_map_head(m, nb, S, out + static_cast<size_t>(b0) * m->vis.D, s));
  }
  return 0;
}

// ---- forward, host buffers ----
static int ensure_copy_stream(jimm_model* m) {
  if (m->copy_stream) return 0;
  JIMM_CUDA_CHECK(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < jimm_model::kHostSlices; ++i) {
    JIMM_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_copied[i], cudaEventDisableTiming));
    JIMM_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_consumed[i], cudaEventDisableTiming));
  }
  JIMM_CUDA_CHECK(cudaEventCreateWithFlags(&m->ev_start, cudaEventDisableTiming));
  return 0;
}

// Slice schedule of one super-chunk of nb images on the host path.  Two slices: a head slice whose H2D copy is the only exposed
// one, chosen between nb/head_div and nb/3 so that BOTH slices quantise well into waves of 256-row pair tiles (a badly chosen
// split costs an extra wave in every GEMM: 64 images take 3.3 ms on ViT-B/16 where 62 take 2.8 ms).  JIMM_HOST_SLICES (comma
// separated sizes) overrides it for experiments.
static void host_slices(const jimm_model* m, int nb, int* sizes, size_t bytes_per_image = 0) {
  for (int i = 0; i < jimm_model::kHostSlices; ++i) sizes[i] = 0;
  sizes[0] = nb;
  if (const char* env = getenv("JIMM_HOST_SLICES")) {
    int k = 0, acc = 0;
    for (const char* q = env; *q && k < jimm_model::kHostSlices - 1;) {
      const int v = atoi(q);
      if (v <= 0 || acc + v >= nb) break;
      sizes[k++] = v;
      acc += v;
      while (*q && *q != ',') ++q;
      if (*q == ',') ++q;
    }
    sizes[k] = nb - acc;
    return;
  }
  if (nb < 128) return;
  // Slicing hides all but the first slice's copy but costs GEMM waves and launches (~0.45 ms on ViT-B/16 at 256 images): only worth it
  // when the whole copy is long.  Raw uint8 frames (38 MB for 256 x 224 x 224 x 3, 0.7 ms over PCIe) go in one piece: measured 10.82 ms
  // unsliced against 11.28 ms sliced, device-resident 10.35 ms (scripts/gpu_e2e_probe.py).
  if (bytes_per_image && static_cast<size_t>(nb) * bytes_per_image < (static_cast<size_t>(64) << 20)) return;
  static int head_div = -1;
  if (head_div < 0) { const char* env = getenv("JIMM_HOST_HEAD_DIV"); head_div = (env && atoi(env) > 0) ? atoi(env) : 4; }
  const int S = m->vis.S, D = m->vis.D, Mm = m->vis.enc.c.M;
  const int pairs = device_sm_count() / 2;
  auto cost = [&](int n) {
    const long mt = (static_cast<long>(n) * S + 255) / 256;
    auto rounds = [&](int N) { return (mt * ((N + 255) / 256) + pairs - 1) / pairs; };
    return static_cast<double>(D) * rounds(3 * D) + static_cast<double>(D) * rounds(D) + static_cast<double>(D) * rounds(Mm) +
           static_cast<double>(Mm) * rounds(D);
  };
  int best = nb / head_div;
  double best_cost = 1e30;
  for (int c0 = nb / head_div; c0 <= nb / 3; ++c0) {
    const double cst = cost(c0) + cost(nb - c0) + 1e-3 * c0 * D;  // tie-break towards the smaller exposed copy
    if (cst < best_cost) { best_cost = cst; best = c0; }
  }
  sizes[0] = best;
  sizes[1] = nb - best;
}

// Host-buffer vision forward.  pre == nullptr: img_host holds NHWC images of in_dtype at the model's resolution.  pre != nullptr:
// img_host holds raw uint8 RGB frames [B,Hin,Win,3]; each slice is copied as bytes (4x fewer than fp32 pixels), run through the image
// front-end on the compute stream (resize / crop / rescale / normalise into the tower's operand dtype) and then through the tower.
static int vit_forward_host_impl(jimm_model_t* m, const void* img_host, int in_dtype, int B, float* out_host, cudaStream_t s,
                                 jimm_preproc_t* pre, int Hin, int Win) {
  JIMM_TRY(ensure_copy_stream(m));
  const size_t img_elems = static_cast<size_t>(m->vis.img) * m->vis.img * m->vis.C;
  const size_t src_bytes = pre ? static_cast<size_t>(Hin) * Win * 3 : img_elems * dtype_size(in_dtype);  // per image, on the host
  const int tower_dtype = pre ? (m->cdt == DT_TF32 ? JIMM_F32 : m->cdt) : in_dtype;
  const int od = vision_out_dim(m);
  const int kind = pre ? 1 : 0;
  if (pre) {
    const size_t need = static_cast<size_t>(m->max_batch) * src_bytes;
    if (need > m->ws.in_u8_bytes) {  // first call (or larger frames): grow the byte staging buffer
      JIMM_CUDA_CHECK(cudaDeviceSynchronize());
      if (m->ws.in_u8) cudaFree(m->ws.in_u8);
      m->ws.in_u8 = nullptr; m->ws.in_u8_bytes = 0;
      JIMM_CUDA_CHECK(cudaMalloc(&m->ws.in_u8, need));
      m->ws.in_u8_bytes = need;
      m->host_chain = false;
    }
  }
  // Sliced pipeline per super-chunk of <= max_batch images: slice i+1 is copied on the side stream while slice i is in the
  // tower, and the next super-chunk's first copy overlaps this one's last forward.  The slices partition the staging buffer
  // (max_batch images), one event pair each; one D2H of the super-chunk's result at its end.
  for (int b0 = 0; b0 < B; b0 += m->max_batch) {
    const int nb = B - b0 < m->max_batch ? B - b0 : m->max_batch;
    int sizes[jimm_model::kHostSlices];
    host_slices(m, nb, sizes, src_bytes);
    bool same_layout = m->host_chain && m->host_chain_stream == s && m->host_chain_kind == kind;
    for (int i = 0; i < jimm_model::kHostSlices; ++i) same_layout = same_layout && sizes[i] == m->host_chain_sizes[i];
    if (!same_layout) {
      // earlier work on the caller's stream may still read the staging buffer in another layout: order the copies after all of it
      JIMM_CUDA_CHECK(cudaEventRecord(m->ev_start, s));
      JIMM_CUDA_CHECK(cudaStreamWaitEvent(m->copy_stream, m->ev_start, 0));
      for (int i = 0; i < jimm_model::kHostSlices; ++i) {
        // ... and after the slices of an earlier host call, which may have run on another stream
        if (m->slot_recorded[i]) JIMM_CUDA_CHECK(cudaStreamWaitEvent(m->copy_stream, m->ev_consumed[i], 0));
        m->slot_recorded[i] = false;
        m->host_chain_sizes[i] = sizes[i];
      }
      m->host_chain = true;
      m->host_chain_stream = s;
      m->host_chain_kind = kind;
    }
    int off = 0;
    for (int slot = 0; slot < jimm_model::kHostSlices; ++slot) {
      const int n = sizes[slot];
      if (n <= 0) continue;
      uint8_t* img_dst = static_cast<uint8_t*>(m->ws.in_img) + static_cast<size_t>(off) * img_elems * sizeof(float);
      uint8_t* copy_dst = pre ? m->ws.in_u8 + static_cast<size_t>(off) * src_bytes : img_dst;
      float* out_d = m->ws.out_dev + static_cast<size_t>(off) * od;
      if (m->slot_recorded[slot]) JIMM_CUDA_CHECK(cudaStreamWaitEvent(m->copy_stream, m->ev_consumed[slot], 0));
      JIMM_CUDA_CHECK(cudaMemcpyAsync(copy_dst, static_cast<const uint8_t*>(img_host) + static_cast<size_t>(b0 + off) * src_bytes, n * src_bytes,
                                      cudaMemcpyHostToDevice, m->copy_stream));
      JIMM_CUDA_CHECK(cudaEventRecord(m->ev_copied[slot], m->copy_stream));
      JIMM_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_copied[slot], 0));
      if (pre) {
        if (int rc = jimm_preproc_run(pre, copy_dst, n, Hin, Win, img_dst, tower_dtype, s)) return rc;
        // the byte staging slice is free as soon as the front-end has read it: the next call's copy runs under THIS call's tower
        // (the front-end's output slice is only rewritten by the next call's front-end, which is stream-ordered after this tower)
        JIMM_CUDA_CHECK(cudaEventRecord(m->ev_consumed[slot], s));
      }
      JIMM_TRY(exec_vision(m, img_dst, tower_dtype, n, out_d, s));
      if (!pre) JIMM_CUDA_CHECK(cudaEventRecord(m->ev_consumed[slot], s));
      m->slot_recorded[slot] = true;
      off += n;
    }
    JIMM_CUDA_CHECK(cudaMemcpyAsync(out_host + static_cast<size_t>(b0) * od, m->ws.out_dev, static_cast<size_t>(nb) * od * sizeof(float),
                                    cudaMemcpyDeviceToHost, s));
  }
  return 0;
}

int jimm_vit_forward_host(jimm_model_t* m, const void* img_host, int in_dtype, int B, float* out_host, void* stream) {
  JIMM_TRY(check_ready(m, B));
  if (in_dtype < JIMM_F32 || in_dtype > JIMM_BF16) { set_last_error("bad image dtype %d", in_dtype); return JIMM_EINVAL; }
  if (m->cfg.kind != JIMM_VIT && m->cfg.kind != JIMM_TOWER) { set_last_error("jimm_vit_forward_host on a dual-tower model"); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  return vit_forward_host_impl(m, img_host, in_dtype, B, out_host, static_cast<cudaStream_t>(stream), nullptr, 0, 0);
}

int jimm_vit_forward_host_u8(jimm_model_t* m, jimm_preproc_t* pre, const uint8_t* img_host, int B, int H, int W, float* out_host, void* stream) {
  JIMM_TRY(check_ready(m, B));
  if (!pre || !img_host || !out_host) { set_last_error("jimm_vit_forward_host_u8: null argument"); return JIMM_EINVAL; }
  if (m->cfg.kind != JIMM_VIT && m->cfg.kind != JIMM_TOWER) { set_last_error("jimm_vit_forward_host_u8 on a dual-tower model"); return JIMM_EINVAL; }
  if (m->vis.C != 3) { set_last_error("the image front-end produces 3-channel images; the model takes %d", m->vis.C); return JIMM_EINVAL; }
  int oh = 0, ow = 0;
  if (int rc = jimm_preproc_output_size(pre, H, W, &oh, &ow)) return rc;
  if (oh != m->vis.img || ow != m->vis.img) {
    set_last_error("front-end output %dx%d for %dx%d frames does not match the model's %dx%d input", oh, ow, H, W, m->vis.img, m->vis.img);
    return JIMM_EINVAL;
  }
  JIMM_TRY(set_device(m));
  return vit_forward_host_impl(m, img_host, JIMM_F32, B, out_host, static_cast<cudaStream_t>(stream), pre, H, W);
}

int jimm_dual_forward_host(jimm_model_t* m, const void* img_host, int in_dtype, int Bi, const int32_t* ids_host, int Bt, int T,
                           float* logits_host, void* stream) {
  JIMM_TRY(check_ready(m, Bi));
  if (!m->txt.present) { set_last_error("model has no text tower"); return JIMM_EINVAL; }
  if (Bi > m->max_batch || Bt > m->max_batch) { set_last_error("dual_forward_host: batch (%d,%d) exceeds max_batch %d", Bi, Bt, m->max_batch); return JIMM_EINVAL; }
  if (in_dtype < JIMM_F32 || in_dtype > JIMM_BF16) { set_last_error("bad image dtype %d", in_dtype); return JIMM_EINVAL; }
  if (T <= 0 || T > m->txt.T) { set_last_error("sequence length %d outside (0, context_length=%d]", T, m->txt.T); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  JIMM_TRY(ensure_copy_stream(m));
  const size_t img_elems = static_cast<size_t>(m->vis.img) * m->vis.img * m->vis.C;
  const size_t img_bytes = img_elems * dtype_size(in_dtype);
  const int E = m->txt.D;
  // The (large) image copy goes to the side stream while the caller's stream takes the token ids and runs the text tower,
  // which hides it (CLIP-B/32 B=256: copy 2.8 ms, text tower 2.8 ms; measured 5.94 ms end to end against 5.85 ms device
  // resident).  Slicing the images as well only costs GEMM waves here (6.3 ms with 64+192), so it is one slice unless
  // JIMM_HOST_SLICES asks otherwise.
  // The token ids go first: H2D copies share one copy engine, so ids submitted after the images would queue behind them and
  // hold the text tower back.
  m->host_chain = false;
  JIMM_CUDA_CHECK(cudaEventRecord(m->ev_start, s));
  JIMM_CUDA_CHECK(cudaStreamWaitEvent(m->copy_stream, m->ev_start, 0));
  cudaStream_t ts = s;
  JIMM_TRY(fork_text(m, s, &ts));  // ids copy + text tower on the side stream, concurrently with the image copy and the vision tower
  JIMM_CUDA_CHECK(cudaMemcpyAsync(m->ws.in_ids, ids_host, static_cast<size_t>(Bt) * T * sizeof(int32_t), cudaMemcpyHostToDevice, ts));
  int sizes[jimm_model::kHostSlices] = {Bi, 0, 0, 0};
  if (getenv("JIMM_HOST_SLICES")) host_slices(m, Bi, sizes);
  int off = 0;
  for (int slot = 0; slot < jimm_model::kHostSlices; ++slot) {
    const int n = sizes[slot];
    if (n <= 0) continue;
    uint8_t* dst = static_cast<uint8_t*>(m->ws.in_img) + static_cast<size_t>(off) * img_elems * sizeof(float);
    JIMM_CUDA_CHECK(cudaMemcpyAsync(dst, static_cast<const uint8_t*>(img_host) + static_cast<size_t>(off) * img_bytes, n * img_bytes,
                                    cudaMemcpyHostToDevice, m->copy_stream));
    JIMM_CUDA_CHECK(cudaEventRecord(m->ev_copied[slot], m->copy_stream));
    off += n;
  }
  JIMM_TRY(exec_text(m, m->ws.in_ids, Bt, T, m->ws.emb_t, ts));
  off = 0;
  for (int slot = 0; slot < jimm_model::kHostSlices; ++slot) {
    const int n = sizes[slot];
    if (n <= 0) continue;
    const uint8_t* src = static_cast<const uint8_t*>(m->ws.in_img) + static_cast<size_t>(off) * img_elems * sizeof(float);
    JIMM_CUDA_CHECK(cudaStreamWaitEvent(s, m->ev_copied[slot], 0));
    JIMM_TRY(exec_vision(m, src, in_dtype, n, m->ws.emb_i + static_cast<size_t>(off) * E, s));
    off += n;
  }
  JIMM_TRY(join_text(m, s, ts));
  JIMM_TRY(jimm_contrastive_logits(m, m->ws.emb_i, Bi, m->ws.emb_t, Bt, m->ws.out_dev, stream));
  JIMM_CUDA_CHECK(cudaMemcpyAsync(logits_host, m->ws.out_dev, static_cast<size_t>(Bi) * Bt * sizeof(float), cudaMemcpyDeviceToHost, s));
  return 0;
}

// ---- multi-GPU contrastive head ----
int jimm_comm_init(jimm_model_t* m, int rank, int world, int max_rows_per_rank, unsigned char* handle_out) {
  JIMM_TRY(check_ready(m, 0));
  if (!m->txt.present) { set_last_error("model has no text tower"); return JIMM_EINVAL; }
  JIMM_TRY(set_device(m));
  return comm_init(&m->comm, rank, world, max_rows_per_rank, m->txt.D, handle_out);
}
int jimm_comm_connect(jimm_model_t* m, const unsigned char* handles) {
  JIMM_TRY(check_ready(m, 0));
  JIMM_TRY(set_device(m));
  return comm_connect(&m->comm, handles);
}
int jimm_comm_contrastive_logits(jimm_model_t* m, const float* img_e, const float* txt_e, int B_local, float* logits_local, void* stream) {
  JIMM_TRY(check_ready(m, B_local));
  JIMM_TRY(set_device(m));
  return comm_contrastive_logits(&m->comm, img_e, txt_e, B_local, m->logit_scale, m->logit_bias, logits_local, static_cast<cudaStream_t>(stream));
}
int jimm_comm_status(jimm_model_t* m) {
  if (!m) { set_last_error("null model"); return JIMM_EINVAL; }
  return comm_status(&m->comm);
}
int jimm_comm_gathered(jimm_model_t* m, float** gathered, int* row_stride) {
  if (!m || !m->comm.ready) { set_last_error("comm not initialised"); return JIMM_ESTATE; }
  if (gathered) *gathered = m->comm.local_buf;
  if (row_stride) *row_stride = 2 * m->comm.E;
  return 0;
}

int jimm_profile_begin(jimm_model_t* m) {
  JIMM_TRY(check_ready(m, 0));
  m->prof_on = true;
  m->prof_used = 0;
  m->prof_flops = 0.0;
  m->prof_launches = 0;
  return 0;
}
int jimm_profile_end(jimm_model_t* m, double* gemm_ms, double* gemm_flops, long long* gemm_launches) {
  JIMM_TRY(check_ready(m, 0));
  JIMM_TRY(set_device(m));
  m->prof_on = false;
  JIMM_CUDA_CHECK(cudaDeviceSynchronize());
  double ms = 0.0;
  for (size_t i = 0; i + 1 < m->prof_used; i += 2) {
    float t = 0.f;
    JIMM_CUDA_CHECK(cudaEventElapsedTime(&t, m->prof_ev[i], m->prof_ev[i + 1]));
    ms += t;
  }
  if (gemm_ms) *gemm_ms = ms;
  if (gemm_flops) *gemm_flops = m->prof_flops;
  if (gemm_launches) *gemm_launches = m->prof_launches;
  m->prof_used = 0;
  return 0;
}

// ---- per-kernel entry points ----
int jimm_k_gemm(int impl, int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias, int act,
                const float* rowadd, const float* residual, int ldr, void* out, int out_type, int ldo, int rows_in, int rows_out,
                int row_off, int epi_mode, void* stream) {
  if (impl == 1) {
    GemmEpilogue e;
    e.bias = bias; e.act = act; e.rowadd = rowadd; e.residual = residual; e.ldr = ldr; e.out = out; e.out_type = out_type; e.ldo = ldo;
    e.rows_in = rows_in; e.rows_out = rows_out; e.row_off = row_off; e.mode = epi_mode;
    return gemm_simt_run(dtype, A, lda, B, ldb, M, N, K, e, static_cast<cudaStream_t>(stream));
  }
  return jimm_k_gemm_ex(dtype, A, lda, B, ldb, M, N, K, bias, act, rowadd, residual, ldr, out, out_type, ldo, rows_in, rows_out, row_off, 0, 0, 0, 0, 0,
                        epi_mode, stream);
}
int jimm_k_gemm_ex(int dtype, const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias, int act,
                   const float* rowadd, const float* residual, int ldr, void* out, int out_type, int ldo, int rows_in, int rows_out,
                   int row_off, int tok_pad, int tok_off, int tok_S, int run_M, int reverse, int epi_mode, void* stream) {
  if (run_M < 0 || run_M > M) { set_last_error("jimm_k_gemm_ex: run_M %d outside [0, M = %d]", run_M, M); return JIMM_EINVAL; }
  if (tok_pad < 0 || (tok_pad > 0 && (residual != out || ldr != ldo || out_type != JIMM_F32 || epi_mode != 2 || rowadd || rows_in != 0 ||
                                      tok_off < 0 || tok_S <= 0))) {
    set_last_error("jimm_k_gemm_ex: token scatter needs residual == out, ldr == ldo, fp32 output, epi_mode 2, no row remap, tok_S > 0");
    return JIMM_EINVAL;
  }
  GemmEpilogue e;
  e.bias = bias; e.act = act; e.rowadd = rowadd; e.residual = residual; e.ldr = ldr; e.out = out; e.out_type = out_type; e.ldo = ldo;
  e.rows_in = rows_in; e.rows_out = rows_out; e.row_off = row_off; e.mode = epi_mode;
  e.tok_pad = tok_pad; e.tok_off = tok_off; e.tok_S = tok_S;
  GemmPlan p;
  JIMM_TRY(gemm_plan_init(&p, dtype, A, lda, B, ldb, M, N, K, e));
  if (tok_pad > 0 && p.epi.mode != 2) { set_last_error("jimm_k_gemm_ex: token-scatter epilogue unavailable (alignment)"); return JIMM_EINVAL; }
  return gemm_plan_run(&p, run_M > 0 ? run_M : M, static_cast<cudaStream_t>(stream), reverse != 0);
}
int jimm_k_layernorm(const float* x, int ldx, int group, int row_off, const int32_t* row_index, const float* scale, const float* bias,
                     float eps, void* out, int out_type, int ldy, int rows, int D, void* stream) {
  return jimm_k_layernorm_ex(x, ldx, group, row_off, row_index, scale, bias, eps, out, out_type, ldy, rows, D, 0, stream);
}
int jimm_k_layernorm_ex(const float* x, int ldx, int group, int row_off, const int32_t* row_index, const float* scale, const float* bias,
                        float eps, void* out, int out_type, int ldy, int rows, int D, int reverse, void* stream) {
  return layernorm_run(x, ldx, group, row_off, row_index, scale, bias, eps, out, out_type, ldy, rows, D, static_cast<cudaStream_t>(stream), reverse != 0);
}
int jimm_k_attention(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, void* stream) {
  return jimm_k_attention_ex(qkv, io_type, out, out_type, B, S, H, causal, 0, stream);
}
int jimm_k_attention_ex(const void* qkv, int io_type, void* out, int out_type, int B, int S, int H, int causal, int reverse, void* stream) {
  return attention_run(qkv, io_type, out, out_type, B, S, H, causal, static_cast<cudaStream_t>(stream), reverse != 0);
}
int jimm_k_map_attention(const float* q, const void* kv, int io_type, void* out, int out_type, int B, int S, int H, void* stream) {
  return map_attention_run(q, kv, io_type, out, out_type, B, S, H, static_cast<cudaStream_t>(stream));
}
int jimm_k_patchify(const void* img, int in_type, int B, int H, int W, int C, int P, void* out, int out_type, void* stream) {
  return patchify_run(img, in_type, B, H, W, C, P, out, out_type, static_cast<cudaStream_t>(stream));
}
int jimm_k_activation(const float* x, float* y, long long n, int act, void* stream) {
  if (n < 0 || (n > 0 && (!x || !y))) { set_last_error("jimm_k_activation: bad arguments"); return JIMM_EINVAL; }
  return activation_run(x, y, static_cast<size_t>(n), act, static_cast<cudaStream_t>(stream));
}
int jimm_k_embed(const int32_t* ids, const float* table, const float* pos, float* x, int B, int T, int D, int vocab, void* stream) {
  return embed_run(ids, table, pos, x, B, T, D, vocab, static_cast<cudaStream_t>(stream));
}
int jimm_k_l2_normalize(const float* x, float* out, int ldo, int B, int E, void* stream) {
  return l2_normalize_run(x, out, ldo, B, E, static_cast<cudaStream_t>(stream));
}
int jimm_k_logits(const float* img, const float* txt, const float* logit_scale, const float* logit_bias, float* logits, int Bi, int Bt,
                  int E, int ldl, void* stream) {
  return logits_run(img, txt, logit_scale, logit_bias, logits, Bi, Bt, E, ldl, static_cast<cudaStream_t>(stream));
}

}  // extern "C"

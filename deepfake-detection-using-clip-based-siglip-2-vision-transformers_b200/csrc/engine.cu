// dfd_engine: owns the repacked SigLIP vision-tower weights and the activation workspace of one
// (device, model config) and strings the kernels into the backbone forward:
//
//   pixels ─patchify→ patches ─GEMM(+bias+pos)→ x
//   L × { LN → GEMM qkv → attention → GEMM out(+residual) → LN → GEMM fc1(+gelu_tanh) → GEMM fc2(+residual) }
//   post-LN → [last_hidden] → GEMM kv → MAP attention → GEMM out → LN → GEMM fc1(+gelu) → GEMM fc2(+residual) → pooled
//
// = HF SiglipVisionModel.forward (HF:modeling_siglip.py:175-186,340-362,586-654), the model the reference
// instantiates at Siglip2sidafrozen.py:753 and calls at :787; identical math to open_clip's
// encode_image (inference_ai_human_images.py:148).  Everything is enqueue-only on the caller's stream.
#include "dfd_common.cuh"

#include <atomic>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace dfd {

extern std::atomic<int64_t> g_launches;

namespace {

// dst[r, c] (dst_dtype, leading dim dst_ld) = src[r, c] (src_dtype, dense [rows, cols]); columns
// cols..dst_cols-1 of each destination row are zero filled (K padding of the patch-embedding weight).
__global__ void convert_rows_kernel(const void* __restrict__ src, int src_bf16, int64_t rows, int64_t cols,
                                    void* __restrict__ dst, int dst_bf16, int64_t dst_ld, int64_t dst_cols) {
  const int64_t total = rows * dst_cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / dst_cols, c = i % dst_cols;
    float v = 0.f;
    if (c < cols) {
      v = src_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[r * cols + c])
                   : reinterpret_cast<const float*>(src)[r * cols + c];
    }
    if (dst_bf16) reinterpret_cast<__nv_bfloat16*>(dst)[r * dst_ld + c] = __float2bfloat16(v);
    else reinterpret_cast<float*>(dst)[r * dst_ld + c] = v;
  }
}

// q[j] = bq[j] + sum_k probe[k] * Wq[j, k]   (one warp per output)
__global__ void probe_query_kernel(const float* __restrict__ probe, const __nv_bfloat16* __restrict__ Wq,
                                   const float* __restrict__ bq, float* __restrict__ q, int D) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= D) return;
  float acc = 0.f;
  for (int k = lane; k < D; k += 32) acc += probe[k] * __bfloat162float(Wq[(int64_t)j * D + k]);
  acc = warp_sum(acc);
  if (lane == 0) q[j] = acc + bq[j];
}

// LayerNorm folded through a Linear (one warp per output row n), in place:
//   W'[n,k] = bf16(W[n,k]·gamma[k]);  colsum[n] = sum_k W'[n,k];  bias[n] += sum_k W[n,k]·beta[k]
// so that  Linear(LN(x)) = rstd·(x·W'^T − mean·colsum) + bias'   (the GEMM epilogue applies the right-hand side)
__global__ void fold_ln_kernel(__nv_bfloat16* __restrict__ W, float* __restrict__ bias, float* __restrict__ colsum,
                               const float* __restrict__ gamma, const float* __restrict__ beta, int N, int K) {
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float cs = 0.f, bs = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = __bfloat162float(W[(int64_t)n * K + k]);
    const __nv_bfloat16 wf = __float2bfloat16(w * gamma[k]);
    W[(int64_t)n * K + k] = wf;
    cs += __bfloat162float(wf);
    bs += w * beta[k];
  }
  cs = warp_sum(cs);
  bs = warp_sum(bs);
  if (lane == 0) {
    colsum[n] = cs;
    bias[n] += bs;
  }
}

struct Layer {
  float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
  __nv_bfloat16 *w_qkv, *w_o, *w_fc1, *w_fc2;
  float *b_qkv, *b_o, *b_fc1, *b_fc2;
  float *cs_qkv, *cs_fc1;  // column sums of the LN-folded weights (fuse_ln)
};

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

}  // namespace
}  // namespace dfd

struct dfd_engine {
  dfd_config cfg;
  int device, max_batch;
  int S, P, G, N, D, I, L, H, hd, Kpe, Kpad;
  bool finalized;
  // weights
  uint8_t* wslab;
  int64_t wbytes;
  __nv_bfloat16* w_pe;
  float *b_pe, *pos;
  std::vector<dfd::Layer> layers;
  float *post_g, *post_b;
  float *probe, *q_probe;
  __nv_bfloat16 *w_in, *w_mo, *w_mfc1, *w_mfc2;
  float *b_in, *b_mo, *hln_g, *hln_b, *b_mfc1, *b_mfc2;
  std::vector<std::string> missing;  // names still to be set
  // workspace
  uint8_t* aslab;
  int64_t abytes;
  __nv_bfloat16 *patches, *x, *h, *qkv, *att, *mlp, *ao, *r, *h2, *m2;
  __nv_bfloat16* x_lo;       // low half of the two-bf16 residual stream (precise mode), allocated on first use
  bool precise;
  float *stats_a, *stats_b;  // per-row (sum, sum of squares) of the residual stream (fuse_ln)
  bool folded;
  void* hidden_tap;          // optional [L+1, B, N, D] bf16 destination of the per-layer hidden states
  float* attn_tap;           // optional [L, B, (H,) N, N] fp32 destination of the per-layer attention probabilities
  int attn_per_head;         // 1: [L, B, H, N, N]; 0: head mean [L, B, N, N]
  float* map_tap;            // optional [B, H, N] fp32 destination of the MAP probe attention
  void* staging;
  int64_t staging_bytes;
  // optional per-launch CUDA-event timing of the forward (bench.py roofline): family 0 GEMM, 1 attention,
  // 2 LayerNorm, 3 patchify, 4 MAP attention
  bool prof_on;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<int> prof_fam;
  int prof_n;
  int prof_cap;  // launches the current profiling session may record
  // CUDA graphs of the forward, one per call signature (see dfd_engine_set_graphs)
  struct GraphKey {
    const void *pixels, *pooled, *last_hidden;
    int fmt, B, Hin, Win, resize_mode;
    bool operator==(const GraphKey& o) const {
      return pixels == o.pixels && pooled == o.pooled && last_hidden == o.last_hidden && fmt == o.fmt && B == o.B &&
             Hin == o.Hin && Win == o.Win && resize_mode == o.resize_mode;
    }
  };
  struct GraphEntry {
    GraphKey key;
    cudaGraphExec_t exec;  // nullptr: the signature has been seen (and run eagerly) once
    int64_t launches;      // kernel launches one replay stands for
    uint64_t last_use;
  };
  bool graphs_on;
  std::vector<GraphEntry> graphs;
  uint64_t graph_clock;
  cudaStream_t capture_stream;
  int64_t graph_replays;
};

namespace dfd {
namespace {

struct Carver {
  uint8_t* base;
  int64_t off;
  template <typename T>
  T* take(int64_t n) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += align_up(n * (int64_t)sizeof(T), 256);
    return p;
  }
};

void carve_weights(dfd_engine* e, uint8_t* base, int64_t* total) {
  Carver c{base, 0};
  const int64_t D = e->D, I = e->I, N = e->N;
  e->w_pe = c.take<__nv_bfloat16>(D * e->Kpad);
  e->b_pe = c.take<float>(D);
  e->pos = c.take<float>(N * D);
  e->layers.resize(e->L);
  for (auto& l : e->layers) {
    l.ln1_g = c.take<float>(D); l.ln1_b = c.take<float>(D);
    l.ln2_g = c.take<float>(D); l.ln2_b = c.take<float>(D);
    l.w_qkv = c.take<__nv_bfloat16>(3 * D * D); l.b_qkv = c.take<float>(3 * D);
    l.w_o = c.take<__nv_bfloat16>(D * D); l.b_o = c.take<float>(D);
    l.w_fc1 = c.take<__nv_bfloat16>(I * D); l.b_fc1 = c.take<float>(I);
    l.w_fc2 = c.take<__nv_bfloat16>(D * I); l.b_fc2 = c.take<float>(D);
    l.cs_qkv = c.take<float>(3 * D); l.cs_fc1 = c.take<float>(I);
  }
  e->post_g = c.take<float>(D); e->post_b = c.take<float>(D);
  e->probe = c.take<float>(D); e->q_probe = c.take<float>(D);
  e->w_in = c.take<__nv_bfloat16>(3 * D * D); e->b_in = c.take<float>(3 * D);
  e->w_mo = c.take<__nv_bfloat16>(D * D); e->b_mo = c.take<float>(D);
  e->hln_g = c.take<float>(D); e->hln_b = c.take<float>(D);
  e->w_mfc1 = c.take<__nv_bfloat16>(I * D); e->b_mfc1 = c.take<float>(I);
  e->w_mfc2 = c.take<__nv_bfloat16>(D * I); e->b_mfc2 = c.take<float>(D);
  *total = c.off;
}

void carve_acts(dfd_engine* e, uint8_t* base, int64_t* total) {
  Carver c{base, 0};
  const int64_t B = e->max_batch, M = B * e->N, D = e->D, I = e->I;
  e->patches = c.take<__nv_bfloat16>(M * e->Kpad);
  e->x = c.take<__nv_bfloat16>(M * D);
  e->h = c.take<__nv_bfloat16>(M * D);
  e->qkv = c.take<__nv_bfloat16>(M * 3 * D);
  e->att = c.take<__nv_bfloat16>(M * D);
  e->mlp = c.take<__nv_bfloat16>(M * I);
  e->ao = c.take<__nv_bfloat16>(B * D);
  e->r = c.take<__nv_bfloat16>(B * D);
  e->h2 = c.take<__nv_bfloat16>(B * D);
  e->m2 = c.take<__nv_bfloat16>(B * I);
  // row statistics of the residual stream: one (Σx, Σx²) pair per 64-column chunk and row, [ceil(D/64)][M][2]
  const int64_t parts = (D + 63) / 64;
  e->stats_a = c.take<float>(parts * M * 2);
  e->stats_b = c.take<float>(parts * M * 2);
  *total = c.off;
}

struct Slot {
  void* dst;
  int dst_bf16;
  int64_t rows, cols, dst_ld, dst_cols;
};

// name -> destination.  Returns false if the name is not part of the vision tower.
bool resolve(dfd_engine* e, const std::string& name, Slot* s) {
  const int64_t D = e->D, I = e->I, N = e->N;
  auto mk = [&](void* dst, int bf, int64_t rows, int64_t cols) {
    *s = Slot{dst, bf, rows, cols, cols, cols};
    return true;
  };
  if (name == "embeddings.patch_embedding.weight") {
    *s = Slot{e->w_pe, 1, D, e->Kpe, e->Kpad, e->Kpad};
    return true;
  }
  if (name == "embeddings.patch_embedding.bias") return mk(e->b_pe, 0, 1, D);
  if (name == "embeddings.position_embedding.weight") return mk(e->pos, 0, N, D);
  if (name == "post_layernorm.weight") return mk(e->post_g, 0, 1, D);
  if (name == "post_layernorm.bias") return mk(e->post_b, 0, 1, D);
  if (name == "head.probe") return mk(e->probe, 0, 1, D);
  if (name == "head.attention.in_proj_weight") return mk(e->w_in, 1, 3 * D, D);
  if (name == "head.attention.in_proj_bias") return mk(e->b_in, 0, 1, 3 * D);
  if (name == "head.attention.out_proj.weight") return mk(e->w_mo, 1, D, D);
  if (name == "head.attention.out_proj.bias") return mk(e->b_mo, 0, 1, D);
  if (name == "head.layernorm.weight") return mk(e->hln_g, 0, 1, D);
  if (name == "head.layernorm.bias") return mk(e->hln_b, 0, 1, D);
  if (name == "head.mlp.fc1.weight") return mk(e->w_mfc1, 1, I, D);
  if (name == "head.mlp.fc1.bias") return mk(e->b_mfc1, 0, 1, I);
  if (name == "head.mlp.fc2.weight") return mk(e->w_mfc2, 1, D, I);
  if (name == "head.mlp.fc2.bias") return mk(e->b_mfc2, 0, 1, D);
  const char* pre = "encoder.layers.";
  if (name.compare(0, strlen(pre), pre) != 0) return false;
  size_t pos = strlen(pre);
  size_t dot = name.find('.', pos);
  if (dot == std::string::npos) return false;
  int li = -1;
  try { li = std::stoi(name.substr(pos, dot - pos)); } catch (...) { return false; }
  if (li < 0 || li >= e->L) return false;
  Layer& l = e->layers[li];
  const std::string t = name.substr(dot + 1);
  if (t == "layer_norm1.weight") return mk(l.ln1_g, 0, 1, D);
  if (t == "layer_norm1.bias") return mk(l.ln1_b, 0, 1, D);
  if (t == "layer_norm2.weight") return mk(l.ln2_g, 0, 1, D);
  if (t == "layer_norm2.bias") return mk(l.ln2_b, 0, 1, D);
  if (t == "self_attn.q_proj.weight") return mk(l.w_qkv, 1, D, D);
  if (t == "self_attn.k_proj.weight") return mk(l.w_qkv + D * D, 1, D, D);
  if (t == "self_attn.v_proj.weight") return mk(l.w_qkv + 2 * D * D, 1, D, D);
  if (t == "self_attn.q_proj.bias") return mk(l.b_qkv, 0, 1, D);
  if (t == "self_attn.k_proj.bias") return mk(l.b_qkv + D, 0, 1, D);
  if (t == "self_attn.v_proj.bias") return mk(l.b_qkv + 2 * D, 0, 1, D);
  if (t == "self_attn.qkv.weight") return mk(l.w_qkv, 1, 3 * D, D);  // timm fused layout (q, k, v)
  if (t == "self_attn.qkv.bias") return mk(l.b_qkv, 0, 1, 3 * D);
  if (t == "self_attn.out_proj.weight") return mk(l.w_o, 1, D, D);
  if (t == "self_attn.out_proj.bias") return mk(l.b_o, 0, 1, D);
  if (t == "mlp.fc1.weight") return mk(l.w_fc1, 1, I, D);
  if (t == "mlp.fc1.bias") return mk(l.b_fc1, 0, 1, I);
  if (t == "mlp.fc2.weight") return mk(l.w_fc2, 1, D, I);
  if (t == "mlp.fc2.bias") return mk(l.b_fc2, 0, 1, D);
  return false;
}

void list_required(dfd_engine* e) {
  auto& m = e->missing;
  m = {"embeddings.patch_embedding.weight", "embeddings.patch_embedding.bias",
       "embeddings.position_embedding.weight", "post_layernorm.weight", "post_layernorm.bias", "head.probe",
       "head.attention.in_proj_weight", "head.attention.in_proj_bias", "head.attention.out_proj.weight",
       "head.attention.out_proj.bias", "head.layernorm.weight", "head.layernorm.bias", "head.mlp.fc1.weight",
       "head.mlp.fc1.bias", "head.mlp.fc2.weight", "head.mlp.fc2.bias"};
  const char* per[] = {"layer_norm1.weight", "layer_norm1.bias", "layer_norm2.weight", "layer_norm2.bias",
                       "self_attn.q_proj.weight", "self_attn.k_proj.weight", "self_attn.v_proj.weight",
                       "self_attn.q_proj.bias", "self_attn.k_proj.bias", "self_attn.v_proj.bias",
                       "self_attn.out_proj.weight", "self_attn.out_proj.bias", "mlp.fc1.weight", "mlp.fc1.bias",
                       "mlp.fc2.weight", "mlp.fc2.bias"};
  for (int i = 0; i < e->L; ++i)
    for (const char* p : per) m.push_back("encoder.layers." + std::to_string(i) + "." + p);
}

void mark_set(dfd_engine* e, const std::string& name) {
  auto erase = [&](const std::string& n) {
    for (size_t i = 0; i < e->missing.size(); ++i)
      if (e->missing[i] == n) { e->missing.erase(e->missing.begin() + i); return; }
  };
  const size_t p = name.find("self_attn.qkv.");
  if (p != std::string::npos) {  // fused tensor satisfies the three split names
    const std::string head = name.substr(0, p), tail = name.substr(p + strlen("self_attn.qkv."));
    erase(head + "self_attn.q_proj." + tail);
    erase(head + "self_attn.k_proj." + tail);
    erase(head + "self_attn.v_proj." + tail);
  } else {
    erase(name);
  }
}

struct DeviceGuard {
  int prev;
  bool ok;
  explicit DeviceGuard(int dev) : prev(-1), ok(false) {
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    ok = (prev == dev) || (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

}  // namespace
}  // namespace dfd

using namespace dfd;

extern "C" DFD_API int dfd_engine_create(const dfd_config* cfg, int device, int max_batch, dfd_engine** out) {
  DFD_REQUIRE(cfg && out, DFD_ERR_BAD_ARG, "engine_create: null pointer");
  *out = nullptr;
  DFD_REQUIRE(max_batch > 0, DFD_ERR_BAD_ARG, "engine_create: max_batch must be positive");
  DFD_REQUIRE(cfg->patch > 0 && cfg->image_size >= cfg->patch && cfg->hidden > 0 && cfg->inter > 0 &&
                  cfg->layers > 0 && cfg->heads > 0,
              DFD_ERR_BAD_ARG, "engine_create: bad config");
  DFD_REQUIRE(cfg->hidden % cfg->heads == 0, DFD_ERR_SHAPE, "engine_create: hidden %% heads != 0");
  const int hd = cfg->hidden / cfg->heads;
  DFD_REQUIRE(hd == 64 || hd == 72, DFD_ERR_UNSUPPORTED, "engine_create: head dim %d unsupported (64, 72)", hd);
  DFD_REQUIRE(cfg->hidden % 8 == 0 && cfg->inter % 8 == 0, DFD_ERR_SHAPE,
              "engine_create: hidden and inter must be multiples of 8");
  DFD_REQUIRE(cfg->gelu_tanh == 1, DFD_ERR_UNSUPPORTED, "engine_create: only gelu_pytorch_tanh backbones");
  DFD_REQUIRE(cfg->fuse_ln == 0 || cfg->fuse_ln == 1, DFD_ERR_BAD_ARG, "engine_create: fuse_ln must be 0 or 1");
  int ndev = 0;
  DFD_CUDA(cudaGetDeviceCount(&ndev));
  DFD_REQUIRE(device >= 0 && device < ndev, DFD_ERR_NO_DEVICE, "engine_create: device %d of %d", device, ndev);
  cudaDeviceProp prop;
  DFD_CUDA(cudaGetDeviceProperties(&prop, device));
  DFD_REQUIRE(prop.major == 10, DFD_ERR_UNSUPPORTED,
              "engine_create: device %d is sm_%d%d; this library is sm_100a only", device, prop.major, prop.minor);
  DeviceGuard guard(device);
  DFD_REQUIRE(guard.ok, DFD_ERR_CUDA, "engine_create: cudaSetDevice(%d) failed", device);

  dfd_engine* e = new dfd_engine();
  e->cfg = *cfg;
  e->device = device;
  e->max_batch = max_batch;
  e->S = cfg->image_size; e->P = cfg->patch; e->G = e->S / e->P; e->N = e->G * e->G;
  e->D = cfg->hidden; e->I = cfg->inter; e->L = cfg->layers; e->H = cfg->heads; e->hd = hd;
  e->Kpe = 3 * e->P * e->P;
  e->Kpad = (int)align_up(e->Kpe, 64);
  e->finalized = false;
  e->folded = false;
  e->hidden_tap = nullptr;
  e->attn_tap = nullptr;
  e->attn_per_head = 0;
  e->map_tap = nullptr;
  e->wslab = e->aslab = nullptr;
  e->staging = nullptr;
  e->staging_bytes = 0;
  e->prof_on = false;
  e->prof_n = 0;
  e->prof_cap = 0;
  e->x_lo = nullptr;
  e->precise = false;
  e->graphs_on = false;
  e->graph_clock = 0;
  e->capture_stream = nullptr;
  e->graph_replays = 0;
  carve_weights(e, nullptr, &e->wbytes);
  carve_acts(e, nullptr, &e->abytes);
  cudaError_t err = cudaMalloc(&e->wslab, e->wbytes);
  if (err == cudaSuccess) err = cudaMalloc(&e->aslab, e->abytes);
  if (err != cudaSuccess) {
    if (e->wslab) cudaFree(e->wslab);
    delete e;
    return cuda_fail(err, "cudaMalloc(engine slabs)", __FILE__, __LINE__);
  }
  carve_weights(e, e->wslab, &e->wbytes);
  carve_acts(e, e->aslab, &e->abytes);
  cudaMemset(e->wslab, 0, e->wbytes);
  list_required(e);
  *out = e;
  return DFD_OK;
}

extern "C" DFD_API int dfd_engine_destroy(dfd_engine* e) {
  if (!e) return DFD_OK;
  DeviceGuard guard(e->device);
  cudaDeviceSynchronize();
  if (e->wslab) cudaFree(e->wslab);
  if (e->aslab) cudaFree(e->aslab);
  if (e->staging) cudaFree(e->staging);
  if (e->x_lo) cudaFree(e->x_lo);
  for (cudaEvent_t ev : e->prof_ev) cudaEventDestroy(ev);
  for (auto& g : e->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (e->capture_stream) cudaStreamDestroy(e->capture_stream);
  delete e;
  return DFD_OK;
}

extern "C" DFD_API int64_t dfd_engine_workspace_bytes(const dfd_engine* e) {
  return e ? e->wbytes + e->abytes : 0;
}

extern "C" DFD_API int dfd_engine_set_tensor(dfd_engine* e, const char* name, const void* data, int dtype,
                                             int ndim, const int64_t* shape, int on_host) {
  DFD_REQUIRE(e && name && data && shape, DFD_ERR_BAD_ARG, "set_tensor: null pointer");
  DFD_REQUIRE(dtype == 0 || dtype == 1, DFD_ERR_BAD_ARG, "set_tensor: dtype must be 0 (f32) or 1 (bf16)");
  DFD_REQUIRE(ndim >= 0 && ndim <= 8, DFD_ERR_BAD_ARG, "set_tensor: bad ndim");
  Slot s;
  DFD_REQUIRE(resolve(e, name, &s), DFD_ERR_BAD_ARG, "set_tensor: unknown tensor name '%s'", name);
  int64_t numel = 1;
  for (int i = 0; i < ndim; ++i) numel *= shape[i];
  DFD_REQUIRE(numel == s.rows * s.cols, DFD_ERR_SHAPE, "set_tensor: '%s' has %lld elements, expected %lld", name,
              (long long)numel, (long long)(s.rows * s.cols));
  DeviceGuard guard(e->device);
  DFD_REQUIRE(guard.ok, DFD_ERR_CUDA, "set_tensor: cudaSetDevice failed");
  const void* src = data;
  if (on_host) {
    const int64_t bytes = numel * (dtype ? 2 : 4);
    if (bytes > e->staging_bytes) {
      if (e->staging) { cudaDeviceSynchronize(); cudaFree(e->staging); e->staging = nullptr; }
      DFD_CUDA(cudaMalloc(&e->staging, bytes));
      e->staging_bytes = bytes;
    }
    DFD_CUDA(cudaMemcpy(e->staging, data, bytes, cudaMemcpyHostToDevice));
    src = e->staging;
  }
  const int64_t total = s.rows * s.dst_cols;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 4096) blocks = 4096;
  // Stream ordered on the legacy default stream: the H2D copy into the staging buffer (which returns once the pageable
  // source has been consumed), this kernel, and the next tensor's copy into the same buffer run in order, so no device
  // synchronisation is needed per tensor — dfd_engine_finalize synchronises once (448 tensors for so400m).
  convert_rows_kernel<<<blocks, 256>>>(src, dtype, s.rows, s.cols, s.dst, s.dst_bf16, s.dst_ld, s.dst_cols);
  DFD_LAUNCH_CHECK();
  mark_set(e, name);
  e->finalized = false;
  if (e->folded) {  // weights were folded in place: a partial reload would mix folded and raw tensors
    e->folded = false;
    list_required(e);
    mark_set(e, name);
  }
  return DFD_OK;
}

extern "C" DFD_API int dfd_engine_finalize(dfd_engine* e) {
  DFD_REQUIRE(e, DFD_ERR_BAD_ARG, "finalize: null engine");
  if (!e->missing.empty()) {
    set_last_error("finalize: %zu tensors not set, first: %s", e->missing.size(), e->missing[0].c_str());
    return DFD_ERR_STATE;
  }
  DeviceGuard guard(e->device);
  DFD_REQUIRE(guard.ok, DFD_ERR_CUDA, "finalize: cudaSetDevice failed");
  // the MAP query is batch independent: q = probe · W_qᵀ + b_q  (first D rows of in_proj)
  probe_query_kernel<<<(e->D + 7) / 8, 256>>>(e->probe, e->w_in, e->b_in, e->q_probe, e->D);
  DFD_LAUNCH_CHECK();
  if (e->cfg.fuse_ln && !e->folded) {
    for (auto& l : e->layers) {
      fold_ln_kernel<<<(3 * e->D + 7) / 8, 256>>>(l.w_qkv, l.b_qkv, l.cs_qkv, l.ln1_g, l.ln1_b, 3 * e->D, e->D);
      fold_ln_kernel<<<(e->I + 7) / 8, 256>>>(l.w_fc1, l.b_fc1, l.cs_fc1, l.ln2_g, l.ln2_b, e->I, e->D);
    }
    DFD_LAUNCH_CHECK();
    e->folded = true;
  }
  DFD_CUDA(cudaDeviceSynchronize());
  e->finalized = true;
  return DFD_OK;
}

#define DFD_TRY(expr)            \
  do {                           \
    const int _rc = (expr);      \
    if (_rc != DFD_OK) return _rc; \
  } while (0)

// run one launch, bracketed by events when profiling is on
#define DFD_OP(fam, expr)                                                                   \
  do {                                                                                      \
    const bool _p = e->prof_on && e->prof_n < e->prof_cap;                                       \
    if (_p) DFD_CUDA(cudaEventRecord(e->prof_ev[2 * e->prof_n], st));                        \
    DFD_TRY(expr);                                                                          \
    if (_p) {                                                                               \
      DFD_CUDA(cudaEventRecord(e->prof_ev[2 * e->prof_n + 1], st));                          \
      e->prof_fam[e->prof_n++] = (fam);                                                     \
    }                                                                                       \
  } while (0)

// hidden_states tap (Siglip2sidafrozen.py:787-793: output_hidden_states=True): when set, the next forwards copy the
// embedding output and every encoder layer's output into buf[(l) * B * N * D ...] (bf16, B = that forward's batch).
extern "C" DFD_API int dfd_engine_set_hidden_tap(dfd_engine* e, void* buf) {
  DFD_REQUIRE(e, DFD_ERR_BAD_ARG, "set_hidden_tap: null engine");
  e->hidden_tap = buf;
  return DFD_OK;
}

// attention-map tap (HF output_attentions=True): when attn is set, the next forwards write each layer's attention
// probabilities right after that layer's attention launch, while its qkv is still live; when map_p is set, the MAP
// kernel also writes the probe attention.  Not profiled, and the forward runs eagerly while either is set.
extern "C" DFD_API int dfd_engine_set_attention_tap(dfd_engine* e, float* attn, int per_head, float* map_p) {
  DFD_REQUIRE(e, DFD_ERR_BAD_ARG, "set_attention_tap: null engine");
  DFD_REQUIRE(per_head == 0 || per_head == 1, DFD_ERR_BAD_ARG, "set_attention_tap: per_head must be 0 or 1");
  DFD_REQUIRE(((uintptr_t)attn % 4 == 0) && ((uintptr_t)map_p % 4 == 0), DFD_ERR_BAD_ARG,
              "set_attention_tap: buffers must be 4-byte aligned");
  e->attn_tap = attn;
  e->attn_per_head = per_head;
  e->map_tap = map_p;
  return DFD_OK;
}

extern "C" DFD_API int dfd_engine_profile(dfd_engine* e, int enable) {
  DFD_REQUIRE(e, DFD_ERR_BAD_ARG, "profile: null engine");
  DeviceGuard guard(e->device);
  // enable = how many forwards the event buffer must hold: launches keep being recorded across forwards (no host
  // synchronisation inside a timed loop) until dfd_engine_profile_read sums and clears them
  if (enable > 0) {
    const size_t n = (size_t)(16 + 8 * e->L) * (size_t)enable;
    const size_t have = e->prof_ev.size();
    if (have < 2 * n) {
      e->prof_ev.resize(2 * n);
      for (size_t i = have; i < 2 * n; ++i) DFD_CUDA(cudaEventCreate(&e->prof_ev[i]));
      e->prof_fam.resize(n, 0);
    }
  }
  e->prof_on = enable > 0;
  e->prof_cap = enable > 0 ? (16 + 8 * e->L) * enable : 0;
  e->prof_n = 0;
  return DFD_OK;
}

// Sums the event-timed durations of every launch recorded since the last read (or since profiling was switched on) per
// kernel family (ms) and the launch counts, then clears the record.  Synchronises on the last recorded event.
// Families: 0 GEMM (patch embedding, pooling head), 1 attention, 2 LayerNorm, 3 patchify, 4 MAP attention, 5 qkv GEMM,
// 6 out-projection GEMM, 7 fc1 GEMM, 8 fc2 GEMM.
extern "C" DFD_API int dfd_engine_profile_read(dfd_engine* e, float* ms, int* count) {
  DFD_REQUIRE(e && ms && count, DFD_ERR_BAD_ARG, "profile_read: null pointer");
  DeviceGuard guard(e->device);
  for (int i = 0; i < 9; ++i) { ms[i] = 0.f; count[i] = 0; }
  if (e->prof_n == 0) return DFD_OK;
  DFD_CUDA(cudaEventSynchronize(e->prof_ev[2 * e->prof_n - 1]));
  for (int i = 0; i < e->prof_n; ++i) {
    float t = 0.f;
    DFD_CUDA(cudaEventElapsedTime(&t, e->prof_ev[2 * i], e->prof_ev[2 * i + 1]));
    const int f = e->prof_fam[i];
    ms[f] += t;
    count[f] += 1;
  }
  e->prof_n = 0;
  return DFD_OK;
}

// The launches of one forward, enqueued on st (which may be a capturing stream).
static int forward_body(dfd_engine* e, const void* pixels, int pix_format, int B, int Hin, int Win, int resize_mode,
                        void* pooled, void* last_hidden, cudaStream_t st) {
  const int N = e->N, D = e->D, I = e->I, H = e->H, hd = e->hd;
  const int M = B * N;
  const float eps = e->cfg.ln_eps;
  const float scale = 1.0f / sqrtf((float)hd);

  DFD_OP(3, patchify(pixels, pix_format, B, Hin, Win, e->S, e->P, resize_mode, e->patches, e->Kpad, st));
  const bool fuse = e->cfg.fuse_ln != 0;
  const int ln_parts = (D + 63) / 64;  // partial statistics per row written by the GEMM that produced the residual stream
  {
    dfd_gemm_epilogue ep{};
    ep.bias = e->b_pe;
    ep.pos = e->pos;
    ep.pos_rows = N;
    if (fuse) ep.stats_out = e->stats_a;
    DFD_OP(0, gemm_bf16_dispatch(e->patches, e->Kpad, e->w_pe, e->Kpad, e->x, D, M, D, e->Kpad, &ep, 0, st));
  }
  const size_t hid_bytes = (size_t)M * D * sizeof(__nv_bfloat16);
  // precise mode: x = hi + lo.  The patch embedding leaves lo = 0 (one bf16 rounding, as for every branch input); each
  // residual GEMM then reads and rewrites both halves, so the additions of all 2·L branches accumulate at ~16 mantissa bits
  __nv_bfloat16* lo = e->precise ? e->x_lo : nullptr;
  if (lo) DFD_CUDA(cudaMemsetAsync(lo, 0, (size_t)((M + 127) / 128) * 128 * ((D + 63) / 64) * 64 * sizeof(__nv_bfloat16), st));
  if (e->hidden_tap) DFD_CUDA(cudaMemcpyAsync(e->hidden_tap, e->x, hid_bytes, cudaMemcpyDeviceToDevice, st));
  for (int li = 0; li < e->L; ++li) {
    const Layer& l = e->layers[li];
    if (fuse) {
      // LN1 folded into the qkv GEMM: row statistics came from the GEMM that produced x
      dfd_gemm_epilogue ep{};
      ep.bias = l.b_qkv;
      ep.ln_rowstats = e->stats_a;
      ep.ln_parts = ln_parts;
      ep.ln_colsum = l.cs_qkv;
      ep.ln_dim = D;
      ep.ln_eps = eps;
      DFD_OP(5, gemm_bf16_dispatch(e->x, D, l.w_qkv, D, e->qkv, 3 * D, M, 3 * D, D, &ep, 0, st));
    } else {
      DFD_OP(2, layernorm_bf16(e->x, D, lo, e->h, D, l.ln1_g, l.ln1_b, M, D, eps, st));
      dfd_gemm_epilogue ep{};
      ep.bias = l.b_qkv;
      DFD_OP(5, gemm_bf16_dispatch(e->h, D, l.w_qkv, D, e->qkv, 3 * D, M, 3 * D, D, &ep, 0, st));
    }
    DFD_OP(1, attention_auto_bf16(e->qkv, 3 * D, e->att, D, B, N, H, hd, scale, st));
    if (e->attn_tap)
      DFD_TRY(attention_probs(e->qkv, 3 * D, B, N, H, hd, scale, e->attn_per_head,
                              e->attn_tap + (int64_t)li * B * (e->attn_per_head ? H : 1) * N * N, st));
    {
      dfd_gemm_epilogue ep{};
      ep.bias = l.b_o;
      ep.residual = e->x;
      ep.ldr = D;
      ep.residual_lo = lo;
      if (fuse) ep.stats_out = e->stats_b;
      DFD_OP(6, gemm_bf16_dispatch(e->att, D, l.w_o, D, e->x, D, M, D, D, &ep, 0, st));
    }
    if (fuse) {
      dfd_gemm_epilogue ep{};
      ep.bias = l.b_fc1;
      ep.act = 1;
      ep.ln_rowstats = e->stats_b;
      ep.ln_parts = ln_parts;
      ep.ln_colsum = l.cs_fc1;
      ep.ln_dim = D;
      ep.ln_eps = eps;
      DFD_OP(7, gemm_bf16_dispatch(e->x, D, l.w_fc1, D, e->mlp, I, M, I, D, &ep, 0, st));
    } else {
      DFD_OP(2, layernorm_bf16(e->x, D, lo, e->h, D, l.ln2_g, l.ln2_b, M, D, eps, st));
      dfd_gemm_epilogue ep{};
      ep.bias = l.b_fc1;
      ep.act = 1;
      DFD_OP(7, gemm_bf16_dispatch(e->h, D, l.w_fc1, D, e->mlp, I, M, I, D, &ep, 0, st));
    }
    {
      dfd_gemm_epilogue ep{};
      ep.bias = l.b_fc2;
      ep.residual = e->x;
      ep.ldr = D;
      ep.residual_lo = lo;
      if (fuse && li + 1 < e->L) ep.stats_out = e->stats_a;  // for the next layer's LN1 (the post-LN runs as a kernel)
      DFD_OP(8, gemm_bf16_dispatch(e->mlp, I, l.w_fc2, I, e->x, D, M, D, I, &ep, 0, st));
    }
    if (e->hidden_tap)
      DFD_CUDA(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(e->hidden_tap) + (size_t)(li + 1) * hid_bytes, e->x, hid_bytes,
                               cudaMemcpyDeviceToDevice, st));
  }
  __nv_bfloat16* xp = last_hidden ? reinterpret_cast<__nv_bfloat16*>(last_hidden) : e->h;
  DFD_OP(2, layernorm_bf16(e->x, D, lo, xp, D, e->post_g, e->post_b, M, D, eps, st));
  {  // K | V projection of every token (rows D..3D of in_proj)
    dfd_gemm_epilogue ep{};
    ep.bias = e->b_in + D;
    DFD_OP(0, gemm_bf16_dispatch(xp, D, e->w_in + (int64_t)D * D, D, e->qkv, 2 * D, M, 2 * D, D, &ep, 0, st));
  }
  DFD_OP(4, map_attention_bf16(e->qkv, 2 * D, e->q_probe, e->ao, D, B, N, H, hd, scale, e->map_tap, st));
  {
    dfd_gemm_epilogue ep{};
    ep.bias = e->b_mo;
    DFD_OP(0, gemm_bf16_dispatch(e->ao, D, e->w_mo, D, e->r, D, B, D, D, &ep, 0, st));
  }
  DFD_OP(2, layernorm_bf16(e->r, D, nullptr, e->h2, D, e->hln_g, e->hln_b, B, D, eps, st));
  {
    dfd_gemm_epilogue ep{};
    ep.bias = e->b_mfc1;
    ep.act = 1;
    DFD_OP(0, gemm_bf16_dispatch(e->h2, D, e->w_mfc1, D, e->m2, I, B, I, D, &ep, 0, st));
  }
  {
    dfd_gemm_epilogue ep{};
    ep.bias = e->b_mfc2;
    ep.residual = e->r;
    ep.ldr = D;
    DFD_OP(0, gemm_bf16_dispatch(e->m2, I, e->w_mfc2, I, pooled, D, B, D, I, &ep, 0, st));
  }
  return DFD_OK;
}

// CUDA graphs of the forward (SURVEY.md §7 step 9).  A forward is 7·L + 13 launches, each with 3-4 tensor maps encoded on
// the host; for small batches (multicrop: 6-9 views; base-224 at any batch below ~64) the host cannot keep ahead of the
// device.  With graphs on, a call signature (pointers, batch, input geometry) runs eagerly the first time it is seen, is
// captured the second time (on a private stream: the caller's may be the legacy default stream, which cannot capture) and
// is replayed with ONE cudaGraphLaunch on the caller's stream from then on: tensor maps and kernel arguments are baked into
// the graph.  Up to kMaxGraphs signatures are kept (least recently used out).  Profiling, hidden-state and attention taps
// run eagerly.
extern "C" DFD_API int dfd_engine_set_graphs(dfd_engine* e, int enable) {
  DFD_REQUIRE(e, DFD_ERR_BAD_ARG, "set_graphs: null engine");
  e->graphs_on = enable != 0;
  if (!e->graphs_on) {
    DeviceGuard guard(e->device);
    cudaDeviceSynchronize();
    for (auto& g : e->graphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    e->graphs.clear();
  }
  return DFD_OK;
}

// Residual-stream precision.  0 (default): the stream is one bf16 tensor, rounded after each of the 2·L residual additions.
// 1: two bf16 tensors (hi + lo, ~16 mantissa bits) — the additions accumulate like the fp32 residual stream the reference keeps
// under autocast (HF:modeling_siglip.py:352,359); branch inputs are still the bf16 value hi.  Costs one extra [B·N, D] bf16
// buffer (allocated here) and 4 more bytes per element and residual GEMM of HBM traffic.
extern "C" DFD_API int dfd_engine_set_precise_residual(dfd_engine* e, int enable) {
  DFD_REQUIRE(e, DFD_ERR_BAD_ARG, "set_precise_residual: null engine");
  DeviceGuard guard(e->device);
  DFD_REQUIRE(guard.ok, DFD_ERR_CUDA, "set_precise_residual: cudaSetDevice failed");
  if (enable && e->x_lo == nullptr)
    DFD_CUDA(cudaMalloc(&e->x_lo, (size_t)(((int64_t)e->max_batch * e->N + 127) / 128) * 128 * ((e->D + 63) / 64) * 64 *
                                      sizeof(__nv_bfloat16)));   // tiled: whole 128-row x 64-column blocks
  if ((enable != 0) != e->precise) {   // captured graphs bake the mode in
    cudaDeviceSynchronize();
    for (auto& g : e->graphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    e->graphs.clear();
  }
  e->precise = enable != 0;
  return DFD_OK;
}

// Graph replays since the engine was created (tests / bench: proves that the graph path ran).
extern "C" DFD_API int64_t dfd_engine_graph_replays(const dfd_engine* e) { return e ? e->graph_replays : 0; }

extern "C" DFD_API int dfd_engine_forward(dfd_engine* e, const void* pixels, int pix_format, int B, int Hin,
                                          int Win, int resize_mode, void* pooled, void* last_hidden,
                                          void* stream) {
  DFD_REQUIRE(e && pixels && pooled, DFD_ERR_BAD_ARG, "forward: null pointer");
  DFD_REQUIRE(e->finalized, DFD_ERR_STATE, "forward: engine not finalized");
  DFD_REQUIRE(B > 0 && B <= e->max_batch, DFD_ERR_SHAPE, "forward: batch %d outside 1..%d", B, e->max_batch);
  {
    // kernels are launched on the CURRENT device: refuse to run against another device's pointers (the stream handed in
    // belongs to the caller's device as well)
    int cur = -1;
    DFD_CUDA(cudaGetDevice(&cur));
    DFD_REQUIRE(cur == e->device, DFD_ERR_STATE,
                "forward: the engine lives on device %d but device %d is current (cudaSetDevice / torch.cuda.device first)",
                e->device, cur);
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool eager =
      !e->graphs_on || e->prof_on || e->hidden_tap != nullptr || e->attn_tap != nullptr || e->map_tap != nullptr;
  if (eager) return forward_body(e, pixels, pix_format, B, Hin, Win, resize_mode, pooled, last_hidden, st);

  constexpr size_t kMaxGraphs = 16;
  const dfd_engine::GraphKey key{pixels, pooled, last_hidden, pix_format, B, Hin, Win, resize_mode};
  dfd_engine::GraphEntry* hit = nullptr;
  for (auto& g : e->graphs)
    if (g.key == key) { hit = &g; break; }
  if (hit != nullptr && hit->exec != nullptr) {
    hit->last_use = ++e->graph_clock;
    DFD_CUDA(cudaGraphLaunch(hit->exec, st));
    g_launches.fetch_add(hit->launches, std::memory_order_relaxed);
    ++e->graph_replays;
    return DFD_OK;
  }
  if (hit == nullptr) {
    // first sight: run eagerly (also takes care of one-time function attributes) and remember the signature
    if (e->graphs.size() >= kMaxGraphs) {
      size_t lru = 0;
      for (size_t i = 1; i < e->graphs.size(); ++i)
        if (e->graphs[i].last_use < e->graphs[lru].last_use) lru = i;
      if (e->graphs[lru].exec) cudaGraphExecDestroy(e->graphs[lru].exec);
      e->graphs.erase(e->graphs.begin() + lru);
    }
    e->graphs.push_back(dfd_engine::GraphEntry{key, nullptr, 0, ++e->graph_clock});
    return forward_body(e, pixels, pix_format, B, Hin, Win, resize_mode, pooled, last_hidden, st);
  }
  // second sight: capture, instantiate, launch
  if (e->capture_stream == nullptr) DFD_CUDA(cudaStreamCreateWithFlags(&e->capture_stream, cudaStreamNonBlocking));
  const int64_t l0 = g_launches.load(std::memory_order_relaxed);
  DFD_CUDA(cudaStreamBeginCapture(e->capture_stream, cudaStreamCaptureModeThreadLocal));
  const int rc = forward_body(e, pixels, pix_format, B, Hin, Win, resize_mode, pooled, last_hidden, e->capture_stream);
  cudaGraph_t graph = nullptr;
  const cudaError_t cerr = cudaStreamEndCapture(e->capture_stream, &graph);
  const int64_t captured = g_launches.load(std::memory_order_relaxed) - l0;
  g_launches.fetch_sub(captured, std::memory_order_relaxed);   // nothing ran yet
  if (rc != DFD_OK) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  if (cerr != cudaSuccess) return cuda_fail(cerr, "cudaStreamEndCapture(forward)", __FILE__, __LINE__);
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ierr = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ierr != cudaSuccess) return cuda_fail(ierr, "cudaGraphInstantiate(forward)", __FILE__, __LINE__);
  hit->exec = exec;
  hit->launches = captured;
  hit->last_use = ++e->graph_clock;
  DFD_CUDA(cudaGraphLaunch(exec, st));
  g_launches.fetch_add(captured, std::memory_order_relaxed);
  ++e->graph_replays;
  return DFD_OK;
}

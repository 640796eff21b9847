// MAP pooling head attention (HF:modeling_siglip.py:639-646): softmax_n(q_h·k_n)·v_n for the ONE learned probe query per
// head, over the N patch tokens of an image.  HBM bound: K and V of a head are read exactly once.
// (The encoder's self-attention kernels are attention_dq.cu / attention_ws.cu; the round-1 mma.sync and per-tile tcgen05
// kernels that used to live here and in attention_tc.cu / attention_pq.cu were superseded and removed from the library.)
#include "dfd_common.cuh"

#include <algorithm>
#include <atomic>

namespace dfd {

extern std::atomic<int64_t> g_launches;

namespace {

// ---- MAP pooling attention: one CTA per (image, head), one query --------------------------------
// HBM-bound (K and V of one head are read exactly once, N x 2 x HD bf16).  Both passes walk the rows in 16-byte chunks
// with consecutive threads on consecutive chunks, so every row's HD*2 bytes are fetched as whole sectors and a CTA keeps
// 256 independent 16-byte loads in flight: the scores pass leaves one partial dot product per chunk in shared memory, the
// P·V pass gives each thread one chunk column and every (256 / chunks)-th key.
constexpr int kMapThreads = 256;

// kProbs: also write the probabilities probs[b, h, n] (the attention-map tap); the product instantiations have it off
template <int HD, bool kProbs>
__global__ void __launch_bounds__(kMapThreads)
map_attention_kernel(const __nv_bfloat16* __restrict__ kv, int64_t ldkv, const float* __restrict__ q,
                     __nv_bfloat16* __restrict__ out, int64_t ldo, int N, int H, float scale, float* __restrict__ probs) {
  constexpr int kC = HD / 8;             // 16-byte chunks per row
  constexpr int kG = kMapThreads / kC;   // key groups of the P·V pass
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float* sc = reinterpret_cast<float*>(smem_raw);   // [N] scores -> probabilities
  float* ps = sc + ((N + 3) & ~3);                  // [max(N*kC, kG*HD)] chunk partials, later the P·V partials
  __shared__ __align__(16) float sq[HD];
  __shared__ float red[kMapThreads / 32];
  const int h = blockIdx.x, b = blockIdx.y;
  const int D = H * HD;
  const __nv_bfloat16* gK = kv + (int64_t)b * N * ldkv + h * HD;
  const __nv_bfloat16* gV = gK + D;

  if (threadIdx.x < HD) sq[threadIdx.x] = __ldg(q + h * HD + threadIdx.x) * scale;
  __syncthreads();
  for (int i = threadIdx.x; i < N * kC; i += kMapThreads) {
    const int n = i / kC, c = i - n * kC;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(gK + (int64_t)n * ldkv) + c);
    const float4 q0 = *reinterpret_cast<const float4*>(sq + c * 8), q1 = *reinterpret_cast<const float4*>(sq + c * 8 + 4);
    const float2 a = unpack_bf16x2(v.x), b2 = unpack_bf16x2(v.y), c2 = unpack_bf16x2(v.z), d2 = unpack_bf16x2(v.w);
    ps[i] = ((a.x * q0.x + a.y * q0.y) + (b2.x * q0.z + b2.y * q0.w)) + ((c2.x * q1.x + c2.y * q1.y) + (d2.x * q1.z + d2.y * q1.w));
  }
  __syncthreads();
  float lmax = -INFINITY;
  for (int n = threadIdx.x; n < N; n += kMapThreads) {
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < kC; ++c) acc += ps[n * kC + c];
    sc[n] = acc;
    lmax = fmaxf(lmax, acc);
  }
  lmax = warp_max(lmax);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = lmax;
  __syncthreads();
  float gmax = red[0];
#pragma unroll
  for (int i = 1; i < kMapThreads / 32; ++i) gmax = fmaxf(gmax, red[i]);
  __syncthreads();
  float lsum = 0.f;
  for (int n = threadIdx.x; n < N; n += kMapThreads) {
    const float p = __expf(sc[n] - gmax);
    sc[n] = p;
    lsum += p;
  }
  lsum = warp_sum(lsum);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = lsum;
  __syncthreads();
  float gsum = 0.f;
#pragma unroll
  for (int i = 0; i < kMapThreads / 32; ++i) gsum += red[i];
  if constexpr (kProbs) {
    for (int n = threadIdx.x; n < N; n += kMapThreads) probs[((int64_t)b * H + h) * N + n] = sc[n] / gsum;
  }

  // out[d] = sum_n p[n] v[n,d] / gsum
  const int g = threadIdx.x / kC, c = threadIdx.x - g * kC;
  if (g < kG) {
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int n = g; n < N; n += kG) {
      const float p = sc[n];
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(gV + (int64_t)n * ldkv) + c);
      const float2 v0 = unpack_bf16x2(v.x), v1 = unpack_bf16x2(v.y), v2 = unpack_bf16x2(v.z), v3 = unpack_bf16x2(v.w);
      a[0] += p * v0.x; a[1] += p * v0.y; a[2] += p * v1.x; a[3] += p * v1.y;
      a[4] += p * v2.x; a[5] += p * v2.y; a[6] += p * v3.x; a[7] += p * v3.y;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) ps[g * HD + c * 8 + j] = a[j];
  }
  __syncthreads();
  if (threadIdx.x < HD) {
    const int d = threadIdx.x;
    float v = 0.f;
#pragma unroll 4
    for (int k = 0; k < kG; ++k) v += ps[k * HD + d];
    out[(int64_t)b * ldo + h * HD + d] = __float2bfloat16(v / gsum);
  }
}

}  // namespace
int map_attention_bf16(const void* kv, int64_t ldkv, const float* q, void* out, int64_t ldo, int B, int N,
                       int H, int hd, float scale, float* probs, cudaStream_t st) {
  DFD_REQUIRE(kv && q && out, DFD_ERR_BAD_ARG, "map_attention: null pointer");
  DFD_REQUIRE(B > 0 && N > 0 && H > 0, DFD_ERR_SHAPE, "map_attention: B, N, H must be positive");
  DFD_REQUIRE(hd == 64 || hd == 72, DFD_ERR_UNSUPPORTED, "map_attention: head dim %d not supported (64, 72)", hd);
  DFD_REQUIRE(ldkv % 8 == 0 && ldkv >= 2 * H * hd && ldo >= H * hd, DFD_ERR_SHAPE,
              "map_attention: bad leading dimensions");
  DFD_REQUIRE(B <= 65535, DFD_ERR_SHAPE, "map_attention: B must be <= 65535");
  DFD_REQUIRE(((uintptr_t)kv % 16 == 0), DFD_ERR_BAD_ARG, "map_attention: kv must be 16-byte aligned");
  const int chunks = hd / 8, groups = kMapThreads / chunks;
  const int64_t part_words = std::max<int64_t>((int64_t)N * chunks, (int64_t)groups * hd);
  const int64_t smem64 = (((int64_t)N + 3) & ~3ll) * 4 + part_words * 4;
  DFD_REQUIRE(smem64 <= 200 * 1024, DFD_ERR_UNSUPPORTED, "map_attention: N=%d too long", N);
  const int smem = (int)smem64;
  dim3 grid(H, B);
  static SmemOptIn smem_once[4];
  const __nv_bfloat16* k = reinterpret_cast<const __nv_bfloat16*>(kv);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
#define DFD_MAP_LAUNCH(HD_, PROBS_, SLOT_)                                                                          \
  do {                                                                                                              \
    if (int rc = ensure_dynamic_smem(smem_once[SLOT_], map_attention_kernel<HD_, PROBS_>, 200 * 1024)) return rc;   \
    map_attention_kernel<HD_, PROBS_><<<grid, kMapThreads, smem, st>>>(k, ldkv, q, o, ldo, N, H, scale, probs);     \
  } while (0)
  if (hd == 64) {
    if (probs) DFD_MAP_LAUNCH(64, true, 2); else DFD_MAP_LAUNCH(64, false, 0);
  } else {
    if (probs) DFD_MAP_LAUNCH(72, true, 3); else DFD_MAP_LAUNCH(72, false, 1);
  }
#undef DFD_MAP_LAUNCH
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

}  // namespace dfd

extern "C" DFD_API int dfd_map_attention_bf16(const void* kv, int64_t ldkv, const float* q, void* out,
                                              int64_t ldo, int B, int N, int H, int hd, float scale,
                                              void* stream) {
  return dfd::map_attention_bf16(kv, ldkv, q, out, ldo, B, N, H, hd, scale, nullptr,
                                 reinterpret_cast<cudaStream_t>(stream));
}

// The pieces of SegFormerStrongDecoder / SigLIP2_MTL (Siglip2sidafrozen.py:698-803) that are not GEMMs.  All 1x1
// convolutions and the LinearProj layers are tcgen05 GEMMs on token-major [B·H·W, C] matrices (gemm_tcgen05.cu, with the
// erf-GELU / sigmoid / gating epilogues); what is left is HBM-bound streaming work:
//
//   dwconv3x3_kernel     depthwise 3x3 convolution, zero padding 1, on the H x W token grid (channels innermost)
//   seg_head_kernel      1x1 convolution E -> 1 on the LOW-resolution grid ...
//   upsample_kernel      ... followed by the bilinear (align_corners=False) resize to the image size.  The reference
//                        upsamples E channels first and applies the head afterwards (:740-741); both maps are linear and
//                        commute exactly, so the head runs on 1/(S/H)² of the pixels and the resize moves 1 channel, not E
//   linear_small_kernel  Linear(hidden, 3) classification head on the pooled embedding (:773-777,789)
#include "dfd_common.cuh"

#include <atomic>

namespace dfd {

extern std::atomic<int64_t> g_launches;

namespace {

// one thread = 8 channels of one token
__global__ void __launch_bounds__(256)
dwconv3x3_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const float* __restrict__ w /*[E][9]*/,
                 const float* __restrict__ bias, __nv_bfloat16* __restrict__ out, int64_t ldo, int H, int W, int E,
                 int64_t total) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int e8 = E / 8;
  const int c0 = (int)(idx % e8) * 8;
  const int64_t tok = idx / e8;
  const int xw = (int)(tok % W), yh = (int)((tok / W) % H);
  const int64_t img0 = tok - (int64_t)yh * W - xw;  // first token of this image
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = bias ? __ldg(bias + c0 + i) : 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int yy = yh + dy;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int xx = xw + dx;
      if (xx < 0 || xx >= W) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(x + (img0 + (int64_t)yy * W + xx) * ldx + c0);
      const float2 p0 = unpack_bf16x2(v.x), p1 = unpack_bf16x2(v.y), p2 = unpack_bf16x2(v.z), p3 = unpack_bf16x2(v.w);
      const float in[8] = {p0.x, p0.y, p1.x, p1.y, p2.x, p2.y, p3.x, p3.y};
      const int t = (dy + 1) * 3 + (dx + 1);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = fmaf(in[i], __ldg(w + (c0 + i) * 9 + t), acc[i]);
    }
  }
  uint4 o;
  o.x = pack_bf16x2(acc[0], acc[1]);
  o.y = pack_bf16x2(acc[2], acc[3]);
  o.z = pack_bf16x2(acc[4], acc[5]);
  o.w = pack_bf16x2(acc[6], acc[7]);
  *reinterpret_cast<uint4*>(out + tok * ldo + c0) = o;
}

// one warp per token: low[tok] = bias + sum_e x[tok][e] * w[e]
__global__ void __launch_bounds__(256)
seg_head_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const float* __restrict__ w, float bias,
                float* __restrict__ low, int64_t tokens, int E) {
  const int64_t tok = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (tok >= tokens) return;
  float acc = 0.f;
  for (int e = lane * 8; e < E; e += 256) {
    const uint4 v = *reinterpret_cast<const uint4*>(x + tok * ldx + e);
    const float2 p0 = unpack_bf16x2(v.x), p1 = unpack_bf16x2(v.y), p2 = unpack_bf16x2(v.z), p3 = unpack_bf16x2(v.w);
    acc += p0.x * __ldg(w + e) + p0.y * __ldg(w + e + 1) + p1.x * __ldg(w + e + 2) + p1.y * __ldg(w + e + 3) +
           p2.x * __ldg(w + e + 4) + p2.y * __ldg(w + e + 5) + p3.x * __ldg(w + e + 6) + p3.y * __ldg(w + e + 7);
  }
  acc = warp_sum(acc);
  if (lane == 0) low[tok] = acc + bias;
}

// one warp per (row, output): out[b][n] = bias[n] + sum_k x[b][k] * w[n][k]
__global__ void __launch_bounds__(256)
linear_small_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const float* __restrict__ w,
                    const float* __restrict__ bias, float* __restrict__ out, int B, int N, int K) {
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (o >= B * N) return;
  const int b = o / N, n = o % N;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc += __bfloat162float(x[(int64_t)b * ldx + k]) * __ldg(w + (int64_t)n * K + k);
  acc = warp_sum(acc);
  if (lane == 0) out[o] = acc + (bias ? __ldg(bias + n) : 0.f);
}

// F.interpolate(mode="bilinear", align_corners=False) of gain·low: src = (dst + 0.5) * in/out - 0.5, clamped at 0
__global__ void __launch_bounds__(256)
upsample_kernel(const float* __restrict__ low, float gain, float* __restrict__ out, int H, int W, int S, float sy, float sx) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= S) return;
  const float fy = fmaxf((y + 0.5f) * sy - 0.5f, 0.f), fx = fmaxf((x + 0.5f) * sx - 0.5f, 0.f);
  const int y0 = (int)fy, x0 = (int)fx;
  const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
  const float ly = fy - y0, lx = fx - x0;
  const float* img = low + (int64_t)b * H * W;
  const float v00 = gain * img[y0 * W + x0], v01 = gain * img[y0 * W + x1], v10 = gain * img[y1 * W + x0],
              v11 = gain * img[y1 * W + x1];
  out[((int64_t)b * S + y) * S + x] = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
}

}  // namespace

// the segmentation head's resize and the attention-rollout heatmap (attention_probs.cu)
int upsample_bilinear(const float* low, float gain, float* out, int B, int H, int W, int S, cudaStream_t st) {
  upsample_kernel<<<dim3((S + 255) / 256, S, B), 256, 0, st>>>(low, gain, out, H, W, S, (float)H / (float)S,
                                                              (float)W / (float)S);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

}  // namespace dfd

extern "C" DFD_API int dfd_dwconv3x3_bf16(const void* x, int64_t ldx, const float* w9, const float* bias, void* out,
                                          int64_t ldo, int B, int H, int W, int E, void* stream) {
  using namespace dfd;
  DFD_REQUIRE(x && w9 && out, DFD_ERR_BAD_ARG, "dwconv3x3: null pointer");
  DFD_REQUIRE(B > 0 && H > 0 && W > 0 && E > 0 && E % 8 == 0 && ldx >= E && ldo >= E && ldx % 8 == 0 && ldo % 8 == 0,
              DFD_ERR_SHAPE, "dwconv3x3: bad shape (channels and leading dimensions must be multiples of 8)");
  DFD_REQUIRE((uintptr_t)x % 16 == 0 && (uintptr_t)out % 16 == 0, DFD_ERR_BAD_ARG, "dwconv3x3: pointers must be 16-byte aligned");
  const int64_t total = (int64_t)B * H * W * (E / 8);
  DFD_REQUIRE((total + 255) / 256 < (1ll << 31), DFD_ERR_SHAPE, "dwconv3x3: too large");
  dwconv3x3_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), ldx, w9, bias, reinterpret_cast<__nv_bfloat16*>(out), ldo, H, W, E, total);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

extern "C" DFD_API int dfd_seg_head_upsample(const void* x, int64_t ldx, const float* w, float bias, int B, int H, int W,
                                             int E, int S, float* low_scratch, float* out, void* stream) {
  using namespace dfd;
  DFD_REQUIRE(x && w && low_scratch && out, DFD_ERR_BAD_ARG, "seg_head_upsample: null pointer");
  DFD_REQUIRE(B > 0 && H > 0 && W > 0 && S > 0 && E > 0 && E % 8 == 0 && ldx >= E && ldx % 8 == 0 && B <= 65535 && S <= 65535,
              DFD_ERR_SHAPE, "seg_head_upsample: bad shape");
  DFD_REQUIRE((uintptr_t)x % 16 == 0, DFD_ERR_BAD_ARG, "seg_head_upsample: x must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t tokens = (int64_t)B * H * W;
  seg_head_kernel<<<(unsigned)((tokens + 7) / 8), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), ldx, w, bias,
                                                                low_scratch, tokens, E);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return upsample_bilinear(low_scratch, 1.0f, out, B, H, W, S, st);
}

extern "C" DFD_API int dfd_linear_small(const void* x, int64_t ldx, const float* w, const float* bias, float* out, int B,
                                        int N, int K, void* stream) {
  using namespace dfd;
  DFD_REQUIRE(x && w && out, DFD_ERR_BAD_ARG, "linear_small: null pointer");
  DFD_REQUIRE(B > 0 && N > 0 && K > 0 && ldx >= K, DFD_ERR_SHAPE, "linear_small: bad shape");
  const int64_t outs = (int64_t)B * N;
  linear_small_kernel<<<(unsigned)((outs + 7) / 8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), ldx, w, bias, out, B, N, K);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

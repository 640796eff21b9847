// HBM-bound row kernels of the backbone: LayerNorm, fused preprocess + im2col.
//
//   dfd_layernorm_bf16  one warp per token row, 16-byte loads, fp32 two-pass statistics
//                       (HF:modeling_siglip.py:348,357,618 — nn.LayerNorm(eps=1e-6) under autocast runs in fp32)
//   dfd_patchify        u8 NHWC / f32 NCHW pixels → normalised bf16 patch matrix, optional nearest /
//                       bilinear resample (inference_ai_human_images.py:200-204; train_fusion_head_only.py:67-74,103-104;
//                       cifake_binary_classifier.py:716-717; HF:modeling_siglip.py:124-130,178)
#include "dfd_common.cuh"

#include <atomic>

namespace dfd {

extern std::atomic<int64_t> g_launches;

namespace {

constexpr int kRowThreads = 256;  // 8 warps = 8 rows per CTA
constexpr int kMaxVec = 8;        // rows up to 8*32*8 = 2048 elements stay in registers

// elements 2j, 2j+1 of a 16-byte vector of a row (plus those of its low half)
template <bool LO>
__device__ __forceinline__ float2 ln_val(const uint4& hi, const uint4& lo, int j) {
  const uint32_t h[4] = {hi.x, hi.y, hi.z, hi.w};
  float2 a = unpack_bf16x2(h[j]);
  if (LO) {
    const uint32_t l[4] = {lo.x, lo.y, lo.z, lo.w};
    const float2 b = unpack_bf16x2(l[j]);
    a.x += b.x;
    a.y += b.y;
  }
  return a;
}

// LO: the row is the sum of two bf16 tensors (x + lo: the two-bf16 residual stream of the precise engine mode)
template <bool LO>
__global__ void __launch_bounds__(kRowThreads)
layernorm_bf16_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, const __nv_bfloat16* __restrict__ lo,
                      __nv_bfloat16* __restrict__ y, int64_t ldy, const float* __restrict__ gamma,
                      const float* __restrict__ beta, int M, int D, float eps) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (kRowThreads / 32) + warp;
  if (row >= M) return;
  const int nvec = D >> 3;
  const uint4* xr = reinterpret_cast<const uint4*>(x + (int64_t)row * ldx);
  // the low halves are stored in the GEMM epilogue's order: [row block of 128][64-column chunk][8-column group][row][8]
  const int nch = (D + 63) >> 6;
  const uint4* lr = LO ? reinterpret_cast<const uint4*>(lo) + (int64_t)(row >> 7) * nch * 1024 + (row & 127) : nullptr;
  uint4 v[kMaxVec], w[LO ? kMaxVec : 1];
  w[0] = make_uint4(0u, 0u, 0u, 0u);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
      v[i] = __ldg(xr + c);
      if (LO) w[i] = __ldg(lr + (c >> 3) * 1024 + (c & 7) * 128);
      const float2 a = ln_val<LO>(v[i], w[LO ? i : 0], 0), b = ln_val<LO>(v[i], w[LO ? i : 0], 1), c2 = ln_val<LO>(v[i], w[LO ? i : 0], 2),
                   d = ln_val<LO>(v[i], w[LO ? i : 0], 3);
      sum += ((a.x + a.y) + (b.x + b.y)) + ((c2.x + c2.y) + (d.x + d.y));
    }
  }
  const float mean = warp_sum(sum) / (float)D;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 a = ln_val<LO>(v[i], w[LO ? i : 0], j);
        const float d0 = a.x - mean, d1 = a.y - mean;
        sq += d0 * d0 + d1 * d1;
      }
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)D + eps);
  uint4* yr = reinterpret_cast<uint4*>(y + (int64_t)row * ldy);
#pragma unroll
  for (int i = 0; i < kMaxVec; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma) + 2 * c);
      const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma) + 2 * c + 1);
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta) + 2 * c);
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(beta) + 2 * c + 1);
      const float2 a = ln_val<LO>(v[i], w[LO ? i : 0], 0), b = ln_val<LO>(v[i], w[LO ? i : 0], 1), c2 = ln_val<LO>(v[i], w[LO ? i : 0], 2),
                   d = ln_val<LO>(v[i], w[LO ? i : 0], 3);
      uint4 o;
      o.x = pack_bf16x2((a.x - mean) * rstd * g0.x + b0.x, (a.y - mean) * rstd * g0.y + b0.y);
      o.y = pack_bf16x2((b.x - mean) * rstd * g0.z + b0.z, (b.y - mean) * rstd * g0.w + b0.w);
      o.z = pack_bf16x2((c2.x - mean) * rstd * g1.x + b1.x, (c2.y - mean) * rstd * g1.y + b1.y);
      o.w = pack_bf16x2((d.x - mean) * rstd * g1.z + b1.z, (d.y - mean) * rstd * g1.w + b1.w);
      yr[c] = o;
    }
  }
}

// ---- preprocess + im2col -----------------------------------------------------------------------
struct PatchArgs {
  const void* pixels;
  int fmt;  // 0 u8 NHWC, 1 f32 NCHW
  int B, Hin, Win, S, P, G, K, mode;
  int flip;  // 1: every image is read mirrored left-right (the TTA "H-Flip" view, inference_ai_human_images.py:207-214)
  float sy, sx;  // Hin/S, Win/S (fp32, as ATen computes them)
  __nv_bfloat16* A;
  int64_t lda;
};

__device__ __forceinline__ float fetch_pixel(const PatchArgs& a, int b, int c, int y, int x) {
  if (a.flip) x = a.Win - 1 - x;  // the flip acts on the SOURCE image, i.e. before any in-model resample, as the transform does
  if (a.fmt == 0) {
    const uint8_t* p = reinterpret_cast<const uint8_t*>(a.pixels);
    const float u = (float)__ldg(p + (((int64_t)b * a.Hin + y) * a.Win + x) * 3 + c);
    // ToTensor (/255) then Normalize(mean .5, std .5), both in fp32 like torchvision
    return (u / 255.0f - 0.5f) / 0.5f;
  }
  const float* p = reinterpret_cast<const float*>(a.pixels);
  return __ldg(p + (((int64_t)b * 3 + c) * a.Hin + y) * a.Win + x);
}

__device__ __forceinline__ float sample_pixel(const PatchArgs& a, int b, int c, int y, int x) {
  if (a.mode == 0) return fetch_pixel(a, b, c, y, x);
  if (a.mode == 1) {
    // ATen nearest: src = min(floor(dst * scale), in - 1), scale = in / out in fp32
    const int ys = min((int)floorf((float)y * a.sy), a.Hin - 1);
    const int xs = min((int)floorf((float)x * a.sx), a.Win - 1);
    return fetch_pixel(a, b, c, ys, xs);
  }
  // ATen bilinear, align_corners=False: src = max(scale * (dst + .5) - .5, 0)
  const float fy = fmaxf(a.sy * ((float)y + 0.5f) - 0.5f, 0.f);
  const float fx = fmaxf(a.sx * ((float)x + 0.5f) - 0.5f, 0.f);
  const int y0 = min((int)fy, a.Hin - 1), x0 = min((int)fx, a.Win - 1);
  const int y1 = min(y0 + 1, a.Hin - 1), x1 = min(x0 + 1, a.Win - 1);
  const float ly = fy - (float)y0, lx = fx - (float)x0;
  const float hy = 1.f - ly, hx = 1.f - lx;
  return hy * (hx * fetch_pixel(a, b, c, y0, x0) + lx * fetch_pixel(a, b, c, y0, x1)) +
         ly * (hx * fetch_pixel(a, b, c, y1, x0) + lx * fetch_pixel(a, b, c, y1, x1));
}

// one thread = 8 consecutive columns of one patch row (one 16-byte store)
__global__ void __launch_bounds__(256) patchify_kernel(PatchArgs a) {
  const int vec_per_row = (int)(a.lda >> 3);
  const int64_t total = (int64_t)a.B * a.G * a.G * vec_per_row;
  const int PP = a.P * a.P;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int vcol = (int)(idx % vec_per_row);
    const int64_t prow = idx / vec_per_row;
    const int gx = (int)(prow % a.G);
    const int gy = (int)((prow / a.G) % a.G);
    const int b = (int)(prow / ((int64_t)a.G * a.G));
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = vcol * 8 + j;
      if (k < a.K) {
        const int c = k / PP;
        const int r = k - c * PP;
        const int ky = r / a.P, kx = r - ky * a.P;
        v[j] = sample_pixel(a, b, c, gy * a.P + ky, gx * a.P + kx);
      } else {
        v[j] = 0.f;  // K padding
      }
    }
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]);
    o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]);
    o.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(a.A + prow * a.lda + (int64_t)vcol * 8) = o;
  }
}

// Fast path for the case every shipped caller hits (u8 NHWC input already on the patch grid, no resample): one CTA per
// (image, patch row).  The P image rows of a patch row are one contiguous span of P*Win*3 bytes, and its G output rows
// one contiguous span of G*lda bf16 — both are moved with 16-byte accesses through shared memory; the k -> (c, ky, kx)
// index arithmetic becomes a table built once per CTA; the bf16 result is bit-identical to the generic kernel's.
__global__ void __launch_bounds__(256) patchify_u8_rows_kernel(PatchArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int span = a.P * a.Win * 3;
  uint16_t* koff = reinterpret_cast<uint16_t*>(smem + 1024);           // [lda] (0xffff = K padding); 16-byte aligned
  uint8_t* pix = smem + 1024 + (((int)a.lda * 2 + 15) & ~15);          // [span + 16]
  const int b = blockIdx.x / a.G, gy = blockIdx.x - b * a.G;
  const uint8_t* src = reinterpret_cast<const uint8_t*>(a.pixels) + ((int64_t)b * a.Hin + (int64_t)gy * a.P) * a.Win * 3;
  const int head = (int)(reinterpret_cast<uintptr_t>(src) & 15);       // pix[head + i] = src[i]
  const int tid = threadIdx.x;
  const int PP = a.P * a.P;
  for (int k = tid; k < (int)a.lda; k += 256) {
    if (k < a.K) {
      const int c = k / PP, r = k - c * PP;
      const int ky = r / a.P, kx = r - ky * a.P;
      // mirrored: patch gx, column kx reads source pixel Win-1-(gx P + kx); the gx part moves into `base` below
      koff[k] = (uint16_t)((ky * a.Win + (a.flip ? a.Win - 1 - kx : kx)) * 3 + c);
    } else {
      koff[k] = 0xffffu;
    }
  }
  // aligned body with 16-byte loads, ragged ends byte by byte (never touches memory outside the span)
  const int lead = head ? 16 - head : 0;
  const int body = (span - lead) >> 4;
  for (int i = tid; i < lead && i < span; i += 256) pix[head + i] = __ldg(src + i);
  const uint4* src16 = reinterpret_cast<const uint4*>(src + lead);
  uint4* pix16 = reinterpret_cast<uint4*>(pix + head + lead);
  for (int i = tid; i < body; i += 256) pix16[i] = __ldg(src16 + i);
  for (int i = lead + (body << 4) + tid; i < span; i += 256) pix[head + i] = __ldg(src + i);
  __syncthreads();
  const int vec_per_row = (int)(a.lda >> 3);
  uint4* dst = reinterpret_cast<uint4*>(a.A + ((int64_t)b * a.G + gy) * a.G * a.lda);
  for (int idx = tid; idx < a.G * vec_per_row; idx += 256) {
    const int gx = idx / vec_per_row, vcol = idx - gx * vec_per_row;
    const uint8_t* base = a.flip ? pix + head - gx * a.P * 3 : pix + head + gx * a.P * 3;
    // the eight source offsets of this 16-byte output piece come as ONE 16-byte shared load; ToTensor + Normalize is one FMA:
    // fmaf(x, 2/255, -1) differs from fetch_pixel's ((x / 255) - 0.5) / 0.5 by an fp32 ulp for some x but rounds to the same
    // bf16 for all 256 byte values (checked exhaustively, tests/test_abi_cpu.py).  The first version did three shared loads per
    // element (offset, byte, a 256-entry value table) and sat at the L1 / shared-memory pipe's limit (ncu: l1tex 99 % busy)
    const uint4 kq = *reinterpret_cast<const uint4*>(koff + vcol * 8);
    const uint32_t kw[4] = {kq.x, kq.y, kq.z, kq.w};
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t o = (kw[j >> 1] >> (16 * (j & 1))) & 0xffffu;
      v[j] = o == 0xffffu ? 0.f : fmaf((float)base[o], 2.0f / 255.0f, -1.0f);
    }
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]);
    o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]);
    o.w = pack_bf16x2(v[6], v[7]);
    dst[idx] = o;
  }
}

}  // namespace

int layernorm_bf16(const void* x, int64_t ldx, const void* lo, void* y, int64_t ldy, const float* gamma,
                   const float* beta, int M, int D, float eps, cudaStream_t st) {
  DFD_REQUIRE(x && y && gamma && beta, DFD_ERR_BAD_ARG, "layernorm: null pointer");
  DFD_REQUIRE(M > 0 && D > 0, DFD_ERR_SHAPE, "layernorm: M and D must be positive");
  DFD_REQUIRE(D % 8 == 0 && D <= kMaxVec * 256, DFD_ERR_SHAPE,
              "layernorm: D must be a multiple of 8 and <= %d (D=%d)", kMaxVec * 256, D);
  DFD_REQUIRE(ldx % 8 == 0 && ldy % 8 == 0 && ldx >= D && ldy >= D, DFD_ERR_SHAPE,
              "layernorm: leading dimensions must be multiples of 8 and >= D");
  const int rows_per_cta = kRowThreads / 32;
  const int grid = (M + rows_per_cta - 1) / rows_per_cta;
  if (lo != nullptr)
    layernorm_bf16_kernel<true><<<grid, kRowThreads, 0, st>>>(
        reinterpret_cast<const __nv_bfloat16*>(x), ldx, reinterpret_cast<const __nv_bfloat16*>(lo),
        reinterpret_cast<__nv_bfloat16*>(y), ldy, gamma, beta, M, D, eps);
  else
    layernorm_bf16_kernel<false><<<grid, kRowThreads, 0, st>>>(
        reinterpret_cast<const __nv_bfloat16*>(x), ldx, nullptr, reinterpret_cast<__nv_bfloat16*>(y), ldy, gamma, beta,
        M, D, eps);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

int patchify(const void* pixels, int pix_format, int B, int Hin, int Win, int S, int P, int resize_mode,
             void* A, int64_t lda, cudaStream_t st) {
  DFD_REQUIRE(pixels && A, DFD_ERR_BAD_ARG, "patchify: null pointer");
  DFD_REQUIRE(pix_format == 0 || pix_format == 1, DFD_ERR_BAD_ARG, "patchify: pix_format must be 0 or 1");
  const int flip = (resize_mode >> 4) & 1;   // DFD_FLIP_H
  resize_mode &= 0xF;
  DFD_REQUIRE(resize_mode >= 0 && resize_mode <= 2, DFD_ERR_BAD_ARG, "patchify: resize_mode must be 0..2 (| DFD_FLIP_H)");
  DFD_REQUIRE(B > 0 && Hin > 0 && Win > 0 && S > 0 && P > 0 && P <= S, DFD_ERR_SHAPE,
              "patchify: bad shape");
  // mode 0 reads the top-left G*P x G*P pixels only (conv padding='valid'), so any input on the same patch grid
  // is accepted: so400m-patch14 takes 378..391-pixel sides for its 27x27 grid.
  const int GP = (S / P) * P;
  DFD_REQUIRE(resize_mode != 0 || (Hin >= GP && Hin < GP + P && Win >= GP && Win < GP + P), DFD_ERR_SHAPE,
              "patchify: resize_mode 0 needs %d..%d-pixel sides, got %dx%d", GP, GP + P - 1, Hin, Win);
  const int K = 3 * P * P;
  DFD_REQUIRE(lda % 8 == 0 && lda >= K, DFD_ERR_SHAPE, "patchify: lda must be a multiple of 8 and >= 3*P*P");
  PatchArgs a;
  a.pixels = pixels;
  a.fmt = pix_format;
  a.B = B; a.Hin = Hin; a.Win = Win; a.S = S; a.P = P; a.G = S / P; a.K = K;
  // images at the model resolution take the patch grid directly; with a resample mode given, every other size is resampled
  // to S x S first, exactly like the reference's `if x.shape[-1] != res: F.interpolate(...)` (train_fusion_head_only.py:103-104,
  // cifake_binary_classifier.py:716-717) — also sizes that happen to cover the patch grid (S < side < GP + P)
  a.mode = (Hin == S && Win == S) ? 0 : resize_mode;
  a.flip = flip;
  a.sy = (float)Hin / (float)S;
  a.sx = (float)Win / (float)S;
  a.A = reinterpret_cast<__nv_bfloat16*>(A);
  a.lda = lda;
  const int64_t fast_smem = 1024 + ((lda * 2 + 15) & ~15ll) + (int64_t)P * Win * 3 + 16;
  if (a.fmt == 0 && a.mode == 0 && fast_smem <= 48 * 1024 && (int64_t)P * Win * 3 < 0xffff && (int64_t)P * Win * 3 >= 64 &&
      (int64_t)B * a.G < (1ll << 31) &&
      (reinterpret_cast<uintptr_t>(A) & 15) == 0) {
    patchify_u8_rows_kernel<<<B * a.G, 256, (size_t)fast_smem, st>>>(a);
    DFD_LAUNCH_CHECK();
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return DFD_OK;
  }
  const int64_t total = (int64_t)B * a.G * a.G * (lda >> 3);
  int64_t blocks = (total + 255) / 256;
  if (blocks > (int64_t)kNumSMs * 32) blocks = (int64_t)kNumSMs * 32;
  patchify_kernel<<<(int)blocks, 256, 0, st>>>(a);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

}  // namespace dfd

extern "C" DFD_API int dfd_layernorm_bf16(const void* x, int64_t ldx, const void* lo, void* y, int64_t ldy,
                                          const float* gamma, const float* beta, int M, int D, float eps, void* stream) {
  return dfd::layernorm_bf16(x, ldx, lo, y, ldy, gamma, beta, M, D, eps, reinterpret_cast<cudaStream_t>(stream));
}
extern "C" DFD_API int dfd_patchify(const void* pixels, int pix_format, int B, int Hin, int Win, int S,
                                    int P, int resize_mode, void* A, int64_t lda, void* stream) {
  return dfd::patchify(pixels, pix_format, B, Hin, Win, S, P, resize_mode, A, lda,
                       reinterpret_cast<cudaStream_t>(stream));
}

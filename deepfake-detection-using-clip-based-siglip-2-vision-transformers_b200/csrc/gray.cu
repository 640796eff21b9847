// gray256 on the GPU: u8 RGB images -> the 256x256 gray image every frequency feature is computed from.
//
// Reference (train_fusion_head_only.py:142-148, deepfake-detector-v2/app.py:736-749):
//     ImageOps.exif_transpose(pil).convert("L") -> [cv2 CLAHE(2.0, 8x8)] -> resize((256,256), BICUBIC) -> f32 / 255
// i.e. Pillow's integer luma, OpenCV's CLAHE and Pillow's 22-bit fixed-point antialiased bicubic resample.  All of it
// is byte / integer work (plus four fp32 multiply-adds per pixel in CLAHE's LUT interpolation, done here in the
// library's operation order without fused multiply-add), so the result is bit-exact with the libraries; the oracle
// restatement is oracle/gray_ref.py, pinned against Pillow 12.2.0 / OpenCV 4.13.0.
//
//   luma_kernel              RGB u8 NHWC -> L u8                         (Pillow Convert.c rgb2l)
//   clahe_lut_kernel         per (image, tile): histogram in shared memory, clip + redistribute, prefix sum -> LUT
//   clahe_apply_kernel       per pixel: bilinear blend of the 4 surrounding tile LUTs        (OpenCV clahe.cpp)
//   resize_rows_kernel       horizontal pass, u8 -> u8                    (Pillow Resample.c, 8bpc)
//   resize_cols_kernel       vertical pass, u8 -> f32 / 255
// HBM-bound streaming kernels; ~1.3 MB of traffic per 384x384 image, < 0.1 % of the detection step.
#include "dfd_common.cuh"

#include <atomic>
#include <cmath>

namespace dfd {

extern std::atomic<int64_t> g_launches;

namespace {

constexpr int kOut = 256;
constexpr int kPrecisionBits = 32 - 8 - 2;  // Resample.c PRECISION_BITS
constexpr int kTiles = 8;

// ---------------------------------------------------------------------------------------------------------
// Pillow rgb2l
// ---------------------------------------------------------------------------------------------------------
__global__ void luma_kernel(const uint8_t* __restrict__ rgb, uint8_t* __restrict__ L, int64_t npix) {
  // 4 pixels (12 bytes in, 4 bytes out) per thread
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t p0 = q * 4;
  if (p0 >= npix) return;
  if (p0 + 4 <= npix) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(rgb + p0 * 3);  // 12-byte groups are 4-byte aligned
    const uint32_t a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
    const uint32_t px[12] = {a & 255u, (a >> 8) & 255u, (a >> 16) & 255u, a >> 24,
                             b & 255u, (b >> 8) & 255u, (b >> 16) & 255u, b >> 24,
                             c & 255u, (c >> 8) & 255u, (c >> 16) & 255u, c >> 24};
    uint32_t out = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t l = (px[3 * i] * 19595u + px[3 * i + 1] * 38470u + px[3 * i + 2] * 7471u + 0x8000u) >> 16;
      out |= l << (8 * i);
    }
    *reinterpret_cast<uint32_t*>(L + p0) = out;
  } else {
    for (int64_t p = p0; p < npix; ++p)
      L[p] = (uint8_t)((rgb[3 * p] * 19595u + rgb[3 * p + 1] * 38470u + rgb[3 * p + 2] * 7471u + 0x8000u) >> 16);
  }
}

// The same for a rectangle of a larger image (a crop given by base pointer + strides): one thread per pixel, rows of the crop
// are row_stride bytes apart, images image_stride bytes.  Output packed [B, H, W] like luma_kernel's.
__global__ void __launch_bounds__(256)
luma_strided_kernel(const uint8_t* __restrict__ rgb, int64_t row_stride, int64_t image_stride, uint8_t* __restrict__ L, int H,
                    int W) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, b = blockIdx.z;
  if (x >= W) return;
  const uint8_t* p = rgb + (int64_t)b * image_stride + (int64_t)y * row_stride + 3 * x;
  L[((int64_t)b * H + y) * W + x] = (uint8_t)((p[0] * 19595u + p[1] * 38470u + p[2] * 7471u + 0x8000u) >> 16);
}

// ---------------------------------------------------------------------------------------------------------
// OpenCV CLAHE (8-bit, histSize 256)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
  return i;
}

// OpenCV's tile geometry for an H x W plane: tile size (the image extended to a multiple of 8 when 8 does not divide it),
// histogram clip limit (clipLimit 2.0 scaled to the tile area, at least 1) and the LUT scale 255 / area
struct ClaheGeometry {
  int tw, th, clip;
  float lut_scale;
};
ClaheGeometry clahe_geometry(int H, int W) {
  ClaheGeometry g;
  if (W % kTiles == 0 && H % kTiles == 0) {
    g.tw = W / kTiles;
    g.th = H / kTiles;
  } else {
    g.tw = (W + (kTiles - W % kTiles)) / kTiles;
    g.th = (H + (kTiles - H % kTiles)) / kTiles;
  }
  const int area = g.tw * g.th;
  g.lut_scale = 255.0f / (float)area;
  g.clip = (int)(2.0 * area / 256);
  if (g.clip < 1) g.clip = 1;
  return g;
}

// grid (64 tiles, B·C planes), 256 threads.  tile (tw x th) of the image extended by BORDER_REFLECT_101 to a multiple of 8.
// C = interleaved channels of the input (1: the luma plane of gray256; 3: one plane per colour channel of an RGB image, the
// per-channel CLAHE of train_fusion_head_only.py:60-65); plane p = image p / C, channel p % C.
__global__ void __launch_bounds__(256)
clahe_lut_kernel(const uint8_t* __restrict__ L, uint8_t* __restrict__ luts, int H, int W, int C, int tw, int th, int clip,
                 float lut_scale) {
  __shared__ int hist[256];
  __shared__ int scan[256];
  __shared__ int s_clipped;
  const int tile = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  const int ty = tile / kTiles, tx = tile % kTiles;
  const uint8_t* img = L + (int64_t)(b / C) * H * W * C + (b % C);
  hist[t] = 0;
  if (t == 0) s_clipped = 0;
  __syncthreads();
  for (int i = t; i < tw * th; i += 256) {
    const int y = reflect101(ty * th + i / tw, H), x = reflect101(tx * tw + i % tw, W);
    atomicAdd(&hist[img[((int64_t)y * W + x) * C]], 1);
  }
  __syncthreads();
  int h = hist[t];
  if (clip > 0) {
    if (h > clip) {
      atomicAdd(&s_clipped, h - clip);
      h = clip;
    }
    __syncthreads();
    const int clipped = s_clipped;
    const int batch = clipped / 256;
    const int residual = clipped - batch * 256;
    h += batch;
    if (residual != 0) {
      // for (i = 0; i < 256 && residual > 0; i += step, residual--) hist[i]++
      const int step = max(256 / residual, 1);
      if (t % step == 0 && t / step < residual) h += 1;
    }
  }
  // inclusive prefix sum over the 256 bins
  scan[t] = h;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const int v = t >= o ? scan[t - o] : 0;
    __syncthreads();
    scan[t] += v;
    __syncthreads();
  }
  // saturate_cast<uchar>(sum * lutScale): one fp32 multiply, round half to even, clamp
  const int r = __float2int_rn(__fmul_rn((float)scan[t], lut_scale));
  luts[((int64_t)b * kTiles * kTiles + tile) * 256 + t] = (uint8_t)min(max(r, 0), 255);
}

__global__ void __launch_bounds__(256)
clahe_apply_kernel(const uint8_t* __restrict__ L, const uint8_t* __restrict__ luts, uint8_t* __restrict__ out, int H,
                   int W, int C, float inv_tw, float inv_th) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;   // b = plane (image, channel)
  if (x >= W) return;
  const float txf = __fsub_rn(__fmul_rn((float)x, inv_tw), 0.5f);
  const float tyf = __fsub_rn(__fmul_rn((float)y, inv_th), 0.5f);
  int tx1 = (int)floorf(txf), ty1 = (int)floorf(tyf);
  const float xa = __fsub_rn(txf, (float)tx1), ya = __fsub_rn(tyf, (float)ty1);
  const float xa1 = __fsub_rn(1.0f, xa), ya1 = __fsub_rn(1.0f, ya);
  const int tx2 = min(tx1 + 1, kTiles - 1), ty2 = min(ty1 + 1, kTiles - 1);
  tx1 = max(tx1, 0);
  ty1 = max(ty1, 0);
  const int64_t pix = (((int64_t)(b / C) * H + y) * W + x) * C + (b % C);
  const int v = L[pix];
  const uint8_t* lb = luts + (int64_t)b * kTiles * kTiles * 256 + v;
  const float l11 = (float)__ldg(lb + (ty1 * kTiles + tx1) * 256), l12 = (float)__ldg(lb + (ty1 * kTiles + tx2) * 256);
  const float l21 = (float)__ldg(lb + (ty2 * kTiles + tx1) * 256), l22 = (float)__ldg(lb + (ty2 * kTiles + tx2) * 256);
  // (l11*xa1 + l12*xa)*ya1 + (l21*xa1 + l22*xa)*ya, every operation rounded separately (no FMA) as in clahe.cpp
  const float top = __fadd_rn(__fmul_rn(l11, xa1), __fmul_rn(l12, xa));
  const float bot = __fadd_rn(__fmul_rn(l21, xa1), __fmul_rn(l22, xa));
  const float res = __fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya));
  out[pix] = (uint8_t)min(max(__float2int_rn(res), 0), 255);
}

// Fast paths for single-channel images whose tiles divide the image (W % 8 == 0, H % 8 == 0 — no border extension) and whose
// tile width is a multiple of 4 bytes: the shapes of the detection step (384², 224², any 32-aligned crop).  The generic kernels
// above issue one byte load / shared atomic / byte gather per thread and pixel and ran at 11 % of the HBM roofline
// (profiles/r01_mem_kernels.md); here
//   * clahe_lut_rows_kernel: one CTA per (tile row, image), one WARP per tile with a private histogram — word loads, no
//     block-wide barrier; clip / redistribute / prefix sum run on 8 bins per lane with shuffles;
//   * clahe_apply_band_kernel: one CTA per (band of rows with the same tile-row pair, image).  The four LUT values a pixel
//     blends — (ty1,tx1) (ty1,tx2) (ty2,tx1) (ty2,tx2) at its gray level — are packed into ONE 32-bit word of a shared table
//     built per band ([9 tile-column pairs][256 levels]), so a pixel costs one shared-memory gather instead of four byte
//     gathers; four pixels per thread through 32-bit loads / stores, row-wise factors hoisted.
// Same arithmetic in the same order as the generic kernels: bit-exact with OpenCV (tests/test_ops_gpu.py).
__global__ void __launch_bounds__(256)
clahe_lut_rows_kernel(const uint8_t* __restrict__ L, uint8_t* __restrict__ luts, int H, int W, int tw, int th, int clip,
                      float lut_scale) {
  __shared__ int hist[kTiles][256];
  const int ty = blockIdx.x, b = blockIdx.y;
  const int tx = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* h = hist[tx];
#pragma unroll
  for (int i = 0; i < 8; ++i) h[lane + 32 * i] = 0;
  __syncwarp();
  const int wq = tw >> 2;                       // 32-bit words per tile row
  const int rows_per_it = 32 / wq > 0 ? 32 / wq : 1;
  const uint8_t* base = L + ((int64_t)b * H + (int64_t)ty * th) * W + tx * tw;
  if (wq <= 32) {
    const int r_off = lane / wq, w_off = lane - r_off * wq;
    if (r_off < rows_per_it) {
      for (int r = r_off; r < th; r += rows_per_it) {
        const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(base + (int64_t)r * W) + w_off);
        atomicAdd(&h[v & 255u], 1);
        atomicAdd(&h[(v >> 8) & 255u], 1);
        atomicAdd(&h[(v >> 16) & 255u], 1);
        atomicAdd(&h[v >> 24], 1);
      }
    }
  } else {
    for (int r = 0; r < th; ++r)
      for (int w = lane; w < wq; w += 32) {
        const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(base + (int64_t)r * W) + w);
        atomicAdd(&h[v & 255u], 1);
        atomicAdd(&h[(v >> 8) & 255u], 1);
        atomicAdd(&h[(v >> 16) & 255u], 1);
        atomicAdd(&h[v >> 24], 1);
      }
  }
  __syncwarp();
  // lane owns bins 8·lane .. 8·lane+7 (contiguous: the prefix sum is a per-lane running sum plus an exclusive warp scan)
  int v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = h[lane * 8 + i];
  if (clip > 0) {
    int clipped = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (v[i] > clip) { clipped += v[i] - clip; v[i] = clip; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) clipped += __shfl_xor_sync(0xffffffffu, clipped, o);
    const int batch = clipped / 256;
    const int residual = clipped - batch * 256;
    const int step = residual != 0 ? max(256 / residual, 1) : 1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int t = lane * 8 + i;
      v[i] += batch;
      if (residual != 0 && t % step == 0 && t / step < residual) v[i] += 1;
    }
  }
  int run = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { run += v[i]; v[i] = run; }
  int incl = run;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  const int excl = incl - run;
  uint32_t w0 = 0, w1 = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = __float2int_rn(__fmul_rn((float)(v[i] + excl), lut_scale));
    const uint32_t byte = (uint32_t)min(max(r, 0), 255);
    if (i < 4) w0 |= byte << (8 * i); else w1 |= byte << (8 * (i - 4));
  }
  uint2* dst = reinterpret_cast<uint2*>(luts + ((int64_t)b * kTiles * kTiles + ty * kTiles + tx) * 256) + lane;
  *dst = make_uint2(w0, w1);
}

__global__ void __launch_bounds__(256)
clahe_apply_band_kernel(const uint8_t* __restrict__ L, const uint8_t* __restrict__ luts, uint8_t* __restrict__ out, int H,
                        int W, int th, float inv_tw, float inv_th) {
  __shared__ uint32_t tab[(kTiles + 1) * 256];   // [tile-column pair p = tx1 + 1][gray level] = l11 | l12 << 8 | l21 << 16 | l22 << 24
  const int band = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  const int ty1u = band - 1;                     // unclamped upper tile row of this band
  const int ty1 = max(ty1u, 0), ty2 = min(ty1u + 1, kTiles - 1);
  const uint8_t* lb = luts + (int64_t)b * kTiles * kTiles * 256;
  for (int p = 0; p <= kTiles; ++p) {
    const int tx1 = max(p - 1, 0), tx2 = min(p, kTiles - 1);
    tab[p * 256 + t] = (uint32_t)__ldg(lb + (ty1 * kTiles + tx1) * 256 + t) | ((uint32_t)__ldg(lb + (ty1 * kTiles + tx2) * 256 + t) << 8) |
                       ((uint32_t)__ldg(lb + (ty2 * kTiles + tx1) * 256 + t) << 16) |
                       ((uint32_t)__ldg(lb + (ty2 * kTiles + tx2) * 256 + t) << 24);
  }
  __syncthreads();
  // candidate rows of the band (one spare row on either side; every row re-checks its own tile row with the generic kernel's
  // float expression, so the split into bands cannot disagree with it)
  const int y_lo = max(ty1u * th + th / 2 - 1, 0), y_hi = min((ty1u + 1) * th + th / 2 + 1, H - 1);
  const int wq = W >> 2;
  const int items = (y_hi - y_lo + 1) * wq;
  for (int idx = t; idx < items; idx += 256) {
    const int yr = idx / wq, q = idx - yr * wq;
    const int y = y_lo + yr;
    const float tyf = __fsub_rn(__fmul_rn((float)y, inv_th), 0.5f);
    const int tyi = (int)floorf(tyf);
    if (tyi != ty1u) continue;
    const float ya = __fsub_rn(tyf, (float)tyi), ya1 = __fsub_rn(1.0f, ya);
    const int64_t off = ((int64_t)b * H + y) * W + 4 * q;
    const uint32_t px = __ldg(reinterpret_cast<const uint32_t*>(L + off));
    uint32_t res4 = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int x = 4 * q + i;
      const float txf = __fsub_rn(__fmul_rn((float)x, inv_tw), 0.5f);
      const int txi = (int)floorf(txf);
      const float xa = __fsub_rn(txf, (float)txi), xa1 = __fsub_rn(1.0f, xa);
      const uint32_t e = tab[(txi + 1) * 256 + ((px >> (8 * i)) & 255u)];
      const float l11 = (float)(e & 255u), l12 = (float)((e >> 8) & 255u), l21 = (float)((e >> 16) & 255u), l22 = (float)(e >> 24);
      const float top = __fadd_rn(__fmul_rn(l11, xa1), __fmul_rn(l12, xa));
      const float bot = __fadd_rn(__fmul_rn(l21, xa1), __fmul_rn(l22, xa));
      const float r = __fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya));
      res4 |= (uint32_t)min(max(__float2int_rn(r), 0), 255) << (8 * i);
    }
    *reinterpret_cast<uint32_t*>(out + off) = res4;
  }
}

// ---------------------------------------------------------------------------------------------------------
// Pillow 8bpc resample passes.  Coefficient tables (host: dfd_resample_coeffs_host): xmin[o], count[o], kk[o][ksize].
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int clip8(int acc) { return min(max(acc >> kPrecisionBits, 0), 255); }

// Fast forms of the two passes for tables with at most kTapMax taps (384 -> 256: 7, 224 -> 256: 5).  Rows pass: a thread owns
// one output column, keeps that column's window and coefficients in registers and walks kRowsPerCta image rows staged in shared
// memory by word loads (the generic kernel re-reads the table for every output pixel and runs one CTA per row).  Columns
// pass: a thread produces 4 adjacent pixels of 4 output rows from 32-bit loads and writes float4s.
constexpr int kTapMax = 8;
constexpr int kRowsPerCta = 16;
__global__ void __launch_bounds__(kOut)
resample_rows_fast_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int H, int W,
                          const int* __restrict__ xmin, const int* __restrict__ count, const int* __restrict__ kk, int ksize) {
  extern __shared__ uint8_t rows_s[];            // [kRowsPerCta][W]  (W % 4 == 0)
  const int xx = threadIdx.x, y0 = blockIdx.x * kRowsPerCta, b = blockIdx.y;
  const int nrows = min(kRowsPerCta, H - y0);
  const int wq = W >> 2;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(in + ((int64_t)b * H + y0) * W);
  uint32_t* dst_s = reinterpret_cast<uint32_t*>(rows_s);
  for (int i = xx; i < nrows * wq; i += kOut) dst_s[i] = __ldg(src + i);
  const int x0 = xmin[xx], n = count[xx];
  int k[kTapMax];
#pragma unroll
  for (int i = 0; i < kTapMax; ++i) k[i] = (i < n) ? __ldg(kk + xx * ksize + i) : 0;
  __syncthreads();
  // taps past the window multiply a clamped (in-row) byte by a zero coefficient
  int xi[kTapMax];
#pragma unroll
  for (int i = 0; i < kTapMax; ++i) xi[i] = min(x0 + i, W - 1);
  uint8_t* o = out + ((int64_t)b * H + y0) * kOut + xx;
  for (int r = 0; r < nrows; ++r) {
    const uint8_t* row = rows_s + r * W;
    int acc = 1 << (kPrecisionBits - 1);
#pragma unroll
    for (int i = 0; i < kTapMax; ++i) acc += (int)row[xi[i]] * k[i];
    o[(int64_t)r * kOut] = (uint8_t)clip8(acc);
  }
}

// grid (256 / 16, B), 256 threads: thread = (x quad 0..63, row group 0..3); output rows 16·blockIdx.x + 4·group + j
__global__ void __launch_bounds__(256)
resample_cols_fast_kernel(const uint8_t* __restrict__ in, float* __restrict__ out, int H, const int* __restrict__ ymin,
                          const int* __restrict__ count, const int* __restrict__ kk, int ksize) {
  const int xq = threadIdx.x & 63, grp = threadIdx.x >> 6, b = blockIdx.y;
  const uint32_t* img = reinterpret_cast<const uint32_t*>(in + (int64_t)b * H * kOut) + xq;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int yy = blockIdx.x * 16 + grp * 4 + j;
    const int y0 = __ldg(ymin + yy), n = __ldg(count + yy);
    int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll
    for (int i = 0; i < kTapMax; ++i) {
      if (i < n) {
        const int c = __ldg(kk + yy * ksize + i);
        const uint32_t v = __ldg(img + (int64_t)(y0 + i) * (kOut / 4));
        a0 += (int)(v & 255u) * c;
        a1 += (int)((v >> 8) & 255u) * c;
        a2 += (int)((v >> 16) & 255u) * c;
        a3 += (int)(v >> 24) * c;
      }
    }
    float4 o;
    o.x = __fdiv_rn((float)clip8(a0), 255.0f);
    o.y = __fdiv_rn((float)clip8(a1), 255.0f);
    o.z = __fdiv_rn((float)clip8(a2), 255.0f);
    o.w = __fdiv_rn((float)clip8(a3), 255.0f);
    reinterpret_cast<float4*>(out + ((int64_t)b * kOut + yy) * kOut)[xq] = o;
  }
}

// Generic Pillow 8bpc passes for interleaved images (C = 1 or 3 channels): dfd_resize_u8, and gray256 where the fast forms do
// not apply (C = 1, OW = OH = 256, f32 output)
// in [B, H, W, C] -> out [B, H, OW, C]
__global__ void __launch_bounds__(256)
resize_rows_kernel(const uint8_t* __restrict__ in, int64_t row_stride, int64_t image_stride, uint8_t* __restrict__ out, int H,
                   int OW, int C, const int* __restrict__ xmin, const int* __restrict__ count, const int* __restrict__ kk,
                   int ksize) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;  // (xx, c) within the output row
  const int y = blockIdx.y, b = blockIdx.z;
  if (e >= OW * C) return;
  const int xx = e / C, c = e - xx * C;
  const uint8_t* row = in + (int64_t)b * image_stride + (int64_t)y * row_stride + c;   // dense input: strides W·C and H·W·C
  const int x0 = xmin[xx], n = count[xx];
  const int* k = kk + xx * ksize;
  int acc = 1 << (kPrecisionBits - 1);
  for (int i = 0; i < n; ++i) acc += (int)row[(x0 + i) * C] * __ldg(k + i);
  out[((int64_t)b * H + y) * OW * C + e] = (uint8_t)clip8(acc);
}
__device__ __forceinline__ void store_px(uint8_t* p, int v) { *p = (uint8_t)v; }
__device__ __forceinline__ void store_px(float* p, int v) { *p = __fdiv_rn((float)v, 255.0f); }
// in [B, H, OW, C] -> out [B, OH, OW, C], u8 or f32 = u8 / 255
template <typename T>
__global__ void __launch_bounds__(256)
resize_cols_kernel(const uint8_t* __restrict__ in, T* __restrict__ out, int H, int OH, int OWC,
                   const int* __restrict__ ymin, const int* __restrict__ count, const int* __restrict__ kk, int ksize) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int yy = blockIdx.y, b = blockIdx.z;
  if (e >= OWC) return;
  const uint8_t* img = in + (int64_t)b * H * OWC + e;
  const int y0 = ymin[yy], n = count[yy];
  const int* k = kk + yy * ksize;
  int acc = 1 << (kPrecisionBits - 1);
  for (int i = 0; i < n; ++i) acc += (int)img[(int64_t)(y0 + i) * OWC] * __ldg(k + i);
  store_px(out + ((int64_t)b * OH + yy) * OWC + e, clip8(acc));
}

double bilinear_filter(double x) {
  if (x < 0.0) x = -x;
  if (x < 1.0) return 1.0 - x;
  return 0.0;
}
double bicubic_filter(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

}  // namespace

// filter: DFD_FILTER_BILINEAR (support 1) or DFD_FILTER_BICUBIC (support 2)
int resample_ksize(int in_size, int out_size, int filter) {
  double filterscale = (double)in_size / out_size;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = (filter == DFD_FILTER_BILINEAR ? 1.0 : 2.0) * filterscale;
  return (int)std::ceil(support) * 2 + 1;
}

}  // namespace dfd

extern "C" DFD_API int dfd_resample_ksize(int in_size, int out_size, int filter) {
  if (in_size <= 0 || out_size <= 0 || (filter != DFD_FILTER_BILINEAR && filter != DFD_FILTER_BICUBIC)) return 0;
  return dfd::resample_ksize(in_size, out_size, filter);
}

// Pillow precompute_coeffs + normalize_coeffs_8bpc over the whole axis (host, double precision, the library's operation
// order).  kk must hold out_size * dfd_resample_ksize(in, out, filter) ints.
extern "C" DFD_API int dfd_resample_coeffs_host(int in_size, int out_size, int filter, int32_t* xmin_host,
                                                int32_t* count_host, int32_t* kk_host) {
  DFD_REQUIRE(in_size > 0 && out_size > 0 && xmin_host && count_host && kk_host, DFD_ERR_BAD_ARG,
              "resample_coeffs: bad argument");
  DFD_REQUIRE(filter == DFD_FILTER_BILINEAR || filter == DFD_FILTER_BICUBIC, DFD_ERR_UNSUPPORTED,
              "resample_coeffs: filter %d not supported (bilinear, bicubic)", filter);
  double scale = (double)in_size / out_size, filterscale = scale;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = (filter == DFD_FILTER_BILINEAR ? 1.0 : 2.0) * filterscale;
  const int ksize = (int)std::ceil(support) * 2 + 1;
  const double ss = 1.0 / filterscale;
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    double ww = 0.0;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    double k[64];
    DFD_REQUIRE(ksize <= 64, DFD_ERR_UNSUPPORTED, "resample_coeffs: downscale factor too large (ksize %d)", ksize);
    for (int x = 0; x < ksize; ++x) k[x] = 0.0;
    for (int x = 0; x < xmax; ++x) {
      const double arg = (x + xmin - center + 0.5) * ss;
      const double w = filter == DFD_FILTER_BILINEAR ? dfd::bilinear_filter(arg) : dfd::bicubic_filter(arg);
      k[x] = w;
      ww += w;
    }
    for (int x = 0; x < xmax; ++x)
      if (ww != 0.0) k[x] /= ww;
    for (int x = 0; x < ksize; ++x)
      kk_host[xx * ksize + x] = k[x] < 0 ? (int)(-0.5 + k[x] * (1 << dfd::kPrecisionBits))
                                         : (int)(0.5 + k[x] * (1 << dfd::kPrecisionBits));
    xmin_host[xx] = xmin;
    count_host[xx] = xmax;
  }
  return DFD_OK;
}

extern "C" DFD_API int64_t dfd_gray256_scratch_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  const int64_t hw = ((int64_t)H * W + 255) / 256 * 256;
  // L, CLAHE output, tile LUTs, horizontally resampled image
  return (int64_t)B * (2 * hw + dfd::kTiles * dfd::kTiles * 256 + (int64_t)H * dfd::kOut);
}

// The source may be a rectangle of a larger image: the crop's rows are row_stride bytes apart and consecutive crops
// image_stride bytes (0 / 0 = dense [B,H,W,3]).  A crop of a resident image is (base + (y0·W_img + x0)·3,
// row_stride = W_img·3): the views of detect_core / the patch grid are produced from ONE upload of the original without a
// copy per view.
extern "C" DFD_API int dfd_gray256(const void* rgb_u8, int64_t row_stride, int64_t image_stride, int B, int H, int W,
                                   int clahe, const int32_t* xmin_w, const int32_t* count_w, const int32_t* kk_w,
                                   int ksize_w, const int32_t* xmin_h, const int32_t* count_h, const int32_t* kk_h,
                                   int ksize_h, void* scratch, float* gray256, void* stream) {
  using namespace dfd;
  if (row_stride == 0) row_stride = (int64_t)W * 3;
  if (image_stride == 0) image_stride = (int64_t)H * row_stride;
  DFD_REQUIRE(row_stride >= (int64_t)W * 3, DFD_ERR_SHAPE, "gray256: row stride smaller than a row");
  // the dense kernel reads 12-byte pixel groups as words: packed images at a 4-byte aligned address only
  const bool dense = row_stride == (int64_t)W * 3 && (B == 1 || image_stride == (int64_t)H * W * 3) && (uintptr_t)rgb_u8 % 4 == 0;
  DFD_REQUIRE(rgb_u8 && scratch && gray256, DFD_ERR_BAD_ARG, "gray256: null pointer");
  DFD_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535 && H <= 65535, DFD_ERR_SHAPE, "gray256: bad shape");
  DFD_REQUIRE(xmin_w && count_w && kk_w && xmin_h && count_h && kk_h, DFD_ERR_BAD_ARG,
              "gray256: resample tables missing");
  DFD_REQUIRE(ksize_w == resample_ksize(W, kOut, DFD_FILTER_BICUBIC) && ksize_h == resample_ksize(H, kOut, DFD_FILTER_BICUBIC),
              DFD_ERR_BAD_ARG,
              "gray256: resample tables were built for another size");
  DFD_REQUIRE((uintptr_t)scratch % 4 == 0, DFD_ERR_BAD_ARG, "gray256: scratch must be 4-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t npix = (int64_t)B * H * W;
  const int64_t hw = ((int64_t)H * W + 255) / 256 * 256;
  uint8_t* L = reinterpret_cast<uint8_t*>(scratch);
  uint8_t* C = L + (int64_t)B * hw;
  uint8_t* luts = C + (int64_t)B * hw;
  uint8_t* rows = luts + (int64_t)B * kTiles * kTiles * 256;
  DFD_REQUIRE((npix + 3) / 4 / 256 + 1 < (1ll << 31), DFD_ERR_SHAPE, "gray256: batch too large");
  // images are packed back to back in L (B*H*W bytes); the per-image stride hw is only used for sizing
  if (dense)
    luma_kernel<<<(unsigned)(((npix + 3) / 4 + 255) / 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(rgb_u8), L, npix);
  else
    luma_strided_kernel<<<dim3((W + 255) / 256, H, B), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(rgb_u8), row_stride,
                                                                    image_stride, L, H, W);
  DFD_LAUNCH_CHECK();
  int launches = 1;
  const uint8_t* src = L;
  if (clahe) {
    const ClaheGeometry g = clahe_geometry(H, W);
    // tiles that divide the image and are whole words wide (384², 224², ...): the warp-per-tile / band kernels; images are packed
    // back to back, so every row start is word aligned when W % 4 == 0
    const bool fast = (W % kTiles == 0) && (H % kTiles == 0) && (g.tw % 4 == 0) && ((uintptr_t)scratch % 8 == 0);
    if (fast) {
      clahe_lut_rows_kernel<<<dim3(kTiles, B), 256, 0, st>>>(L, luts, H, W, g.tw, g.th, g.clip, g.lut_scale);
      DFD_LAUNCH_CHECK();
      clahe_apply_band_kernel<<<dim3(kTiles + 1, B), 256, 0, st>>>(L, luts, C, H, W, g.th, 1.0f / (float)g.tw,
                                                                   1.0f / (float)g.th);
      DFD_LAUNCH_CHECK();
    } else {
      clahe_lut_kernel<<<dim3(kTiles * kTiles, B), 256, 0, st>>>(L, luts, H, W, 1, g.tw, g.th, g.clip, g.lut_scale);
      DFD_LAUNCH_CHECK();
      clahe_apply_kernel<<<dim3((W + 255) / 256, H, B), 256, 0, st>>>(L, luts, C, H, W, 1, 1.0f / (float)g.tw,
                                                                    1.0f / (float)g.th);
      DFD_LAUNCH_CHECK();
    }
    launches += 2;
    src = C;
  }
  // Pillow skips a pass whose size does not change; here the identity tables (count 1, weight 2^22) reproduce the
  // input exactly, so both passes always run
  if (ksize_w <= kTapMax && W % 4 == 0 && (int64_t)kRowsPerCta * W <= 48 * 1024 && (uintptr_t)scratch % 4 == 0)
    resample_rows_fast_kernel<<<dim3((H + kRowsPerCta - 1) / kRowsPerCta, B), kOut, kRowsPerCta * W, st>>>(src, rows, H, W, xmin_w,
                                                                                                            count_w, kk_w, ksize_w);
  else
    resize_rows_kernel<<<dim3(1, H, B), kOut, 0, st>>>(src, W, (int64_t)H * W, rows, H, kOut, 1, xmin_w, count_w, kk_w, ksize_w);
  DFD_LAUNCH_CHECK();
  if (ksize_h <= kTapMax && (uintptr_t)gray256 % 16 == 0)   // float4 stores
    resample_cols_fast_kernel<<<dim3(kOut / 16, B), 256, 0, st>>>(rows, gray256, H, xmin_h, count_h, kk_h, ksize_h);
  else
    resize_cols_kernel<<<dim3(1, kOut, B), kOut, 0, st>>>(rows, gray256, H, kOut, kOut, xmin_h, count_h, kk_h, ksize_h);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(launches + 2, std::memory_order_relaxed);
  return DFD_OK;
}

// OpenCV CLAHE(clipLimit 2.0, tileGridSize 8x8) of every channel of dense u8 images [B, H, W, C] (C = 1 or 3), each channel on
// its own: the `apply_clahe` that precedes Resize in the reference's training preprocess (train_fusion_head_only.py:60-65:
// `for chan in range(3): arr[:, :, chan] = clahe.apply(arr[:, :, chan])`).  Same kernels as the gray256 stage, one plane per
// (image, channel); bit-exact with the library.  scratch: dfd_clahe_scratch_bytes(B, C) bytes (the tile LUTs).  src != dst.
extern "C" DFD_API int64_t dfd_clahe_scratch_bytes(int B, int C) {
  if (B <= 0 || C <= 0) return 0;
  return (int64_t)B * C * dfd::kTiles * dfd::kTiles * 256;
}

extern "C" DFD_API int dfd_clahe_u8(const void* src, int B, int H, int W, int C, void* scratch, void* dst, void* stream) {
  using namespace dfd;
  DFD_REQUIRE(src && dst && scratch, DFD_ERR_BAD_ARG, "clahe: null pointer");
  DFD_REQUIRE(src != dst, DFD_ERR_BAD_ARG, "clahe: in-place operation is not supported (every pixel reads four tile LUTs built from the input)");
  DFD_REQUIRE(B > 0 && H > 0 && W > 0 && (C == 1 || C == 3), DFD_ERR_SHAPE, "clahe: bad shape (B, H, W > 0; C = 1 or 3)");
  DFD_REQUIRE((int64_t)B * C <= 65535 && H <= 65535, DFD_ERR_SHAPE, "clahe: B*C and H must be <= 65535");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const ClaheGeometry g = clahe_geometry(H, W);
  uint8_t* luts = reinterpret_cast<uint8_t*>(scratch);
  clahe_lut_kernel<<<dim3(kTiles * kTiles, B * C), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(src), luts, H, W, C, g.tw,
                                                                g.th, g.clip, g.lut_scale);
  DFD_LAUNCH_CHECK();
  clahe_apply_kernel<<<dim3((W + 255) / 256, H, B * C), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(src), luts,
                                                                     reinterpret_cast<uint8_t*>(dst), H, W, C,
                                                                     1.0f / (float)g.tw, 1.0f / (float)g.th);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(2, std::memory_order_relaxed);
  return DFD_OK;
}

// Pillow Image.resize((OW, OH), BILINEAR | BICUBIC) for batches of same-size 8-bit images, 1 or 3 interleaved channels:
// what torchvision's transforms.Resize does to a PIL image (inference_ai_human_images.py:200-204,
// train_fusion_head_only.py:67-74) — horizontal pass, u8, vertical pass.  scratch: B*H*OW*C bytes.
// The source may be a rectangle of a larger image (strides in bytes; 0 / 0 = dense), see dfd_gray256.
extern "C" DFD_API int dfd_resize_u8(const void* src, int64_t row_stride, int64_t image_stride, int B, int H, int W, int C,
                                     int OH, int OW, const int32_t* xmin_w, const int32_t* count_w, const int32_t* kk_w,
                                     int ksize_w, const int32_t* xmin_h, const int32_t* count_h, const int32_t* kk_h,
                                     int ksize_h, void* scratch, void* dst, void* stream) {
  using namespace dfd;
  if (row_stride == 0) row_stride = (int64_t)W * C;
  if (image_stride == 0) image_stride = (int64_t)H * row_stride;
  DFD_REQUIRE(row_stride >= (int64_t)W * C, DFD_ERR_SHAPE, "resize: row stride smaller than a row");
  DFD_REQUIRE(src && dst && scratch, DFD_ERR_BAD_ARG, "resize: null pointer");
  DFD_REQUIRE(B > 0 && H > 0 && W > 0 && OH > 0 && OW > 0 && (C == 1 || C == 3), DFD_ERR_SHAPE, "resize: bad shape");
  DFD_REQUIRE(B <= 65535 && H <= 65535 && OH <= 65535, DFD_ERR_SHAPE, "resize: B, H, OH must be <= 65535");
  DFD_REQUIRE(xmin_w && count_w && kk_w && xmin_h && count_h && kk_h && ksize_w > 0 && ksize_h > 0, DFD_ERR_BAD_ARG,
              "resize: resample tables missing");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* rows = reinterpret_cast<uint8_t*>(scratch);
  resize_rows_kernel<<<dim3((OW * C + 255) / 256, H, B), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(src), row_stride,
                                                                      image_stride, rows, H, OW, C, xmin_w, count_w, kk_w,
                                                                      ksize_w);
  DFD_LAUNCH_CHECK();
  resize_cols_kernel<<<dim3((OW * C + 255) / 256, OH, B), 256, 0, st>>>(rows, reinterpret_cast<uint8_t*>(dst), H, OH,
                                                                       OW * C, xmin_h, count_h, kk_h, ksize_h);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(2, std::memory_order_relaxed);
  return DFD_OK;
}

// Common device/host helpers for the dfd sm_100a kernels.
//
// PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and a
// few vector load/store helpers.  Everything here is sm_100a-only; there is no fallback path.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dfd.h"

#ifndef DFD_SPIN_TIMEOUT_NS
// A wait that lasts longer than this traps instead of hanging the GPU (a trap kills the context with
// an error the host sees; a hang costs the whole box).
#define DFD_SPIN_TIMEOUT_NS 4000000000ull
#endif

namespace dfd {

constexpr int kNumSMs = 148;

// ---------------------------------------------------------------------------------------------
// host-side error plumbing (thread-local last-error string, int status codes across the C ABI)
// ---------------------------------------------------------------------------------------------
void set_last_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define DFD_CUDA(expr)                                                         \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) return ::dfd::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define DFD_REQUIRE(cond, code, ...)        \
  do {                                      \
    if (!(cond)) {                          \
      ::dfd::set_last_error(__VA_ARGS__);   \
      return (code);                        \
    }                                       \
  } while (0)

#define DFD_LAUNCH_CHECK()                                                       \
  do {                                                                           \
    cudaError_t _e = cudaGetLastError();                                         \
    if (_e != cudaSuccess) return ::dfd::cuda_fail(_e, "kernel launch", __FILE__, __LINE__); \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-(function, DEVICE) setting: remember it per device, so that a
// process that drives several GPUs (or changes device between calls) still launches correctly.  One instance per kernel
// instantiation (a function-local static at the launch site).
struct SmemOptIn {
  unsigned long long done = 0;  // bit d = set on device d (benign race: at worst the attribute is set twice)
};
#if defined(__CUDACC__)
template <typename F>
inline int ensure_dynamic_smem(SmemOptIn& once, F func, int bytes) {
  int dev = 0;
  DFD_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if (once.done & bit) return DFD_OK;
  DFD_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  once.done |= bit;
  return DFD_OK;
}
#endif

// ---------------------------------------------------------------------------------------------
// internal (cross translation unit) entry points; the extern "C" wrappers and the engine call these
// ---------------------------------------------------------------------------------------------
int gemm_bf16_dispatch(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                       int M, int N, int K, const dfd_gemm_epilogue* epi, int force_bn, cudaStream_t st);
int layernorm_bf16(const void* x, int64_t ldx, const void* lo, void* y, int64_t ldy, const float* gamma,
                   const float* beta, int M, int D, float eps, cudaStream_t st);
int patchify(const void* pixels, int pix_format, int B, int Hin, int Win, int S, int P, int resize_mode,
             void* A, int64_t lda, cudaStream_t st);
int attention_dq_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N, int H, int hd,
                      float scale, cudaStream_t st);
int attention_auto_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N, int H, int hd,
                        float scale, cudaStream_t st);
int attention_ws_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N, int H, int hd,
                      float scale, cudaStream_t st);
// probs != NULL: also writes the probe attention probs[b, h, n] (fp32 [B, H, N])
int map_attention_bf16(const void* kv, int64_t ldkv, const float* q, void* out, int64_t ldo, int B, int N,
                       int H, int hd, float scale, float* probs, cudaStream_t st);
int attention_probs(const void* qkv, int64_t ldqkv, int B, int N, int H, int hd, float scale, int per_head, float* out,
                    cudaStream_t st);
// out[b, S, S] = bilinear (align_corners=False) resize of gain·low[b, H, W]
int upsample_bilinear(const float* low, float gain, float* out, int B, int H, int W, int S, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// The same with a suspend-time hint: the hardware parks the thread until the phase completes or the hint (ns) runs out, instead of
// returning after its short default window.  Without it the waiting warps of a warp-specialised kernel (TMA producer, MMA issuer,
// idle epilogue / softmax warps) poll: a third of all instructions the attention kernel issued in round 2 were SYNCS / BRA / the
// loop's bookkeeping (profiles/r02_attention.md), taking issue slots from the working warps of the same scheduler and power from
// a power-capped step.
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
  return t;
}
#ifndef DFD_MBAR_SUSPEND_NS
#define DFD_MBAR_SUSPEND_NS 1000000u   // 1 ms per hardware-suspended attempt
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint64_t t0 = 0;
  while (!mbar_try_wait_hint(bar, parity, DFD_MBAR_SUSPEND_NS)) {
    // (an attempt only fails after its suspend window: this path runs about once per millisecond of waiting)
    const uint64_t now = global_timer_ns();
    if (t0 == 0) t0 = now;
    else if (now - t0 > DFD_SPIN_TIMEOUT_NS) __trap();
  }
}

// ---- proxies / fences ---------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ void sts_zero16(uint32_t smem_addr) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};\n" ::"r"(smem_addr), "r"(0u) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
}

// ---- TMA ----------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load global -> shared, completion on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];\n" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 2-D tiled store shared -> global (bulk async group).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;\n" ::"n"(N) : "memory");
}

// ---- clusters / CTA pairs -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// arrive on the mbarrier at the same shared offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
// 2-CTA TMA load: data lands in THIS CTA's shared memory, the transaction bytes are signalled on the
// mbarrier of the pair's leader (even) CTA (peer bit 24 of the shared::cluster address cleared).
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];\n" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_dst)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(kCols) : "memory");
}
// D[tmem, both CTAs] (+)= A * B with M = 256 split over the CTA pair; issued by ONE thread of the leader CTA.
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                                  uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued pair-MMAs arrive (once) on the mbarrier at this offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}

// ---- tcgen05 / TMEM -----------------------------------------------------------------------------
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
  static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                   smem_u32(smem_dst)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(kCols)
               : "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 tile written by TMA with SWIZZLE_128B:
// rows are 128 B (64 bf16) apart, 8-row groups 1024 B apart (SBO), LBO unused (=1), version 1.
__device__ __forceinline__ uint64_t umma_desc_sw128_kmajor(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address  [0,14)
  d |= static_cast<uint64_t>(1) << 16;                      // LBO (ignored)  [16,30)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // SBO = 1024 B   [32,46)
  d |= static_cast<uint64_t>(1) << 46;                      // version = 1    [46,48)
  d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B   [61,64)
  return d;
}

// Instruction descriptor, kind::f16: bf16 x bf16 -> f32, both operands K-major.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4)                                  // c_format = F32
         | (1u << 7)                                // a_format = BF16
         | (1u << 10)                               // b_format = BF16
         | (static_cast<uint32_t>(n >> 3) << 17)    // n_dim
         | (static_cast<uint32_t>(m >> 4) << 24);   // m_dim
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Make all previously issued MMAs arrive on an mbarrier when they complete.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(
                   smem_u32(bar))
               : "memory");
}

// TMEM -> registers: 32 lanes x 32 consecutive fp32 columns (thread t <- lane base+t).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// 4-D tiled load (used by attention: dims = head-dim, head, token, image), completion on an mbarrier.
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// Generic shared-memory matrix descriptor (version 1 = Blackwell): layout 2 = SWIZZLE_128B, 6 = SWIZZLE_32B.
// K-major operands: SBO = byte distance between 8-row groups.  MN-major operands (tile stored [k][mn] with mn
// contiguous): SBO = byte distance between 8-k groups, LBO = byte distance between swizzle-wide mn blocks.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout_type & 7u) << 61;
  return d;
}
// kind::f16 instruction descriptor with explicit operand majorness (0 = K-major, 1 = MN-major)
__host__ __device__ constexpr uint32_t umma_idesc_bf16_major(int m, int n, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) |
         (static_cast<uint32_t>(b_mn) << 16) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
// D[tmem] (+)= A[tmem] * B[smem]  (A operand read from tensor memory: lane = row, 2 bf16 per 32-bit column)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// registers -> TMEM: 32 lanes x 32 consecutive 32-bit columns (thread t -> lane base+t)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
      "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]),
      "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]),
      "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
      "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;\n" : "=f"(y) : "f"(x));
  return y;
}

// ---- packed fp32 pairs (Blackwell FFMA2 / FADD2 / FMUL2: two fp32 lanes per issue slot) ------------------------
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "mul.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

// ---- misc math / packing ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
// gelu_pytorch_tanh: 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))   (HF modeling_siglip MLP)
__device__ __forceinline__ float gelu_tanh(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  // tanh(u) = 1 - 2 / (1 + exp(2u)); exp via ex2.approx is accurate to ~1e-7 relative here
  float e = __expf(2.0f * u);
  float t = 1.0f - __fdividef(2.0f, 1.0f + e);
  return 0.5f * x * (1.0f + t);
}
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

#endif  // __CUDACC__

}  // namespace dfd

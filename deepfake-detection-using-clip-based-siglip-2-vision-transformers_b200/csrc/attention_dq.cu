// Non-causal attention on tcgen05 + TMEM, two query tiles per CTA ("dq"): the product kernel for the 729..1024-token
// SigLIP sequences.
//
// What round 1 measured (profiles/r01_attention_full.md, r01_ubench_tma.txt, r01_ubench_tc.txt): with one 128-row query tile
// per CTA every K/V tile is fetched from L2 once per 128 query rows; at so400m shapes that is 7.6 TB/s of L2 -> SM traffic
// and the K/V ring, not the tensor pipe (33 % busy) or the MUFU unit, bounded the kernel.  Here
//   * one persistent CTA per SM owns 256 query rows (two 128-row tiles) of an (image, head): each K/V tile is read from
//     L2 once per 256 rows (half the traffic per FLOP), in 128-key boxes (half the TMA instructions per byte);
//   * Q lives in TMEM (bf16 pairs, A operand of S = Q·Kᵀ): an M128 N64 K16 MMA then takes ~42 cycles instead of ~75
//     (the SS form re-reads the 128-row Q operand from shared memory for every key tile);
//   * each query tile has its own softmax warpgroup (one thread per row, no shuffles), its own double-buffered S in
//     TMEM and its own O accumulator, so the two tiles ping-pong on the tensor pipe while both warpgroups keep the MUFU
//     unit busy; P (bf16) aliases S and is the TMEM A operand of O += P·V;
//   * O leaves through a shared-memory staging tile and ONE TMA store per tile (the per-lane 16-byte global stores of the
//     round-1 kernels cost 2.05x the output bytes in SM -> L2 traffic).
//
//   warp 0       TMA loader: next item's Q (prefetched while the current item runs), K/V in 128-key stages (3-deep ring)
//   warps 1, 2   MMA issuers (one elected thread each): S_t,j = Q_t·K_jᵀ, O_t += P_t,j·V_j for query tile t = warp - 1
//   warps 3-6    softmax / output of query tile 0 (one thread per row)
//   warps 7-10   softmax / output of query tile 1
//
// TMEM (512 columns):  S[t][buf] fp32 128x64 at (2t+buf)·64 | O[t] fp32 128x80 at 256+80t | Q[t] bf16x2 128x40 at 416+40t
//
// Reference semantics: HF:modeling_siglip.py:229-249,293-306 (softmax(q·kᵀ/sqrt(hd)) v, fp32 softmax, no mask).
#include "dfd_common.cuh"

#include <atomic>
#include <mutex>

namespace dfd {

extern std::atomic<int64_t> g_launches;

namespace {

constexpr int kQ = 128;          // query rows per tile
constexpr int kKV = 64;          // keys per S tile
constexpr int kStageKeys = 128;  // keys per ring stage (two S tiles)
constexpr int kStages = 3;
constexpr int kThreads = 352;    // loader, 2 MMA warps, 2 x 4 softmax warps
constexpr int kTmemCols = 512;
constexpr int kColO = 256;
constexpr int kColQ = 416;
// kHandoff = pairs of exponentials (of 32 per row and tile) a tile issues before it hands the MUFU turn to the other tile: measured on
// B200 at so400m shapes (64 images): 8 -> 0.253 ms, 16 -> 0.247, 24 -> 0.249, 32 (strict alternation) -> 0.277
constexpr int kHandoff = 16;

// 2^x for a pair on the FMA pipe (x <= ~8): round to the nearest integer with the 1.5·2^23 trick, degree-3 minimax polynomial
// of 2^f on [-0.5, 0.5] (7.5e-5 relative: P is rounded to bf16, 2e-3, right after), exponent added as an integer.  The MUFU
// unit takes 8 cycles per warp-wide EX2 and the softmax warps are what bounds this kernel (scripts/ubench_softmax.cu:
// 10.8 cycles per exponential and scheduler with two warps per scheduler, all on the MUFU unit; 9.0 with every third pair
// here), so a share of the exponentials goes through six packed FMA-pipe instructions per pair instead: every kPoly-th pair
// (every 3rd and all on the MUFU unit measured slower, profiles/r02_attention.md §C).
constexpr int kPoly = 4;
__device__ __forceinline__ float2 poly_exp2x2(float2 x) {
  const float kMagic = 12582912.0f;
  x.x = fmaxf(x.x, -120.0f);
  x.y = fmaxf(x.y, -120.0f);
  const float2 t = fadd2(x, make_float2(kMagic, kMagic));
  const float2 n = fadd2(t, make_float2(-kMagic, -kMagic));
  const float2 f = fadd2(x, make_float2(-n.x, -n.y));
  float2 p = ffma2(f, make_float2(0.05517153f, 0.05517153f), make_float2(0.24261111f, 0.24261111f));
  p = ffma2(p, f, make_float2(0.69326103f, 0.69326103f));
  p = ffma2(p, f, make_float2(0.99992806f, 0.99992806f));
  float2 r;
  r.x = __uint_as_float(__float_as_uint(p.x) + (__float_as_uint(t.x) << 23));
  r.y = __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(t.y) << 23));
  return r;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;\n" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

template <int HD>
struct DqSmem {
  static constexpr bool kTail = (HD % 64) != 0;
  static constexpr int kQMainTile = kQ * 128;                        // 128 rows x 128 B, SWIZZLE_128B
  static constexpr int kQTailTile = kTail ? kQ * 32 : 0;             // 128 rows x 32 B, SWIZZLE_32B
  static constexpr int kQMain = 2 * kQMainTile, kQBytes = kQMain + 2 * kQTailTile;
  static constexpr int kMain = kStageKeys * 128;                     // K or V main box of one stage
  static constexpr int kTailB = kTail ? kStageKeys * 32 : 0;
  static constexpr int kStageBytes = 2 * kMain + 2 * kTailB;         // K main | V main | K tail | V tail
  static constexpr int kOutTile = kQ * HD * 2;                       // output staging of one query tile
  static constexpr int kBarBytes = 256;
  static constexpr int kOffKV = kQBytes;
  static constexpr int kOffOut = kOffKV + kStages * kStageBytes;
  static constexpr int kOffBar = kOffOut + 2 * kOutTile;
  static constexpr int kTotal = kOffBar + kBarBytes + 1024;
  static_assert(kTotal <= 227 * 1024, "shared memory budget");
  static_assert(kQBytes % 1024 == 0 && kStageBytes % 1024 == 0 && kOutTile % 1024 == 0, "swizzle alignment");
};

__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"r"(taddr),
               "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_u4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void bar_sync_named(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
// 4-D tiled store shared -> global (bulk async group); rows past the tensor's extent are clipped by the TMA unit
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];\n" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

template <int HD>
__global__ void __launch_bounds__(kThreads, 1)
attention_dq_kernel(const __grid_constant__ CUtensorMap tmMain, const __grid_constant__ CUtensorMap tmTail,
                    const __grid_constant__ CUtensorMap tmOut, int N, int H, int n_items, float scale_log2) {
  using S = DqSmem<HD>;
  constexpr bool kTail = S::kTail;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sQ = smem;
  uint8_t* sKV = smem + S::kOffKV;
  uint8_t* sOut = smem + S::kOffOut;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kOffBar);
  uint64_t* q_full = bars;                    // TMA: the item's two Q tiles are in shared memory
  uint64_t* q_copied = bars + 1;              // [2] tile t's Q is in TMEM (8 warps)
  uint64_t* kv_full = q_copied + 2;           // [kStages]
  uint64_t* kv_empty = kv_full + kStages;     // [kStages] both MMA warps are done with the stage
  uint64_t* s_full = kv_empty + kStages;      // [2 tiles][2 buffers]
  uint64_t* p_full = s_full + 4;              // [2][2] (8 warps)
  uint64_t* o_done = p_full + 4;              // [2] phase g: the g-th P·V of tile t (of this CTA) has retired
  uint64_t* o_full = o_done + 2;              // [2] phase i: the last P·V of tile t of this CTA's i-th active item has retired
  uint64_t* turn = o_full + 2;                // [2] tile t may start its exponentials (4 warps of the other tile arrive)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(turn + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = (N + kKV - 1) / kKV;                  // S tiles (64 keys) per item
  const int TS = (N + kStageKeys - 1) / kStageKeys;   // ring stages per item
  const int QP = (N + 2 * kQ - 1) / (2 * kQ);         // 256-row query pairs per (image, head)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmMain);
    if (kTail) tma_prefetch_desc(&tmTail);
    tma_prefetch_desc(&tmOut);
    mbar_init(q_full, 1);
    mbar_init(&q_copied[0], 4);
    mbar_init(&q_copied[1], 4);
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 2);
    }
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 4);
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbar_init(&o_done[s], 1);
      mbar_init(&o_full[s], 1);
      mbar_init(&turn[s], 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<kTmemCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------ TMA loader ------------------------------------
    if (elect_one()) {
      uint32_t ku0 = 0, ku1 = 0, ku2 = 0;   // uses of each ring stage so far (stages restart at 0 with every item)
      uint32_t it = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const int qp = item % QP, h = (item / QP) % H, b = item / (QP * H);
        mbar_wait(&q_copied[0], (it & 1u) ^ 1u);  // the previous item's Q tiles have been copied out of shared memory
        mbar_wait(&q_copied[1], (it & 1u) ^ 1u);
        mbar_expect_tx(q_full, S::kQBytes);
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          tma_load_4d(&tmMain, q_full, sQ + t * S::kQMainTile, 0, h, qp * 2 * kQ + t * kQ, b);
          if (kTail)
            tma_load_4d(&tmTail, q_full, sQ + S::kQMain + t * S::kQTailTile, HD - 16, h, qp * 2 * kQ + t * kQ, b);
        }
        int st = 0;
        for (int jj = 0; jj < TS; ++jj) {
          const uint32_t n = st == 0 ? ku0++ : (st == 1 ? ku1++ : ku2++);
          mbar_wait(&kv_empty[st], (n & 1u) ^ 1u);
          mbar_expect_tx(&kv_full[st], S::kStageBytes);
          uint8_t* base = sKV + st * S::kStageBytes;
          tma_load_4d(&tmMain, &kv_full[st], base, 0, H + h, jj * kStageKeys, b);
          tma_load_4d(&tmMain, &kv_full[st], base + S::kMain, 0, 2 * H + h, jj * kStageKeys, b);
          if (kTail) {
            // tail boxes = columns HD-16..HD-1, in bounds (boxes that cross the tensor edge are served slowly); the 8
            // columns they share with the main box meet zeros on the Q side and unread accumulator columns in P·V
            tma_load_4d(&tmTail, &kv_full[st], base + 2 * S::kMain, HD - 16, H + h, jj * kStageKeys, b);
            tma_load_4d(&tmTail, &kv_full[st], base + 2 * S::kMain + S::kTailB, HD - 16, 2 * H + h, jj * kStageKeys, b);
          }
          st = (st + 1 == kStages) ? 0 : st + 1;
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ------------------------------------ MMA issuers ------------------------------------
    // One issuing thread per query tile: with a single thread walking both tiles in a fixed order a late P of one tile
    // held back the other tile's P·V and next S (head-of-line blocking); the tensor pipe itself still runs in issue order.
    if (elect_one()) {
      const int t = warp - 1;
      const uint64_t dK0 = umma_desc(smem_u32(sKV), 16, 1024, 2);
      const uint64_t dV0 = umma_desc(smem_u32(sKV + S::kMain), 16, 1024, 2);  // MN-major, 8-key groups 1024 B apart
      const uint64_t dKt0 = umma_desc(smem_u32(sKV + 2 * S::kMain), 16, 256, 6);
      const uint64_t dVt0 = umma_desc(smem_u32(sKV + 2 * S::kMain + S::kTailB), 16, 256, 6);
      constexpr uint64_t kStageStep = S::kStageBytes >> 4;       // descriptor start addresses count 16-byte units
      constexpr uint64_t kHalfMain = (kKV * 128) >> 4;           // second 64 keys of a stage
      constexpr uint64_t kHalfTail = (kKV * 32) >> 4;
      constexpr uint32_t idesc_qk_full = umma_idesc_bf16_major(kQ, kKV, 0, 0);
      constexpr uint32_t idesc_pv = umma_idesc_bf16_major(kQ, 64, 0, 1);
      constexpr uint32_t idesc_pvt = umma_idesc_bf16_major(kQ, 16, 0, 1);
      const uint32_t tQ = tmem_base + kColQ + static_cast<uint32_t>(40 * t);
      const uint32_t tO = tmem_base + kColO + static_cast<uint32_t>(80 * t);
      uint32_t ku[kStages] = {0, 0, 0};   // kv_full uses per stage      (constant indices after unrolling)
      uint32_t pu[2] = {0, 0};            // p_full uses per S buffer
      // S_j = Q_t · K_jᵀ into S buffer j & 1.  u = j mod 6 (stage = u / 2, half = u % 2) is a constant after unrolling.
      auto issue_qk = [&](int j, int u) {
        const int st = u >> 1, hf = u & 1, sb = u & 1;
        if (hf == 0) {  // first use of the stage by this item
          mbar_wait(&kv_full[st], ku[st]++ & 1u);
          tc_fence_after();
        }
        const uint32_t tS = tmem_base + static_cast<uint32_t>((2 * t + sb) * kKV);
        const uint64_t dK = dK0 + st * kStageStep + hf * kHalfMain;
        const int valid = N - j * kKV;
        const uint32_t idesc_qk = valid >= kKV ? idesc_qk_full : umma_idesc_bf16_major(kQ, (valid + 15) & ~15, 0, 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_ts(tS, tQ + static_cast<uint32_t>(8 * k), dK + static_cast<uint64_t>(2 * k), idesc_qk, k != 0);
        if (kTail) umma_bf16_ts(tS, tQ + 32, dKt0 + st * kStageStep + hf * kHalfTail, idesc_qk, 1u);
        umma_commit(&s_full[2 * t + sb]);
      };
      uint32_t it = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const int qp = item % QP;
        if (qp * 2 * kQ + t * kQ >= N) {
          // (only tile 1) no real query rows: just hand the K/V stages back
          for (int j6 = 0; j6 < TS; j6 += kStages) {
#pragma unroll
            for (int st = 0; st < kStages; ++st) {
              if (j6 + st < TS) {
                mbar_wait(&kv_full[st], ku[st]++ & 1u);
                mbar_arrive(&kv_empty[st]);
              }
            }
          }
          continue;
        }
        mbar_wait(&q_copied[t], it & 1u);
        tc_fence_after();
        issue_qk(0, 0);
        if (T > 1) issue_qk(1, 1);
        for (int j6 = 0; j6 < T; j6 += 2 * kStages) {
#pragma unroll
          for (int u = 0; u < 2 * kStages; ++u) {
            const int j = j6 + u;
            if (j < T) {
              const int st = u >> 1, hf = u & 1, sb = u & 1;
              const uint64_t dV = dV0 + st * kStageStep + hf * kHalfMain;
              const uint64_t dVt = dVt0 + st * kStageStep + hf * kHalfTail;
              const int valid = N - j * kKV;
              // ---- O (+)= P_j · V_j ----  (P written by the tile's softmax warps into the S columns)
              mbar_wait(&p_full[2 * t + sb], pu[sb]++ & 1u);
              tc_fence_after();
              const uint32_t tP = tmem_base + static_cast<uint32_t>((2 * t + sb) * kKV);
              if (valid >= kKV) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                  // 16 keys per step: 16 rows x 128 B (main) / 16 rows x 32 B (tail); P: 8 packed columns per step
                  const uint32_t acc = (kk != 0) ? 1u : (j != 0 ? 1u : 0u);
                  umma_bf16_ts(tO, tP + static_cast<uint32_t>(8 * kk), dV + static_cast<uint64_t>(kk * 128), idesc_pv, acc);
                  if (kTail)
                    umma_bf16_ts(tO + 64, tP + static_cast<uint32_t>(8 * kk), dVt + static_cast<uint64_t>(kk * 32),
                                 idesc_pvt, acc);
                }
              } else {
                const int ksteps = (valid + 15) >> 4;
                for (int kk = 0; kk < ksteps; ++kk) {
                  const uint32_t acc = (j | kk) != 0 ? 1u : 0u;
                  umma_bf16_ts(tO, tP + static_cast<uint32_t>(8 * kk), dV + static_cast<uint64_t>(kk * 128), idesc_pv, acc);
                  if (kTail)
                    umma_bf16_ts(tO + 64, tP + static_cast<uint32_t>(8 * kk), dVt + static_cast<uint64_t>(kk * 32),
                                 idesc_pvt, acc);
                }
              }
              umma_commit(&o_done[t]);
              if (j == T - 1) umma_commit(&o_full[t]);
              // this tile is done with the stage after its second half (or the item's last tile)
              if (hf == 1 || j == T - 1) umma_commit(&kv_empty[st]);
              // the tensor pipe executes in issue order, so S buffer sb / P_j are free for tile j+2 right here
              if (j + 2 < T) issue_qk(j + 2, (u + 2) % (2 * kStages));
            }
          }
        }
      }
    }
  } else {
    // ------------------------------------ softmax / output ------------------------------------
    // 8 warps: query tile t = (warp - 3) / 4, one thread per query row (no shuffles, no shared-memory exchange).
    //
    // Measured on B200 (clock64 traces of this loop, profiles/r02_attention.md): per 64-key tile a warp spends ~90 cycles on
    // the s_full wait, ~35 on the TMEM load, ~220 on the row maximum, ~850 in the exponentials (one warp can issue a
    // MUFU.EX2 only every ~13 cycles; the unit itself takes one per 8) and ~70 on the P store + arrive.  Left alone, the two
    // tiles' warps on a scheduler drift into lock step: both exponentiate (sharing the MUFU unit, ~1050 cycles), then both
    // sit in their TMEM round trips with the unit idle - 1650 cycles per 64-key step.  So the exponential phases take turns:
    // two mbarriers hand a token back and forth between the tiles (a warpgroup ping-pong), each tile's loads, maxima,
    // stores and barrier traffic run under the other tile's exponentials; the token is passed after HALF of a tile's
    // exponentials (kHandoff), so the tail of one tile's MUFU stream is interleaved with the head of the other's: ~1400
    // cycles per step, 635 TFLOP/s at so400m shapes (557 without turns), 298 at base-224 (SDPA: 657 / 281).  (mbarriers, not named
    // barriers: bar.sync / bar.arrive sit in the same basic block as the exponentials and ptxas moved all 64 MUFU.EX2 above
    // the bar.sync - the turn then orders nothing; the wait loop and the one-lane arrive are control flow it cannot cross.)
    // Tried and rejected on the way (all parity-green, all slower): two threads per row (16 softmax warps; maximum
    // exchanged through shared memory or recomputed) with and without turns, 468-584 TFLOP/s; a degree-3 polynomial exp2
    // on the FMA pipe for every 2nd / 3rd / 4th element (the loop is issue bound for ONE warp, extra instructions cost more
    // than the MUFU slots they free); truncating bf16 conversion by PRMT instead of F2FP (no change); fetching S_{j+1}
    // ahead of tile j's exponentials (it only exists once P_{j-1} has gone through the MMA warp: the warp then waits for
    // the tensor pipe instead of exponentiating); round 2: a speculative tile that takes the exponentials against the current
    // reference maximum without waiting for the row maximum (tracked on the side with FMNMX3, tile redone if it moved) and
    // overlaps the second half of the TMEM load with the first half's exponentials — bit-identical, 612-640 against 665 TFLOP/s:
    // the maximum pass is not on the critical path, the two warps of a scheduler are bound by their own instruction streams
    // (scripts/ubench_softmax.cu: 1230 cycles per 64-key step for two warps with no MMA or TMEM wait at all).
    const int sw = warp - 3;
    const int t = sw >> 2;                    // query tile of this warp
    const int quad = warp & 3;                // TMEM lane quadrant this warp may access
    const int row = quad * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t tO = tmem_base + lane_off + kColO + static_cast<uint32_t>(80 * t);
    const uint32_t tQ = tmem_base + lane_off + kColQ + static_cast<uint32_t>(40 * t);
    constexpr int kOChunks = (HD + 15) / 16;  // 16-column chunks of O
    const uint32_t q_row = smem_u32(sQ + t * S::kQMainTile) + static_cast<uint32_t>(row * 128);
    const uint32_t q_tail = smem_u32(sQ + S::kQMain + t * S::kQTailTile) + static_cast<uint32_t>(row * 32);
    uint8_t* out_tile = sOut + t * S::kOutTile;
    const uint32_t out_row = smem_u32(out_tile) + static_cast<uint32_t>(row * HD * 2);
    const bool store_thread = (sw & 3) == 0 && lane == 0;   // issues (and waits for) the tile's TMA stores
    uint32_t turns = 0;                                     // turns this tile has taken (phase of turn[t])
    // Q row of item `it_q`: shared memory (TMA, swizzled) -> registers -> TMEM as bf16 pairs
    auto copy_q = [&](uint32_t it_q) {
      mbar_wait(q_full, it_q & 1u);
      uint32_t qw[32];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint4 v = lds_u4(q_row + static_cast<uint32_t>((c ^ (row & 7)) << 4));
        qw[4 * c] = v.x; qw[4 * c + 1] = v.y; qw[4 * c + 2] = v.z; qw[4 * c + 3] = v.w;
      }
      tmem_st_32x32b_x32(tQ, qw);
      if (kTail) {
        // tail k-step = columns 56..71; 56..63 already went through the main box: Q contributes zeros there
        uint32_t t8[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        const uint4 v = lds_u4(q_tail + static_cast<uint32_t>((1 ^ ((row >> 2) & 1)) << 4));
        t8[4] = v.x; t8[5] = v.y; t8[6] = v.z; t8[7] = v.w;
        tmem_st_32x32b_x8(tQ + 32, t8);
      }
      tmem_st_wait();
      // generic-proxy reads of the Q tile precede its TMA refill: proxy fence before the release (see gemm_tcgen05.cu)
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&q_copied[t]);
    };
    uint32_t su0 = 0, su1 = 0;   // s_full uses per S buffer
    uint32_t g = 0, it = 0;      // running count of this tile's P·V products (o_done phases), item count
    uint32_t act_items = 0;      // items in which this tile was active (o_full phases)
    if (t == 1 && lane == 0) mbar_arrive(&turn[0]);   // tile 0 takes the first turn
    if (blockIdx.x < n_items) copy_q(0);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int qp = item % QP, h = (item / QP) % H, b = item / (QP * H);
      const int row0 = qp * 2 * kQ + t * kQ;   // first query row of this tile
      const bool has_next = item + (int)gridDim.x < n_items;
      if (row0 >= N) {  // (only tile 1) nothing to do for this item; keep the turn-taking and the Q hand-shake going
        // (turns first: the next item's Q only arrives after the loader has placed all of THIS item's K/V stages, and
        //  those drain only as tile 0 advances - which needs its turns)
        for (int j = 0; j < T; ++j) {
          mbar_wait(&turn[t], turns++ & 1u);
          __syncwarp();
          if (lane == 0) mbar_arrive(&turn[t ^ 1]);
        }
        if (has_next) copy_q(it + 1);
        continue;
      }
      float m = -INFINITY, l = 0.f;             // m is kept in log2 units (already multiplied by scale_log2)
      for (int j = 0; j < T; ++j, ++g) {
        const int sb = j & 1;
        const int valid = min(kKV, N - j * kKV);
        const uint32_t tS = tmem_base + lane_off + static_cast<uint32_t>((2 * t + sb) * kKV);
        const uint32_t par = sb ? su1 : su0;
        if (sb) ++su1; else ++su0;
        mbar_wait(&s_full[2 * t + sb], par & 1u);
        tc_fence_after();
        uint32_t s[64];
        tmem_ld_32x32b_x32(tS, *reinterpret_cast<uint32_t(*)[32]>(&s[0]));
        tmem_ld_32x32b_x32(tS + 32, *reinterpret_cast<uint32_t(*)[32]>(&s[32]));
        tmem_ld_wait();
        if (valid < kKV) {  // last tile: keys past the sequence end (zero-filled K rows) never win
#pragma unroll
          for (int c = 0; c < 64; ++c)
            if (c >= valid) s[c] = __float_as_uint(-INFINITY);
        }
        // four independent chains of three-input maxima (FMNMX3: 32 instructions instead of 63)
        float mx4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c)
          mx4[c] = fmax3(__uint_as_float(s[c]), __uint_as_float(s[4 + c]), __uint_as_float(s[8 + c]));
#pragma unroll
        for (int c = 12; c < 60; c += 8)
#pragma unroll
          for (int k = 0; k < 4; ++k) mx4[k] = fmax3(mx4[k], __uint_as_float(s[c + k]), __uint_as_float(s[c + 4 + k]));
#pragma unroll
        for (int k = 0; k < 4; ++k) mx4[k] = fmaxf(mx4[k], __uint_as_float(s[60 + k]));
        float mx = fmaxf(fmax3(mx4[0], mx4[1], mx4[2]), mx4[3]);
        mx *= scale_log2;  // scale > 0
        // lazy rescale: keep the old reference max unless the new one is more than 2^8 larger
        const float m_new = (mx > m + 8.0f) ? mx : m;
        const bool moved = m_new != m;
        const float alpha = (j == 0) ? 0.f : fast_exp2(m - m_new);
        if (j > 0 && __any_sync(0xffffffffu, moved)) {
          mbar_wait(&o_done[t], (g - 1) & 1u);  // the previous P·V has retired: O is stable
          tc_fence_after();
#pragma unroll
          for (int c = 0; c < kOChunks; ++c) {
            uint32_t o[16];
            tmem_ld_32x32b_x16(tO + static_cast<uint32_t>(16 * c), o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_32x32b_x16(tO + static_cast<uint32_t>(16 * c), o);
          }
        }
        m = m_new;
        float2 sum4[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
        const float2 sc2 = make_float2(scale_log2, scale_log2), nm2 = make_float2(-m, -m);
        mbar_wait(&turn[t], turns++ & 1u);      // ---- this tile's turn on the MUFU unit ----
        // packed FFMA2 / FADD2 around the exponentials; every kPoly-th pair is computed on the FMA pipe instead
        auto exps = [&](int c) {
          const float2 x = ffma2(make_float2(__uint_as_float(s[2 * c]), __uint_as_float(s[2 * c + 1])), sc2, nm2);
          float2 p;
          if (c % kPoly == kPoly - 1) p = poly_exp2x2(x);
          else p = make_float2(fast_exp2(x.x), fast_exp2(x.y));
          sum4[c & 3] = fadd2(sum4[c & 3], p);
          s[c] = pack_bf16x2(p.x, p.y);  // in place: s[2c], s[2c+1] (indices >= c) are consumed first
        };
#pragma unroll
        for (int c = 0; c < kHandoff; ++c) exps(c);
        // ---- hand the MUFU unit to the other tile after kHandoff of the 32 pairs: its first exponentials then fill the
        // gaps of this warp's last ones (one warp cannot saturate the unit).  The arrive is predicated on a partial row sum
        // (never negative; ptxas cannot know): a data dependence on the exponentials before it, otherwise the predicated
        // arrive is scheduled ahead of most of them
        const float2 pa = fadd2(fadd2(sum4[0], sum4[1]), fadd2(sum4[2], sum4[3]));
        __syncwarp();
        if (lane == 0 && pa.x + pa.y >= 0.f) mbar_arrive(&turn[t ^ 1]);
        if (valid > 2 * kHandoff) {
#pragma unroll
          for (int c = kHandoff; c < 32; ++c) exps(c);
        } else {
          // short last tile (so400m: 25 of 64 keys): the rest of the row is all padding, P = 0 without exponentials
#pragma unroll
          for (int c = kHandoff; c < 32; ++c) s[c] = 0u;
        }
        const float2 sa = fadd2(fadd2(sum4[0], sum4[1]), fadd2(sum4[2], sum4[3]));
        const float lsum = sa.x + sa.y;
        l = l * alpha + lsum;
        tmem_st_32x32b_x32(tS, *reinterpret_cast<const uint32_t(*)[32]>(&s[0]));   // P (bf16 pairs) aliases S
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[2 * t + sb]);
      }
      // every Q_t·Kᵀ of this item has retired (its last S tile has been consumed): the next item's Q may replace it in
      // TMEM now, so that the MMA warp can start the next item's S tiles while this item's output is written
      if (has_next) copy_q(it + 1);
      // ---- O / l -> bf16 -> staging tile -> one TMA store ----
      mbar_wait(&o_full[t], act_items++ & 1u);
      tc_fence_after();
      if (store_thread) tma_store_wait_read<0>();   // the previous store of this tile has finished reading the staging tile
      bar_sync_named(1 + t, 128);
      const float inv = 1.0f / l;
#pragma unroll
      for (int c = 0; c < kOChunks; ++c) {
        uint32_t o[16];
        tmem_ld_32x32b_x16(tO + static_cast<uint32_t>(16 * c), o);
        tmem_ld_wait();
        if (kTail && c == kOChunks - 1) {  // tail accumulator = columns 56..71: its upper half is columns 64..71
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] = o[8 + i];
        }
        uint4 lo, hi;
        lo.x = pack_bf16x2(__uint_as_float(o[0]) * inv, __uint_as_float(o[1]) * inv);
        lo.y = pack_bf16x2(__uint_as_float(o[2]) * inv, __uint_as_float(o[3]) * inv);
        lo.z = pack_bf16x2(__uint_as_float(o[4]) * inv, __uint_as_float(o[5]) * inv);
        lo.w = pack_bf16x2(__uint_as_float(o[6]) * inv, __uint_as_float(o[7]) * inv);
        hi.x = pack_bf16x2(__uint_as_float(o[8]) * inv, __uint_as_float(o[9]) * inv);
        hi.y = pack_bf16x2(__uint_as_float(o[10]) * inv, __uint_as_float(o[11]) * inv);
        hi.z = pack_bf16x2(__uint_as_float(o[12]) * inv, __uint_as_float(o[13]) * inv);
        hi.w = pack_bf16x2(__uint_as_float(o[14]) * inv, __uint_as_float(o[15]) * inv);
        if (HD == 64) {   // 128-byte rows: SWIZZLE_128B staging (16-byte chunk index XOR row mod 8), conflict free
          sts_u4(out_row + static_cast<uint32_t>(((2 * c) ^ (row & 7)) << 4), lo);
          sts_u4(out_row + static_cast<uint32_t>(((2 * c + 1) ^ (row & 7)) << 4), hi);
        } else {          // 144-byte rows, no swizzle: consecutive rows are 9 chunks apart, conflict free as they are
          sts_u4(out_row + static_cast<uint32_t>(32 * c), lo);
          if (16 * c + 8 < HD) sts_u4(out_row + static_cast<uint32_t>(32 * c + 16), hi);
        }
      }
      fence_proxy_async_smem();
      // order this item's TMEM reads before the p_full arrive that lets the next item's first P·V overwrite O
      tc_fence_before();
      bar_sync_named(1 + t, 128);
      if (store_thread) {
        tma_store_4d(&tmOut, out_tile, 0, h, row0, b);   // rows >= N are clipped
        tma_store_commit();
      }
    }
    if (store_thread) tma_store_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled dq_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

// [B*N, ld] bf16 viewed as (hd, heads, N, B); box = box_cols x 1 x box_rows x 1
int make_tmap_heads(CUtensorMap* out, const void* base, int hd, int heads, int N, int B, int64_t ld, int box_cols,
                    int box_rows, CUtensorMapSwizzle sw, bool store) {
  PFN_encodeTiled fn = dq_encode_fn();
  DFD_REQUIRE(fn != nullptr, DFD_ERR_NO_DEVICE, "cuTensorMapEncodeTiled unavailable (no CUDA driver on this host)");
  cuuint64_t gdim[4] = {(cuuint64_t)hd, (cuuint64_t)heads, (cuuint64_t)N, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)hd * 2, (cuuint64_t)ld * 2, (cuuint64_t)N * (cuuint64_t)ld * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_cols, 1, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  store ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DFD_REQUIRE(r == CUDA_SUCCESS, DFD_ERR_CUDA, "cuTensorMapEncodeTiled(heads 4-D) failed (%d)", (int)r);
  return DFD_OK;
}

}  // namespace

// shared with attention_ws.cu: qkv [B*N, ld] viewed as (hd, 3H, N, B), box = box_cols x 1 x box_rows x 1
int make_tmap_qkv_4d(CUtensorMap* out, const void* base, int hd, int heads3, int N, int B, int64_t ld, int box_cols,
                     int box_rows, int swizzle32) {
  return make_tmap_heads(out, base, hd, heads3, N, B, ld, box_cols, box_rows,
                         swizzle32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B, false);
}

int attention_dq_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N, int H, int hd,
                      float scale, cudaStream_t st) {
  DFD_REQUIRE(qkv && out, DFD_ERR_BAD_ARG, "attention: null pointer");
  DFD_REQUIRE(B > 0 && N > 0 && H > 0, DFD_ERR_SHAPE, "attention: B, N, H must be positive");
  DFD_REQUIRE(hd == 64 || hd == 72, DFD_ERR_UNSUPPORTED, "attention: head dim %d not supported (64, 72)", hd);
  DFD_REQUIRE(ldqkv % 8 == 0 && ldqkv >= 3 * H * hd && ldo % 8 == 0 && ldo >= H * hd, DFD_ERR_SHAPE,
              "attention: bad leading dimensions");
  DFD_REQUIRE(((uintptr_t)qkv % 16 == 0) && ((uintptr_t)out % 16 == 0), DFD_ERR_BAD_ARG,
              "attention: pointers must be 16-byte aligned");
  const int64_t items64 = (int64_t)((N + 2 * kQ - 1) / (2 * kQ)) * H * B;
  DFD_REQUIRE(items64 < (1ll << 31), DFD_ERR_SHAPE, "attention: too many work items");
  CUtensorMap tmMain, tmTail, tmOut;
  int rc = make_tmap_heads(&tmMain, qkv, hd, 3 * H, N, B, ldqkv, 64, kStageKeys, CU_TENSOR_MAP_SWIZZLE_128B, false);
  if (rc != DFD_OK) return rc;
  tmTail = tmMain;
  if (hd == 72) {
    rc = make_tmap_heads(&tmTail, qkv, hd, 3 * H, N, B, ldqkv, 16, kStageKeys, CU_TENSOR_MAP_SWIZZLE_32B, false);
    if (rc != DFD_OK) return rc;
  }
  rc = make_tmap_heads(&tmOut, out, hd, H, N, B, ldo, hd, kQ,
                       hd == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, true);
  if (rc != DFD_OK) return rc;
  const float scale_log2 = scale * 1.4426950408889634f;
  const int n_items = (int)items64;
  const int grid = n_items < kNumSMs ? n_items : kNumSMs;
  static SmemOptIn smem_once[2];
#define DFD_DQ_LAUNCH(HD_)                                                                                                  \
  do {                                                                                                                      \
    if (int rc2 = ensure_dynamic_smem(smem_once[HD_ == 64 ? 0 : 1], attention_dq_kernel<HD_>, DqSmem<HD_>::kTotal))         \
      return rc2;                                                                                                           \
    attention_dq_kernel<HD_><<<grid, kThreads, DqSmem<HD_>::kTotal, st>>>(tmMain, tmTail, tmOut, N, H, n_items, scale_log2); \
  } while (0)
  if (hd == 64) DFD_DQ_LAUNCH(64); else DFD_DQ_LAUNCH(72);
#undef DFD_DQ_LAUNCH
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

}  // namespace dfd

namespace dfd {

// Product dispatch.  Measured on B200 (scripts/kbench.py attn, profiles/r02_kbench_attention.txt): the dual-query-tile
// kernel is ahead from the 196-token sequences of base-224 up (298 vs 232 TFLOP/s there, 635 vs 505 at 729 tokens);
// sequences that do not even fill one 128-row query tile keep the persistent single-tile kernel (two CTAs per SM).
int attention_auto_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N, int H, int hd,
                        float scale, cudaStream_t st) {
  if (N <= 128) return attention_ws_bf16(qkv, ldqkv, out, ldo, B, N, H, hd, scale, st);
  return attention_dq_bf16(qkv, ldqkv, out, ldo, B, N, H, hd, scale, st);
}

}  // namespace dfd

extern "C" DFD_API int dfd_attention_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B,
                                          int N, int H, int hd, float scale, void* stream) {
  return dfd::attention_auto_bf16(qkv, ldqkv, out, ldo, B, N, H, hd, scale, reinterpret_cast<cudaStream_t>(stream));
}

// Test / A-B hook: impl 2 = persistent single-tile kernel (attention_ws.cu), 5 = dual-query-tile kernel (this file),
// for any sequence length.
extern "C" DFD_API int dfd_attention_bf16_impl(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N,
                                               int H, int hd, float scale, int impl, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (impl == 2) return dfd::attention_ws_bf16(qkv, ldqkv, out, ldo, B, N, H, hd, scale, st);
  if (impl == 5) return dfd::attention_dq_bf16(qkv, ldqkv, out, ldo, B, N, H, hd, scale, st);
  dfd::set_last_error("attention: impl must be 2 (single-tile persistent) or 5 (dual-query-tile)");
  return DFD_ERR_BAD_ARG;
}

// Persistent, warp-specialised bf16 GEMM for sm_100a:  C[M,N] = epi(A[M,K] · W[N,K]ᵀ)
//
//   warp 0      TMA producer   (cp.async.bulk.tensor, SWIZZLE_128B, kStages-deep mbarrier ring)
//   warp 1      MMA issuer     (one thread issues tcgen05.mma cta_group::1 kind::f16, M=128, N=BN, K=16;
//                               accumulators live in TMEM, two accumulator stages)
//   warps 2..5  epilogue       (tcgen05.ld 32x32b → registers → fused epilogue → bf16 global stores)
//
// Replaces the cuBLAS/cuDNN calls behind nn.Linear / nn.Conv2d in the reference's backbone
// (HF:modeling_siglip.py:178,285-287,308,324-326; SURVEY.md §2.2 K2,K4,K6,K7,K8,K9).
#include "dfd_common.cuh"

#include <atomic>
#include <mutex>

namespace dfd {

extern std::atomic<int64_t> g_launches;
static std::atomic<int> g_last_variant{0};  // BN + 1000·CG + 10000·RES + 100000·EPI of the last GEMM launch (tests)
static std::atomic<int64_t> g_variant_launches[3 * 2 * 2 * 8];  // launches per instantiation since load (tests)
static int variant_slot(int bn, int cg, int res, int epi) {
  const int b = bn == 256 ? 2 : (bn == 192 ? 1 : 0);
  return ((b * 2 + (cg - 1)) * 2 + res) * 8 + epi;
}

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int kEpiWarps = 8;                       // two groups of 4 warps (one warp per TMEM lane quadrant)
constexpr int kGemmThreads = (3 + kEpiWarps) * 32;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue, warp 10 residual TMA
constexpr int kResSlotsMax = 4;                     // residual ring: 2 epilogue groups x up to 2 chunks in flight
constexpr int kChunkN = 64;                         // epilogue / TMA-store granularity along N
constexpr int kStageCBytes = BM * kChunkN * 2;      // 16 KB staging tile per epilogue group

struct EpiArgs {
  const float* bias;
  int act;
  const float* pos;
  int pos_rows;
  const __nv_bfloat16* residual;
  int64_t ldr;
  const float* ln_rowstats;
  const float* ln_colsum;
  float ln_inv_dim;
  float ln_eps;
  float* stats_out;
  int residual_op;  // 0: v += residual, 1: v *= residual
  int ln_parts;     // ln_rowstats holds this many partial (Σx, Σx²) pairs per row: [ln_parts][M][2]
  __nv_bfloat16* lo;  // low half of a two-bf16 ("hi + lo") residual stream, tiled (see the epilogue): read with the residual,
                      // written with C
};

// CG = CTAs per MMA (1, or 2 = cta_group::2: a 256 x BN tile shared by an SM pair, each CTA staging its own
// 128 rows of A and HALF of the B tile, which roughly halves shared-memory traffic per MMA)
// RES = the epilogue adds a bf16 residual tile; it is prefetched chunk by chunk with TMA into its own ring.
// Persistent schedule (shared by the kernel and by the host-side dfd_gemm_schedule, which tests/test_abi_cpu.py uses to check
// that every tile is taken exactly once).  In round r the U units (CTAs / CTA pairs) take the tiles [r U, (r + 1) U) in N-fastest
// order, so the units working at the same time share A row blocks through L2.  Within a round the assignment is rotated by
// r * rot: with a fixed assignment unit u would only ever see the n-tiles (u + r U) mod num_n — 74 units and 14 n-tiles: odd units
// alone get the half-width tail tile, run ahead of their row-block peers and turn the shared A reads into DRAM re-reads.
// rot = the smallest shift for which a unit's n-tile index advances by a step coprime to num_n, i.e. for which every unit cycles
// through ALL n-tiles (74 units: 14 n-tiles -> 1, 5 n-tiles -> 0; a shift of 1 would pin each unit to one n-tile there).
__host__ __device__ inline int sched_rotation(int units, int num_n) {
  for (int rot = 0; rot < num_n; ++rot) {
    int a = (units + rot) % num_n, b = num_n;
    while (b) { const int t = a % b; a = b; b = t; }
    if (a == 1) return rot;
  }
  return 0;
}
__host__ __device__ inline int sched_tile(int round, int unit, int units, int rot) {
  return round * units + (unit + round * rot) % units;
}

template <int BN, int CG, int RES>
struct GemmSmem {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (BN / CG) * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // residual chunks in flight per epilogue group; group g owns slots [g kResDepth, (g + 1) kResDepth).  Measured on
  // B200 (so400m out-projection, K = 1152): depth 2 costs one of the five 32 KB pipeline stages and is 9 % SLOWER than
  // depth 1 (1090 vs 1197 TFLOP/s) — the mainloop needs the stages more than the epilogue needs the prefetch.
  static constexpr int kResDepth = 1;
  static constexpr int kResBytes = RES ? 2 * kResDepth * kStageCBytes : 0;
  static constexpr int kColTabBytes = 2 * 2 * kChunkN * 4;  // per epilogue group: 64 LayerNorm column sums + 64 biases
  static constexpr int kAvail = 227 * 1024 - 2 * kStageCBytes - kResBytes - 256 - kColTabBytes - 1024;
  static constexpr int kStages = kAvail / kStageBytes > 8 ? 8 : kAvail / kStageBytes;
  static constexpr int kTileBytes = kStages * kStageBytes;
  static constexpr int kCBytes = 2 * kStageCBytes + kResBytes;  // C staging (2) then the residual ring
  static constexpr int kBarBytes = 256;
  static constexpr int kTotal = kTileBytes + kCBytes + kBarBytes + kColTabBytes + 1024;  // +1024 alignment slack
  static constexpr int kTmemCols = (2 * BN <= 256) ? 256 : 512;
  static_assert(kTotal <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
// gelu_pytorch_tanh with the single-MUFU tanh (abs error ~5e-4 of a value that is rounded to bf16 anyway),
// for a pair: 0.5 x (1 + tanh(x (k0 + k0 k1 x²))) in five packed FP instructions + two MUFU.TANH
__device__ __forceinline__ float2 gelu_tanh_fast2(float2 x) {
  const float k0 = 0.7978845608028654f, k01 = 0.7978845608028654f * 0.044715f;
  const float2 w = ffma2(fmul2(x, x), make_float2(k01, k01), make_float2(k0, k0));
  const float2 u = fmul2(x, w);
  float2 t;
  asm("tanh.approx.f32 %0, %1;\n" : "=f"(t.x) : "f"(u.x));
  asm("tanh.approx.f32 %0, %1;\n" : "=f"(t.y) : "f"(u.y));
  const float2 hx = fmul2(x, make_float2(0.5f, 0.5f));
  return ffma2(hx, t, hx);
}

__device__ __noinline__ float2 act_rare(float2 v, int act) {
  if (act == 2) return make_float2(gelu_erf(v.x), gelu_erf(v.y));   // exact erf GELU (nn.GELU() default)
  return make_float2(1.f / (1.f + __expf(-v.x)), 1.f / (1.f + __expf(-v.y)));  // act == 3: sigmoid
}

// EPI selects a compile-time epilogue: 0 = generic (every fused option is a run-time flag), otherwise exactly one of the
// combinations the backbone launches, with everything else compiled out:
//   1 LayerNorm fold + bias (qkv)           2 LayerNorm fold + bias + tanh-GELU (fc1)      5 bias        6 bias + tanh-GELU
//   3 bias + residual add + row statistics (out-projection / fc2 under fuse_ln)            4 bias + residual add
//   7 as 3 on a two-bf16 residual stream: v = acc + bias + hi + lo, C = hi' = bf16(v), lo' = bf16(v - hi') (row statistics of
//     hi', the operand the next LayerNorm-folded GEMM reads, only if stats_out is given)
// The generic epilogue if-converts its run-time options into predicated code: ~880 issued instructions per 64-column chunk
// per warp for bias + residual (clock64 trace: 3600 of the 4900 cycles of a chunk), which made every GEMM with a short K
// loop epilogue bound (K = 768 / 1152 out-projections at 45-75 % of the tensor peak).
template <int BN, int CG, int RES, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA,
                         const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmC,
                         const __grid_constant__ CUtensorMap tmR, int M, int N, int K, EpiArgs epi) {
  using S = GemmSmem<BN, CG, RES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);

  uint8_t* smem_c = smem + S::kTileBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::kTileBytes + S::kCBytes);
  uint64_t* empty_bar = full_bar + S::kStages;
  uint64_t* tfull_bar = empty_bar + S::kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* rfull_bar = tempty_bar + 2;
  uint64_t* rempty_bar = rfull_bar + kResSlotsMax;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty_bar + kResSlotsMax);
  uint8_t* smem_r = smem_c + 2 * kStageCBytes;
  float* col_tab = reinterpret_cast<float*>(smem + S::kTileBytes + S::kCBytes + S::kBarBytes);  // [group][colsum 64 | bias 64]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
  const bool is_leader = cta_rank == 0;
  const int num_m = (M + BM * CG - 1) / (BM * CG);
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + BK - 1) / BK;
  const int first_tile = blockIdx.x / CG;   // this unit's index
  const int tile_step = gridDim.x / CG;     // units
  const int rot = sched_rotation(tile_step, num_n);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
#pragma unroll
    for (int s = 0; s < S::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], kEpiWarps * CG);
    }
#pragma unroll
    for (int r = 0; r < kResSlotsMax; ++r) {
      mbar_init(&rfull_bar[r], 1);
      mbar_init(&rempty_bar[r], 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    if (CG == 2) tmem_alloc_pair<S::kTmemCols>(tmem_slot);
    else tmem_alloc<S::kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all();  // peer barriers are initialised before anything signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------- TMA producer -------------------------------
    // elect.sync rather than `lane == 0`: ptxas then knows exactly one thread is active and emits the TMA / MMA /
    // commit instructions bare; behind `lane == 0` every one of them sits in an ELECT..BRA.U.ANY loop that costs
    // ~100 cycles per issue (scripts/ubench_tc.cu) — as much as a 128x256x16 MMA takes to execute.
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int rr = 0; rr * tile_step < num_tiles; ++rr) {
        const int tile = sched_tile(rr, first_tile, tile_step, rot);  // rotated within the round, see sched_rotation
        if (tile >= num_tiles) break;  // only in the last, partial round
        // N fastest: CTAs working at the same time share A row blocks through L2; the weights (<= 10 MB)
        // stay L2 resident for the whole GEMM
        const int m0 = (tile / num_n) * (BM * CG) + (int)cta_rank * BM;
        // the last N tile is only as wide as it has to be (multiple of 16): a pair MMA of width n_eff takes n_eff / 2
        // columns of B from each CTA, so CTA 1's rows start at n_eff / 2, not BN / 2
        const int nt0 = (tile % num_n) * BN;
        const int n_eff = min(BN, (N - nt0 + 15) & ~15);
        const int n0 = nt0 + (int)cta_rank * (n_eff / CG) * (CG - 1);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          uint8_t* sa = smem + stage * S::kStageBytes;
          uint8_t* sb = sa + S::kABytes;
          if (CG == 2) {
            // the leader's barrier collects the bytes of both CTAs
            if (is_leader) mbar_expect_tx(&full_bar[stage], 2 * S::kStageBytes);
            tma_load_2d_pair(&tmA, &full_bar[stage], sa, kb * BK, m0);
            tma_load_2d_pair(&tmB, &full_bar[stage], sb, kb * BK, n0);
          } else {
            mbar_expect_tx(&full_bar[stage], S::kStageBytes);
            tma_load_2d(&tmA, &full_bar[stage], sa, kb * BK, m0);
            tma_load_2d(&tmB, &full_bar[stage], sb, kb * BK, n0);
          }
          if (++stage == S::kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer ---------------------------------
    if (is_leader && elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int rr = 0; rr * tile_step < num_tiles; ++rr) {
        const int tile = sched_tile(rr, first_tile, tile_step, rot);  // rotated within the round, see sched_rotation
        if (tile >= num_tiles) break;  // only in the last, partial round
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN);
        // N tail: an MMA of width n_eff (multiple of 16) instead of BN — a half-empty 256-wide tile (N = 1152: the fifth
        // one) then costs half, not all, of a full tile's tensor-pipe time
        const int n_eff = min(BN, (N - (tile % num_n) * BN + 15) & ~15);
        const uint32_t idesc = umma_idesc_bf16(BM * CG, n_eff);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * S::kStageBytes);
          const uint64_t da = umma_desc_sw128_kmajor(sa);
          const uint64_t db = umma_desc_sw128_kmajor(sa + S::kABytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 bf16 = 32 B along K inside the 128-byte swizzle row: +2 in 16-byte units
            if (CG == 2)
              umma_bf16_ss_pair(d_tmem, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k),
                                idesc, (kb | k) != 0 ? 1u : 0u);
            else
              umma_bf16_ss(d_tmem, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k),
                           idesc, (kb | k) != 0 ? 1u : 0u);
          }
          // frees this smem stage (in both CTAs) when the MMAs retire
          if (CG == 2) umma_commit_pair(&empty_bar[stage]);
          else umma_commit(&empty_bar[stage]);
          if (++stage == S::kStages) { stage = 0; phase ^= 1u; }
        }
        // accumulator complete -> epilogue warps (of both CTAs)
        if (CG == 2) umma_commit_pair(&tfull_bar[acc]);
        else umma_commit(&tfull_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp == 2 + kEpiWarps) {
    // ------------------------------- residual producer --------------------------
    if (RES && elect_one()) {
      tma_prefetch_desc(&tmR);
      // epilogue group g (chunks c ≡ g mod 2) owns a ring of kResDepth slots: each slot has exactly one consumer, so
      // the parity waits stay one phase apart whatever the number of chunks per tile (a shared ring broke for odd
      // counts)
      uint32_t uses[2] = {0, 0};
      for (int rr = 0; rr * tile_step < num_tiles; ++rr) {
        const int tile = sched_tile(rr, first_tile, tile_step, rot);  // rotated within the round, see sched_rotation
        if (tile >= num_tiles) break;  // only in the last, partial round
        const int m0 = (tile / num_n) * (BM * CG) + (int)cta_rank * BM;
        const int n0 = (tile % num_n) * BN;
        const int nvalid = min(BN / kChunkN, (N - n0 + kChunkN - 1) / kChunkN);
        for (int c = 0; c < nvalid; ++c) {
          const uint32_t u = uses[c & 1]++;
          const int slot = (c & 1) * S::kResDepth + (int)(u % S::kResDepth);
          mbar_wait(&rempty_bar[slot], ((u / S::kResDepth) & 1u) ^ 1u);
          mbar_expect_tx(&rfull_bar[slot], kStageCBytes);
          tma_load_2d(&tmR, &rfull_bar[slot], smem_r + slot * kStageCBytes, n0 + c * kChunkN, m0);
        }
      }
    }
  } else {
    // ------------------------------- epilogue -----------------------------------
    // 8 warps = 2 groups; group g takes the 64-column chunks c ≡ g (mod 2) of every tile.  A chunk goes
    // TMEM -> registers -> fused math -> bf16 -> 128B-swizzled staging tile -> one TMA store.
    const int ew = warp - 2;
    const int grp = ew >> 2;
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int row_in_tile = quad * 32 + lane;
    const bool store_warp = (ew & 3) == 0;  // its elected lane issues (and waits for) the group's TMA stores
    uint8_t* stage_c = smem_c + grp * kStageCBytes;
    const uint32_t stage_row = smem_u32(stage_c) + static_cast<uint32_t>(row_in_tile * 128);
    const int sw = row_in_tile & 7;
    constexpr int kChunks = BN / kChunkN;
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t res_uses = 0;  // residual chunks this group has consumed from its ring

    // Per-column epilogue parameters (LayerNorm column sums, bias) of the group's CURRENT chunk live in a 512-byte
    // shared table; the values of its NEXT chunk are fetched with one LDG per thread while the current chunk is being
    // computed and stored into the table between the group's two barriers.  (Reading them with __ldg per 8-column
    // group left every such group waiting on the long scoreboard: 20 % of all samples of the fc1 GEMM.)
    float* tab = col_tab + grp * (2 * kChunkN);
    const int tab_t = (ew & 3) * 32 + lane;           // 0..127 within the group
    constexpr bool kSpec = EPI != 0;
    const bool f_ln = kSpec ? (EPI == 1 || EPI == 2) : (epi.ln_colsum != nullptr);
    const bool f_bias = kSpec ? true : (epi.bias != nullptr);
    const int f_act = kSpec ? ((EPI == 2 || EPI == 6) ? 1 : 0) : epi.act;
    const bool f_pos = kSpec ? false : (epi.pos != nullptr);
    const bool f_mul = kSpec ? false : (epi.residual_op != 0);
    const bool f_stats = kSpec ? (EPI == 3 || (EPI == 7 && epi.stats_out != nullptr)) : (epi.stats_out != nullptr);
    // two-bf16 residual stream: the low halves go straight between registers and global memory, one 128-byte row segment
    // per thread and chunk (whole lines); read only where a residual is added, written wherever C is
    const bool f_lo = EPI == 7;   // (the generic kernel has no registers left for it: EPI 7 exists for every tile shape)
    const float* tab_src = (tab_t < kChunkN) ? epi.ln_colsum : epi.bias;
    const int tab_e = tab_t & (kChunkN - 1);
    auto next_chunk_col = [&](int rr, int c) -> int {  // first column of the group's chunk after (round rr, c); -1: none
      c += 2;
      for (; rr * tile_step < num_tiles; ++rr, c = grp) {
        const int tile = sched_tile(rr, first_tile, tile_step, rot);
        if (tile >= num_tiles) break;
        const int n0t = (tile % num_n) * BN;
        if (c < min(kChunks, (N - n0t + kChunkN - 1) / kChunkN)) return n0t + c * kChunkN;
      }
      return -1;
    };
    auto fetch_col = [&](int col0) -> float {
      const int col = col0 + tab_e;
      return (tab_src != nullptr && col0 >= 0 && col < N) ? __ldg(tab_src + col) : 0.f;
    };
    tab[tab_t] = fetch_col(next_chunk_col(0, grp - 2));
    named_bar_sync(1 + grp, 128);
    const uint32_t tab_addr = smem_u32(tab);

    for (int rr = 0; rr * tile_step < num_tiles; ++rr) {
        const int tile = sched_tile(rr, first_tile, tile_step, rot);  // rotated within the round, see sched_rotation
        if (tile >= num_tiles) break;  // only in the last, partial round
      const int m0 = (tile / num_n) * (BM * CG) + (int)cta_rank * BM;
      const int n0 = (tile % num_n) * BN;
      const int row = m0 + row_in_tile;
      const bool row_ok = row < M;

      float ln_mean = 0.f, ln_rstd = 1.f;
      if (f_ln && row_ok) {
        // the producer GEMM left one (Σx, Σx²) pair per 64-column chunk of the row; they are added here in a fixed
        // order (no atomics anywhere: results are bit-reproducible run to run)
        const float2* rs = reinterpret_cast<const float2*>(epi.ln_rowstats) + row;
        float s_sum = 0.f, s_sq = 0.f;
        for (int p = 0; p < epi.ln_parts; ++p) {
          const float2 st = __ldg(rs + (int64_t)p * M);
          s_sum += st.x;
          s_sq += st.y;
        }
        ln_mean = s_sum * epi.ln_inv_dim;
        const float var = fmaxf(s_sq * epi.ln_inv_dim - ln_mean * ln_mean, 0.f);
        ln_rstd = rsqrtf(var + epi.ln_eps);
      }
      const float* pos_row =
          f_pos ? epi.pos + (int64_t)(row_ok ? (row % epi.pos_rows) : 0) * N : nullptr;

      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(acc * BN);
      // chunks of this tile that hold real columns (the N tail may leave a group without work)
      const int nvalid = min(kChunks, (N - n0 + kChunkN - 1) / kChunkN);
      if (grp >= nvalid) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CG == 2) mbar_arrive_cluster(&tempty_bar[acc], 0);
          else mbar_arrive(&tempty_bar[acc]);
        }
      }
#pragma unroll 1
      for (int c = grp; c < nvalid; c += 2) {
        const int c0 = n0 + c * kChunkN;
        uint4 lo_in[8];
        // low halves live in the epilogue's own order, [row block of 128][64-column chunk][8-column group][row][8]: for a
        // given group the 32 lanes of a warp (32 consecutive rows) touch 512 contiguous bytes.  (Row-major, one 128-byte row
        // segment per thread: 32 lines per load / store instruction, 16x the L1 wavefronts — the out-projection ran at
        // 705 instead of 1219 TFLOP/s.)
        __nv_bfloat16* lo_row = f_lo ? epi.lo + (((int64_t)(row >> 7) * ((N + kChunkN - 1) / kChunkN) + (c0 / kChunkN)) * 8 * BM +
                                                 (row & (BM - 1))) * 8
                                     : nullptr;
        constexpr int kLoGroup = BM * 8;   // elements between consecutive 8-column groups of a row
        if (RES && f_lo) {
          // issued ahead of the TMEM load: the global latency overlaps the TMEM round trip and the residual wait
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            lo_in[g] = make_uint4(0u, 0u, 0u, 0u);
            if (row_ok && c0 + g * 8 < N) lo_in[g] = *reinterpret_cast<const uint4*>(lo_row + g * kLoGroup);
          }
        }
        uint32_t r[64];
        tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c * kChunkN), *reinterpret_cast<uint32_t(*)[32]>(&r[0]));
        tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c * kChunkN + 32),
                           *reinterpret_cast<uint32_t(*)[32]>(&r[32]));
        tmem_ld_wait();
        if (RES && f_lo) {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const uint32_t w4[4] = {lo_in[g].x, lo_in[g].y, lo_in[g].z, lo_in[g].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 l2 = unpack_bf16x2(w4[j]);
              r[g * 8 + 2 * j] = __float_as_uint(__uint_as_float(r[g * 8 + 2 * j]) + l2.x);
              r[g * 8 + 2 * j + 1] = __float_as_uint(__uint_as_float(r[g * 8 + 2 * j + 1]) + l2.y);
            }
          }
        }
        const float tab_next = fetch_col(next_chunk_col(rr, c));  // consumed after the first barrier below
        if (c + 2 >= nvalid) {
          // last chunk of this group for this tile: the accumulator stage can go back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CG == 2) mbar_arrive_cluster(&tempty_bar[acc], 0);
            else mbar_arrive(&tempty_bar[acc]);
          }
        }
        uint4 res[8];
        if (RES) {
          // this chunk's residual tile was prefetched by the residual warp (128B-swizzled, like the C staging)
          const int slot = grp * S::kResDepth + (int)(res_uses % S::kResDepth);
          mbar_wait(&rfull_bar[slot], (res_uses / S::kResDepth) & 1u);
          ++res_uses;
          const uint32_t rrow = smem_u32(smem_r + slot * kStageCBytes) + static_cast<uint32_t>(row_in_tile * 128);
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n"
                         : "=r"(res[g].x), "=r"(res[g].y), "=r"(res[g].z), "=r"(res[g].w)
                         : "r"(rrow + static_cast<uint32_t>((g ^ sw) << 4)));
          }
          // generic-proxy reads above vs the TMA (async-proxy) refill of this slot: the proxy fence makes every
          // lane's loads complete before its warp releases the slot (without it one 16-byte piece of one row was,
          // rarely, read after the refill had landed — tests/test_ops_gpu.py::test_gemm_residual_many_tiles)
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&rempty_bar[slot]);
        }
        uint4 o[8];
        float st_sum = 0.f, st_sq = 0.f;
        // two fp32 lanes per instruction (FFMA2 / FADD2 / FMUL2): the fused epilogues (LayerNorm fold + bias + GELU)
        // were issue bound — fc1 held the tensor pipe at 70 % (profiles/r01_gemm_full.md)
        const float2 nmean2 = make_float2(-ln_mean, -ln_mean), rstd2 = make_float2(ln_rstd, ln_rstd);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const int cc = c0 + g * 8;
          float2 v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            v[j] = make_float2(__uint_as_float(r[g * 8 + 2 * j]), __uint_as_float(r[g * 8 + 2 * j + 1]));
          if (cc < N) {
            if (f_ln) {
              const float4 s0 = lds_f4(tab_addr + static_cast<uint32_t>(g * 32));
              const float4 s1 = lds_f4(tab_addr + static_cast<uint32_t>(g * 32 + 16));
              const float2 cs[4] = {{s0.x, s0.y}, {s0.z, s0.w}, {s1.x, s1.y}, {s1.z, s1.w}};
#pragma unroll
              for (int j = 0; j < 4; ++j) v[j] = fmul2(rstd2, ffma2(nmean2, cs[j], v[j]));
            }
            if (f_bias) {
              const float4 b0 = lds_f4(tab_addr + static_cast<uint32_t>(kChunkN * 4 + g * 32));
              const float4 b1 = lds_f4(tab_addr + static_cast<uint32_t>(kChunkN * 4 + g * 32 + 16));
              v[0] = fadd2(v[0], make_float2(b0.x, b0.y));
              v[1] = fadd2(v[1], make_float2(b0.z, b0.w));
              v[2] = fadd2(v[2], make_float2(b1.x, b1.y));
              v[3] = fadd2(v[3], make_float2(b1.z, b1.w));
            }
            if (f_act == 1) {
#pragma unroll
              for (int j = 0; j < 4; ++j) v[j] = gelu_tanh_fast2(v[j]);
            } else if (f_act >= 2) {  // erf GELU / sigmoid (SegFormer decoder of SigLIP2_MTL): out of line, so that the
              // backbone's epilogue keeps its registers and schedule (inlined erff cost the base-224 engine 10 %)
#pragma unroll
              for (int j = 0; j < 4; ++j) v[j] = act_rare(v[j], f_act);
            }
            if (f_pos) {
              const float4 p0 = __ldg(reinterpret_cast<const float4*>(pos_row + cc));
              const float4 p1 = __ldg(reinterpret_cast<const float4*>(pos_row + cc + 4));
              v[0] = fadd2(v[0], make_float2(p0.x, p0.y));
              v[1] = fadd2(v[1], make_float2(p0.z, p0.w));
              v[2] = fadd2(v[2], make_float2(p1.x, p1.y));
              v[3] = fadd2(v[3], make_float2(p1.z, p1.w));
            }
            if (RES) {
              if (!f_mul) {
                v[0] = fadd2(v[0], unpack_bf16x2(res[g].x));
                v[1] = fadd2(v[1], unpack_bf16x2(res[g].y));
                v[2] = fadd2(v[2], unpack_bf16x2(res[g].z));
                v[3] = fadd2(v[3], unpack_bf16x2(res[g].w));
              } else {  // gate: sigmoid(conv(x)) * x  (SegFormerStrongDecoder.fuse_attn)
                v[0] = fmul2(v[0], unpack_bf16x2(res[g].x));
                v[1] = fmul2(v[1], unpack_bf16x2(res[g].y));
                v[2] = fmul2(v[2], unpack_bf16x2(res[g].z));
                v[3] = fmul2(v[3], unpack_bf16x2(res[g].w));
              }
            }
          }
          o[g].x = pack_bf16x2(v[0].x, v[0].y);
          o[g].y = pack_bf16x2(v[1].x, v[1].y);
          o[g].z = pack_bf16x2(v[2].x, v[2].y);
          o[g].w = pack_bf16x2(v[3].x, v[3].y);
          if (f_lo && row_ok && cc < N) {
            const float2 h0 = unpack_bf16x2(o[g].x), h1 = unpack_bf16x2(o[g].y),
                         h2 = unpack_bf16x2(o[g].z), h3 = unpack_bf16x2(o[g].w);
            uint4 lw;
            lw.x = pack_bf16x2(v[0].x - h0.x, v[0].y - h0.y);
            lw.y = pack_bf16x2(v[1].x - h1.x, v[1].y - h1.y);
            lw.z = pack_bf16x2(v[2].x - h2.x, v[2].y - h2.y);
            lw.w = pack_bf16x2(v[3].x - h3.x, v[3].y - h3.y);
            *reinterpret_cast<uint4*>(lo_row + g * (BM * 8)) = lw;
          }
          if (f_stats && cc < N) {
            const float2 q0 = unpack_bf16x2(o[g].x), q1 = unpack_bf16x2(o[g].y),
                         q2 = unpack_bf16x2(o[g].z), q3 = unpack_bf16x2(o[g].w);
            const float2 sm = fadd2(fadd2(q0, q1), fadd2(q2, q3));
            const float2 sq = ffma2(q0, q0, ffma2(q1, q1, ffma2(q2, q2, fmul2(q3, q3))));
            st_sum += sm.x + sm.y;
            st_sq += sq.x + sq.y;
          }
        }
        // staging tile free? (the previous TMA store of this group has finished reading it)
        if (store_warp && elect_one()) tma_store_wait_read<0>();
        named_bar_sync(1 + grp, 128);
        tab[tab_t] = tab_next;  // every thread of the group is past its reads of the current chunk's parameters
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const uint32_t addr = stage_row + static_cast<uint32_t>((g ^ sw) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(o[g].x), "r"(o[g].y),
                       "r"(o[g].z), "r"(o[g].w)
                       : "memory");
        }
        fence_proxy_async_smem();
        named_bar_sync(1 + grp, 128);
        if (store_warp && elect_one()) {
          tma_store_2d(&tmC, stage_c, c0, m0);  // rows >= M and columns >= N are clipped by the TMA unit
          tma_store_commit();
        }
        // row statistics of the bf16 output, one partial per (64-column chunk, row): every slot is written exactly once
        // per GEMM, 32 consecutive rows per warp store (coalesced), and summed in chunk order by the consumer
        if (f_stats && row_ok)
          reinterpret_cast<float2*>(epi.stats_out)[(int64_t)(c0 / kChunkN) * M + row] = make_float2(st_sum, st_sq);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (store_warp && elect_one()) tma_store_wait<0>();
  }

  tc_fence_before();
  if (CG == 2) cluster_sync_all();  // no CTA of the pair leaves while the other may still touch it
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_pair<S::kTmemCols>(tmem_base);
    else tmem_dealloc<S::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) ==
            cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
  });
  return fn;
}

}  // namespace

// bf16 row-major [rows, cols] with leading dimension ld (elements) -> 2-D tiled map, box = {64, box_rows}
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int64_t ld,
                      int box_rows, bool store = false) {
  PFN_encodeTiled fn = get_encode_fn();
  DFD_REQUIRE(fn != nullptr, DFD_ERR_NO_DEVICE,
              "cuTensorMapEncodeTiled unavailable (no CUDA driver on this host)");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  store ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DFD_REQUIRE(r == CUDA_SUCCESS, DFD_ERR_CUDA,
              "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld box_rows=%d", (int)r,
              (long long)rows, (long long)cols, (long long)ld, box_rows);
  return DFD_OK;
}

template <int BN, int CG, int RES, int EPI = 0>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                       const CUtensorMap& tmR, int M, int N, int K, const EpiArgs& ea, cudaStream_t st) {
  using S = GemmSmem<BN, CG, RES>;
  static SmemOptIn smem_once;
  if (int rc = ensure_dynamic_smem(smem_once, gemm_bf16_tcgen05_kernel<BN, CG, RES, EPI>, S::kTotal)) return rc;
  const int num_tiles = ((M + BM * CG - 1) / (BM * CG)) * ((N + BN - 1) / BN);
  const int max_units = kNumSMs / CG;
  const int units = num_tiles < max_units ? num_tiles : max_units;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(units * CG);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DFD_CUDA(cudaLaunchKernelEx(&cfg, gemm_bf16_tcgen05_kernel<BN, CG, RES, EPI>, tmA, tmB, tmC, tmR, M, N, K, ea));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  g_last_variant.store(BN + 1000 * CG + 10000 * RES + 100000 * EPI, std::memory_order_relaxed);
  g_variant_launches[variant_slot(BN, CG, RES, EPI)].fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

// Tile choice.  Large-M GEMMs run as CTA pairs (256 x BN tiles, cta_group::2); BN = 256 keeps the pair at the
// shared-memory bandwidth limit, narrower tiles only pay off when they remove a mostly-empty N tail.
static void pick_tile(int M, int N, int* bn_out, int* cg_out) {
  const int cg = (M > BM * kNumSMs / 2) ? 2 : 1;
  const int cands[3] = {256, 192, 128};
  const double penalty[3] = {1.0, 1.2, 1.45};
  int best = 128;
  double best_cost = 1e30;
  const int num_m = (M + BM * cg - 1) / (BM * cg);
  const int units = kNumSMs / cg;
  for (int i = 0; i < 3; ++i) {
    const int bn = cands[i];
    const int num_n = (N + bn - 1) / bn;
    const long tiles = (long)num_m * num_n;
    const long waves = (tiles + units - 1) / units;
    const double cost = (double)waves * bn * penalty[i];
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  *bn_out = best;
  *cg_out = cg;
}

int gemm_bf16_dispatch(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                       int M, int N, int K, const dfd_gemm_epilogue* epi, int force_bn,
                       cudaStream_t st) {
  DFD_REQUIRE(A && W && C, DFD_ERR_BAD_ARG, "gemm: null pointer");
  DFD_REQUIRE(M > 0 && N > 0 && K > 0, DFD_ERR_SHAPE, "gemm: M,N,K must be positive (%d,%d,%d)", M, N, K);
  DFD_REQUIRE(K % 8 == 0 && N % 8 == 0, DFD_ERR_SHAPE, "gemm: K and N must be multiples of 8 (K=%d N=%d)", K, N);
  DFD_REQUIRE(lda % 8 == 0 && ldw % 8 == 0 && ldc % 8 == 0, DFD_ERR_SHAPE,
              "gemm: leading dimensions must be multiples of 8 elements");
  DFD_REQUIRE(lda >= K && ldw >= K && ldc >= N, DFD_ERR_SHAPE, "gemm: leading dimension too small");
  DFD_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)W % 16 == 0) && ((uintptr_t)C % 16 == 0),
              DFD_ERR_BAD_ARG, "gemm: pointers must be 16-byte aligned");
  EpiArgs ea{};
  if (epi != nullptr) {
    ea.bias = epi->bias;
    ea.act = epi->act;
    ea.pos = epi->pos;
    ea.pos_rows = epi->pos_rows > 0 ? epi->pos_rows : 1;
    ea.residual = reinterpret_cast<const __nv_bfloat16*>(epi->residual);
    ea.ldr = epi->ldr;
    ea.ln_rowstats = epi->ln_rowstats;
    ea.ln_colsum = epi->ln_colsum;
    ea.ln_inv_dim = epi->ln_dim > 0 ? 1.0f / (float)epi->ln_dim : 0.f;
    ea.ln_eps = epi->ln_eps;
    ea.stats_out = epi->stats_out;
    ea.residual_op = epi->residual_op;
    ea.ln_parts = epi->ln_parts > 0 ? epi->ln_parts : 1;
    ea.lo = reinterpret_cast<__nv_bfloat16*>(epi->residual_lo);
    DFD_REQUIRE(ea.lo == nullptr || (uintptr_t)ea.lo % 16 == 0, DFD_ERR_SHAPE, "gemm: residual_lo must be 16-byte aligned");
    DFD_REQUIRE(ea.lo == nullptr || ea.residual_op == 0, DFD_ERR_BAD_ARG, "gemm: residual_lo goes with an additive residual");
    DFD_REQUIRE(ea.act >= 0 && ea.act <= 3, DFD_ERR_BAD_ARG, "gemm: act must be 0 (none), 1 (gelu_tanh), 2 (gelu_erf) or 3 (sigmoid)");
    DFD_REQUIRE(ea.residual_op == 0 || ea.residual_op == 1, DFD_ERR_BAD_ARG, "gemm: residual_op must be 0 (add) or 1 (multiply)");
    DFD_REQUIRE((ea.ln_colsum == nullptr) == (ea.ln_rowstats == nullptr), DFD_ERR_BAD_ARG,
                "gemm: ln_rowstats and ln_colsum must be given together");
    DFD_REQUIRE(ea.ln_colsum == nullptr || epi->ln_dim > 0, DFD_ERR_BAD_ARG, "gemm: ln_dim must be > 0");
    DFD_REQUIRE(ea.residual == nullptr || (ea.ldr % 8 == 0 && ea.ldr >= N), DFD_ERR_SHAPE,
                "gemm: residual leading dimension invalid");
    DFD_REQUIRE((uintptr_t)ea.residual % 16 == 0, DFD_ERR_BAD_ARG, "gemm: residual must be 16-byte aligned");
  }
  int bn = 0, cg = 1;
  pick_tile(M, N, &bn, &cg);
  if (force_bn > 0) {  // test hook: tile_n, +1000 forces single-CTA tiles, +2000 forces CTA pairs
    bn = force_bn % 1000;
    if (force_bn >= 2000) cg = 2;
    else if (force_bn >= 1000) cg = 1;
  }
  DFD_REQUIRE(bn == 128 || bn == 192 || bn == 256, DFD_ERR_UNSUPPORTED, "gemm: unsupported tile N %d", bn);
  CUtensorMap tmA, tmB, tmC, tmR;
  int rc = make_tmap_bf16_2d(&tmA, A, M, K, lda, BM);
  if (rc != DFD_OK) return rc;
  rc = make_tmap_bf16_2d(&tmB, W, N, K, ldw, bn / cg);
  if (rc != DFD_OK) return rc;
  rc = make_tmap_bf16_2d(&tmC, C, M, N, ldc, BM, true);
  if (rc != DFD_OK) return rc;
  const bool has_res = ea.residual != nullptr;
  tmR = tmC;
  if (has_res) {
    rc = make_tmap_bf16_2d(&tmR, ea.residual, M, N, ea.ldr, BM);
    if (rc != DFD_OK) return rc;
  }
  if (ea.lo != nullptr) {
    // two-bf16 residual stream: one specialised epilogue (bias + residual + lo [+ row statistics]) for every tile shape
    DFD_REQUIRE(has_res && ea.bias != nullptr && ea.pos == nullptr && ea.ln_colsum == nullptr && ea.act == 0, DFD_ERR_UNSUPPORTED,
                "gemm: residual_lo needs bias + additive residual and no other fused option");
#define DFD_GEMM_LO_CASE(BN_, CG_) \
  if (bn == BN_ && cg == CG_) return launch_gemm<BN_, CG_, 1, 7>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
    DFD_GEMM_LO_CASE(256, 2)
    DFD_GEMM_LO_CASE(192, 2)
    DFD_GEMM_LO_CASE(128, 2)
    DFD_GEMM_LO_CASE(256, 1)
    DFD_GEMM_LO_CASE(192, 1)
    DFD_GEMM_LO_CASE(128, 1)
#undef DFD_GEMM_LO_CASE
  }
  // the backbone's own epilogues on its one large-M tile shape get compile-time specialised kernels (see EPI above)
  if (bn == 256 && cg == 2 && ea.bias != nullptr && ea.pos == nullptr) {
    const bool ln = ea.ln_colsum != nullptr, stats = ea.stats_out != nullptr;
    if (!has_res && !stats) {
      if (ln && ea.act == 0) return launch_gemm<256, 2, 0, 1>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
      if (ln && ea.act == 1) return launch_gemm<256, 2, 0, 2>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
      if (!ln && ea.act == 0) return launch_gemm<256, 2, 0, 5>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
      if (!ln && ea.act == 1) return launch_gemm<256, 2, 0, 6>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
    } else if (has_res && !ln && ea.act == 0 && ea.residual_op == 0) {
      if (stats) return launch_gemm<256, 2, 1, 3>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
      return launch_gemm<256, 2, 1, 4>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
    }
  }
#define DFD_GEMM_CASE(BN_, CG_)                                                                   \
  if (bn == BN_ && cg == CG_)                                                                     \
    return has_res ? launch_gemm<BN_, CG_, 1>(tmA, tmB, tmC, tmR, M, N, K, ea, st)                 \
                   : launch_gemm<BN_, CG_, 0>(tmA, tmB, tmC, tmR, M, N, K, ea, st);
  DFD_GEMM_CASE(256, 2)
  DFD_GEMM_CASE(192, 2)
  DFD_GEMM_CASE(128, 2)
  DFD_GEMM_CASE(256, 1)
  DFD_GEMM_CASE(192, 1)
  DFD_GEMM_CASE(128, 1)
#undef DFD_GEMM_CASE
  set_last_error("gemm: unsupported tile N %d", bn);
  return DFD_ERR_UNSUPPORTED;
}

}  // namespace dfd

// Which kernel instantiation the last dfd_gemm_bf16[_tile] call of this process launched:
// BN + 1000·CG + 10000·RES + 100000·EPI (tests assert that the specialised epilogues are the ones being checked).
extern "C" DFD_API int dfd_gemm_last_variant(void) { return dfd::g_last_variant.load(std::memory_order_relaxed); }
// Launches of one instantiation (same encoding) by this process since load; -1 for an encoding that names no kernel.
extern "C" DFD_API int64_t dfd_gemm_variant_launches(int variant) {
  const int bn = variant % 1000, cg = variant / 1000 % 10, res = variant / 10000 % 10, epi = variant / 100000;
  if ((bn != 128 && bn != 192 && bn != 256) || cg < 1 || cg > 2 || res < 0 || res > 1 || epi < 0 || epi > 7) return -1;
  return dfd::g_variant_launches[dfd::variant_slot(bn, cg, res, epi)].load(std::memory_order_relaxed);
}

// Host-only view of the persistent schedule: the tile that `unit` (of `units`) processes in `round`, or -1 when it has none.
extern "C" DFD_API int dfd_gemm_schedule(int num_tiles, int num_n, int units, int unit, int round) {
  if (num_tiles <= 0 || num_n <= 0 || units <= 0 || unit < 0 || unit >= units || round < 0) return -1;
  if ((long long)round * units >= num_tiles) return -1;
  const int tile = dfd::sched_tile(round, unit, units, dfd::sched_rotation(units, num_n));
  return tile < num_tiles ? tile : -1;
}

extern "C" DFD_API int dfd_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, void* C,
                                     int64_t ldc, int M, int N, int K, const dfd_gemm_epilogue* epi,
                                     void* stream) {
  return dfd::gemm_bf16_dispatch(A, lda, W, ldw, C, ldc, M, N, K, epi, 0,
                                 reinterpret_cast<cudaStream_t>(stream));
}

// Test hook: same as dfd_gemm_bf16 with the tile width forced (128/192/256).
extern "C" DFD_API int dfd_gemm_bf16_tile(const void* A, int64_t lda, const void* W, int64_t ldw,
                                          void* C, int64_t ldc, int M, int N, int K,
                                          const dfd_gemm_epilogue* epi, int tile_n, void* stream) {
  return dfd::gemm_bf16_dispatch(A, lda, W, ldw, C, ldc, M, N, K, epi, tile_n,
                                 reinterpret_cast<cudaStream_t>(stream));
}

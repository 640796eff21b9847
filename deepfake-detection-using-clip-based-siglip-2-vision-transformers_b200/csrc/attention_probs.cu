// Attention maps: the probabilities P = softmax(q·kᵀ·scale) that the flash kernels (attention_dq.cu / attention_ws.cu)
// compute and drop, and Abnar & Zuidema's attention rollout over them.
//
//   attention_probs_kernel   one CTA per (image, 128-query tile, head group) on tcgen05 + TMEM.  S = Q·Kᵀ runs on the tensor
//                            cores, 128 keys per MMA tile.  The normaliser needs every key before any probability can be
//                            written, so the CTA sweeps the key tiles twice: sweep 1 keeps a running (max, sum) per row and
//                            head, sweep 2 recomputes S and writes P.  Per-head mode (head group = one head) writes
//                            [B, H, N, N]; head-mean mode (head group = all H heads) walks the heads innermost in sweep 2,
//                            sums P_h/H in registers and writes [B, N, N] once per (image, query tile, key tile).
//                            Warps: 0 TMA loader, 1 MMA issuer, 2..9 softmax (two per TMEM lane quadrant, 64 keys each).
//   rollout_*                r_L = mean_h map_p[b, h, :], then r ← α·(r·Ā_l) + (1 − α)·r for l = L−1 … 0; one launch per
//                            layer, each HBM bound (B·N² fp32 read).  The heatmap is the bilinear upsample of N·r.
//
// Reference semantics: HF:modeling_siglip.py:229-249 (eager_attention_forward: softmax in fp32, returned as attn_weights).
#include "dfd_common.cuh"

#include <atomic>

namespace dfd {

extern std::atomic<int64_t> g_launches;
int make_tmap_qkv_4d(CUtensorMap* out, const void* base, int hd, int heads3, int N, int B, int64_t ld, int box_cols,
                     int box_rows, int swizzle32);

namespace {

constexpr int kPQ = 128;             // query rows per CTA (TMEM lanes)
constexpr int kPK = 128;             // keys per S tile
constexpr int kPStages = 3;          // K tiles in flight
constexpr int kPSoftmaxWarps = 8;    // two per lane quadrant, 64 keys each
constexpr int kPThreads = (2 + kPSoftmaxWarps) * 32;
constexpr int kPStg = 65;            // staging pitch (floats): row-per-lane writes and row-per-warp reads are conflict free
constexpr int kPMaxSmem = 227 * 1024;

template <int HD>
struct ProbsSmem {
  static constexpr bool kTail = (HD % 64) != 0;
  static constexpr int kMain = 128 * 64 * 2;               // 128 rows x 128 B, SWIZZLE_128B (Q tile and K tile alike)
  static constexpr int kTailBytes = kTail ? 128 * 16 * 2 : 0;  // 128 rows x 32 B, SWIZZLE_32B
  static constexpr int kTileBytes = kMain + kTailBytes;
  static constexpr int kStgBytes = kPSoftmaxWarps * 32 * kPStg * 4;
  static constexpr int kXchgBytes = 2 * 2 * kPQ * 2 * 4;  // (max, sum) [head parity][part][row]
  static constexpr int kBarBytes = 256;
  static constexpr int kFixed = 2 * kTileBytes + kPStages * kTileBytes + kStgBytes + kXchgBytes + kBarBytes + 1024;
  // + per-part (max, scale / sum) of every head of the group: [part][head][row][2]
  static constexpr int total(int nh) { return kFixed + 2 * nh * kPQ * 2 * 4; }
};

// named barrier 1 + quad over the two softmax warps of one lane quadrant
__device__ __forceinline__ void pair_bar_sync(int quad) {
  switch (quad) {
    case 0: asm volatile("bar.sync 1, 64;\n" ::: "memory"); break;
    case 1: asm volatile("bar.sync 2, 64;\n" ::: "memory"); break;
    case 2: asm volatile("bar.sync 3, 64;\n" ::: "memory"); break;
    default: asm volatile("bar.sync 4, 64;\n" ::: "memory"); break;
  }
}

// Tile t of a CTA's sequence: sweep 1 = t < nh·T (head-major, key tiles inner), sweep 2 = the rest (key tiles outer,
// heads inner).  Loader, MMA issuer and softmax warps walk the same sequence.
struct TileSeq {
  int nh, T;
  __device__ __forceinline__ int total() const { return 2 * nh * T; }
  __device__ __forceinline__ bool sweep1(int t) const { return t < nh * T; }
  __device__ __forceinline__ int head(int t) const { return sweep1(t) ? t / T : (t - nh * T) % nh; }
  __device__ __forceinline__ int key(int t) const { return sweep1(t) ? t % T : (t - nh * T) / nh; }
  __device__ __forceinline__ bool new_q(int t) const { return t == 0 || head(t) != head(t - 1); }
};

template <int HD>
__global__ void __launch_bounds__(kPThreads, 1)
attention_probs_kernel(const __grid_constant__ CUtensorMap tmMain, const __grid_constant__ CUtensorMap tmTail,
                       float* __restrict__ out, int N, int H, int nh, int per_head, float scale_log2, float out_scale) {
  using S = ProbsSmem<HD>;
  constexpr bool kTail = S::kTail;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sQ = smem;                                   // [2 slots]
  uint8_t* sK = sQ + 2 * S::kTileBytes;                 // [kPStages]
  float* stg = reinterpret_cast<float*>(sK + kPStages * S::kTileBytes);   // [softmax warp][32][kPStg]
  float* xchg = stg + kPSoftmaxWarps * 32 * kPStg;                         // [2][2][128][2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(xchg + 2 * 2 * kPQ * 2);
  uint64_t* q_full = bars;                  // [2]
  uint64_t* q_empty = bars + 2;             // [2]
  uint64_t* k_full = bars + 4;              // [kPStages]
  uint64_t* k_empty = k_full + kPStages;    // [kPStages]
  uint64_t* s_full = k_empty + kPStages;    // [2]
  uint64_t* s_empty = s_full + 2;           // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_empty + 2);
  float* stats = reinterpret_cast<float*>(smem + (S::kFixed - 1024));      // [2][nh][128][2]

  const int qt = blockIdx.x, b = blockIdx.z, h0 = blockIdx.y * nh;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TileSeq seq{nh, (N + kPK - 1) / kPK};
  const int n_tiles = seq.total();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmMain);
    if (kTail) tma_prefetch_desc(&tmTail);
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], kPSoftmaxWarps);
    }
#pragma unroll
    for (int s = 0; s < kPStages; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<2 * kPK>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------ TMA loader ------------------------------------
    if (elect_one()) {
      int qc = -1;
      for (int t = 0; t < n_tiles; ++t) {
        const int h = h0 + seq.head(t), j = seq.key(t);
        if (seq.new_q(t)) {
          ++qc;
          const int slot = qc & 1;
          mbar_wait(&q_empty[slot], ((qc >> 1) & 1) ^ 1);
          mbar_expect_tx(&q_full[slot], S::kTileBytes);
          uint8_t* q = sQ + slot * S::kTileBytes;
#pragma unroll
          for (int i = 0; i < kPQ / 64; ++i) {  // 64-row TMA boxes
            tma_load_4d(&tmMain, &q_full[slot], q + i * 8192, 0, h, qt * kPQ + i * 64, b);
            if (kTail) tma_load_4d(&tmTail, &q_full[slot], q + S::kMain + i * 2048, 64, h, qt * kPQ + i * 64, b);
          }
        }
        const int st = t % kPStages;
        mbar_wait(&k_empty[st], ((t / kPStages) & 1) ^ 1);
        mbar_expect_tx(&k_full[st], S::kTileBytes);
        uint8_t* k = sK + st * S::kTileBytes;
#pragma unroll
        for (int i = 0; i < kPK / 64; ++i) {
          tma_load_4d(&tmMain, &k_full[st], k + i * 8192, 0, H + h, j * kPK + i * 64, b);
          if (kTail) tma_load_4d(&tmTail, &k_full[st], k + S::kMain + i * 2048, 64, H + h, j * kPK + i * 64, b);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------ MMA issuer: S_t = Q · K_tᵀ into TMEM buffer t&1 ------------------------------------
    if (elect_one()) {
      int qc = -1;
      for (int t = 0; t < n_tiles; ++t) {
        if (seq.new_q(t)) {
          ++qc;
          mbar_wait(&q_full[qc & 1], (qc >> 1) & 1);
        }
        const int slot = qc & 1, st = t % kPStages, buf = t & 1;
        mbar_wait(&k_full[st], (t / kPStages) & 1);
        mbar_wait(&s_empty[buf], ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        const int n16 = (min(kPK, N - seq.key(t) * kPK) + 15) & ~15;
        const uint32_t tS = tmem_base + static_cast<uint32_t>(buf * kPK);
        const uint32_t qaddr = smem_u32(sQ + slot * S::kTileBytes), kaddr = smem_u32(sK + st * S::kTileBytes);
        const uint64_t dQ = umma_desc(qaddr, 16, 1024, 2), dK = umma_desc(kaddr, 16, 1024, 2);
        const uint32_t idesc = umma_idesc_bf16_major(kPQ, n16, 0, 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_ss(tS, dQ + static_cast<uint64_t>(2 * k), dK + static_cast<uint64_t>(2 * k), idesc, k != 0);
        if (kTail)
          umma_bf16_ss(tS, umma_desc(qaddr + S::kMain, 16, 256, 6), umma_desc(kaddr + S::kMain, 16, 256, 6), idesc, 1u);
        umma_commit(&k_empty[st]);
        umma_commit(&s_full[buf]);
        if (t + 1 == n_tiles || seq.new_q(t + 1)) umma_commit(&q_empty[slot]);
      }
    }
  } else {
    // ------------------------------------ softmax / output ------------------------------------
    const int w = warp - 2;
    const int quad = warp & 3;     // TMEM lane quadrant this warp may access
    const int part = w >> 2;       // keys [64 part, 64 part + 64) of every tile
    const int row = quad * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
    float* my_stats = stats + part * nh * kPQ * 2;
    float* my_stg = stg + w * 32 * kPStg;
    float m = -INFINITY, l = 0.f;  // running row max (log2 units) and sum of this part's keys, sweep 1
    float acc[64];
#pragma unroll
    for (int c = 0; c < 64; ++c) acc[c] = 0.f;
    for (int t = 0; t < n_tiles; ++t) {
      const int buf = t & 1;
      mbar_wait(&s_full[buf], (t >> 1) & 1);
      tc_fence_after();
      uint32_t s[64];
      {
        uint32_t (&s0)[32] = *reinterpret_cast<uint32_t(*)[32]>(&s[0]);
        uint32_t (&s1)[32] = *reinterpret_cast<uint32_t(*)[32]>(&s[32]);
        const uint32_t tS = tmem_base + lane_off + static_cast<uint32_t>(buf * kPK + 64 * part);
        tmem_ld_32x32b_x32(tS, s0);
        tmem_ld_32x32b_x32(tS + 32, s1);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_empty[buf]);  // S is in registers: the buffer may take tile t + 2
      const int hr = seq.head(t), j = seq.key(t);
      const int valid = min(kPK, N - j * kPK) - 64 * part;  // valid keys among this part's 64 (may be <= 0)
      if (seq.sweep1(t)) {
#pragma unroll
        for (int c = 0; c < 64; ++c)
          if (c >= valid) s[c] = __float_as_uint(-INFINITY);
        float mx = __uint_as_float(s[0]);
#pragma unroll
        for (int c = 1; c < 64; ++c) mx = fmaxf(mx, __uint_as_float(s[c]));
        const float m_new = fmaxf(m, mx * scale_log2);  // scale > 0
        if (m_new != -INFINITY) {
          float sum4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int c = 0; c < 64; ++c) sum4[c & 3] += fast_exp2(fmaf(__uint_as_float(s[c]), scale_log2, -m_new));
          l = l * fast_exp2(m - m_new) + ((sum4[0] + sum4[1]) + (sum4[2] + sum4[3]));
          m = m_new;
        }
        if (j == seq.T - 1) {  // this head's row statistics are complete: merge the two parts
          float* xc = xchg + (hr & 1) * 2 * kPQ * 2;
          xc[(part * kPQ + row) * 2] = m;
          xc[(part * kPQ + row) * 2 + 1] = l;
          pair_bar_sync(quad);
          const float mo = xc[((1 - part) * kPQ + row) * 2], lo = xc[((1 - part) * kPQ + row) * 2 + 1];
          const float mm = fmaxf(m, mo);  // finite: key 0 is valid for part 0
          const float ll = l * fast_exp2(m - mm) + lo * fast_exp2(mo - mm);
          my_stats[(hr * kPQ + row) * 2] = mm;
          my_stats[(hr * kPQ + row) * 2 + 1] = out_scale / ll;
          m = -INFINITY;
          l = 0.f;
        }
      } else {
        const float mm = my_stats[(hr * kPQ + row) * 2], inv = my_stats[(hr * kPQ + row) * 2 + 1];
#pragma unroll
        for (int c = 0; c < 64; ++c) acc[c] += fast_exp2(fmaf(__uint_as_float(s[c]), scale_log2, -mm)) * inv;
        if (hr == nh - 1) {
          // transpose through shared memory so that every store instruction writes 128 contiguous bytes of one row
#pragma unroll
          for (int c = 0; c < 64; ++c) {
            my_stg[lane * kPStg + c] = acc[c];
            acc[c] = 0.f;
          }
          __syncwarp();
          const int64_t plane = per_head ? (int64_t)b * H + h0 : (int64_t)b;
          const int row0 = qt * kPQ + quad * 32;
          const int rows = min(32, N - row0);
          float* obase = out + (plane * N + row0) * (int64_t)N + j * kPK + 64 * part;
          for (int r = 0; r < rows; ++r) {
            if (lane < valid) obase[(int64_t)r * N + lane] = my_stg[r * kPStg + lane];
            if (lane + 32 < valid) obase[(int64_t)r * N + lane + 32] = my_stg[r * kPStg + lane + 32];
          }
          __syncwarp();
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<2 * kPK>(tmem_base);
  }
}

template <int HD>
int launch_probs(const void* qkv, int64_t ldqkv, int B, int N, int H, float scale, int per_head, float* out,
                 cudaStream_t st) {
  using S = ProbsSmem<HD>;
  const int nh = per_head ? 1 : H;
  const int smem = S::total(nh);
  DFD_REQUIRE(smem <= kPMaxSmem, DFD_ERR_UNSUPPORTED, "attention_probs: %d heads do not fit the head-mean kernel", H);
  CUtensorMap tmMain, tmTail;
  int rc = make_tmap_qkv_4d(&tmMain, qkv, HD, 3 * H, N, B, ldqkv, 64, 64, 0);
  if (rc != DFD_OK) return rc;
  tmTail = tmMain;
  if (S::kTail) {
    rc = make_tmap_qkv_4d(&tmTail, qkv, HD, 3 * H, N, B, ldqkv, 16, 64, 1);
    if (rc != DFD_OK) return rc;
  }
  static SmemOptIn smem_once;
  if (int rc2 = ensure_dynamic_smem(smem_once, attention_probs_kernel<HD>, kPMaxSmem)) return rc2;
  const dim3 grid((N + kPQ - 1) / kPQ, per_head ? H : 1, B);
  attention_probs_kernel<HD><<<grid, kPThreads, smem, st>>>(tmMain, tmTail, out, N, H, nh, per_head,
                                                            scale * 1.4426950408889634f, per_head ? 1.0f : 1.0f / H);
  DFD_LAUNCH_CHECK();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return DFD_OK;
}

// ---- rollout ------------------------------------------------------------------------------------------------------------
constexpr int kRollCols = 128;  // output columns per CTA
constexpr int kRollThreads = 256;

// r[b, n] = mean_h map_p[b, h, n]
__global__ void __launch_bounds__(256)
rollout_seed_kernel(const float* __restrict__ map_p, float* __restrict__ r, int B, int N, int H) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * N) return;
  const int64_t b = i / N, n = i % N;
  float s = 0.f;
  for (int h = 0; h < H; ++h) s += map_p[(b * H + h) * N + n];
  r[i] = s / H;
}

// r_out[b, k] = α·Σ_q r_in[b, q]·A[b, q, k] + (1 − α)·r_in[b, k], CTA = (128 columns, image); the warps split the rows and
// each lane reads four columns 32 apart, so a warp reads whole 128-byte row segments
__global__ void __launch_bounds__(kRollThreads)
rollout_step_kernel(const float* __restrict__ A, const float* __restrict__ r_in, float* __restrict__ r_out, int N,
                    float alpha) {
  extern __shared__ float rs[];                            // [N] r_in of this image, then [8][kRollCols] partials
  float* part = rs + ((N + 3) & ~3);
  const int b = blockIdx.y, k0 = blockIdx.x * kRollCols;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int q = threadIdx.x; q < N; q += kRollThreads) rs[q] = r_in[(int64_t)b * N + q];
  __syncthreads();
  const float* Ab = A + (int64_t)b * N * N + k0;
  const int cols = min(kRollCols, N - k0);
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  // four rows per iteration: 16 independent loads in flight per thread
  constexpr int kWarps = kRollThreads / 32;
  for (int q0 = warp; q0 < N; q0 += 4 * kWarps) {
    float v[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int q = q0 + u * kWarps;
      const float* row = Ab + (int64_t)min(q, N - 1) * N;
#pragma unroll
      for (int i = 0; i < 4; ++i) v[u][i] = (q < N && lane + 32 * i < cols) ? __ldg(row + lane + 32 * i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float rq = q0 + u * kWarps < N ? rs[q0 + u * kWarps] : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(rq, v[u][i], acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) part[warp * kRollCols + lane + 32 * i] = acc[i];
  __syncthreads();
  if (threadIdx.x < cols) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kRollThreads / 32; ++w) s += part[w * kRollCols + threadIdx.x];
    const int k = k0 + threadIdx.x;
    r_out[(int64_t)b * N + k] = alpha * s + (1.f - alpha) * rs[k];
  }
}

}  // namespace

int attention_probs(const void* qkv, int64_t ldqkv, int B, int N, int H, int hd, float scale, int per_head, float* out,
                    cudaStream_t st) {
  DFD_REQUIRE(qkv && out, DFD_ERR_BAD_ARG, "attention_probs: null pointer");
  DFD_REQUIRE(B > 0 && N > 0 && H > 0, DFD_ERR_SHAPE, "attention_probs: B, N, H must be positive");
  DFD_REQUIRE(B <= 65535 && H <= 65535, DFD_ERR_SHAPE, "attention_probs: B and H must be <= 65535");
  DFD_REQUIRE(hd == 64 || hd == 72, DFD_ERR_UNSUPPORTED, "attention_probs: head dim %d not supported (64, 72)", hd);
  DFD_REQUIRE(ldqkv % 8 == 0 && ldqkv >= 3 * (int64_t)H * hd, DFD_ERR_SHAPE, "attention_probs: bad leading dimension");
  DFD_REQUIRE(per_head == 0 || per_head == 1, DFD_ERR_BAD_ARG, "attention_probs: per_head must be 0 or 1");
  DFD_REQUIRE(scale > 0.f && scale < INFINITY, DFD_ERR_BAD_ARG, "attention_probs: scale must be positive and finite");
  DFD_REQUIRE((uintptr_t)qkv % 16 == 0, DFD_ERR_BAD_ARG, "attention_probs: qkv must be 16-byte aligned");
  if (hd == 64) return launch_probs<64>(qkv, ldqkv, B, N, H, scale, per_head, out, st);
  return launch_probs<72>(qkv, ldqkv, B, N, H, scale, per_head, out, st);
}

int attention_rollout(const float* attn_mean, const float* map_p, int L, int B, int N, int H, float alpha, int G, int S,
                      float* relevance, float* heatmap, cudaStream_t st) {
  DFD_REQUIRE(attn_mean && map_p && relevance, DFD_ERR_BAD_ARG, "attention_rollout: null pointer");
  DFD_REQUIRE(L >= 0 && B > 0 && N > 0 && H > 0, DFD_ERR_SHAPE, "attention_rollout: bad shape");
  DFD_REQUIRE(B <= 65535, DFD_ERR_SHAPE, "attention_rollout: B must be <= 65535");
  DFD_REQUIRE(alpha >= 0.f && alpha <= 1.f, DFD_ERR_BAD_ARG, "attention_rollout: alpha must be in [0, 1]");
  DFD_REQUIRE(heatmap == nullptr || ((int64_t)G * G == N && S > 0 && S <= 65535), DFD_ERR_SHAPE,
              "attention_rollout: the heatmap needs G*G == N and 0 < S <= 65535");
  const int smem = (((N + 3) & ~3) + (kRollThreads / 32) * kRollCols) * 4;
  DFD_REQUIRE(smem <= 200 * 1024, DFD_ERR_UNSUPPORTED, "attention_rollout: N=%d too long", N);
  static SmemOptIn smem_once;
  if (int rc = ensure_dynamic_smem(smem_once, rollout_step_kernel, 200 * 1024)) return rc;
  // the steps alternate between relevance and a scratch vector so that the last one lands in relevance
  float* scratch = nullptr;
  if (L > 0) DFD_CUDA(cudaMallocAsync(&scratch, (size_t)B * N * sizeof(float), st));
  float* cur = (L % 2 == 0) ? relevance : scratch;
  float* nxt = (L % 2 == 0) ? scratch : relevance;
  int launches = 1;
  rollout_seed_kernel<<<(unsigned)(((int64_t)B * N + 255) / 256), 256, 0, st>>>(map_p, cur, B, N, H);
  int rc = cudaGetLastError() == cudaSuccess ? DFD_OK : DFD_ERR_CUDA;
  for (int l = L - 1; l >= 0 && rc == DFD_OK; --l, ++launches) {
    rollout_step_kernel<<<dim3((N + kRollCols - 1) / kRollCols, B), kRollThreads, smem, st>>>(
        attn_mean + (int64_t)l * B * N * N, cur, nxt, N, alpha);
    if (cudaGetLastError() != cudaSuccess) rc = DFD_ERR_CUDA;
    float* tmp = cur;
    cur = nxt;
    nxt = tmp;
  }
  if (scratch) DFD_CUDA(cudaFreeAsync(scratch, st));
  if (rc != DFD_OK) {
    set_last_error("attention_rollout: kernel launch failed");
    return rc;
  }
  g_launches.fetch_add(launches, std::memory_order_relaxed);
  if (heatmap) return upsample_bilinear(relevance, (float)N, heatmap, B, G, G, S, st);
  return DFD_OK;
}

}  // namespace dfd

extern "C" DFD_API int dfd_attention_probs(const void* qkv, int64_t ldqkv, int B, int N, int H, int hd, float scale,
                                           int per_head, float* out, void* stream) {
  return dfd::attention_probs(qkv, ldqkv, B, N, H, hd, scale, per_head, out, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" DFD_API int dfd_attention_rollout(const float* attn_mean, const float* map_p, int L, int B, int N, int H,
                                             float alpha, int G, int S, float* relevance, float* heatmap, void* stream) {
  return dfd::attention_rollout(attn_mean, map_p, L, B, N, H, alpha, G, S, relevance, heatmap,
                                reinterpret_cast<cudaStream_t>(stream));
}

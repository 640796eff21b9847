/*
 * dfd.h — C ABI of libdfd.so, the B200 (sm_100a) implementation of the deepfake-detection hot path
 * (SigLIP-2 ViT forward + FreqMLP spectrum features + fusion head + temperature/CORAL scoring).
 *
 * The reference (joesound212985/Deepfake-Detection-using-CLIP-Based-SigLIP-2-Vision-Transformers)
 * has no FFI of its own: its seam is Python duck typing of nn.Modules (SURVEY.md §8b).  Each entry
 * point below therefore cites the reference Python call it replaces (file:line under /root/reference,
 * or HF: = transformers/models/siglip/modeling_siglip.py which the reference calls at
 * Siglip2sidafrozen.py:753,787).  INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - every call is enqueue-only on `stream` (a cudaStream_t passed as void*), never synchronises,
 *     except the *_host entry points (which copy, run and synchronise) and dfd_engine_create/destroy;
 *   - return value: 0 = ok, negative = error (enum below); dfd_last_error() gives the text
 *     (thread-local).  No exceptions or aborts cross the ABI.  There is NO CPU fallback: without a
 *     CUDA device every compute entry point returns DFD_ERR_NO_DEVICE / DFD_ERR_CUDA.
 *   - bf16 tensors are row-major with an explicit leading dimension in ELEMENTS.
 */
#ifndef DFD_H_
#define DFD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define DFD_API
#else
#define DFD_API __attribute__((visibility("default")))
#endif

enum {
  DFD_OK = 0,
  DFD_ERR_BAD_ARG = -1,
  DFD_ERR_SHAPE = -2,
  DFD_ERR_UNSUPPORTED = -3,
  DFD_ERR_CUDA = -4,
  DFD_ERR_NO_DEVICE = -5,
  DFD_ERR_UNIMPLEMENTED = -6,
  DFD_ERR_STATE = -7
};

DFD_API const char* dfd_last_error(void);
DFD_API int dfd_version(void);
/* Number of kernels launched by this library in the calling process since load (bench "gpu_launches"). */
DFD_API int64_t dfd_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Op level (each is one kernel family; the engine below strings them together)
 * ---------------------------------------------------------------------------------------------- */

/* Epilogue of the tcgen05 GEMM.  out = epi(A·Wᵀ):
 *   v = acc                                   (fp32, TMEM)
 *   if (ln_colsum) v = rstd_m·(v − mean_m·ln_colsum[n])      — LayerNorm folded through the GEMM:
 *                     mean/rstd from ln_rowstats[m] = (Σx, Σx²) over ln_dim columns, eps ln_eps
 *   if (bias)     v += bias[n]
 *   if (act == 1) v = gelu_tanh(v)             HF:modeling_siglip.py:323-327 (gelu_pytorch_tanh)
 *      act == 2: exact erf GELU, act == 3: sigmoid   (nn.GELU() / nn.Sigmoid() of SegFormerStrongDecoder,
 *                                                     Siglip2sidafrozen.py:704-722)
 *   if (pos)      v += pos[(m % pos_rows)·N + n]   HF:modeling_siglip.py:179-185 (position embedding)
 *   if (residual) v += residual[m·ldr + n]     HF:modeling_siglip.py:354,359 (residual adds)
 *   C[m·ldc + n] = bf16(v)
 *   if (stats_out) stats_out[c][m] = (Σ bf16(v), Σ bf16(v)²) over the columns [64c, 64c+64) of row m — one partial per
 *                  64-column chunk, layout [ceil(N/64)][M][2] fp32, every slot written exactly once (no atomics, no
 *                  zero-fill needed); a consumer GEMM reads them back through ln_rowstats with ln_parts = ceil(N/64)
 *                  and adds them in chunk order, so the LayerNorm-folded path is bit-reproducible
 */
typedef struct dfd_gemm_epilogue {
  const float* bias;         /* [N] fp32 or NULL */
  int act;                   /* 0 none, 1 gelu_tanh, 2 gelu_erf, 3 sigmoid */
  const float* pos;          /* [pos_rows, N] fp32 or NULL */
  int pos_rows;
  const void* residual;      /* bf16 [M, ldr] or NULL; may alias C */
  int64_t ldr;
  const float* ln_rowstats;  /* [ln_parts][M][2] fp32 partial (Σx, Σx²) per row, or NULL */
  const float* ln_colsum;    /* [N] fp32 */
  int ln_dim;
  float ln_eps;
  float* stats_out;          /* [ceil(N/64)][M][2] fp32 partials (see above), or NULL */
  int residual_op;           /* 0: v += residual (default), 1: v *= residual (gating: Siglip2sidafrozen.py:737) */
  int ln_parts;              /* partial pairs per row in ln_rowstats; 0 or 1 = one [M,2] pair per row (whole-row sums) */
  void* residual_lo;         /* bf16 or NULL: low half of a two-bf16 residual stream.  With it the epilogue value is
                              * v = ... + residual + residual_lo (read only when residual is given), C = hi = bf16(v) and
                              * residual_lo = bf16(v - hi) is written back (in place), so the stream carries ~16 mantissa bits
                              * across layers like the fp32 residual of the reference's autocast path.  Layout (private to the
                              * epilogue and dfd_layernorm_bf16, coalesced for the epilogue's row-per-lane mapping):
                              * [ceil(M/128)][ceil(N/64)][8][128][8] = (row block, 64-column chunk, 8-column group, row, column) */
} dfd_gemm_epilogue;

/* C[M,N] (bf16) = epi(A[M,K] (bf16, lda) · W[N,K]ᵀ (bf16, ldw)), fp32 accumulate in TMEM.
 * Replaces nn.Linear / nn.Conv2d-as-GEMM under bf16 autocast: HF:modeling_siglip.py:285-287 (q/k/v),
 * :308 (out_proj), :324,326 (fc1/fc2), :178 (patch embedding).  Requires K%8==0, N%8==0, 16-byte
 * aligned pointers and leading dimensions that are multiples of 8 elements. */
DFD_API int dfd_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, void* C,
                          int64_t ldc, int M, int N, int K, const dfd_gemm_epilogue* epi,
                          void* stream);

/* Host-only view of the GEMM's persistent schedule (no GPU needed): the tile index (m_block * num_n + n_tile, N fastest) that
 * work unit `unit` of `units` (CTAs or CTA pairs) processes in round `round`, or -1 if it has none.  Each round covers `units`
 * consecutive tiles, rotated between rounds so that every unit cycles through all n-tiles (gemm_tcgen05.cu: sched_rotation). */
DFD_API int dfd_gemm_schedule(int num_tiles, int num_n, int units, int unit, int round);
/* Test / audit hooks: which kernel instantiation the last dfd_gemm_bf16[_tile] call of this process launched, encoded
 * as tile_n + 1000·CTAs-per-tile + 10000·has_residual + 100000·EPI (EPI: 0 generic, 1 LN fold + bias, 2 LN fold + bias +
 * tanh-GELU, 3 bias + residual + row statistics, 4 bias + residual, 5 bias, 6 bias + tanh-GELU, 7 = 3 on a two-bf16
 * residual stream), and how often a given
 * instantiation has been launched since load (-1: no such kernel).  The parity tests use them to prove that the
 * specialised kernels bench.py times are the ones being compared with the oracle. */
DFD_API int dfd_gemm_last_variant(void);
DFD_API int64_t dfd_gemm_variant_launches(int variant);

/* y[M,D] (bf16) = LayerNorm(x[M,D] (bf16)) · gamma + beta, fp32 statistics, eps as given.
 * HF:modeling_siglip.py:348,357 (layer_norm1/2), :618 (post_layernorm).  lo = NULL: the rows are x alone; otherwise
 * they are the two-bf16 sum x + lo, lo in the tiled layout of dfd_gemm_epilogue.residual_lo. */
DFD_API int dfd_layernorm_bf16(const void* x, int64_t ldx, const void* lo, void* y, int64_t ldy, const float* gamma,
                               const float* beta, int M, int D, float eps, void* stream);

/* Non-causal multi-head attention over packed qkv[B·N, 3·H·hd] (bf16; q | k | v column blocks, head h at
 * columns h·hd) -> out[B·N, H·hd] (bf16).  softmax(q·kᵀ·scale) in fp32.
 * HF:modeling_siglip.py:229-249,293-306 (SDPA, is_causal=False). hd in {64,72}. */
DFD_API int dfd_attention_bf16(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N,
                               int H, int hd, float scale, void* stream);

/* Same, with the kernel chosen explicitly (A/B tests): impl 5 = dual-query-tile tcgen05 kernel (what dfd_attention_bf16
 * runs for N > 128), impl 2 = persistent single-tile tcgen05 kernel (N <= 128).  Other values: DFD_ERR_BAD_ARG. */
DFD_API int dfd_attention_bf16_impl(const void* qkv, int64_t ldqkv, void* out, int64_t ldo, int B, int N,
                                    int H, int hd, float scale, int impl, void* stream);

/* Fused preprocess + im2col: pixels -> bf16 patch matrix A[B·G·G, Kpad] with column order (c, ky, kx)
 * (= conv weight [D,3,P,P] flattened), value (u8/255 − 0.5)/0.5 (ToTensor + Normalize(.5,.5):
 * inference_ai_human_images.py:200-204; train_fusion_head_only.py:67-74), optional resize of the
 * source to S×S first (resize_mode: 0 none (Hin==S), 1 nearest — train_fusion_head_only.py:103-104,
 * 2 bilinear align_corners=False — cifake_binary_classifier.py:716-717).  Only pixels
 * [0, G·P) of each axis are read (conv padding='valid': HF:modeling_siglip.py:124-130).
 * resize_mode | DFD_FLIP_H reads every source image mirrored left-right first (RandomHorizontalFlip(p=1) of the TTA
 * "H-Flip" transform, inference_ai_human_images.py:207-214): the second TTA pass re-uses the resident pixels.
 * pix_format: 0 = u8 NHWC [B,Hin,Win,3]; 1 = f32 NCHW [B,3,Hin,Win] already normalised. */
#define DFD_FLIP_H 0x10
DFD_API int dfd_patchify(const void* pixels, int pix_format, int B, int Hin, int Win, int S, int P,
                         int resize_mode, void* A, int64_t lda, void* stream);

/* MAP pooling head, single learned query per head (HF:modeling_siglip.py:639-654):
 * attn[b, h·hd..] = softmax_n(q[h]·k[b,n,h]·scale) · v[b,n,h]  with kv[B·N, 2·H·hd] (k | v), q fp32 [H·hd]
 * (the projected probe, batch independent).  out bf16 [B, H·hd]. */
DFD_API int dfd_map_attention_bf16(const void* kv, int64_t ldkv, const float* q, void* out,
                                   int64_t ldo, int B, int N, int H, int hd, float scale,
                                   void* stream);

/* Attention probabilities of the packed qkv that dfd_attention_bf16 reads (same layout, hd in {64,72}, any N >= 1):
 * P = softmax(q·kᵀ·scale) in fp32 (HF eager_attention_forward's attn_weights, HF:modeling_siglip.py:229-249), scale > 0.
 *   per_head = 1: out [B, H, N, N]  (what HF output_attentions returns)
 *   per_head = 0: out [B, N, N] = (1/H)·Σ_h P_h, summed on chip (the input of the rollout below)
 * S = q·kᵀ runs on the tensor cores; two sweeps over the keys (row statistics, then the probabilities). */
DFD_API int dfd_attention_probs(const void* qkv, int64_t ldqkv, int B, int N, int H, int hd, float scale, int per_head,
                                float* out, void* stream);

/* Attention rollout (Abnar & Zuidema 2020) seeded by the MAP probe, which is the query that forms the pooled embedding
 * (SigLIP has no CLS token): r = mean_h map_p[b, h, :], then for l = L-1 ... 0: r <- alpha·(r·attn_mean[l][b]) +
 * (1 - alpha)·r.  relevance [B][N] sums to 1.  heatmap (optional, needs G·G == N) [B][S][S] = the bilinear
 * (align_corners=False) resize of N·relevance on the G×G grid, so 1.0 is a uniform share.  Uses B·N floats of
 * stream-ordered scratch. */
DFD_API int dfd_attention_rollout(const float* attn_mean /*[L][B][N][N]*/, const float* map_p /*[B][H][N]*/, int L, int B,
                                  int N, int H, float alpha, int G, int S, float* relevance /*[B][N]*/,
                                  float* heatmap /*[B][S][S] or NULL*/, void* stream);

/* Classifier head on pooled embeddings (fp32 weights, fp32 math):
 *   f = pooled / (‖pooled‖₂ + norm_eps)                       inference_ai_human_images.py:149; +1e-6: train_fusion_head_only.py:106
 *   then, if kind >= 1: [kind 2: SE gate f·sigmoid(W2·relu(W1·f))  train_fusion_head_only.py:84-89,107]
 *                       -> LayerNorm(ln_g, ln_b, ln_eps) -> a chain of up to 6 dense layers (act: 0 none, 1 relu,
 *                          2 GELU(erf), 3 sigmoid); the last layer must have out_dim 1 and yields the logit.
 *     H-A  LN → Linear(D,D/2)+GELU → Linear(D/2,1)                       inference_ai_human_images.py:131-138
 *     H-B  SE → LN → Linear+GELU → Linear+GELU → Linear(·,1)             train_fusion_head_only.py:90-99,107-108
 *     H-D  LN → [1-token attention ≡ proj(v(x))] → 1-3 layer classifier  cifake_binary_classifier.py:643-684,728-749
 *   prototypes (optional [2,D] real,fake): p_proto = softmax([−‖f−p_r‖, −‖f−p_f‖])[1]        inference_ai_human_images.py:288-295
 * All weights are fp32 device pointers; every layer dimension must be <= dim. */
typedef struct dfd_dense_layer {
  const float *w, *b;       /* [out_dim, in_dim] row-major, [out_dim] (b may be NULL) */
  int out_dim, in_dim, act;
} dfd_dense_layer;
typedef struct dfd_head_weights {
  int kind;                 /* 0 = none (only normalise / prototypes), 1 = LN -> layers, 2 = SE -> LN -> layers */
  int dim;                  /* D */
  float norm_eps;           /* added to the L2 norm (0 or 1e-6) */
  float ln_eps;             /* classifier LayerNorm eps (1e-5) */
  const float *se_w1, *se_b1, *se_w2, *se_b2;          /* [D/16,D],[D/16],[D,D/16],[D] (kind 2) */
  const float *ln_g, *ln_b;                             /* [D] */
  int n_layers;
  dfd_dense_layer layers[6];
} dfd_head_weights;
DFD_API int dfd_head_fwd(const dfd_head_weights* w, const void* pooled_bf16, int64_t ldp, int B,
                         const float* prototypes, float* feat_out /*[B,D] normalised, or NULL*/,
                         float* z_sig /*[B] or NULL*/, float* p_proto /*[B] or NULL*/, void* stream);

/* 24-d frequency feature vector per gray 256×256 fp32 image in [0,1]
 * (train_fusion_head_only.py:150-226 = FreqMLP trainer.py:91-177; app copy deepfake-detector-v2/app.py:752-846):
 * 2-D FFT magnitude band energies, log-spectrum slope, sector anisotropy, phase entropy, 2-level Haar
 * energies, 3 SRM stencil moments.  lut = device pointer to the per-pixel table of the fft-shifted 256² grid that the host builds
 * once with the reference's own torch expressions (scoring.py build_freq_luts) and uploads: word [sx*256 + sy] (transposed, so
 * a warp walking a spectrum column reads it contiguously) = band id (bits 0-7: 0 low, 1 mid, 2 high) | log-radius bin (bits
 * 8-15, int8, -1 = not counted) | sector id (bits 16-23, int8, -1 = none); followed by 40 + 8 int32 bin populations (how many
 * grid positions fall in each log-radius bin / sector — geometry only).  eps: 1e-8 (trainers/app v2) or 1e-6 (appv3.py:570).  zscore!=0 applies the app's per-vector
 * z-scoring (app.py:840-846).  scratch: dfd_freq_scratch_bytes(B) bytes (per image the half spectrum plus the
 * column-pass partial slots and counters). */
DFD_API int dfd_freq_features(const float* gray256, int B, const int32_t* lut /*[256*256 + 48]*/, float eps, int zscore,
                              void* scratch, float* feats /*[B,24]*/, void* stream);
DFD_API int64_t dfd_freq_scratch_bytes(int B);

/* gray256: u8 RGB images [B,H,W,3] (NHWC) -> the 256x256 gray image in [0,1] (fp32) the frequency features are
 * computed from.  Replaces _pil_to_gray256_clahe / _pil_to_gray256 (train_fusion_head_only.py:142-148,
 * deepfake-detector-v2/app.py:736-749): Pillow convert("L") (integer ITU-R 601-2 luma) -> optional
 * cv2.createCLAHE(2.0,(8,8)).apply -> Pillow resize((256,256), BICUBIC) (22-bit fixed-point antialiased resample,
 * horizontal pass then vertical, u8 in between) -> /255.  Bit-exact with Pillow 12.2 / OpenCV 4.13 (oracle/gray_ref.py).
 * The per-axis coefficient tables are built on the HOST by dfd_resample_coeffs_host (double precision, Pillow's
 * precompute_coeffs + normalize_coeffs_8bpc; no GPU needed) and passed as device arrays: xmin[out], count[out],
 * kk[out][ksize] with ksize = dfd_resample_ksize(in_size, out, filter); gray256 takes BICUBIC tables with out = 256.
 * scratch: dfd_gray256_scratch_bytes(B,H,W). */
enum { DFD_FILTER_BILINEAR = 2, DFD_FILTER_BICUBIC = 3 };   /* PIL.Image.BILINEAR / BICUBIC */
DFD_API int dfd_resample_ksize(int in_size, int out_size, int filter);
DFD_API int dfd_resample_coeffs_host(int in_size, int out_size, int filter, int32_t* xmin_host, int32_t* count_host,
                                     int32_t* kk_host);
DFD_API int64_t dfd_gray256_scratch_bytes(int B, int H, int W);

/* Pillow Image.resize((OW,OH), BILINEAR|BICUBIC) for a batch of same-size 8-bit images with 1 or 3 interleaved channels
 * — what torchvision transforms.Resize((S,S)) does to the PIL image in the reference's preprocess
 * (inference_ai_human_images.py:200-204, train_fusion_head_only.py:67-74) and what open_clip's preprocess does with
 * BICUBIC.  Same fixed-point arithmetic as above, bit-exact; tables from dfd_resample_coeffs_host with the same filter.
 * scratch: B*H*OW*C bytes.
 * dfd_resize_u8 and dfd_gray256 read a rectangle of a larger image — rows row_stride bytes apart, consecutive rectangles
 * image_stride bytes apart (0 / 0 = dense).  A crop (x0, y0, w, h) of a resident u8 RGB image of width Wi is
 * (base + (y0·Wi + x0)·3, row_stride = Wi·3): the multicrop views of detect_core (deepfake-detector-v2/app.py:1418-1430,
 * appv3.py:3315-3350) and the patch-grid cells (:1461-1485) come from one upload, without a copy per view. */
DFD_API int dfd_resize_u8(const void* src, int64_t row_stride, int64_t image_stride, int B, int H, int W, int C, int OH,
                          int OW, const int32_t* xmin_w, const int32_t* count_w, const int32_t* kk_w, int ksize_w,
                          const int32_t* xmin_h, const int32_t* count_h, const int32_t* kk_h, int ksize_h, void* scratch,
                          void* dst, void* stream);
DFD_API int dfd_gray256(const void* rgb_u8, int64_t row_stride, int64_t image_stride, int B, int H, int W, int clahe,
                        const int32_t* xmin_w, const int32_t* count_w, const int32_t* kk_w, int ksize_w,
                        const int32_t* xmin_h, const int32_t* count_h, const int32_t* kk_h, int ksize_h, void* scratch,
                        float* gray256 /*[B,256,256]*/, void* stream);

/* Per-channel CLAHE of dense u8 images [B,H,W,C] (C = 1 or 3): cv2.createCLAHE(clipLimit=2.0, tileGridSize=(8,8)).apply on
 * every channel separately — `apply_clahe`, the first stage of the reference's training preprocess
 * (train_fusion_head_only.py:60-65), ahead of Resize (dfd_resize_u8) and ToTensor + Normalize (the patch kernel).  Bit-exact with
 * OpenCV 4.13 (oracle/gray_ref.py:clahe_u8).  scratch: dfd_clahe_scratch_bytes(B, C) bytes; src and dst must differ. */
DFD_API int64_t dfd_clahe_scratch_bytes(int B, int C);
DFD_API int dfd_clahe_u8(const void* src, int B, int H, int W, int C, void* scratch, void* dst, void* stream);

/* FreqMLP (generation 2) forward + backward of mean BCE-with-logits: one training step's
 * `logits = model(xb); loss = criterion(logits, yb); loss.backward()` ("FreqMLP trainer.py":366-369; model :218-301).
 * params6494 = the state dict without its two buffers, flattened in order: contrast.alpha[24], contrast.beta[24],
 * band.gates[4], blocks.{0,1}.{norm.weight[24], norm.bias[24], fc1.weight[64,24], fc1.bias[64], fc2.weight[24,64],
 * fc2.bias[24]}, head.weight[24], head.bias, temp.T.  mean24/std24 = FeatureNormalizer buffers.
 * loss_sum[1] and grads[6494] are ACCUMULATED partial sums with the factor inv_global_batch applied (zero them, then
 * all-reduce-sum across ranks).  grads == NULL: forward only (eval; no dropout).  dropout_p: the blocks' nn.Dropout
 * (0.05 in the reference's train mode; masks come from a counter hash of (seed, sample, element), so they match torch's
 * only in distribution; 0 = deterministic). */
DFD_API int dfd_freqmlp_fwd_bwd(const float* params6494, const float* mean24, const float* std24, const float* feats,
                                const float* y, int B, float inv_global_batch, float dropout_p, uint32_t seed,
                                float* loss_sum, float* grads, float* logits, void* stream);

/* SegFormerStrongDecoder / SigLIP2_MTL (Siglip2sidafrozen.py:698-803), the parts that are not GEMMs.  Activations are
 * token-major bf16 [B·H·W, C] with a leading dimension; the LinearProj and 1x1-convolution layers are dfd_gemm_bf16 calls
 * (act 2 = erf GELU, act 3 = sigmoid, residual_op 1 = gating).
 *   dfd_dwconv3x3_bf16     nn.Conv2d(E, E, 3, padding=1, groups=E) (:711); w9 = weight[E,1,3,3] flattened to [E,9] fp32
 *   dfd_seg_head_upsample  self.head(F.interpolate(x, (S,S), mode="bilinear", align_corners=False)) (:740-741) computed as
 *                          upsample(head(x)) — both linear, so they commute; low_scratch: B·H·W floats; out [B,S,S] fp32
 *   dfd_linear_small       nn.Linear(hidden, 3) on the pooled embedding (:777,789): x bf16 [B,K], w fp32 [N,K] */
DFD_API int dfd_dwconv3x3_bf16(const void* x, int64_t ldx, const float* w9, const float* bias, void* out, int64_t ldo,
                               int B, int H, int W, int E, void* stream);
DFD_API int dfd_seg_head_upsample(const void* x, int64_t ldx, const float* w, float bias, int B, int H, int W, int E,
                                  int S, float* low_scratch, float* out, void* stream);
DFD_API int dfd_linear_small(const void* x, int64_t ldx, const float* w, const float* bias, float* out, int B, int N,
                             int K, void* stream);

/* Score epilogue: FreqMLP + fusion + temperature + CORAL, one warp per sample.
 *  gen 1 (shipped siglip/ safetensors files; deepfake-detector-v2/app.py:601-628,691-709,1355-1396):
 *     z_freq = FreqMLP_G1(feats)  (SafeLayerNorm eps 1e-5 → Linear(24,64) → GELU(erf) → Linear(64,1); eval noise omitted)
 *     z = fc·[σ(z_sig), σ(z_freq/freq_temp)] + b
 *  gen 2 (train_fusion_head_only.py:230-317):
 *     z_freq = FreqMLP_G2(feats) ; z = AdaptiveFusionHead(z_freq, z_sig)
 *  then z_scaled = z / max(coral_temp,1e-3); p_raw = σ(z_scaled); CORAL probs/argmax/μ/var/entropy/blend.
 * If feats==NULL, z_freq_in[B] is used directly.  All outputs are SoA fp32 (risk_idx int32), any may be NULL. */
typedef struct dfd_score_weights {
  int gen;                      /* 1 or 2 */
  /* G1 FreqMLP */
  const float *g1_ln_w, *g1_ln_b, *g1_w1, *g1_b1, *g1_w2, *g1_b2;
  /* G1 fusion */
  float g1_fc_w[2], g1_fc_b, freq_temp;
  /* G2 FreqMLP: normer.mean/std, contrast.alpha/beta, band.gates[4], blocks{0,1}.{norm.w,norm.b,fc1.w,fc1.b,fc2.w,fc2.b}, head.w, head.b, temp.T */
  const float *g2_mean, *g2_std, *g2_alpha, *g2_beta, *g2_gates;
  const float *g2_blk[2][6];
  const float *g2_head_w, *g2_head_b;
  float g2_temp;
  /* G2 fusion: mlp.0.{w[32,3],b[32]}, mlp.2.{w[2,32],b[2]}, temp.T */
  const float *f2_w0, *f2_b0, *f2_w1, *f2_b1;
  float f2_temp;
  /* CORAL */
  float coral_cuts[4];          /* logit-space cutpoints */
  float coral_temp;
} dfd_score_weights;
typedef struct dfd_scores {
  float *z_freq, *z, *z_scaled, *p_raw, *risk_probs /*[B,5]*/, *p_coral, *entropy, *p_blend;
  int32_t* risk_idx;
} dfd_scores;
DFD_API int dfd_score_epilogue(const dfd_score_weights* w, const float* z_sig, const float* feats,
                               const float* z_freq_in, int B, const dfd_scores* out, void* stream);

/* AdaptiveFusionHead forward + backward for head-only training (train_fusion_head_only.py:303-317,423-425):
 * loss = mean BCEWithLogits(head(z_freq,z_sig), y) over the GLOBAL batch (inv_global_batch = 1/B_global);
 * grads[195] (order mlp.0.weight[32,3], mlp.0.bias[32], mlp.2.weight[2,32], mlp.2.bias[2], temp.T) and
 * loss_sum[1] are ACCUMULATED (caller zeroes), so ranks allreduce(sum) them afterwards. logits[B] optional. */
DFD_API int dfd_fusion_fwd_bwd(const float* params195, const float* z_freq, const float* z_sig,
                               const float* y, int B, float inv_global_batch, float* loss_sum,
                               float* grads195, float* logits, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Engine level (owns packed weights + workspaces; one per (device, model config))
 * ---------------------------------------------------------------------------------------------- */
typedef struct dfd_engine dfd_engine;
typedef struct dfd_config {
  int image_size, patch, hidden, inter, layers, heads; /* tokens = (image_size/patch)^2, hd = hidden/heads */
  int gelu_tanh;   /* 1 = HF gelu_pytorch_tanh (default) */
  float ln_eps;    /* 1e-6 */
  int fuse_ln;     /* 1 = LayerNorm folded into the QKV / fc1 / MAP-kv GEMM epilogues (row stats from the
                      producing GEMM); 0 = stand-alone LayerNorm kernels */
} dfd_config;

DFD_API int dfd_engine_create(const dfd_config* cfg, int device, int max_batch, dfd_engine** out);
DFD_API int dfd_engine_destroy(dfd_engine* e);
/* Copy + repack one tensor (device or host pointer; dtype 0=f32, 1=bf16) under its canonical HF name,
 * e.g. "embeddings.patch_embedding.weight", "encoder.layers.3.self_attn.q_proj.bias",
 * "head.attention.in_proj_weight" (Siglip2sidafrozen.py:753 state dict; SURVEY.md App. B). */
DFD_API int dfd_engine_set_tensor(dfd_engine* e, const char* name, const void* data, int dtype,
                                  int ndim, const int64_t* shape, int on_host);
/* Call once after all tensors are set: folds LN affine into weights (fuse_ln), projects the probe. */
DFD_API int dfd_engine_finalize(dfd_engine* e);
/* pixels -> pooled[B,D] (bf16) (+ optional last_hidden[B·N,D] bf16 = post_layernorm output).
 * HF SiglipVisionModel.forward (HF:modeling_siglip.py:586-625) == open_clip encode_image
 * (inference_ai_human_images.py:148). */
DFD_API int dfd_engine_forward(dfd_engine* e, const void* pixels, int pix_format, int B, int Hin,
                               int Win, int resize_mode, void* pooled, void* last_hidden,
                               void* stream);
/* Per-layer hidden states (HF output_hidden_states=True, Siglip2sidafrozen.py:787-793): when buf != NULL the following
 * forwards also copy the embedding output and each encoder layer's output to buf as bf16 [L+1][B][N][D] (B = the
 * batch of that forward).  NULL switches the tap off. */
DFD_API int dfd_engine_set_hidden_tap(dfd_engine* e, void* buf);
/* Attention maps (HF output_attentions=True): when attn != NULL the following forwards write layer l's attention
 * probabilities to attn + l·(per-layer size), in the layout of dfd_attention_probs(per_head): fp32 [L][B][H][N][N]
 * (per_head = 1) or the head mean [L][B][N][N] (per_head = 0).  When map_p != NULL the MAP pooling kernel also writes the
 * probe attention, fp32 [B][H][N].  NULL / NULL switches the tap off.  While it is on, forwards run eagerly (no graph
 * replay); its launches are not profiled. */
DFD_API int dfd_engine_set_attention_tap(dfd_engine* e, float* attn, int per_head, float* map_p);
/* CUDA graphs of the forward: with enable != 0 a call signature (pixels / pooled / last_hidden pointers, batch, input geometry)
 * runs eagerly the first time, is captured the second time and replayed with one cudaGraphLaunch on the caller's stream
 * afterwards (tensor maps and arguments baked in; 16 signatures kept, LRU).  Keep the buffers of a serving loop stable to
 * benefit.  enable == 0 drops every captured graph.  dfd_engine_graph_replays counts replays since creation. */
DFD_API int dfd_engine_set_graphs(dfd_engine* e, int enable);
/* Residual-stream precision: 0 (default) one bf16 tensor, rounded after each of the 2·L residual additions; 1 two bf16 tensors
 * (hi + lo, ~16 mantissa bits), which accumulates the additions like the fp32 residual stream of the reference's autocast path
 * (HF:modeling_siglip.py:352,359).  Allocates one more [max_batch·N, D] bf16 buffer on first use. */
DFD_API int dfd_engine_set_precise_residual(dfd_engine* e, int enable);
DFD_API int64_t dfd_engine_graph_replays(const dfd_engine* e);
DFD_API int64_t dfd_engine_workspace_bytes(const dfd_engine* e);
/* Measurement aid (bench.py roofline): dfd_engine_profile(e, n) with n > 0 makes dfd_engine_forward bracket every launch
 * with CUDA events on the caller's stream, with room for n forwards (launches past that are not recorded); n = 0 switches
 * it off.  dfd_engine_profile_read waits for the last recorded event, sums the durations recorded since the previous read
 * per kernel family and clears the record.  ms[9] / count[9] index: 0 GEMM (patch embedding, pooling head), 1 attention,
 * 2 LayerNorm, 3 patchify, 4 MAP attention, 5 qkv GEMM, 6 out-projection GEMM, 7 fc1 GEMM, 8 fc2 GEMM. */
DFD_API int dfd_engine_profile(dfd_engine* e, int forwards);
DFD_API int dfd_engine_profile_read(dfd_engine* e, float* ms, int* count);

#ifdef __cplusplus
}
#endif
#endif /* DFD_H_ */

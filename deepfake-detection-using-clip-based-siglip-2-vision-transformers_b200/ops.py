"""Torch-tensor wrappers over the op-level C ABI of libdfd.so (include/dfd.h).

PyTorch is used here only for device memory and streams; every function enqueues hand-written
sm_100a kernels on the current CUDA stream and returns torch tensors.  There is no CPU fallback:
non-CUDA tensors raise.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import torch

from . import _lib
from ._lib import GemmEpilogue, HeadWeights, ScoreWeights, Scores, check, current_stream


def _need_cuda(*ts):
    cur = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("dfd ops need CUDA tensors (there is no CPU fallback)")
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            # the kernels are launched on the current device's stream: pointers of another device would fault (or go
            # through peer access) instead of failing here
            raise RuntimeError(f"dfd ops launch on the current device (cuda:{cur}) but an argument lives on {t.device}; "
                               f"wrap the call in `with torch.cuda.device({t.device.index}):`")


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def gemm_bf16(a: torch.Tensor, w: torch.Tensor, *, bias=None, act: int = 0, pos=None, residual=None,
              ln_rowstats=None, ln_colsum=None, ln_dim: int = 0, ln_eps: float = 1e-6, stats_out=None,
              out: Optional[torch.Tensor] = None, tile_n: int = 0, residual_op: int = 0,
              residual_lo: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[M,N] = epilogue(a[M,K] @ w[N,K].T); bf16 in/out, fp32 accumulate in TMEM (dfd_gemm_bf16).
    act: 0 none, 1 gelu_tanh, 2 gelu_erf, 3 sigmoid; residual_op: 0 add, 1 multiply.
    stats_out: fp32 [ceil(N/64), M, 2] per-chunk (sum, sum of squares) of the bf16 output rows (written, not
    accumulated); ln_rowstats: fp32 [M, 2] whole-row sums or [parts, M, 2] partials (a previous GEMM's stats_out)."""
    _need_cuda(a, w, bias, pos, residual, out)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16
    assert a.dim() == 2 and w.dim() == 2 and a.shape[1] == w.shape[1]
    assert a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.bfloat16, device=a.device)
    epi = GemmEpilogue()
    epi.bias = _p(bias)
    epi.act = act
    epi.pos = _p(pos)
    epi.pos_rows = 0 if pos is None else pos.shape[0]
    epi.residual = _p(residual)
    epi.ldr = 0 if residual is None else residual.stride(0)
    epi.ln_rowstats = _p(ln_rowstats)
    epi.ln_colsum = _p(ln_colsum)
    epi.ln_dim = ln_dim
    epi.ln_eps = ln_eps
    epi.stats_out = _p(stats_out)
    epi.residual_op = residual_op
    epi.ln_parts = 0
    # two-bf16 residual stream: residual_lo (tiled, ops.lo_to_tiled) is read with the residual and rewritten in place with the
    # low half of the new value (see dfd_gemm_epilogue.residual_lo)
    epi.residual_lo = _p(residual_lo)
    if residual_lo is not None:
        assert residual_lo.dtype == torch.bfloat16 and residual_lo.is_contiguous() and \
            tuple(residual_lo.shape) == ((M + 127) // 128, (N + 63) // 64, 8, 128, 8), "residual_lo: see ops.lo_to_tiled"
    if ln_rowstats is not None:
        assert ln_rowstats.dtype == torch.float32 and ln_rowstats.is_contiguous() and ln_rowstats.shape[-2:] == (M, 2)
        epi.ln_parts = ln_rowstats.shape[0] if ln_rowstats.dim() == 3 else 1
    if stats_out is not None:
        assert stats_out.dtype == torch.float32 and stats_out.is_contiguous() and \
            tuple(stats_out.shape) == ((N + 63) // 64, M, 2)
    lib = _lib.load()
    if tile_n:
        rc = lib.dfd_gemm_bf16_tile(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), out.data_ptr(),
                                    out.stride(0), M, N, K, C.byref(epi), tile_n, current_stream())
    else:
        rc = lib.dfd_gemm_bf16(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), out.data_ptr(),
                               out.stride(0), M, N, K, C.byref(epi), current_stream())
    check(rc)
    return out


def lo_to_tiled(lo: torch.Tensor) -> torch.Tensor:
    """Row-major bf16 [M, N] -> the tiled layout of dfd_gemm_epilogue.residual_lo: [ceil(M/128)][ceil(N/64)][8][128][8]."""
    M, N = lo.shape
    Mp, Np = (M + 127) // 128 * 128, (N + 63) // 64 * 64
    pad = torch.zeros((Mp, Np), dtype=lo.dtype, device=lo.device)
    pad[:M, :N] = lo
    return pad.view(Mp // 128, 128, Np // 64, 8, 8).permute(0, 2, 3, 1, 4).contiguous()


def lo_from_tiled(t: torch.Tensor, M: int, N: int) -> torch.Tensor:
    """Inverse of lo_to_tiled."""
    mb, nc = t.shape[0], t.shape[1]
    return t.permute(0, 3, 1, 2, 4).reshape(mb * 128, nc * 64)[:M, :N].contiguous()


def layernorm_bf16(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-6,
                   lo: Optional[torch.Tensor] = None) -> torch.Tensor:
    """LayerNorm of the bf16 rows of x (dfd_layernorm_bf16); with lo (tiled, ops.lo_to_tiled) of the two-bf16 rows x + lo."""
    _need_cuda(x, gamma, beta, lo)
    assert x.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1
    assert gamma.dtype == torch.float32 and beta.dtype == torch.float32
    M, D = x.shape
    if lo is not None:
        assert lo.dtype == torch.bfloat16 and lo.is_contiguous() and \
            tuple(lo.shape) == ((M + 127) // 128, (D + 63) // 64, 8, 128, 8), "lo: see ops.lo_to_tiled"
    y = torch.empty_like(x)
    check(_lib.load().dfd_layernorm_bf16(x.data_ptr(), x.stride(0), _p(lo), y.data_ptr(), y.stride(0), gamma.data_ptr(),
                                         beta.data_ptr(), M, D, eps, current_stream()))
    return y


def attention_bf16(qkv: torch.Tensor, B: int, N: int, H: int, hd: int, scale: Optional[float] = None,
                   impl: Optional[int] = None) -> torch.Tensor:
    """qkv [B*N, 3*H*hd] (q | k | v) -> [B*N, H*hd]; non-causal softmax(q k^T scale) v.
    impl None = product dispatch (2 for N <= 128, 5 above); 5 / 2 force the dual-query-tile / single-tile persistent
    tcgen05 kernel for any N (A/B tests); any other value is rejected (DFD_ERR_BAD_ARG)."""
    _need_cuda(qkv)
    assert qkv.dtype == torch.bfloat16 and qkv.shape == (B * N, 3 * H * hd) and qkv.stride(1) == 1
    out = torch.empty((B * N, H * hd), dtype=torch.bfloat16, device=qkv.device)
    scale = (1.0 / math.sqrt(hd)) if scale is None else scale
    lib = _lib.load()
    if impl is None:
        rc = lib.dfd_attention_bf16(qkv.data_ptr(), qkv.stride(0), out.data_ptr(), out.stride(0), B, N, H, hd, scale,
                                    current_stream())
    else:
        rc = lib.dfd_attention_bf16_impl(qkv.data_ptr(), qkv.stride(0), out.data_ptr(), out.stride(0), B, N, H, hd,
                                         scale, impl, current_stream())
    check(rc)
    return out


def attention_probs(qkv: torch.Tensor, B: int, N: int, H: int, hd: int, scale: Optional[float] = None,
                    per_head: bool = True) -> torch.Tensor:
    """The attention probabilities softmax(q k^T scale) of the packed qkv that attention_bf16 reads, in fp32:
    [B, H, N, N] with per_head, else the head mean [B, N, N]."""
    _need_cuda(qkv)
    assert qkv.dtype == torch.bfloat16 and qkv.dim() == 2 and qkv.shape[0] == B * N and qkv.stride(1) == 1
    shape = (B, H, N, N) if per_head else (B, N, N)
    out = torch.empty(shape, dtype=torch.float32, device=qkv.device)
    scale = (1.0 / math.sqrt(hd)) if scale is None else scale
    check(_lib.load().dfd_attention_probs(qkv.data_ptr(), qkv.stride(0), B, N, H, hd, scale, int(bool(per_head)),
                                          out.data_ptr(), current_stream()))
    return out


def attention_rollout(attn_mean: torch.Tensor, map_p: torch.Tensor, alpha: float = 0.5, heatmap_size: int = 0):
    """Attention rollout seeded by the MAP probe: attn_mean fp32 [L, B, N, N] (head-mean probabilities per layer),
    map_p fp32 [B, H, N].  Returns (relevance [B, N], heatmap [B, S, S] | None).  The heatmap (heatmap_size = S > 0,
    needs a square token grid) is the bilinear upsample of N·relevance, so 1.0 marks a uniform share."""
    _need_cuda(attn_mean, map_p)
    assert attn_mean.dtype == torch.float32 and attn_mean.dim() == 4 and attn_mean.is_contiguous()
    assert map_p.dtype == torch.float32 and map_p.dim() == 3 and map_p.is_contiguous()
    L, B, N, _ = attn_mean.shape
    H = map_p.shape[1]
    assert attn_mean.shape == (L, B, N, N) and map_p.shape == (B, H, N)
    rel = torch.empty((B, N), dtype=torch.float32, device=map_p.device)
    heat = (torch.empty((B, heatmap_size, heatmap_size), dtype=torch.float32, device=map_p.device)
            if heatmap_size > 0 else None)
    check(_lib.load().dfd_attention_rollout(attn_mean.data_ptr(), map_p.data_ptr(), L, B, N, H, float(alpha),
                                            math.isqrt(N), heatmap_size, rel.data_ptr(), _p(heat), current_stream()))
    return rel, heat


def map_attention_bf16(kv: torch.Tensor, q: torch.Tensor, B: int, N: int, H: int, hd: int,
                       scale: Optional[float] = None) -> torch.Tensor:
    _need_cuda(kv, q)
    assert kv.dtype == torch.bfloat16 and kv.shape == (B * N, 2 * H * hd) and kv.stride(1) == 1
    assert q.dtype == torch.float32 and q.numel() == H * hd
    out = torch.empty((B, H * hd), dtype=torch.bfloat16, device=kv.device)
    scale = (1.0 / math.sqrt(hd)) if scale is None else scale
    check(_lib.load().dfd_map_attention_bf16(kv.data_ptr(), kv.stride(0), q.data_ptr(), out.data_ptr(),
                                             out.stride(0), B, N, H, hd, scale, current_stream()))
    return out


def gemm_last_variant() -> dict:
    """Which kernel instantiation the last gemm_bf16 call launched: {'bn', 'cg', 'res', 'epi'} (dfd_gemm_last_variant)."""
    v = _lib.load().dfd_gemm_last_variant()
    return {"bn": v % 1000, "cg": v // 1000 % 10, "res": v // 10000 % 10, "epi": v // 100000}


def gemm_variant_launches(bn: int, cg: int, res: int, epi: int) -> int:
    """Launches of the gemm kernel instantiation <bn, cg, res, epi> by this process so far."""
    return int(_lib.load().dfd_gemm_variant_launches(bn + 1000 * cg + 10000 * res + 100000 * epi))


RESIZE_NONE, RESIZE_NEAREST, RESIZE_BILINEAR = 0, 1, 2
FLIP_H = 0x10   # or-ed into resize_mode: the source images are read mirrored left-right (DFD_FLIP_H)


def patchify(pixels: torch.Tensor, S: int, P: int, resize_mode: int = RESIZE_NONE, lda: Optional[int] = None) -> torch.Tensor:
    """u8 NHWC [B,H,W,3] or f32 NCHW [B,3,H,W] -> bf16 patch matrix [B*G*G, lda] (column order c,ky,kx)."""
    _need_cuda(pixels)
    pixels = pixels.contiguous()
    if pixels.dtype == torch.uint8:
        fmt, (B, Hin, Win, ch) = 0, pixels.shape
    elif pixels.dtype == torch.float32:
        fmt, (B, ch, Hin, Win) = 1, pixels.shape
    else:
        raise TypeError("patchify: pixels must be uint8 NHWC or float32 NCHW")
    assert ch == 3
    K = 3 * P * P
    lda = lda or (K + 63) // 64 * 64
    G = S // P
    A = torch.empty((B * G * G, lda), dtype=torch.bfloat16, device=pixels.device)
    check(_lib.load().dfd_patchify(pixels.data_ptr(), fmt, B, Hin, Win, S, P, resize_mode, A.data_ptr(), lda,
                                   current_stream()))
    return A


def _f32(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


ACT_NONE, ACT_RELU, ACT_GELU, ACT_SIGMOID = 0, 1, 2, 3


class HeadParams:
    """Device copy of a classifier head for dfd_head_fwd.
    kind 0: L2-normalise only; 1: LN -> dense chain; 2: SE gate -> LN -> dense chain.
    `layers` = [(weight [out,in], bias [out] | None, act), ...]; the last layer must have one output."""

    def __init__(self, kind: int, dim: int, norm_eps: float, device, ln=None, se=None, layers=(), ln_eps: float = 1e-5):
        self.kind, self.dim = kind, dim
        self._keep = []
        w = HeadWeights()
        w.kind, w.dim, w.norm_eps, w.ln_eps = kind, dim, norm_eps, ln_eps

        def put(t):
            if t is None:
                return None
            d = _f32(t, device)
            self._keep.append(d)
            return d.data_ptr()

        if ln is not None:
            w.ln_g, w.ln_b = put(ln[0]), put(ln[1])
        if se is not None:
            w.se_w1, w.se_b1, w.se_w2, w.se_b2 = (put(t) for t in se)
        assert len(layers) <= 6
        w.n_layers = len(layers)
        for i, (wt, bs, act) in enumerate(layers):
            w.layers[i].w, w.layers[i].b = put(wt), put(bs)
            w.layers[i].out_dim, w.layers[i].in_dim, w.layers[i].act = int(wt.shape[0]), int(wt.shape[1]), int(act)
        self.struct = w


def head_fwd(head: HeadParams, pooled: torch.Tensor, prototypes: Optional[torch.Tensor] = None,
             want_features: bool = False):
    """pooled bf16 [B,D] -> (features f32 [B,D] | None, z_sig f32 [B] | None, p_proto f32 [B] | None)."""
    _need_cuda(pooled, prototypes)
    assert pooled.dtype == torch.bfloat16 and pooled.dim() == 2 and pooled.stride(1) == 1
    B, D = pooled.shape
    assert D == head.dim
    dev = pooled.device
    feats = torch.empty((B, D), dtype=torch.float32, device=dev) if want_features else None
    z = torch.empty((B,), dtype=torch.float32, device=dev) if head.kind != 0 else None
    pp = None
    if prototypes is not None:
        assert prototypes.dtype == torch.float32 and prototypes.shape == (2, D) and prototypes.is_contiguous()
        pp = torch.empty((B,), dtype=torch.float32, device=dev)
    check(_lib.load().dfd_head_fwd(C.byref(head.struct), pooled.data_ptr(), pooled.stride(0), B, _p(prototypes),
                                   _p(feats), _p(z), _p(pp), current_stream()))
    return feats, z, pp


def freq_features(gray256: torch.Tensor, luts: torch.Tensor, eps: float = 1e-8, zscore: bool = False,
                  scratch: Optional[torch.Tensor] = None) -> torch.Tensor:
    """gray256 f32 [B,256,256] in [0,1] -> 24-d features f32 [B,24] (dfd_freq_features)."""
    _need_cuda(gray256)
    assert gray256.dtype == torch.float32 and gray256.shape[1:] == (256, 256) and gray256.is_contiguous()
    B = gray256.shape[0]
    lib = _lib.load()
    need = lib.dfd_freq_scratch_bytes(B)
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty((need,), dtype=torch.uint8, device=gray256.device)
    assert luts.dtype == torch.int32 and luts.numel() == 256 * 256 + 48 and luts.is_contiguous() and luts.device == gray256.device
    feats = torch.empty((B, 24), dtype=torch.float32, device=gray256.device)
    check(lib.dfd_freq_features(gray256.data_ptr(), B, luts.data_ptr(), eps, int(zscore), scratch.data_ptr(),
                                feats.data_ptr(), current_stream()))
    return feats


FILTERS = {"bilinear": 2, "bicubic": 3}   # PIL.Image.BILINEAR / BICUBIC


def resample_coeffs(in_size: int, out_size: int = 256, filter: str = "bicubic"):
    """Pillow's 8bpc resample tables for one axis (host, dfd_resample_coeffs_host): (xmin, count, kk) int32
    numpy arrays, kk [out_size, ksize].  Works without a GPU."""
    import numpy as np

    lib = _lib.load()
    f = FILTERS[filter]
    ks = lib.dfd_resample_ksize(in_size, out_size, f)
    xmin, cnt = np.zeros(out_size, np.int32), np.zeros(out_size, np.int32)
    kk = np.zeros((out_size, ks), np.int32)
    check(lib.dfd_resample_coeffs_host(in_size, out_size, f, xmin.ctypes.data, cnt.ctypes.data, kk.ctypes.data))
    return xmin, cnt, kk


_RESAMPLE_TABLES: dict = {}


def _resample_tables(size: int, device, out_size: int = 256, filter: str = "bicubic") -> tuple:
    key = (size, out_size, filter, str(device))
    if key not in _RESAMPLE_TABLES:
        _RESAMPLE_TABLES[key] = tuple(torch.from_numpy(a).to(device) for a in resample_coeffs(size, out_size, filter))
    return _RESAMPLE_TABLES[key]


def _rect_strides(images: torch.Tensor):
    """(tensor, row_stride_bytes, image_stride_bytes) of a u8 [B,H,W,C] tensor whose pixels are contiguous within a row — a dense
    batch or a rectangle cut out of a larger image (`img[y0:y1, x0:x1][None]`); anything else is copied."""
    B, H, W, Cn = images.shape
    if images.stride(3) != 1 or images.stride(2) != Cn or (H > 1 and images.stride(1) < W * Cn):
        images = images.contiguous()
    return images, images.stride(1) if H > 1 else W * Cn, images.stride(0) if B > 1 else 0


def resize_u8(images: torch.Tensor, out_h: int, out_w: int, filter: str = "bilinear") -> torch.Tensor:
    """u8 images [B,H,W,C] (C = 1 or 3, device; dense or a rectangle view of a larger image) -> [B,out_h,out_w,C] u8, bit-exact
    with PIL `Image.resize((out_w, out_h), BILINEAR|BICUBIC)` — torchvision `transforms.Resize` on PIL inputs
    (inference_ai_human_images.py:200-204)."""
    _need_cuda(images)
    assert images.dtype == torch.uint8 and images.dim() == 4 and images.shape[3] in (1, 3)
    images, rs, ims = _rect_strides(images)
    B, H, W, C = images.shape
    xw, cw, kw = _resample_tables(W, images.device, out_w, filter)
    xh, ch, kh = _resample_tables(H, images.device, out_h, filter)
    scratch = torch.empty((B, H, out_w, C), dtype=torch.uint8, device=images.device)
    out = torch.empty((B, out_h, out_w, C), dtype=torch.uint8, device=images.device)
    check(_lib.load().dfd_resize_u8(images.data_ptr(), rs, ims, B, H, W, C, out_h, out_w, xw.data_ptr(), cw.data_ptr(),
                                    kw.data_ptr(), kw.shape[1], xh.data_ptr(), ch.data_ptr(), kh.data_ptr(), kh.shape[1],
                                    scratch.data_ptr(), out.data_ptr(), current_stream()))
    return out


def clahe_u8(images: torch.Tensor) -> torch.Tensor:
    """Per-channel cv2 CLAHE(clipLimit 2.0, 8x8 tiles) of dense u8 images [B,H,W,C] (C = 1 or 3, device) -> u8 of the same shape,
    bit-exact with `for c in range(3): arr[:, :, c] = clahe.apply(arr[:, :, c])` (train_fusion_head_only.py:60-65) (dfd_clahe_u8)."""
    _need_cuda(images)
    assert images.dtype == torch.uint8 and images.dim() == 4 and images.shape[3] in (1, 3)
    images = images.contiguous()
    B, H, W, C = images.shape
    lib = _lib.load()
    scratch = torch.empty((lib.dfd_clahe_scratch_bytes(B, C),), dtype=torch.uint8, device=images.device)
    out = torch.empty_like(images)
    check(lib.dfd_clahe_u8(images.data_ptr(), B, H, W, C, scratch.data_ptr(), out.data_ptr(), current_stream()))
    return out


def gray256_from_rgb(images: torch.Tensor, clahe: bool, scratch: Optional[torch.Tensor] = None,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """u8 RGB images [B,H,W,3] (NHWC, device; dense or a rectangle view of a larger image) -> gray256 f32 [B,256,256] in [0,1]
    (dfd_gray256): Pillow 'L' luma, optional OpenCV CLAHE(2.0, 8x8), Pillow bicubic resize, /255 —
    train_fusion_head_only.py:142-148 (clahe=True), deepfake-detector-v2/app.py:736-749.  EXIF orientation is the decoder's
    business (apply ImageOps.exif_transpose before handing pixels over, as the reference does)."""
    _need_cuda(images)
    assert images.dtype == torch.uint8 and images.dim() == 4 and images.shape[3] == 3
    images, rs, ims = _rect_strides(images)
    B, H, W, _ = images.shape
    lib = _lib.load()
    need = lib.dfd_gray256_scratch_bytes(B, H, W)
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty((need,), dtype=torch.uint8, device=images.device)
    xw, cw, kw = _resample_tables(W, images.device)
    xh, ch, kh = _resample_tables(H, images.device)
    if out is None:
        out = torch.empty((B, 256, 256), dtype=torch.float32, device=images.device)
    check(lib.dfd_gray256(images.data_ptr(), rs, ims, B, H, W, int(clahe), xw.data_ptr(), cw.data_ptr(), kw.data_ptr(),
                          kw.shape[1], xh.data_ptr(), ch.data_ptr(), kh.data_ptr(), kh.shape[1], scratch.data_ptr(),
                          out.data_ptr(), current_stream()))
    return out


class ScoreParams:
    """Device copy of FreqMLP + fusion + CORAL parameters for dfd_score_epilogue (gen 1 or 2)."""

    def __init__(self, gen: int, device, *, freq_state: Optional[dict] = None, fusion_state: Optional[dict] = None,
                 coral_cuts_logit=(0.0, 0.0, 0.0, 0.0), coral_temp: float = 1.0, freq_temp: float = 1.25):
        self.gen = gen
        self._keep = []
        w = ScoreWeights()
        w.gen = gen
        w.freq_temp = freq_temp

        def put(t):
            d = _f32(t, device)
            self._keep.append(d)
            return d.data_ptr()

        if freq_state is not None:
            if gen == 1:
                w.g1_ln_w, w.g1_ln_b = put(freq_state["net.0.weight"]), put(freq_state["net.0.bias"])
                w.g1_w1, w.g1_b1 = put(freq_state["net.1.weight"]), put(freq_state["net.1.bias"])
                w.g1_w2, w.g1_b2 = put(freq_state["net.3.weight"]), put(freq_state["net.3.bias"])
            else:
                w.g2_mean, w.g2_std = put(freq_state["normer.mean"]), put(freq_state["normer.std"])
                w.g2_alpha, w.g2_beta = put(freq_state["contrast.alpha"]), put(freq_state["contrast.beta"])
                w.g2_gates = put(freq_state["band.gates"])
                for b in range(2):
                    names = ("norm.weight", "norm.bias", "fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")
                    for i, n in enumerate(names):
                        w.g2_blk[b][i] = put(freq_state[f"blocks.{b}.{n}"])
                w.g2_head_w, w.g2_head_b = put(freq_state["head.weight"]), put(freq_state["head.bias"])
                w.g2_temp = float(freq_state["temp.T"])
        if fusion_state is not None:
            if gen == 1:
                fw = fusion_state["fc.weight"].detach().float().reshape(-1).tolist()
                w.g1_fc_w[0], w.g1_fc_w[1] = fw[0], fw[1]
                w.g1_fc_b = float(fusion_state["fc.bias"].detach().float().reshape(-1)[0])
            else:
                w.f2_w0, w.f2_b0 = put(fusion_state["mlp.0.weight"]), put(fusion_state["mlp.0.bias"])
                w.f2_w1, w.f2_b1 = put(fusion_state["mlp.2.weight"]), put(fusion_state["mlp.2.bias"])
                w.f2_temp = float(fusion_state["temp.T"])
        for i in range(4):
            w.coral_cuts[i] = float(coral_cuts_logit[i])
        w.coral_temp = float(coral_temp)
        self.struct = w


SCORE_FIELDS = ("z_freq", "z", "z_scaled", "p_raw", "risk_probs", "p_coral", "entropy", "p_blend", "risk_idx")


def score_epilogue(params: ScoreParams, z_sig: torch.Tensor, feats: Optional[torch.Tensor] = None,
                   z_freq: Optional[torch.Tensor] = None) -> dict:
    """One warp per sample: FreqMLP -> fusion -> temperature -> CORAL.  Returns a dict of SoA tensors."""
    _need_cuda(z_sig, feats, z_freq)
    assert z_sig.dtype == torch.float32 and z_sig.is_contiguous()
    B = z_sig.numel()
    dev = z_sig.device
    if feats is not None:
        assert feats.dtype == torch.float32 and feats.shape == (B, 24) and feats.is_contiguous()
    if z_freq is not None:
        assert z_freq.dtype == torch.float32 and z_freq.numel() == B and z_freq.is_contiguous()
    out = {k: torch.empty((B,), dtype=torch.float32, device=dev) for k in SCORE_FIELDS}
    out["risk_probs"] = torch.empty((B, 5), dtype=torch.float32, device=dev)
    out["risk_idx"] = torch.empty((B,), dtype=torch.int32, device=dev)
    s = Scores()
    for k in SCORE_FIELDS:
        setattr(s, k, out[k].data_ptr())
    check(_lib.load().dfd_score_epilogue(C.byref(params.struct), z_sig.data_ptr(), _p(feats), _p(z_freq), B,
                                         C.byref(s), current_stream()))
    out["z_sig"] = z_sig
    return out


FUSION_PARAM_ORDER = ("mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias", "temp.T")


def dwconv3x3_bf16(x: torch.Tensor, w9: torch.Tensor, bias: Optional[torch.Tensor], B: int, H: int, W: int,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Depthwise 3x3 convolution (zero padding 1) on token-major bf16 activations x [B*H*W, E]; w9 fp32 [E, 9]."""
    _need_cuda(x, w9, bias, out)
    assert x.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1 and x.shape[0] == B * H * W
    E = x.shape[1]
    assert w9.dtype == torch.float32 and w9.shape == (E, 9) and w9.is_contiguous()
    if out is None:
        out = torch.empty((B * H * W, E), dtype=torch.bfloat16, device=x.device)
    check(_lib.load().dfd_dwconv3x3_bf16(x.data_ptr(), x.stride(0), w9.data_ptr(), _p(bias), out.data_ptr(), out.stride(0),
                                         B, H, W, E, current_stream()))
    return out


def seg_head_upsample(x: torch.Tensor, w: torch.Tensor, bias: float, B: int, H: int, W: int, S: int) -> torch.Tensor:
    """1x1 conv E -> 1 then bilinear (align_corners=False) resize to S x S: x bf16 [B*H*W, E] -> fp32 [B, 1, S, S]."""
    _need_cuda(x, w)
    assert x.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1 and x.shape[0] == B * H * W
    assert w.dtype == torch.float32 and w.numel() == x.shape[1] and w.is_contiguous()
    low = torch.empty((B * H * W,), dtype=torch.float32, device=x.device)
    out = torch.empty((B, 1, S, S), dtype=torch.float32, device=x.device)
    check(_lib.load().dfd_seg_head_upsample(x.data_ptr(), x.stride(0), w.data_ptr(), float(bias), B, H, W, x.shape[1], S,
                                            low.data_ptr(), out.data_ptr(), current_stream()))
    return out


def linear_small(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """x bf16 [B,K] @ w fp32 [N,K].T + bias -> fp32 [B,N] (tiny heads: one warp per output)."""
    _need_cuda(x, w, bias)
    assert x.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1
    assert w.dtype == torch.float32 and w.dim() == 2 and w.shape[1] == x.shape[1] and w.is_contiguous()
    out = torch.empty((x.shape[0], w.shape[0]), dtype=torch.float32, device=x.device)
    check(_lib.load().dfd_linear_small(x.data_ptr(), x.stride(0), w.data_ptr(), _p(bias), out.data_ptr(), x.shape[0],
                                       w.shape[0], x.shape[1], current_stream()))
    return out


FREQMLP_PARAM_ORDER = ("contrast.alpha", "contrast.beta", "band.gates") + tuple(
    f"blocks.{b}.{n}" for b in range(2)
    for n in ("norm.weight", "norm.bias", "fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")) + ("head.weight", "head.bias", "temp.T")
FREQMLP_PARAM_SHAPES = ((24,), (24,), (4,)) + ((24,), (24,), (64, 24), (64,), (24, 64), (24,)) * 2 + ((1, 24), (1,), ())
FREQMLP_NUM_PARAMS = 6494


def freqmlp_fwd_bwd(params: torch.Tensor, mean: torch.Tensor, std: torch.Tensor, feats: torch.Tensor,
                    y: Optional[torch.Tensor] = None, inv_global_batch: Optional[float] = None, dropout_p: float = 0.0,
                    seed: int = 0, want_grads: bool = True, want_logits: bool = False):
    """FreqMLP G2 forward (+ backward of mean BCE-with-logits).  Returns (loss[1] | None, grads[6494] | None,
    logits[B] | None); loss / grads are this rank's partial sums (all-reduce-sum them)."""
    _need_cuda(params, mean, std, feats)
    for t in (params, mean, std, feats):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert params.numel() == FREQMLP_NUM_PARAMS and mean.numel() == 24 and std.numel() == 24 and feats.shape[1] == 24
    B, dev = feats.shape[0], feats.device
    loss = grads = None
    if want_grads:
        assert y is not None and y.dtype == torch.float32 and y.is_contiguous() and y.numel() == B
        loss = torch.zeros((1,), dtype=torch.float32, device=dev)
        grads = torch.zeros((FREQMLP_NUM_PARAMS,), dtype=torch.float32, device=dev)
    logits = torch.empty((B,), dtype=torch.float32, device=dev) if (want_logits or not want_grads) else None
    inv = (1.0 / B) if inv_global_batch is None else inv_global_batch
    check(_lib.load().dfd_freqmlp_fwd_bwd(params.data_ptr(), mean.data_ptr(), std.data_ptr(), feats.data_ptr(), _p(y), B,
                                          inv, float(dropout_p), int(seed) & 0xFFFFFFFF, _p(loss), _p(grads), _p(logits),
                                          current_stream()))
    return loss, grads, logits


def fusion_fwd_bwd(params195: torch.Tensor, z_freq: torch.Tensor, z_sig: torch.Tensor, y: torch.Tensor,
                   inv_global_batch: Optional[float] = None, want_logits: bool = False):
    """AdaptiveFusionHead forward + backward of mean BCE-with-logits. Returns (loss[1], grads[195], logits|None);
    loss and grads are this rank's partial sums (allreduce-sum them across ranks)."""
    _need_cuda(params195, z_freq, z_sig, y)
    for t in (params195, z_freq, z_sig, y):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert params195.numel() == 195
    B = z_freq.numel()
    dev = z_freq.device
    loss = torch.zeros((1,), dtype=torch.float32, device=dev)
    grads = torch.zeros((195,), dtype=torch.float32, device=dev)
    logits = torch.empty((B,), dtype=torch.float32, device=dev) if want_logits else None
    inv = (1.0 / B) if inv_global_batch is None else inv_global_batch
    check(_lib.load().dfd_fusion_fwd_bwd(params195.data_ptr(), z_freq.data_ptr(), z_sig.data_ptr(), y.data_ptr(), B,
                                         inv, loss.data_ptr(), grads.data_ptr(), _p(logits), current_stream()))
    return loss, grads, logits

"""SiglipEngine — Python handle on a dfd_engine (include/dfd.h): packed SigLIP vision-tower weights +
workspace on one GPU, forward = hand-written sm_100a kernels only.

Accepts the two weight layouts the reference uses (SURVEY.md App. B):
  * HuggingFace `SiglipVisionModel` state dicts (`vision_model.*`, split q/k/v)  — Siglip2sidafrozen.py:753
  * open_clip/timm SigLIP state dicts (`visual.trunk.*`, fused qkv, `attn_pool.*`) — inference_ai_human_images.py:124-128
"""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import _lib
from ._lib import EngineConfig, check, current_stream


@dataclass(frozen=True)
class VisionArch:
    image_size: int
    patch_size: int
    hidden_size: int
    intermediate_size: int
    num_hidden_layers: int
    num_attention_heads: int
    layer_norm_eps: float = 1e-6

    @property
    def grid(self) -> int:
        return self.image_size // self.patch_size

    @property
    def tokens(self) -> int:
        return self.grid * self.grid

    @property
    def head_dim(self) -> int:
        return self.hidden_size // self.num_attention_heads

    def flops_per_image(self) -> float:
        """Algorithmic FLOPs (SURVEY.md §8d): 2MNK per GEMM, 4·N²·D per attention layer, MAP head included."""
        N, D, I, L, P = self.tokens, self.hidden_size, self.intermediate_size, self.num_hidden_layers, self.patch_size
        pe = 2 * N * 3 * P * P * D
        layer = 8 * N * D * D + 4 * N * D * I + 4 * N * N * D
        mp = 4 * N * D * D + 4 * D * D + 4 * N * D + 4 * D * I
        return float(pe + L * layer + mp)


# SURVEY.md App. C / C.1: names the reference passes to open_clip / HF, plus small shapes for tests
ARCHS: Dict[str, VisionArch] = {
    "google/siglip2-base-patch16-224": VisionArch(224, 16, 768, 3072, 12, 12),
    "google/siglip2-so400m-patch14-384": VisionArch(384, 14, 1152, 4304, 27, 16),
    "google/siglip2-large-patch16-384": VisionArch(384, 16, 1024, 4096, 24, 16),
    "ViT-B-16-SigLIP": VisionArch(224, 16, 768, 3072, 12, 12),
    "ViT-B-16-SigLIP-256": VisionArch(256, 16, 768, 3072, 12, 12),
    "ViT-B-16-SigLIP-384": VisionArch(384, 16, 768, 3072, 12, 12),
    "ViT-L-16-SigLIP-384": VisionArch(384, 16, 1024, 4096, 24, 16),
    "ViT-SO400M-16-SigLIP2-512": VisionArch(512, 16, 1152, 4304, 27, 16),
    "tiny-hd64": VisionArch(64, 16, 128, 256, 2, 2),
    "tiny-hd72": VisionArch(60, 14, 144, 304, 2, 2),
    "small-hd72": VisionArch(210, 14, 288, 1080, 3, 4),
}
ARCHS["siglip2-base-patch16-224"] = ARCHS["google/siglip2-base-patch16-224"]
ARCHS["siglip2-so400m-patch14-384"] = ARCHS["google/siglip2-so400m-patch14-384"]
ARCHS["siglip2-large-patch16-384"] = ARCHS["google/siglip2-large-patch16-384"]


_TIMM_BLOCK = re.compile(r"^blocks\.(\d+)\.(.+)$")
_TIMM_MAP = {
    "norm1.weight": "layer_norm1.weight", "norm1.bias": "layer_norm1.bias",
    "norm2.weight": "layer_norm2.weight", "norm2.bias": "layer_norm2.bias",
    "attn.qkv.weight": "self_attn.qkv.weight", "attn.qkv.bias": "self_attn.qkv.bias",
    "attn.proj.weight": "self_attn.out_proj.weight", "attn.proj.bias": "self_attn.out_proj.bias",
    "mlp.fc1.weight": "mlp.fc1.weight", "mlp.fc1.bias": "mlp.fc1.bias",
    "mlp.fc2.weight": "mlp.fc2.weight", "mlp.fc2.bias": "mlp.fc2.bias",
}


def canonicalize_state_dict(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """Map an HF (`vision_model.*`) or open_clip/timm (`[backbone.]visual.trunk.*`) state dict to the engine's
    canonical tensor names.  Text-tower and unrelated keys are dropped (train_fusion_head_only.py:111-116)."""
    out: Dict[str, torch.Tensor] = {}
    for k, v in sd.items():
        key = k
        for pre in ("backbone.", "encoder.", "model.", "_orig_mod."):
            if key.startswith(pre) and not key.startswith("encoder.layers."):
                key = key[len(pre):]
        if key.startswith("vision_model."):
            out[key[len("vision_model."):]] = v
            continue
        if key.startswith(("embeddings.", "encoder.layers.", "post_layernorm.", "head.")):
            out[key] = v
            continue
        if not key.startswith("visual.trunk."):
            continue
        t = key[len("visual.trunk."):]
        m = _TIMM_BLOCK.match(t)
        if m and m.group(2) in _TIMM_MAP:
            out[f"encoder.layers.{m.group(1)}.{_TIMM_MAP[m.group(2)]}"] = v
        elif t == "patch_embed.proj.weight":
            out["embeddings.patch_embedding.weight"] = v
        elif t == "patch_embed.proj.bias":
            out["embeddings.patch_embedding.bias"] = v
        elif t == "pos_embed":
            out["embeddings.position_embedding.weight"] = v.reshape(v.shape[-2], v.shape[-1])
        elif t in ("norm.weight", "norm.bias"):
            out["post_layernorm." + t.split(".")[1]] = v
        elif t == "attn_pool.latent":
            out["head.probe"] = v
        elif t in ("attn_pool.q.weight", "attn_pool.kv.weight", "attn_pool.q.bias", "attn_pool.kv.bias"):
            out["__timm_" + t] = v
        elif t.startswith("attn_pool.proj."):
            out["head.attention.out_proj." + t.split(".")[-1]] = v
        elif t.startswith("attn_pool.norm."):
            out["head.layernorm." + t.split(".")[-1]] = v
        elif t.startswith("attn_pool.mlp."):
            out["head.mlp." + t[len("attn_pool.mlp."):]] = v
    if "__timm_attn_pool.q.weight" in out:  # timm keeps q and kv separately; HF packs [q; k; v]
        out["head.attention.in_proj_weight"] = torch.cat(
            [out.pop("__timm_attn_pool.q.weight"), out.pop("__timm_attn_pool.kv.weight")], 0)
        out["head.attention.in_proj_bias"] = torch.cat(
            [out.pop("__timm_attn_pool.q.bias"), out.pop("__timm_attn_pool.kv.bias")], 0)
    return out


def arch_from_state_dict(sd: Dict[str, torch.Tensor], num_heads: Optional[int] = None) -> VisionArch:
    sd = canonicalize_state_dict(sd)
    w = sd["embeddings.patch_embedding.weight"]
    D, P = w.shape[0], w.shape[-1]
    N = sd["embeddings.position_embedding.weight"].shape[0]
    G = int(round(N ** 0.5))
    L = 1 + max(int(k.split(".")[2]) for k in sd if k.startswith("encoder.layers."))
    I = sd["encoder.layers.0.mlp.fc1.weight"].shape[0]
    if num_heads is None:
        num_heads = D // 72 if D % 72 == 0 and D % 64 != 0 else D // 64
    return VisionArch(G * P, P, D, I, L, num_heads)


class SiglipEngine:
    """One engine per (device, architecture).  `forward` accepts uint8 NHWC images (preprocess fused into the
    im2col kernel) or float32 NCHW tensors that are already normalised, and returns bf16 pooled embeddings."""

    def __init__(self, arch: VisionArch, device: int | torch.device = 0, max_batch: int = 64, fuse_ln: bool = False,
                 graphs: bool = False, precise_residual: bool = False):
        if not torch.cuda.is_available():
            raise RuntimeError("SiglipEngine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.arch = arch
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        self.max_batch = int(max_batch)
        # fuse_ln: LayerNorm1/2 folded into the qkv / fc1 GEMMs; the row statistics are left by the GEMM that wrote the
        # residual stream as per-64-column partial sums and added in a fixed order (no atomics: bit-reproducible)
        self.fuse_ln = bool(fuse_ln)
        self._lib = _lib.load()
        cfg = EngineConfig(arch.image_size, arch.patch_size, arch.hidden_size, arch.intermediate_size,
                           arch.num_hidden_layers, arch.num_attention_heads, 1, arch.layer_norm_eps, int(self.fuse_ln))
        h = C.c_void_p()
        check(self._lib.dfd_engine_create(C.byref(cfg), self.device.index or 0, self.max_batch, C.byref(h)))
        self._h = h
        self._finalized = False
        # graphs: a forward whose buffers and shape have been seen before is replayed as ONE CUDA graph launch (tensor maps
        # and arguments baked in) instead of 7·L + 13 launches — for small batches, where the host cannot keep ahead of the
        # device.  The engine then writes into output buffers it keeps per batch size (stable pointers) and hands out copies.
        self.graphs = False
        self._out: Dict[tuple, torch.Tensor] = {}
        if graphs:
            self.set_graphs(True)
        # precise_residual: the residual stream is carried as two bf16 tensors (hi + lo), so the 2·L residual additions
        # accumulate like the fp32 stream of the reference's autocast path instead of being rounded to bf16 each time
        self.precise_residual = False
        if precise_residual:
            self.set_precise_residual(True)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dfd_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_graphs(self, on: bool) -> None:
        check(self._lib.dfd_engine_set_graphs(self._h, int(bool(on))))
        self.graphs = bool(on)
        if not on:
            self._out.clear()

    def set_precise_residual(self, on: bool) -> None:
        check(self._lib.dfd_engine_set_precise_residual(self._h, int(bool(on))))
        self.precise_residual = bool(on)

    @property
    def graph_replays(self) -> int:
        return int(self._lib.dfd_engine_graph_replays(self._h))

    @property
    def workspace_bytes(self) -> int:
        return int(self._lib.dfd_engine_workspace_bytes(self._h))

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> "SiglipEngine":
        canon = canonicalize_state_dict(sd)
        if not canon:
            raise KeyError("no SigLIP vision-tower tensors found in the state dict")
        for name, t in canon.items():
            t = t.detach()
            if t.dtype not in (torch.float32, torch.bfloat16):
                t = t.float()
            t = t.contiguous()
            shape = (C.c_int64 * max(t.dim(), 1))(*(t.shape if t.dim() else (1,)))
            on_host = 0 if t.is_cuda else 1
            if t.is_cuda and t.device != self.device:
                t = t.to(self.device)
            check(self._lib.dfd_engine_set_tensor(self._h, name.encode(), t.data_ptr(),
                                                  1 if t.dtype == torch.bfloat16 else 0, max(t.dim(), 1), shape,
                                                  on_host))
        check(self._lib.dfd_engine_finalize(self._h))
        self._finalized = True
        return self

    def forward_hidden(self, pixels: torch.Tensor, resize_mode: int = 0):
        """Like forward(), plus the L+1 per-layer hidden states (HF `output_hidden_states=True`):
        returns (pooled [B,D], last_hidden [B,N,D], hidden [L+1,B,N,D]) in bf16.  B <= max_batch."""
        B = pixels.shape[0]
        if B > self.max_batch:
            raise ValueError("forward_hidden: batch must fit the engine workspace (max_batch)")
        a = self.arch
        hidden = torch.empty((a.num_hidden_layers + 1, B, a.tokens, a.hidden_size), dtype=torch.bfloat16,
                             device=self.device)
        check(self._lib.dfd_engine_set_hidden_tap(self._h, hidden.data_ptr()))
        try:
            pooled, last = self.forward(pixels, resize_mode, want_last_hidden=True)
        finally:
            check(self._lib.dfd_engine_set_hidden_tap(self._h, None))
        return pooled, last, hidden

    def forward_attentions(self, pixels: torch.Tensor, resize_mode: int = 0, per_head: bool = False,
                           hidden: bool = False):
        """One forward that also returns the attention maps (HF `output_attentions=True`): (pooled [B,D] bf16,
        attentions fp32 [L,B,N,N] (head mean) or [L,B,H,N,N] (per_head), map_attention fp32 [B,H,N] = the MAP probe's
        attention over the tokens[, hidden [L+1,B,N,D] bf16 with hidden=True]).  Rows sum to 1.  B <= max_batch."""
        pooled, _, attn, map_p, hid = self._forward_tapped(pixels, resize_mode, per_head, hidden, False)
        return (pooled, attn, map_p, hid) if hidden else (pooled, attn, map_p)

    def _forward_tapped(self, pixels, resize_mode, per_head, hidden, want_last_hidden):
        B = pixels.shape[0]
        if B > self.max_batch:
            raise ValueError("forward_attentions: batch must fit the engine workspace (max_batch)")
        a = self.arch
        L, H, N = a.num_hidden_layers, a.num_attention_heads, a.tokens
        shape = (L, B, H, N, N) if per_head else (L, B, N, N)
        attn = torch.empty(shape, dtype=torch.float32, device=self.device)
        map_p = torch.empty((B, H, N), dtype=torch.float32, device=self.device)
        hid = (torch.empty((L + 1, B, N, a.hidden_size), dtype=torch.bfloat16, device=self.device) if hidden else None)
        check(self._lib.dfd_engine_set_attention_tap(self._h, attn.data_ptr(), int(bool(per_head)), map_p.data_ptr()))
        try:
            if hid is not None:
                check(self._lib.dfd_engine_set_hidden_tap(self._h, hid.data_ptr()))
            pooled, last = self.forward(pixels, resize_mode, want_last_hidden=want_last_hidden)
        finally:
            check(self._lib.dfd_engine_set_attention_tap(self._h, None, 0, None))
            check(self._lib.dfd_engine_set_hidden_tap(self._h, None))
        return pooled, last, attn, map_p, hid

    def forward(self, pixels: torch.Tensor, resize_mode: int = 0, want_last_hidden: bool = False):
        """pixels: uint8 [B,H,W,3] or float32 [B,3,H,W] on this engine's device.  Batches larger than
        max_batch are processed in chunks.  Returns (pooled bf16 [B,D], last_hidden bf16 [B,N,D] | None)."""
        if not self._finalized:
            raise RuntimeError("load_state_dict() first")
        if not pixels.is_cuda:
            raise RuntimeError("pixels must be a CUDA tensor (there is no CPU fallback)")
        pixels = pixels.contiguous()
        if pixels.dtype == torch.uint8:
            fmt, (B, Hin, Win, ch) = 0, pixels.shape
        elif pixels.dtype == torch.float32:
            fmt, (B, ch, Hin, Win) = 1, pixels.shape
        else:
            raise TypeError("pixels must be uint8 NHWC or float32 NCHW")
        if ch != 3:
            raise ValueError("pixels must have 3 channels")
        a = self.arch
        stable = self.graphs and B <= self.max_batch
        if stable:   # stable output pointers, so that the call signature repeats and its graph is replayed
            pooled = self._out.get(("p", B))
            if pooled is None:
                pooled = self._out[("p", B)] = torch.empty((B, a.hidden_size), dtype=torch.bfloat16, device=self.device)
            last = None
            if want_last_hidden:
                last = self._out.get(("l", B))
                if last is None:
                    last = self._out[("l", B)] = torch.empty((B, a.tokens, a.hidden_size), dtype=torch.bfloat16,
                                                               device=self.device)
        else:
            pooled = torch.empty((B, a.hidden_size), dtype=torch.bfloat16, device=self.device)
            last = (torch.empty((B, a.tokens, a.hidden_size), dtype=torch.bfloat16, device=self.device)
                    if want_last_hidden else None)
        if pixels.device != self.device:
            raise RuntimeError(f"pixels live on {pixels.device}, this engine on {self.device}")
        # launch on THIS engine's device and on its current stream, whatever device the caller has selected
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            for b0 in range(0, B, self.max_batch):
                nb = min(self.max_batch, B - b0)
                check(self._lib.dfd_engine_forward(self._h, pixels[b0:b0 + nb].data_ptr(), fmt, nb, Hin, Win, resize_mode,
                                                   pooled[b0:b0 + nb].data_ptr(),
                                                   None if last is None else last[b0:b0 + nb].data_ptr(), st))
        if stable:   # the kept buffers are overwritten by the next call of this batch size: hand out copies
            return pooled.clone(), (None if last is None else last.clone())
        return pooled, last

    __call__ = forward

    def profile(self, forwards: int = 1) -> None:
        """Bracket every launch of the following forwards with CUDA events (bench.py roofline).  `forwards` = how many
        forwards the event buffer holds before profile_read() must be called; 0 / False switches profiling off."""
        check(self._lib.dfd_engine_profile(self._h, int(forwards)))

    FAMILIES = ("gemm", "attention", "layernorm", "patchify", "map_attention")
    GEMM_TYPES = ("gemm_other", "gemm_qkv", "gemm_out", "gemm_fc1", "gemm_fc2")

    def profile_read(self, by_gemm_type: bool = False) -> dict:
        """Per kernel family, summed over every forward since the last read: {'gemm': (ms, launches), 'attention': ...,
        'layernorm': ..., 'patchify': ..., 'map_attention': ...}; with by_gemm_type also 'gemm_qkv' / 'gemm_out' / 'gemm_fc1' /
        'gemm_fc2' / 'gemm_other' (patch embedding + pooling head), which add up to 'gemm'.  Waits for the last recorded launch."""
        ms, cnt = (C.c_float * 9)(), (C.c_int * 9)()
        check(self._lib.dfd_engine_profile_read(self._h, ms, cnt))
        out = {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.FAMILIES)}
        gm = [0, 5, 6, 7, 8]
        out["gemm"] = (float(sum(ms[i] for i in gm)), int(sum(cnt[i] for i in gm)))
        if by_gemm_type:
            for k, i in zip(self.GEMM_TYPES, gm):
                out[k] = (float(ms[i]), int(cnt[i]))
        return out

    def gemm_flops_by_type(self, batch: int) -> dict:
        a = self.arch
        N, D, I, L, P = a.tokens, a.hidden_size, a.intermediate_size, a.num_hidden_layers, a.patch_size
        return {"gemm_qkv": 6.0 * N * D * D * L * batch, "gemm_out": 2.0 * N * D * D * L * batch,
                "gemm_fc1": 2.0 * N * D * I * L * batch, "gemm_fc2": 2.0 * N * D * I * L * batch,
                "gemm_other": float(2 * N * 3 * P * P * D + 4 * N * D * D + 2 * D * D + 4 * D * I) * batch}

    def gemm_flops(self, batch: int) -> float:
        """Algorithmic FLOPs of all GEMM launches of one forward of `batch` images (2·M·N·K each; the
        patch-embedding K is the unpadded 3·P²)."""
        a = self.arch
        N, D, I, L, P = a.tokens, a.hidden_size, a.intermediate_size, a.num_hidden_layers, a.patch_size
        per_img = 2 * N * 3 * P * P * D + L * (8 * N * D * D + 4 * N * D * I) + 4 * N * D * D + 2 * D * D + 4 * D * I
        return float(per_img) * batch
